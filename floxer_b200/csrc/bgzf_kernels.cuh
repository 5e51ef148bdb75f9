// bgzf_kernels.cuh -- BGZF compression on the device for sm_100a: the blocks of the BAM image (fxg_write_bam_device) and
// of the compressed SAM text (fxg_write_sam_device with bgzf = 1).
//
// The stream is cut into BGZF blocks at the 0xff00-byte boundaries bam_output.cpp uses, so every block has the host
// block's ISIZE and CRC32 and only the deflate payloads differ from the host writer's:
//   deflate   bgzf_deflate_kernel: one CTA per 0xff00-byte chunk -- LZ77 over hash chains in shared memory, a greedy
//             parse per 512-byte segment, dynamic Huffman codes (15-bit limit, code-length code 7 bits), bit offsets by
//             a scan over the segments, packing into words; a stored block when that is smaller.  CRC32 per segment,
//             folded by GF(2) multiplication;
//   offsets   an exclusive scan of the block sizes (cub, on the host's stream);
//   assemble  bgzf_assemble_kernel: BGZF header, payload and trailer of every block at its scanned offset, then the
//             end-of-file block.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace fxg {

constexpr uint32_t kBgzfChunk = 0xff00;              // raw bytes per BGZF block (as bam_output.cpp cuts them)
constexpr uint32_t kBgzfSlotWords = 65536 / 4;       // a block's deflate payload area in the work buffer
constexpr int kDeflateThreads = 512;
constexpr int kDeflateHashBits = 12;
constexpr uint32_t kDeflateSeg = 512;                // parse segment: a match never crosses one's end
constexpr uint32_t kDeflateMaxSegs = (kBgzfChunk + kDeflateSeg - 1) / kDeflateSeg;
constexpr int kDeflateChain = 8;                     // candidates tried per position
constexpr uint32_t kDeflateNice = 64;                // a match this long ends the search
constexpr uint32_t kNoPrev = 0xffff;

// per BGZF block: its deflate payload (or stored) length, CRC32 and input size
struct BgzfBlockInfo { uint32_t payload, crc, isize, stored; };

__device__ __forceinline__ void put_le(uint8_t* p, uint32_t v, int n) { for (int i = 0; i < n; ++i) p[i] = uint8_t(v >> (8 * i)); }

// ------------------------------------------------------------------------------------------------ deflate

// CRC32 (reflected polynomial 0xedb88320) helpers after zlib's crc32_combine: multiplication modulo the polynomial
__device__ inline uint32_t crc_multmodp(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) { p ^= b; if ((a & (m - 1)) == 0) break; }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ 0xedb88320u : b >> 1;
    }
    return p;
}
__device__ inline uint32_t crc_x8n(uint32_t n) {                       // x^(8n) modulo the polynomial
    uint32_t p = 1u << 31, sq = 1u << 23;                              // x^0, x^8
    for (; n; n >>= 1) { if (n & 1) p = crc_multmodp(sq, p); sq = crc_multmodp(sq, sq); }
    return p;
}

// length 3..258 -> (symbol 257..285, extra bits, their value); distance 1..32768 -> (symbol 0..29, extra bits, value)
__device__ __forceinline__ void deflate_len_sym(uint32_t len, uint32_t& sym, uint32_t& eb, uint32_t& ev) {
    uint32_t const l = len - 3;
    if (len == 258) { sym = 285; eb = 0; ev = 0; return; }
    if (l < 8) { sym = 257 + l; eb = 0; ev = 0; return; }
    eb = (31 - __clz(l)) - 2;
    sym = 257 + 4 * (eb + 1) + ((l >> eb) & 3);
    ev = l & ((1u << eb) - 1);
}
__device__ __forceinline__ void deflate_dist_sym(uint32_t dist, uint32_t& sym, uint32_t& eb, uint32_t& ev) {
    uint32_t const d = dist - 1;
    if (d < 4) { sym = d; eb = 0; ev = 0; return; }
    eb = (31 - __clz(d)) - 1;
    sym = 2 * (eb + 1) + ((d >> eb) & 1);
    ev = d & ((1u << eb) - 1);
}

// LSB-first bit writer into a zeroed word buffer shared with other writers (the words at range ends are shared)
struct BitWriter {
    uint32_t* out; uint64_t acc = 0; uint32_t nbits, word;
    __device__ BitWriter(uint32_t* o, uint32_t bitpos) : out(o), nbits(bitpos & 31), word(bitpos >> 5) {}
    __device__ __forceinline__ void put(uint32_t v, uint32_t n) {
        acc |= uint64_t(v) << nbits;
        nbits += n;
        if (nbits >= 32) { atomicOr(out + word, uint32_t(acc)); ++word; acc >>= 32; nbits -= 32; }
    }
    __device__ __forceinline__ void flush() { if (nbits) atomicOr(out + word, uint32_t(acc)); }
};

struct DeflateSmem {
    uint8_t buf[kBgzfChunk + 8];
    uint16_t prev[kBgzfChunk];                   // nearest earlier position with the same 3-byte hash (kNoPrev: none)
    uint32_t head[1 << kDeflateHashBits];        // latest position + 1 per hash, as of the current tile
    uint32_t lit_freq[288], dist_freq[32], cl_freq[20];
    uint8_t lit_len[288], dist_len[32], cl_len[20];
    uint16_t lit_code[288], dist_code[32], cl_code[20];     // bit-reversed canonical codes
    uint32_t sort_key[288 + 32]; uint16_t sort_sym[288 + 32];
    uint8_t rle_sym[288 + 32], rle_extra[288 + 32];
    uint32_t seg_bits[kDeflateMaxSegs], seg_crc[kDeflateMaxSegs];
    uint32_t crc_table[256];
    uint32_t n_rle, hlit, hdist, hclen, hdr_bits, stored, crc;
};

// Code lengths of a length-limited Huffman code for the n >= 2 symbols key/sym sorted by ascending frequency (key):
// minimum-redundancy lengths in place (Moffat and Katajainen), then the counts per length moved under `limit` with the
// Kraft sum restored, and the lengths handed out -- the shortest to the most frequent.  One thread.
__device__ inline void huffman_lengths(uint32_t* key, const uint16_t* sym, int n, int limit, uint8_t* len_out) {
    key[0] += key[1];
    int root = 0, leaf = 2;
    for (int next = 1; next < n - 1; ++next) {
        if (leaf >= n || key[root] < key[leaf]) { key[next] = key[root]; key[root++] = uint32_t(next); }
        else key[next] = key[leaf++];
        if (leaf >= n || (root < next && key[root] < key[leaf])) { key[next] += key[root]; key[root++] = uint32_t(next); }
        else key[next] += key[leaf++];
    }
    key[n - 2] = 0;
    for (int next = n - 3; next >= 0; --next) key[next] = key[key[next]] + 1;
    int avbl = 1, used = 0, dpth = 0, next = n - 1;
    root = n - 2;
    while (avbl > 0) {
        while (root >= 0 && int(key[root]) == dpth) { ++used; --root; }
        while (avbl > used) { key[next--] = uint32_t(dpth); --avbl; }
        avbl = 2 * used; ++dpth; used = 0;
    }
    uint32_t count[33] = {0};
    for (int i = 0; i < n; ++i) count[min(key[i], 32u)]++;
    for (int i = limit + 1; i <= 32; ++i) { count[limit] += count[i]; count[i] = 0; }
    uint32_t total = 0;
    for (int i = limit; i > 0; --i) total += count[i] << (limit - i);
    while (total != (1u << limit)) {
        count[limit]--;
        for (int i = limit - 1; i > 0; --i) if (count[i]) { count[i]--; count[i + 1] += 2; break; }
        total--;
    }
    int j = n;
    for (int l = 1; l <= limit; ++l)
        for (uint32_t c = count[l]; c > 0; --c) len_out[sym[--j]] = uint8_t(l);
}

__device__ inline void canonical_codes(const uint8_t* len, uint16_t* code, int n) {
    uint32_t count[16] = {0}, next[16];
    for (int s = 0; s < n; ++s) count[len[s]]++;
    count[0] = 0;
    uint32_t c = 0;
    for (int l = 1; l < 16; ++l) { c = (c + count[l - 1]) << 1; next[l] = c; }
    for (int s = 0; s < n; ++s)
        if (len[s]) code[s] = uint16_t(__brev(next[len[s]]++) >> (32 - len[s]));
}

// sorts symbols 0..n-1 with a non-zero frequency by (frequency, symbol) into key/sym: one thread per symbol
__device__ __forceinline__ void rank_sort(const uint32_t* freq, int n, int s, uint32_t* key, uint16_t* sym) {
    uint32_t const f = freq[s];
    if (!f) return;
    int rank = 0;
    for (int t = 0; t < n; ++t) rank += freq[t] && (freq[t] < f || (freq[t] == f && t < s));
    key[rank] = f; sym[rank] = uint16_t(s);
}

// One CTA per kBgzfChunk bytes of `raw`: the chunk's deflate payload (one final block, dynamic codes) into its
// 64 KB slot of `slots`, or -- when a stored block is not larger -- nothing but the decision; CRC32 and size into info.
__global__ void __launch_bounds__(kDeflateThreads, 1)
bgzf_deflate_kernel(const uint8_t* raw, uint64_t raw_len, uint32_t* work, uint32_t* slots, BgzfBlockInfo* info, uint64_t* block_size,
                    uint32_t n_chunks) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    DeflateSmem& S = *reinterpret_cast<DeflateSmem*>(smem_raw);
    uint32_t const tid = threadIdx.x, lane = tid & 31;
    uint32_t const c = blockIdx.x;
    uint64_t const at = uint64_t(c) * kBgzfChunk;
    uint32_t const n = uint32_t(min(uint64_t(kBgzfChunk), raw_len - at));
    uint32_t* const out = slots + size_t(c) * kBgzfSlotWords;
    uint32_t* const tok = work + at;              // per position: its match (len << 16 | dist, 0: none), then the tokens

    // ---- load the chunk, clear the payload slot and the tables ----
    {
        const uint4* src = reinterpret_cast<const uint4*>(raw + at);          // (chunks start at multiples of 16 bytes)
        for (uint32_t i = tid; i < n / 16; i += kDeflateThreads) reinterpret_cast<uint4*>(S.buf)[i] = src[i];
        for (uint32_t i = (n / 16) * 16 + tid; i < n + 8; i += kDeflateThreads) S.buf[i] = i < n ? raw[at + i] : 0;
        for (uint32_t i = tid; i < kBgzfSlotWords / 4; i += kDeflateThreads) reinterpret_cast<uint4*>(out)[i] = make_uint4(0, 0, 0, 0);
        for (uint32_t i = tid; i < (1u << kDeflateHashBits); i += kDeflateThreads) S.head[i] = 0;
        for (uint32_t i = tid; i < 288; i += kDeflateThreads) { S.lit_freq[i] = i == 256; S.lit_len[i] = 0; }   // (one end-of-block)
        if (tid < 32) { S.dist_freq[tid] = 0; S.dist_len[tid] = 0; }
        if (tid < 20) { S.cl_freq[tid] = 0; S.cl_len[tid] = 0; }
        if (tid < 256) {
            uint32_t v = tid;
            for (int k = 0; k < 8; ++k) v = v & 1 ? (v >> 1) ^ 0xedb88320u : v >> 1;
            S.crc_table[tid] = v;
        }
        if (c == 0 && tid == 0) { block_size[n_chunks] = 28; block_size[n_chunks + 1] = 0; }     // the end-of-file block
    }
    __syncthreads();

    // ---- hash chains, one tile of kDeflateThreads positions at a time: a position's candidate is the nearest earlier
    //      one with its hash in its warp, else the latest one before the tile (atomicMax keeps this deterministic) ----
    for (uint32_t base = 0; base < n; base += kDeflateThreads) {
        uint32_t const i = base + tid;
        bool const valid = i + 3 <= n;
        uint32_t h = 0;
        if (valid) h = ((uint32_t(S.buf[i]) | uint32_t(S.buf[i + 1]) << 8 | uint32_t(S.buf[i + 2]) << 16) * 2654435761u) >> (32 - kDeflateHashBits);
        uint32_t const peers = __match_any_sync(0xffffffffu, valid ? h : (0x80000000u | lane));
        uint32_t const lower = peers & ((1u << lane) - 1);
        if (i < n) {
            uint32_t cand = kNoPrev;
            if (valid) {
                if (lower) cand = i - (lane - (31 - __clz(lower)));
                else if (S.head[h]) cand = S.head[h] - 1;
            }
            S.prev[i] = uint16_t(cand);
        }
        __syncthreads();
        if (valid && (peers >> lane) == 1u) atomicMax(&S.head[h], i + 1);          // the highest lane of its hash
        __syncthreads();
    }

    // ---- the longest match of every position over up to kDeflateChain candidates ----
    for (uint32_t i = tid; i < n; i += kDeflateThreads) {
        uint32_t best_len = 0, best_dist = 0;
        if (i + 3 <= n) {
            uint32_t const max_len = min(258u, n - i);
            uint32_t cand = S.prev[i];
            for (int step = 0; step < kDeflateChain && cand != kNoPrev; ++step) {
                uint32_t const dist = i - cand;
                if (dist > 32768) break;
                if (S.buf[cand + best_len] == S.buf[i + best_len]) {       // (only a longer match can win)
                    uint32_t l = 0;
                    while (l < max_len && S.buf[cand + l] == S.buf[i + l]) ++l;
                    if (l > best_len) { best_len = l; best_dist = dist; if (l >= kDeflateNice || l == max_len) break; }
                }
                cand = S.prev[cand];
            }
        }
        if (best_len < 3 || (best_len == 3 && best_dist > 4096)) best_len = 0;    // a far 3-byte match costs more than literals
        tok[i] = best_len ? best_len << 16 | best_dist : 0u;
    }
    __syncthreads();

    // ---- greedy parse per segment (tokens overwrite the matches in place: a token never lies behind its position),
    //      histograms, CRC32 per segment ----
    uint32_t const n_seg = (n + kDeflateSeg - 1) / kDeflateSeg;
    uint32_t n_tok = 0;
    if (tid < n_seg) {
        uint32_t const s0 = tid * kDeflateSeg, s1 = min(n, s0 + kDeflateSeg);
        uint32_t t = s0;
        for (uint32_t i = s0; i < s1;) {
            uint32_t const m = tok[i];
            uint32_t len = min(m >> 16, s1 - i);
            uint32_t const dist = m & 0xffffu;
            if (len >= 3 && !(len == 3 && dist > 4096)) {
                uint32_t sym, eb, ev;
                deflate_len_sym(len, sym, eb, ev); atomicAdd(&S.lit_freq[sym], 1u);
                deflate_dist_sym(dist, sym, eb, ev); atomicAdd(&S.dist_freq[sym], 1u);
                tok[t++] = len << 16 | dist;
                i += len;
            } else {
                atomicAdd(&S.lit_freq[S.buf[i]], 1u);
                tok[t++] = S.buf[i];
                ++i;
            }
        }
        n_tok = t - s0;
        uint32_t crc = ~0u;
        for (uint32_t i = s0; i < s1; ++i) crc = S.crc_table[(crc ^ S.buf[i]) & 0xff] ^ (crc >> 8);
        S.seg_crc[tid] = ~crc;
    }
    __syncthreads();
    if (tid == 0) {                                                    // a code needs two symbols at least
        int used = 0;
        for (int s = 0; s < 30; ++s) used += S.dist_freq[s] != 0;
        if (used < 2) { if (!S.dist_freq[0]) S.dist_freq[0] = 1; else S.dist_freq[1] = 1; }
        if (used == 0) S.dist_freq[1] = 1;
    }
    __syncthreads();

    // ---- Huffman codes: rank sort, code lengths (literal/length and distance on two threads), CRC fold on a third ----
    int const n_lit = __syncthreads_count(tid < 286 && S.lit_freq[tid] != 0);
    int const n_dist = __syncthreads_count(tid >= 286 && tid < 316 && S.dist_freq[tid - 286] != 0);
    if (tid < 286) rank_sort(S.lit_freq, 286, int(tid), S.sort_key, S.sort_sym);
    else if (tid < 316) rank_sort(S.dist_freq, 30, int(tid - 286), S.sort_key + 288, S.sort_sym + 288);
    __syncthreads();
    if (tid == 0) huffman_lengths(S.sort_key, S.sort_sym, n_lit, 15, S.lit_len);
    if (tid == 32) huffman_lengths(S.sort_key + 288, S.sort_sym + 288, n_dist, 15, S.dist_len);
    if (tid == 64) {
        uint32_t crc = S.seg_crc[0];
        uint32_t const op = crc_x8n(kDeflateSeg);
        for (uint32_t k = 1; k < n_seg; ++k) {
            uint32_t const len = min(n, (k + 1) * kDeflateSeg) - k * kDeflateSeg;
            crc = crc_multmodp(len == kDeflateSeg ? op : crc_x8n(len), crc) ^ S.seg_crc[k];
        }
        S.crc = crc;
    }
    __syncthreads();

    // ---- the code-length code: run-length coded lengths (16: repeat 3..6, 17: 3..10 zeros, 18: 11..138 zeros) ----
    if (tid == 0) {
        uint32_t hlit = 286, hdist = 30;
        while (hlit > 257 && !S.lit_len[hlit - 1]) --hlit;
        while (hdist > 1 && !S.dist_len[hdist - 1]) --hdist;
        uint32_t const total = hlit + hdist;
        auto len_at = [&](uint32_t k) -> uint32_t { return k < hlit ? S.lit_len[k] : S.dist_len[k - hlit]; };
        uint32_t nr = 0;
        for (uint32_t k = 0; k < total;) {
            uint32_t const l = len_at(k);
            uint32_t run = 1;
            while (k + run < total && len_at(k + run) == l) ++run;
            k += run;
            if (l == 0) {
                while (run >= 11) { uint32_t const r = min(run, 138u); S.rle_sym[nr] = 18; S.rle_extra[nr++] = uint8_t(r - 11); run -= r; }
                if (run >= 3) { S.rle_sym[nr] = 17; S.rle_extra[nr++] = uint8_t(run - 3); run = 0; }
            } else {
                S.rle_sym[nr] = uint8_t(l); S.rle_extra[nr++] = 0; --run;
                while (run >= 3) { uint32_t const r = min(run, 6u); S.rle_sym[nr] = 16; S.rle_extra[nr++] = uint8_t(r - 3); run -= r; }
            }
            while (run) { S.rle_sym[nr] = uint8_t(l); S.rle_extra[nr++] = 0; --run; }
        }
        for (uint32_t k = 0; k < nr; ++k) S.cl_freq[S.rle_sym[k]]++;
        int used = 0;
        for (int s = 0; s < 19; ++s) used += S.cl_freq[s] != 0;
        for (int s = 0; used < 2; ++s) if (!S.cl_freq[s]) { S.cl_freq[s] = 1; ++used; }
        uint32_t key[19]; uint16_t sym[19];                             // insertion sort of the (at most 19) used symbols
        int m = 0;
        for (int s = 0; s < 19; ++s) {
            if (!S.cl_freq[s]) continue;
            int j = m++;
            while (j > 0 && key[j - 1] > S.cl_freq[s]) { key[j] = key[j - 1]; sym[j] = sym[j - 1]; --j; }
            key[j] = S.cl_freq[s]; sym[j] = uint16_t(s);
        }
        huffman_lengths(key, sym, m, 7, S.cl_len);
        canonical_codes(S.lit_len, S.lit_code, 286);
        canonical_codes(S.dist_len, S.dist_code, 30);
        canonical_codes(S.cl_len, S.cl_code, 19);
        const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
        uint32_t hclen = 19;
        while (hclen > 4 && !S.cl_len[order[hclen - 1]]) --hclen;
        uint32_t bits = 3 + 5 + 5 + 4 + 3 * hclen;
        for (uint32_t k = 0; k < nr; ++k) bits += S.cl_len[S.rle_sym[k]] + (S.rle_sym[k] == 16 ? 2 : S.rle_sym[k] == 17 ? 3 : S.rle_sym[k] == 18 ? 7 : 0);
        S.n_rle = nr; S.hlit = hlit; S.hdist = hdist; S.hclen = hclen; S.hdr_bits = bits;
    }
    __syncthreads();

    // ---- bits per segment, their offsets, the choice between the coded and the stored block ----
    if (tid < n_seg) {
        uint32_t bits = 0;
        for (uint32_t k = 0; k < n_tok; ++k) {
            uint32_t const t = tok[tid * kDeflateSeg + k];
            if (t < 256) { bits += S.lit_len[t]; continue; }
            uint32_t sym, eb, ev;
            deflate_len_sym(t >> 16, sym, eb, ev); bits += S.lit_len[sym] + eb;
            deflate_dist_sym(t & 0xffffu, sym, eb, ev); bits += S.dist_len[sym] + eb;
        }
        S.seg_bits[tid] = bits;
    }
    __syncthreads();
    if (tid == 0) {
        uint32_t sum = S.hdr_bits;
        for (uint32_t k = 0; k < n_seg; ++k) { uint32_t const b = S.seg_bits[k]; S.seg_bits[k] = sum; sum += b; }
        uint32_t const coded = (sum + S.lit_len[256] + 7) / 8;
        S.stored = coded >= n + 5;
        uint32_t const payload = S.stored ? n + 5 : coded;
        info[c] = BgzfBlockInfo{payload, S.crc, n, S.stored};
        block_size[c] = 18 + uint64_t(payload) + 8;
        if (!S.stored) {
            BitWriter w(out, 0);
            w.put(1, 1); w.put(2, 2);                                  // the final block, dynamic codes
            w.put(S.hlit - 257, 5); w.put(S.hdist - 1, 5); w.put(S.hclen - 4, 4);
            const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
            for (uint32_t k = 0; k < S.hclen; ++k) w.put(S.cl_len[order[k]], 3);
            for (uint32_t k = 0; k < S.n_rle; ++k) {
                uint32_t const s = S.rle_sym[k];
                w.put(S.cl_code[s], S.cl_len[s]);
                if (s == 16) w.put(S.rle_extra[k], 2);
                else if (s == 17) w.put(S.rle_extra[k], 3);
                else if (s == 18) w.put(S.rle_extra[k], 7);
            }
            w.flush();
            BitWriter e(out, sum);
            e.put(S.lit_code[256], S.lit_len[256]);
            e.flush();
        }
    }
    __syncthreads();

    // ---- the tokens, every segment at its bit offset ----
    if (!S.stored && tid < n_seg) {
        BitWriter w(out, S.seg_bits[tid]);
        for (uint32_t k = 0; k < n_tok; ++k) {
            uint32_t const t = tok[tid * kDeflateSeg + k];
            if (t < 256) { w.put(S.lit_code[t], S.lit_len[t]); continue; }
            uint32_t sym, eb, ev;
            deflate_len_sym(t >> 16, sym, eb, ev);
            w.put(S.lit_code[sym], S.lit_len[sym]);
            if (eb) w.put(ev, eb);
            deflate_dist_sym(t & 0xffffu, sym, eb, ev);
            w.put(S.dist_code[sym], S.dist_len[sym]);
            if (eb) w.put(ev, eb);
        }
        w.flush();
    }
}

// Block c of the image at offset[c]: BGZF header (BSIZE = block size - 1), payload, CRC32, ISIZE; block n_chunks is the
// end-of-file block.
__global__ void bgzf_assemble_kernel(const uint8_t* raw, const uint32_t* slots, const BgzfBlockInfo* info, const uint64_t* offset,
                                     uint32_t n_chunks, uint8_t* image) {
    uint32_t const c = blockIdx.x;
    uint8_t* const dst = image + offset[c];
    const uint8_t head[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
    if (c == n_chunks) {
        if (threadIdx.x < 28) dst[threadIdx.x] = threadIdx.x < 16 ? head[threadIdx.x] : threadIdx.x == 16 ? 0x1b : threadIdx.x == 18 ? 3 : 0;
        return;
    }
    BgzfBlockInfo const I = info[c];
    if (threadIdx.x < 16) dst[threadIdx.x] = head[threadIdx.x];
    if (threadIdx.x == 0) {
        put_le(dst + 16, 18 + I.payload + 8 - 1, 2);
        put_le(dst + 18 + I.payload, I.crc, 4);
        put_le(dst + 22 + I.payload, I.isize, 4);
    }
    uint8_t* const p = dst + 18;
    if (I.stored) {                                                    // BFINAL, BTYPE 00, LEN, NLEN, the bytes
        if (threadIdx.x == 0) { p[0] = 1; put_le(p + 1, I.isize, 2); put_le(p + 3, ~I.isize, 2); }
        const uint8_t* const src = raw + uint64_t(c) * kBgzfChunk;
        for (uint32_t i = threadIdx.x; i < I.isize; i += blockDim.x) p[5 + i] = src[i];
    } else {
        const uint8_t* const src = reinterpret_cast<const uint8_t*>(slots + size_t(c) * kBgzfSlotWords);
        for (uint32_t i = threadIdx.x; i < I.payload; i += blockDim.x) p[i] = src[i];
    }
}

}  // namespace fxg

