// seed_kernels.cuh -- device code of the batch seeder (fxg_gpu_seeder_create / fxg_seed_reads) for sm_100a.
//
// The same q-gram seeder as seeder.cpp, for every (read, orientation, leaf) of a batch at once:
//   index     seed_index_count_kernel / seed_index_fill_kernel: a counting sort of the q-grams of the resident 4-bit store
//             (positions in the unpadded concatenation, as the host seeder numbers them);
//   plan      seed_plan_kernel: one thread per seed -- its e + 1 pigeonhole pieces, the q-gram occurrences they have;
//   emit      seed_emit_kernel: (seed, nominal start) keys, radix-sorted and made unique on the host's stream;
//   check     seed_check_kernel<E>: one thread per distinct nominal start checks the starts nominal - e .. nominal + e that
//             no smaller nominal of its seed covers (so every distinct candidate start is checked once), with the host's
//             banded prefix_distance, band in registers;
//   caps      seed_caps_kernel on hits sorted by (seed, errors, position): hard cap, soft cap;
//   erase     seed_erase_kernel on kept hits sorted by (seed, position): the host's erase_useless per (seed, reference);
//   output    seed_output_kernel<J>: the survivors in seed order -- fxg_anchor records (fxg_seed_reads) or a verification job's
//             AnchorRec16 (fxg_seed_verify_reads) -- and counts per (read, orientation).
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace fxg {

constexpr int kSeedMaxErrors = 8;                 // fxg_seeder_search refuses leaves with more
constexpr int kSeedKeyShift = 33;                 // emit keys: seed << 33 | (nominal + e)
constexpr int kHitKeyShift = 36;                  // hit keys: seed << 36 | errors << 32 | position
constexpr uint64_t kSeedSentinel = ~uint64_t(0);

// a seed packed into one word: position of its first base in the device query pool (forward pool, then the reverse
// complement pool) in bits 0..39, length in bits 40..59, errors in bits 60..63
__host__ __device__ __forceinline__ uint64_t seed_pack(uint64_t qpos, uint32_t m, uint32_t e) { return qpos | (uint64_t(m) << 40) | (uint64_t(e) << 60); }
__device__ __forceinline__ uint64_t seed_qpos(uint64_t s) { return s & ((uint64_t(1) << 40) - 1); }
__device__ __forceinline__ uint32_t seed_len(uint64_t s) { return uint32_t(s >> 40) & ((1u << 20) - 1); }
__device__ __forceinline__ uint32_t seed_err(uint64_t s) { return uint32_t(s >> 60); }

struct SeedRefs {
    const uint32_t* packed;      // the context's 4-bit store (every reference at a multiple of 32 bases)
    const uint64_t* ubase;       // start of reference r in the unpadded concatenation
    const uint64_t* pbase;       // ... and in the store
    const uint64_t* len;
    uint32_t n_refs;
};

// last r with ubase[r] <= g (std::upper_bound - 1, as seeder.cpp picks the reference of a candidate)
__device__ __forceinline__ uint32_t seed_ref_of(const uint64_t* __restrict__ ubase, uint32_t n, uint64_t g) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) { uint32_t const mid = (lo + hi) >> 1; if (ubase[mid] <= g) lo = mid + 1; else hi = mid; }
    return lo - 1;
}

// first i in [lo, hi) with a[i] > v
template <class T>
__device__ __forceinline__ uint64_t seed_upper_bound(const T* __restrict__ a, uint64_t lo, uint64_t hi, T v) {
    while (lo < hi) { uint64_t const mid = (lo + hi) >> 1; if (a[mid] <= v) lo = mid + 1; else hi = mid; }
    return lo;
}

__device__ __forceinline__ void seed_add(unsigned long long* ctr, uint64_t v) {      // warp-aggregated counter
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(ctr, (unsigned long long)v);
}

// ------------------------------------------------------------------------------------------------ index

// code of the q-gram at unpadded position g, or false if it crosses the end of its reference or holds a rank outside 1..4
__device__ __forceinline__ bool seed_ref_gram(SeedRefs const& R, uint64_t g, uint32_t q, uint32_t& code) {
    uint32_t const r = seed_ref_of(R.ubase, R.n_refs, g);
    uint64_t const p = g - R.ubase[r];
    if (p + q > R.len[r]) return false;
    uint64_t const at = R.pbase[r] + p;
    uint32_t c = 0;
    for (uint32_t i = 0; i < q; ++i) {
        uint32_t const b = packed_base(R.packed, at + i);
        if (b < 1 || b > 4) return false;
        c = (c << 2) | (b - 1);
    }
    code = c;
    return true;
}

__global__ void seed_index_count_kernel(SeedRefs R, uint64_t total, uint32_t q, uint32_t* __restrict__ counts) {
    for (uint64_t g = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; g < total; g += uint64_t(gridDim.x) * blockDim.x) {
        uint32_t code;
        if (seed_ref_gram(R, g, q, code)) atomicAdd(&counts[code], 1u);
    }
}

// The positions of a bucket land in whatever order the atomics hand out the slots.  That is enough: every user of a
// bucket (seed_emit_kernel) sorts and de-duplicates its candidates before it looks at them, as the host seeder does.
__global__ void seed_index_fill_kernel(SeedRefs R, uint64_t total, uint32_t q, uint32_t* __restrict__ cursor, uint32_t* __restrict__ pos) {
    for (uint64_t g = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x; g < total; g += uint64_t(gridDim.x) * blockDim.x) {
        uint32_t code;
        if (seed_ref_gram(R, g, q, code)) pos[atomicAdd(&cursor[code], 1u)] = uint32_t(g);
    }
}

// ------------------------------------------------------------------------------------------------ seeds

struct SeedBatch {
    const uint8_t* pool;             // forward pool, then the reverse-complement pool (pool_len bytes each)
    uint64_t pool_len;
    const uint32_t* seed_base;       // per read (+1): first seed id; seeds of read r: forward leaves, then reverse leaves
    const uint32_t* leaf_base;       // per read (+1): first entry of `leaves`
    const uint64_t* leaves;          // per (read, leaf): seed_pack(query_offset + from, m, e)
    uint32_t n_reads, n_seeds;
    const uint32_t* bucket;          // the index
    const uint32_t* pos;
    uint32_t q;
};

// piece k of a seed of length m with e errors starts at m * k / (e + 1) (seeder.cpp)
__device__ __forceinline__ bool seed_piece_code(const uint8_t* __restrict__ s, uint32_t q, uint32_t& code) {
    uint32_t c = 0;
    for (uint32_t i = 0; i < q; ++i) {
        uint32_t const r = s[i];
        if (r < 1 || r > 4) return false;
        c = (c << 2) | (r - 1);
    }
    code = c;
    return true;
}

// per seed: its packed descriptor and the q-gram occurrences of its pieces
__global__ void seed_plan_kernel(SeedBatch B, uint64_t* __restrict__ info, uint64_t* __restrict__ occ) {
    uint32_t const s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= B.n_seeds) return;
    uint32_t const r = uint32_t(seed_upper_bound(B.seed_base, 0, B.n_reads + 1, s)) - 1;
    uint32_t const local = s - B.seed_base[r], nl = B.leaf_base[r + 1] - B.leaf_base[r];
    uint32_t const strand = local >= nl, li = local - strand * nl;
    uint64_t const d = B.leaves[B.leaf_base[r] + li] + (strand ? B.pool_len : 0);
    info[s] = d;
    uint32_t const m = seed_len(d), e = seed_err(d);
    const uint8_t* q = B.pool + seed_qpos(d);
    uint64_t n = 0;
    for (uint32_t k = 0; k <= e; ++k) {
        uint32_t code;
        if (seed_piece_code(q + uint64_t(m) * k / (e + 1), B.q, code)) n += B.bucket[code + 1] - B.bucket[code];
    }
    occ[s] = n;
}

// seeds [s0, s1): every occurrence of every piece as key (seed - s0) << 33 | (nominal + e); nominals below -e give no
// candidate start >= 0 and become the sentinel.  ctr[0] += candidate starts >= 0 before de-duplication.
__global__ void seed_emit_kernel(SeedBatch B, const uint64_t* __restrict__ info, const uint64_t* __restrict__ off, uint32_t s0, uint32_t s1,
                                 uint64_t* __restrict__ keys, unsigned long long* __restrict__ ctr) {
    uint32_t const s = s0 + blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t cand = 0;
    if (s < s1) {
        uint64_t const d = info[s];
        uint32_t const m = seed_len(d), e = seed_err(d);
        const uint8_t* q = B.pool + seed_qpos(d);
        uint64_t at = off[s] - off[s0];
        for (uint32_t k = 0; k <= e; ++k) {
            uint32_t const po = uint32_t(uint64_t(m) * k / (e + 1));
            uint32_t code;
            if (!seed_piece_code(q + po, B.q, code)) continue;
            for (uint32_t x = B.bucket[code]; x < B.bucket[code + 1]; ++x) {
                int64_t const nominal = int64_t(B.pos[x]) - int64_t(po);
                if (nominal >= -int64_t(e)) {
                    keys[at++] = (uint64_t(s - s0) << kSeedKeyShift) | uint64_t(nominal + e);
                    cand += uint64_t(nominal >= int64_t(e) ? 2 * e + 1 : nominal + e + 1);
                } else {
                    keys[at++] = kSeedSentinel;
                }
            }
        }
    }
    seed_add(&ctr[0], cand);
}

// seeder.cpp's prefix_distance with the band in registers: min over prefixes t of the text (at most text_len bases) of
// the edit distance of the seed and t if <= E, else E + 1.  The text is read from the store; win[x] holds the base the
// cell at band index x compares against (text[i + x - E - 1]).
template <int E>
__device__ __forceinline__ uint32_t seed_prefix_distance(const uint8_t* __restrict__ seed, uint32_t m, const uint32_t* __restrict__ packed,
                                                         uint64_t text_at, uint32_t text_len) {
    constexpr uint32_t inf = E + 1;
    constexpr int W = 2 * E + 1;
    uint32_t prev[W], cur[W], win[W];
#pragma unroll
    for (int x = 0; x < W; ++x) {
        int const j = x - E;
        prev[x] = j >= 0 && j <= E ? uint32_t(j) : inf;        // row 0: D[0][j] = j
        int64_t const t = int64_t(x) - E;                        // text index of row 1, band index x
        win[x] = t >= 0 && t < int64_t(text_len) ? packed_base(packed, text_at + uint64_t(t)) : 0u;
    }
    for (uint32_t i = 1; i <= m; ++i) {
        if (i > 1) {
#pragma unroll
            for (int x = 0; x + 1 < W; ++x) win[x] = win[x + 1];
            int64_t const t = int64_t(i) + E - 1;
            win[W - 1] = t < int64_t(text_len) ? packed_base(packed, text_at + uint64_t(t)) : 0u;
        }
        uint32_t const sc = seed[i - 1];
        uint32_t row_min = inf;
#pragma unroll
        for (int x = 0; x < W; ++x) {
            int64_t const j = int64_t(i) + x - E;
            uint32_t v = inf;
            if (j >= 0 && j <= int64_t(text_len)) {
                if (j == 0) v = i <= uint32_t(E) ? i : inf;
                else {
                    uint32_t const diag = prev[x] + (sc != win[x] ? 1u : 0u);
                    uint32_t const up = x + 1 < W ? prev[x + 1] + 1 : inf;
                    uint32_t const left = x > 0 ? cur[x - 1] + 1 : inf;
                    v = min(min(diag, up), left);
                    if (v > inf) v = inf;
                }
            }
            cur[x] = v;
            row_min = min(row_min, v);
        }
        if (row_min >= inf) return inf;
#pragma unroll
        for (int x = 0; x < W; ++x) prev[x] = cur[x];
    }
    uint32_t best = inf;
#pragma unroll
    for (int x = 0; x < W; ++x) best = min(best, prev[x]);
    return best;
}

// the starts of one distinct nominal that no smaller nominal of the same seed covers; ctr[1] += checked, ctr[2] += hits
template <int E>
__device__ __forceinline__ void seed_check_starts(SeedRefs const& R, const uint8_t* __restrict__ seed, uint32_t m, uint64_t sl, int64_t nominal,
                                                  int64_t covered_to, uint64_t* __restrict__ hits, uint64_t hit_cap,
                                                  unsigned long long* __restrict__ ctr, uint64_t& checked) {
    for (int64_t x = nominal - E; x <= nominal + E; ++x) {
        if (x < 0 || x <= covered_to) continue;
        uint64_t const g = uint64_t(x);
        uint32_t const r = seed_ref_of(R.ubase, R.n_refs, g);
        uint64_t const p = g - R.ubase[r];
        if (p >= R.len[r]) continue;
        ++checked;
        uint32_t const room = uint32_t(min(R.len[r] - p, uint64_t(m) + E));
        uint32_t const d = seed_prefix_distance<E>(seed, m, R.packed, R.pbase[r] + p, room);
        if (d <= uint32_t(E)) {
            unsigned long long const at = atomicAdd(&ctr[2], 1ull);
            if (at < hit_cap) hits[at] = (sl << kHitKeyShift) | (uint64_t(d) << 32) | g;
        }
    }
}

// one thread per distinct key of a chunk (`uniq`, *n_uniq of them, sorted)
__global__ void seed_check_kernel(SeedRefs R, SeedBatch B, const uint64_t* __restrict__ info, uint32_t s0, const uint64_t* __restrict__ uniq,
                                  const uint32_t* __restrict__ n_uniq, uint64_t* __restrict__ hits, uint64_t hit_cap,
                                  unsigned long long* __restrict__ ctr) {
    uint64_t const i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    uint64_t checked = 0;
    uint64_t const key = i < *n_uniq ? uniq[i] : kSeedSentinel;
    if (key != kSeedSentinel) {
        uint64_t const sl = key >> kSeedKeyShift;
        uint64_t const d = info[s0 + sl];
        uint32_t const m = seed_len(d), e = seed_err(d);
        const uint8_t* seed = B.pool + seed_qpos(d);
        uint64_t const mask = (uint64_t(1) << kSeedKeyShift) - 1;
        int64_t const nominal = int64_t(key & mask) - int64_t(e);
        // starts up to the previous nominal of the seed + e are that nominal's (the key holds nominal + e)
        int64_t covered_to = -1;
        if (i > 0 && (uniq[i - 1] >> kSeedKeyShift) == sl) covered_to = int64_t(uniq[i - 1] & mask);
        switch (e) {
            case 0: seed_check_starts<0>(R, seed, m, sl, nominal, covered_to, hits, hit_cap, ctr, checked); break;
            case 1: seed_check_starts<1>(R, seed, m, sl, nominal, covered_to, hits, hit_cap, ctr, checked); break;
            case 2: seed_check_starts<2>(R, seed, m, sl, nominal, covered_to, hits, hit_cap, ctr, checked); break;
            case 3: seed_check_starts<3>(R, seed, m, sl, nominal, covered_to, hits, hit_cap, ctr, checked); break;
            case 4: seed_check_starts<4>(R, seed, m, sl, nominal, covered_to, hits, hit_cap, ctr, checked); break;
            case 5: seed_check_starts<5>(R, seed, m, sl, nominal, covered_to, hits, hit_cap, ctr, checked); break;
            case 6: seed_check_starts<6>(R, seed, m, sl, nominal, covered_to, hits, hit_cap, ctr, checked); break;
            case 7: seed_check_starts<7>(R, seed, m, sl, nominal, covered_to, hits, hit_cap, ctr, checked); break;
            default: seed_check_starts<8>(R, seed, m, sl, nominal, covered_to, hits, hit_cap, ctr, checked); break;
        }
    }
    seed_add(&ctr[1], checked);
}

// hits sorted by (seed, errors, position): a seed with more than `hard` hits loses all of them (ctr[3]), otherwise the
// first `soft` stay (ctr[4] counts the rest) -- the host's stable_sort by errors of position-ordered hits.  Kept hits
// become seed << 36 | position << 4 | errors, the others the sentinel.
__global__ void seed_caps_kernel(const uint64_t* __restrict__ hits, uint64_t n, uint64_t hard, uint64_t soft, uint64_t* __restrict__ kept,
                                 unsigned long long* __restrict__ ctr) {
    uint64_t const i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    uint64_t dropped = 0, cut = 0;
    if (i < n) {
        uint64_t const sl = hits[i] >> kHitKeyShift;
        // first hit of the seed: last index whose key is below sl << 36, + 1
        uint64_t lo = 0, hi = i;
        while (lo < hi) { uint64_t const mid = (lo + hi) >> 1; if ((hits[mid] >> kHitKeyShift) < sl) lo = mid + 1; else hi = mid; }
        uint64_t const first = lo;
        uint64_t const end = seed_upper_bound(hits, i, n, (sl << kHitKeyShift) | ((uint64_t(1) << kHitKeyShift) - 1));
        uint64_t out = kSeedSentinel;
        if (end - first > hard) dropped = 1;
        else if (i - first >= soft) cut = 1;
        else out = (sl << kHitKeyShift) | ((hits[i] & 0xffffffffull) << 4) | ((hits[i] >> 32) & 15u);
        kept[i] = out;
    }
    seed_add(&ctr[3], dropped);
    seed_add(&ctr[4], cut);
}

// kept hits sorted by (seed, position), n of them: one thread per (seed, reference) run runs seeder.cpp's erase_useless
// (search.cpp:352-389) with the reference's unsigned arithmetic; erased[i] = 1 for the anchors it removes
__global__ void seed_erase_kernel(SeedRefs R, const uint64_t* __restrict__ kept, uint64_t n, uint32_t* __restrict__ erased) {
    uint64_t const lo = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (lo >= n) return;
    auto seed_of = [&](uint64_t i) { return kept[i] >> kHitKeyShift; };
    auto gpos = [&](uint64_t i) { return (kept[i] >> 4) & 0xffffffffull; };
    auto ref = [&](uint64_t i) { return seed_ref_of(R.ubase, R.n_refs, gpos(i)); };
    uint32_t const r = ref(lo);
    if (lo > 0 && seed_of(lo - 1) == seed_of(lo) && ref(lo - 1) == r) return;        // not the first of its run
    uint64_t hi = lo + 1;
    while (hi < n && seed_of(hi) == seed_of(lo) && ref(hi) == r) ++hi;
    if (hi - lo < 2) return;
    auto errs = [&](uint64_t i) -> uint64_t { return erased[i] ? 0xffffffffull : (kept[i] & 15u); };
    auto better = [&](uint64_t x, uint64_t y) {            // anchor_t::is_better_than; positions relative to the same reference
        uint64_t const px = gpos(x), py = gpos(y);
        uint64_t const dist = px < py ? py - px : px - py;
        return errs(x) <= errs(y) && dist <= errs(y) - errs(x);
    };
    for (uint64_t cur = lo; cur < hi - 1;) {
        uint64_t other = cur + 1;
        while (other < hi && better(cur, other)) { erased[other] = 1; ++other; }
        if (other < hi && better(other, cur)) erased[cur] = 1;
        cur = other;
    }
}

// survivors (they go to i - at[i], at = exclusive prefix sum of erased), counted per (read, orientation): as fxg_anchor-shaped
// records (four words: leaf, reference, position, errors), or with kJobRecords as the AnchorRec16 a verification job reads
// (position, leaf, reference; the walks do not use the errors)
template <bool kJobRecords>
__global__ void seed_output_kernel(SeedRefs R, SeedBatch B, uint32_t s0, const uint64_t* __restrict__ kept, uint64_t n,
                                   const uint32_t* __restrict__ erased, const uint32_t* __restrict__ at, void* __restrict__ out,
                                   uint32_t* __restrict__ per_read, unsigned long long* __restrict__ ctr) {
    uint64_t const i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    uint64_t gone = 0;
    if (i < n) {
        if (erased[i]) gone = 1;
        else {
            uint32_t const s = s0 + uint32_t(kept[i] >> kHitKeyShift);
            uint64_t const g = (kept[i] >> 4) & 0xffffffffull;
            uint32_t const rd = uint32_t(seed_upper_bound(B.seed_base, 0, B.n_reads + 1, s)) - 1;
            uint32_t const local = s - B.seed_base[rd], nl = B.leaf_base[rd + 1] - B.leaf_base[rd];
            uint32_t const strand = local >= nl;
            uint32_t const r = seed_ref_of(R.ubase, R.n_refs, g);
            if constexpr (kJobRecords) {
                AnchorRec16& o = static_cast<AnchorRec16*>(out)[i - at[i]];
                o.reference_position = g - R.ubase[r];
                o.pex_leaf_index = local - strand * nl;
                o.reference_id = r;
            } else {
                uint64_t* o = static_cast<uint64_t*>(out) + 4 * (i - at[i]);
                o[0] = local - strand * nl;
                o[1] = r;
                o[2] = g - R.ubase[r];
                o[3] = kept[i] & 15u;
            }
            atomicAdd(&per_read[2 * rd + strand], 1u);
        }
    }
    seed_add(&ctr[5], gone);
}

}  // namespace fxg
