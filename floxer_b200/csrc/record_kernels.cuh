// record_kernels.cuh -- device code of the record writers (fxg_write_bam_device, fxg_write_sam_device) for sm_100a.
//
// The BAM records are those of bam_output.cpp and the SAM text that of sam_output.cpp, byte for byte.  Both formats take
// the same per-read records and arguments from the host, and the same steps:
//   sizes     bam_size_kernel / sam_size_kernel: one warp per read -- the stable order of its alignments by reference
//             id and its primary (the first one in that order with the read's fewest errors), shared as
//             for_each_record_in_order; every record's size (BAM: with its CIGAR spans; SAM: from the decimal digits of
//             its flag, POS, NM and CIGAR lengths plus its name, reference name, SEQ and QUAL lengths);
//   offsets   an exclusive scan of the sizes (cub, on the host's stream) behind the header the host put in front;
//   write     bam_write_kernel: one warp per record, lanes striding over the name, CIGAR, SEQ nibbles and QUAL bytes;
//             sam_write_kernel: one warp per record -- lane 0 writes the short fields, the lanes stride over the name,
//             the reference name, SEQ and QUAL; the CIGAR is written 32 operations at a time, each lane placing its
//             operation's text by a warp prefix sum of the text lengths, so no CIGAR is left to one thread.
// The BGZF blocks of the output are bgzf_kernels.cuh's.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/floxer_gpu.h"
#include "bgzf_kernels.cuh"                           // put_le

namespace fxg {

// one read as the record kernels see it (built by the host from fxg_read / fxg_sam_query)
struct OutReadRec {
    uint64_t seq;                // its ranks in the uploaded forward-pool range
    uint64_t name, qual;         // offsets of its name and its quality string in their buffers (or both in the text)
    uint32_t l_seq, l_name;      // l_seq = 0: SEQ '*' (SAM); l_name: BAM's counts the NUL
    uint32_t l_qual, al0;        // l_qual = 0: no usable quality (SAM: QUAL '*'; BAM: QUAL 0xff)
    uint32_t n_al, rec0;         // its alignments; its first record
};

// one output record (bam_size_kernel -> bam_write_kernel)
struct BamRecord {
    uint64_t qspan, rspan;       // CIGAR spans on the query and on the reference
    uint32_t read, al;           // al = ~0: the read's unmapped record
    uint32_t flag, l_seq;        // l_seq = 0 for a secondary record
};

// one output record (sam_size_kernel -> sam_write_kernel)
struct SamRecord {
    uint64_t cigar_chars;        // the CIGAR's text length ('*' counts 1)
    uint32_t read, al;           // al = ~0: the read's unmapped record
    uint32_t flag, pad;          // flag & 256: secondary (no SEQ / QUAL)
};

struct OutArgs {
    const OutReadRec* reads; uint32_t n_reads;
    const fxg_alignment* al;
    const uint32_t* cigars; uint64_t cigar_lo;       // the uploaded CIGAR range begins at pool offset cigar_lo
    const uint8_t* seq; const char* names; const char* quals;
    const char* ref_names; const uint64_t* ref_off;  // (SAM) reference r's name: ref_names[ref_off[r], ref_off[r + 1])
    void* recs; uint64_t* rec_off;                   // recs: BamRecord / SamRecord; rec_off: sizes, then (scanned in place)
                                                     // offsets; n_rec + 1 entries
    uint8_t* out; uint64_t body;                     // the records start at out + body, behind the header
};

__device__ __forceinline__ unsigned long long warp_sum_u64(unsigned long long v) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long v) {
    for (int o = 16; o; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__device__ __forceinline__ uint32_t bam_nm_bytes(uint32_t nm) { return 3u + (nm < 256 ? 1u : nm < 65536 ? 2u : 4u); }

__device__ __forceinline__ uint32_t bam_reg2bin(int64_t beg, int64_t end) {      // SAM specification, section 5.3
    --end;
    if (beg >> 14 == end >> 14) return uint32_t(((1 << 15) - 1) / 7 + (beg >> 14));
    if (beg >> 17 == end >> 17) return uint32_t(((1 << 12) - 1) / 7 + (beg >> 17));
    if (beg >> 20 == end >> 20) return uint32_t(((1 << 9) - 1) / 7 + (beg >> 20));
    if (beg >> 23 == end >> 23) return uint32_t(((1 << 6) - 1) / 7 + (beg >> 23));
    if (beg >> 26 == end >> 26) return uint32_t(((1 << 3) - 1) / 7 + (beg >> 26));
    return 0;
}

// The record order of one read, for a whole warp (every lane calls emit(k, a, slot, primary) for k = 0 .. n_al-1):
// slot is alignment k's place in the stable order of the read's alignments by reference id, primary tells whether it
// is the first in that order with the read's fewest errors (output.cpp:57-67).  Both formats' size kernels
// share it.
template <class Emit>
__device__ __forceinline__ void for_each_record_in_order(const fxg_alignment* al, uint32_t n_al, uint32_t lane, Emit&& emit) {
    unsigned long long best = ~0ull;
    for (uint32_t k = lane; k < n_al; k += 32) best = min(best, (unsigned long long)al[k].num_errors);
    best = warp_min_u64(best);
    unsigned long long primary = ~0ull;                                // (reference id, index) of the primary
    for (uint32_t k = lane; k < n_al; k += 32)
        if (al[k].num_errors == best) primary = min(primary, (unsigned long long)(uint64_t(al[k].reference_id) << 32 | k));
    primary = warp_min_u64(primary);
    for (uint32_t k = 0; k < n_al; ++k) {
        fxg_alignment const a = al[k];
        unsigned long long before = 0;
        for (uint32_t j = lane; j < n_al; j += 32)
            before += al[j].reference_id < a.reference_id || (al[j].reference_id == a.reference_id && j < k);
        before = warp_sum_u64(before);
        emit(k, a, uint32_t(before), (uint64_t(a.reference_id) << 32 | k) == primary);
    }
}

// ------------------------------------------------------------------------------------------------ BAM records

__global__ void bam_size_kernel(OutArgs A) {
    uint32_t const r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t const lane = threadIdx.x & 31;
    if (r >= A.n_reads) return;
    OutReadRec const R = A.reads[r];
    BamRecord* const recs = static_cast<BamRecord*>(A.recs);
    uint64_t const seq_bytes = (uint64_t(R.l_seq) + 1) / 2 + R.l_seq;
    if (R.n_al == 0) {                                                 // output.cpp:95-107: one unmapped record
        if (lane == 0) {
            recs[R.rec0] = BamRecord{0, 0, r, ~0u, 4u, R.l_seq};
            A.rec_off[R.rec0] = 36 + R.l_name + seq_bytes;
        }
        return;
    }
    for_each_record_in_order(A.al + R.al0, R.n_al, lane, [&](uint32_t k, fxg_alignment const& a, uint32_t before, bool is_primary) {
        const uint32_t* const ops = A.cigars + (a.cigar_offset - A.cigar_lo);
        unsigned long long qs = 0, rs = 0;
        for (uint32_t i = lane; i < a.cigar_len; i += 32) {
            uint32_t const op = ops[i] & 15u, n = ops[i] >> 4;
            if (op == FXG_CIGAR_D || op == FXG_CIGAR_EQ || op == FXG_CIGAR_X) rs += n;
            if (op == FXG_CIGAR_I || op == FXG_CIGAR_EQ || op == FXG_CIGAR_X) qs += n;
        }
        qs = warp_sum_u64(qs); rs = warp_sum_u64(rs);
        if (lane == 0) {
            bool const long_cigar = a.cigar_len > 65535;
            uint32_t const flag = (a.orientation == FXG_REVERSE_COMPLEMENT ? 16u : 0u) | (is_primary ? 0u : 256u);
            uint64_t size = 36 + R.l_name + 4 * uint64_t(long_cigar ? 2 : a.cigar_len) + bam_nm_bytes(a.num_errors);
            if (is_primary) size += seq_bytes;
            if (long_cigar) size += 8 + 4 * uint64_t(a.cigar_len);
            uint32_t const slot = R.rec0 + before;
            recs[slot] = BamRecord{qs, rs, r, R.al0 + k, flag, is_primary ? R.l_seq : 0u};
            A.rec_off[slot] = size;
        }
    });
}

__global__ void bam_write_kernel(OutArgs A, uint32_t n_rec) {
    uint32_t const i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t const lane = threadIdx.x & 31;
    if (i >= n_rec) return;
    BamRecord const rec = static_cast<const BamRecord*>(A.recs)[i];
    OutReadRec const R = A.reads[rec.read];
    uint8_t* p = A.out + A.body + A.rec_off[i];
    uint32_t const size = uint32_t(A.rec_off[i + 1] - A.rec_off[i] - 4);
    bool const mapped = rec.al != ~0u;
    fxg_alignment a{};
    if (mapped) a = A.al[rec.al];
    uint32_t const n_ops = mapped ? a.cigar_len : 0;
    bool const long_cigar = n_ops > 65535;
    uint32_t const n_written = long_cigar ? 2 : n_ops;
    const uint32_t* const ops = mapped ? A.cigars + (a.cigar_offset - A.cigar_lo) : nullptr;
    uint32_t const placeholder[2] = {uint32_t(rec.qspan) << 4 | 4u /* S */, uint32_t(rec.rspan) << 4 | 3u /* N */};
    if (lane == 0) {
        int64_t const pos = mapped ? int64_t(min((unsigned long long)a.start_in_reference, (unsigned long long)INT32_MAX)) : -1;
        int64_t const end = pos + int64_t(max((unsigned long long)rec.rspan, 1ull));
        uint32_t const bin = pos < 0 || end > (int64_t(1) << 29) ? 4680u : bam_reg2bin(pos, end);
        put_le(p, size, 4);
        put_le(p + 4, mapped ? a.reference_id : ~0u, 4);
        put_le(p + 8, uint32_t(int32_t(pos)), 4);
        p[12] = uint8_t(R.l_name); p[13] = 255;                       // MAPQ 255: not available
        put_le(p + 14, bin, 2);
        put_le(p + 16, n_written, 2);
        put_le(p + 18, rec.flag, 2);
        put_le(p + 20, rec.l_seq, 4);
        put_le(p + 24, ~0u, 4); put_le(p + 28, ~0u, 4); put_le(p + 32, 0, 4);     // no mate
    }
    p += 36;
    for (uint32_t j = lane; j < R.l_name; j += 32) p[j] = j + 1 < R.l_name ? uint8_t(A.names[R.name + j]) : uint8_t(0);     // (the NUL)
    p += R.l_name;
    for (uint32_t j = lane; j < n_written; j += 32) put_le(p + 4 * j, long_cigar ? placeholder[j] : ops[j], 4);
    p += 4 * size_t(n_written);
    // ranks 0..5 = $ A C G T N as nibbles of "=ACMGRSVTWYHKDBN" ('$' has no code: N)
    uint32_t const l_seq = rec.l_seq;
    const uint8_t* const seq = A.seq + R.seq;
    for (uint32_t j = lane; j < (l_seq + 1) / 2; j += 32) {
        uint32_t const nib = 0xf8421fu;                                // 15, 1, 2, 4, 8, 15 at 4 bits each (rank 0 low)
        uint32_t const r0 = min(uint32_t(seq[2 * j]), 5u);
        uint32_t const hi = (nib >> (4 * r0)) & 15u;
        uint32_t const lo = 2 * j + 1 < l_seq ? (nib >> (4 * min(uint32_t(seq[2 * j + 1]), 5u))) & 15u : 0u;
        p[j] = uint8_t(hi << 4 | lo);
    }
    p += (l_seq + 1) / 2;
    bool const have_qual = R.l_qual != 0;
    for (uint32_t j = lane; j < l_seq; j += 32) p[j] = have_qual ? uint8_t(A.quals[R.qual + j] - 33) : uint8_t(0xff);
    p += l_seq;
    if (!mapped) return;
    uint32_t const nm = a.num_errors;
    if (lane == 0) {
        p[0] = 'N'; p[1] = 'M';
        if (nm < 256) { p[2] = 'C'; p[3] = uint8_t(nm); }
        else if (nm < 65536) { p[2] = 'S'; put_le(p + 3, nm, 2); }
        else { p[2] = 'I'; put_le(p + 3, nm, 4); }
    }
    p += bam_nm_bytes(nm);
    if (!long_cigar) return;
    if (lane == 0) { p[0] = 'C'; p[1] = 'G'; p[2] = 'B'; p[3] = 'I'; put_le(p + 4, n_ops, 4); }
    p += 8;
    for (uint32_t j = lane; j < n_ops; j += 32) put_le(p + 4 * size_t(j), ops[j], 4);
}

// ------------------------------------------------------------------------------------------------ SAM records

constexpr uint32_t kSamUnmappedFields = 19;          // "\t4\t*\t0\t255\t*\t*\t0\t0\t"

__device__ __forceinline__ uint32_t dec_digits(uint32_t v) {
    uint32_t n = 1;
    for (uint32_t p = 10; n < 10 && v >= p; p *= 10) ++n;
    return n;
}

__device__ __forceinline__ void put_dec(char* p, uint32_t v, uint32_t n) {
    for (uint32_t i = n; i > 0; --i) { p[i - 1] = char('0' + v % 10); v /= 10; }
}

__device__ __forceinline__ char sam_op_char(uint32_t op) {
    return op == FXG_CIGAR_I ? 'I' : op == FXG_CIGAR_D ? 'D' : op == FXG_CIGAR_EQ ? '=' : op == FXG_CIGAR_X ? 'X' : '?';
}

// POS = min(start, INT32_MAX) + 1 (math.hpp:10-16): at most 2^31, which fits 32 bits
__device__ __forceinline__ uint32_t sam_pos1(uint64_t start) { return uint32_t(min((unsigned long long)start, (unsigned long long)INT32_MAX)) + 1u; }

// the lanes copy n bytes
__device__ __forceinline__ void warp_copy(char* dst, const char* src, uint64_t n, uint32_t lane) {
    for (uint64_t j = lane; j < n; j += 32) dst[j] = src[j];
}

// SEQ '\t' QUAL at p (the forward read, rank 0 '$', 1..5 ACGTN, >= 6 N; '*' when empty); returns the bytes written
__device__ __forceinline__ uint64_t sam_seq_qual(char* p, OutArgs const& A, OutReadRec const& R, uint32_t lane) {
    const uint8_t* const seq = A.seq + R.seq;
    for (uint32_t j = lane; j < R.l_seq; j += 32) {
        uint32_t const rk = seq[j];
        p[j] = rk < 6 ? "$ACGTN"[rk] : 'N';
    }
    uint64_t const ls = R.l_seq ? R.l_seq : 1;
    if (lane == 0) {
        if (!R.l_seq) p[0] = '*';
        p[ls] = '\t';
        if (!R.l_qual) p[ls + 1] = '*';
    }
    warp_copy(p + ls + 1, A.quals + R.qual, R.l_qual, lane);
    return ls + 1 + (R.l_qual ? R.l_qual : 1);
}

__global__ void sam_size_kernel(OutArgs A) {
    uint32_t const r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t const lane = threadIdx.x & 31;
    if (r >= A.n_reads) return;
    OutReadRec const R = A.reads[r];
    SamRecord* const recs = static_cast<SamRecord*>(A.recs);
    uint64_t const seq_qual = uint64_t(R.l_seq ? R.l_seq : 1) + 1 + (R.l_qual ? R.l_qual : 1);
    if (R.n_al == 0) {                                                 // output.cpp:95-107: one unmapped record
        if (lane == 0) {
            recs[R.rec0] = SamRecord{1, r, ~0u, 4u, 0};
            A.rec_off[R.rec0] = R.l_name + kSamUnmappedFields + seq_qual + 1;
        }
        return;
    }
    for_each_record_in_order(A.al + R.al0, R.n_al, lane, [&](uint32_t k, fxg_alignment const& a, uint32_t before, bool is_primary) {
        const uint32_t* const ops = A.cigars + (a.cigar_offset - A.cigar_lo);
        unsigned long long chars = 0;
        for (uint32_t i = lane; i < a.cigar_len; i += 32) chars += dec_digits(ops[i] >> 4) + 1;
        chars = warp_sum_u64(chars);
        if (lane == 0) {
            if (a.cigar_len == 0) chars = 1;                           // '*'
            uint32_t const flag = (a.orientation == FXG_REVERSE_COMPLEMENT ? 16u : 0u) | (is_primary ? 0u : 256u);
            uint64_t const l_rname = A.ref_off[a.reference_id + 1] - A.ref_off[a.reference_id];
            // name \t flag \t rname \t pos \t255\t cigar \t*\t0\t0\t (SEQ \t QUAL | *\t*) \tNM:i: nm \n
            uint64_t const size = R.l_name + 1 + dec_digits(flag) + 1 + l_rname + 1 + dec_digits(sam_pos1(a.start_in_reference)) + 5 +
                                  chars + 7 + (is_primary ? seq_qual : 3) + 6 + dec_digits(a.num_errors) + 1;
            uint32_t const slot = R.rec0 + before;
            recs[slot] = SamRecord{chars, r, R.al0 + k, flag, 0};
            A.rec_off[slot] = size;
        }
    });
}

__global__ void sam_write_kernel(OutArgs A, uint32_t n_rec) {
    uint32_t const i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t const lane = threadIdx.x & 31;
    if (i >= n_rec) return;
    SamRecord const rec = static_cast<const SamRecord*>(A.recs)[i];
    OutReadRec const R = A.reads[rec.read];
    char* p = reinterpret_cast<char*>(A.out) + A.body + A.rec_off[i];
    warp_copy(p, A.names + R.name, R.l_name, lane);
    p += R.l_name;
    if (rec.al == ~0u) {                                               // unmapped
        if (lane < kSamUnmappedFields) p[lane] = "\t4\t*\t0\t255\t*\t*\t0\t0\t"[lane];
        p += kSamUnmappedFields;
        p += sam_seq_qual(p, A, R, lane);
        if (lane == 0) *p = '\n';
        return;
    }
    fxg_alignment const a = A.al[rec.al];
    uint64_t const r0 = A.ref_off[a.reference_id], l_rname = A.ref_off[a.reference_id + 1] - r0;
    uint32_t const n_flag = dec_digits(rec.flag), pos1 = sam_pos1(a.start_in_reference), n_pos = dec_digits(pos1);
    if (lane == 0) {
        p[0] = '\t'; put_dec(p + 1, rec.flag, n_flag); p[1 + n_flag] = '\t';
        char* const q = p + 2 + n_flag + l_rname;
        q[0] = '\t'; put_dec(q + 1, pos1, n_pos);
        q[1 + n_pos] = '\t'; q[2 + n_pos] = '2'; q[3 + n_pos] = '5'; q[4 + n_pos] = '5'; q[5 + n_pos] = '\t';
    }
    warp_copy(p + 2 + n_flag, A.ref_names + r0, l_rname, lane);
    p += 2 + n_flag + l_rname + 6 + n_pos;

    // the CIGAR: 32 operations at a time, each one's text placed by a prefix sum of the text lengths (digits + 1)
    const uint32_t* const ops = A.cigars + (a.cigar_offset - A.cigar_lo);
    if (a.cigar_len == 0 && lane == 0) p[0] = '*';
    uint64_t base = 0;
    for (uint32_t j0 = 0; j0 < a.cigar_len; j0 += 32) {
        uint32_t const j = j0 + lane;
        uint32_t const v = j < a.cigar_len ? ops[j] : 0u;
        uint32_t const len = j < a.cigar_len ? dec_digits(v >> 4) + 1 : 0u;
        uint32_t incl = len;
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t const t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= uint32_t(o)) incl += t;
        }
        if (len) {
            char* const q = p + base + (incl - len);
            put_dec(q, v >> 4, len - 1);
            q[len - 1] = sam_op_char(v & 15u);
        }
        base += __shfl_sync(0xffffffffu, incl, 31);
    }
    p += rec.cigar_chars;

    if (lane == 0) { p[0] = '\t'; p[1] = '*'; p[2] = '\t'; p[3] = '0'; p[4] = '\t'; p[5] = '0'; p[6] = '\t'; }
    p += 7;
    if (rec.flag & 256u) {
        if (lane == 0) { p[0] = '*'; p[1] = '\t'; p[2] = '*'; }
        p += 3;
    } else {
        p += sam_seq_qual(p, A, R, lane);
    }
    if (lane == 0) {
        uint32_t const n_nm = dec_digits(a.num_errors);
        p[0] = '\t'; p[1] = 'N'; p[2] = 'M'; p[3] = ':'; p[4] = 'i'; p[5] = ':';
        put_dec(p + 6, a.num_errors, n_nm);
        p[6 + n_nm] = '\n';
    }
}

}  // namespace fxg

