// sam_kernels.cuh -- device code of the SAM writer (fxg_write_sam_device) for sm_100a.
//
// The text is that of sam_output.cpp, byte for byte:
//   sizes     sam_size_kernel: one warp per read -- the record order and primary of bam_size_kernel (the shared
//             for_each_record_in_order), every record's length from the decimal digits of its flag, POS, NM and CIGAR
//             lengths plus its name, reference name, SEQ and QUAL lengths;
//   offsets   an exclusive scan of the lengths (cub, on the host's stream) behind the @HD / @SQ header the host put in front;
//   write     sam_write_kernel: one warp per record -- lane 0 writes the short fields, the lanes stride over the name,
//             the reference name, SEQ and QUAL; the CIGAR is written 32 operations at a time, each lane placing its
//             operation's text by a warp prefix sum of the text lengths, so no CIGAR is left to one thread.
// With bgzf = 1 the text goes through bgzf_deflate_kernel / bgzf_assemble_kernel of bam_kernels.cuh.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/floxer_gpu.h"
#include "bam_kernels.cuh"

namespace fxg {

// one read as the SAM kernels see it (built by the host from fxg_read / fxg_sam_query)
struct SamReadRec {
    uint64_t seq;                // its ranks in the uploaded forward-pool range
    uint64_t name, qual;         // offsets of its name and its quality string in their buffers
    uint32_t l_seq, l_name;      // l_seq = 0: SEQ '*'
    uint32_t l_qual, al0;        // l_qual = 0: QUAL '*' (a null or empty quality)
    uint32_t n_al, rec0;         // its alignments; its first record
};

// one output record (sam_size_kernel -> sam_write_kernel)
struct SamRecord {
    uint64_t cigar_chars;        // the CIGAR's text length ('*' counts 1)
    uint32_t read, al;           // al = ~0: the read's unmapped record
    uint32_t flag, pad;          // flag & 256: secondary (no SEQ / QUAL)
};

struct SamArgs {
    const SamReadRec* reads; uint32_t n_reads;
    const fxg_alignment* al;
    const uint32_t* cigars; uint64_t cigar_lo;       // the uploaded CIGAR range begins at pool offset cigar_lo
    const uint8_t* seq; const char* names; const char* quals;
    const char* ref_names; const uint64_t* ref_off;  // reference r's name: ref_names[ref_off[r], ref_off[r + 1])
    SamRecord* recs; uint64_t* rec_off;              // rec_off: lengths, then (scanned in place) offsets; n_rec + 1 entries
    char* text; uint64_t body;                       // the records start at text + body, behind the header
};

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
__device__ __forceinline__ uint64_t sam_seq_qual(char* p, SamArgs const& A, SamReadRec const& R, uint32_t lane) {
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

__global__ void sam_size_kernel(SamArgs A) {
    uint32_t const r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t const lane = threadIdx.x & 31;
    if (r >= A.n_reads) return;
    SamReadRec const R = A.reads[r];
    uint64_t const seq_qual = uint64_t(R.l_seq ? R.l_seq : 1) + 1 + (R.l_qual ? R.l_qual : 1);
    if (R.n_al == 0) {                                                 // output.cpp:95-107: one unmapped record
        if (lane == 0) {
            A.recs[R.rec0] = SamRecord{1, r, ~0u, 4u, 0};
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
            A.recs[slot] = SamRecord{chars, r, R.al0 + k, flag, 0};
            A.rec_off[slot] = size;
        }
    });
}

__global__ void sam_write_kernel(SamArgs A, uint32_t n_rec) {
    uint32_t const i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t const lane = threadIdx.x & 31;
    if (i >= n_rec) return;
    SamRecord const rec = A.recs[i];
    SamReadRec const R = A.reads[rec.read];
    char* p = A.text + A.body + A.rec_off[i];
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
