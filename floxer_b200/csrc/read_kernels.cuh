// read_kernels.cuh -- device FASTQ parsing (fxg_parse_fastq, fxg_map_fastq) for sm_100a.
//
// A call's text holds whole FASTQ records of four lines each: '@' and a header, the sequence, '+' and anything, the
// quality.  Lines end at '\n', one '\r' before the end of a line is dropped, and the last line may lack its '\n'.  The
// text is uploaded once and the device does the rest:
//   lines     cub::DeviceSelect::If over the byte positions keeps those of '\n' (FastqNewline); line j ends at the j-th
//             of them, or at the end of the text;
//   records   fastq_record_kernel: one thread per whole record -- its four lines, the checks ('@' starts the header,
//             '+' the third line), the id, the sequence and quality spans, the error budget k and the status
//             (fastq_read_status); the first malformed record's index is kept by an atomic minimum;
//   layout    an exclusive scan of the kept reads' lengths (cub) gives each kept read its pool offset;
//   ranks     fastq_ranks_kernel: one warp per record, lanes striding over the sequence -- the forward ranks at the offset,
//             the reverse complement at pool_len + offset + (m - 1 - i), the two pools back to back as a verification
//             job's Pool holds them.
// The id is the header after '@' up to the first space or tab.  The reference's reader cannot be read here, so this cut
// is the project's own choice; it is what most aligners write as QNAME.  Ranks follow input.cpp:165-176: '$' -> 0,
// A C G T in either case -> 1..4, every other byte -> 5; the complement swaps A<->T and C<->G and keeps '$' and N.
// k is query_errors when given, else floating_point_error_aware_ceil(m * error_probability) (math.hpp:22-27,
// input.cpp:26-34).  The PEX trees are built on the host from the lengths (pex_tree.cpp), which reads them there anyway.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/floxer_gpu.h"

namespace fxg {

// one record as fastq_record_kernel leaves it (48 bytes; copied back to the host whole)
struct FastqRec {
    uint64_t id, seq, qual;      // offsets of the id, the sequence and the quality in the text
    uint64_t errors;             // k
    uint32_t l_id, l_seq, l_qual;
    uint8_t status;              // FXG_READ_*
    uint8_t fault;               // kFastq*: why the record is malformed (0: it is not)
    uint16_t pad;
};
static_assert(sizeof(FastqRec) == 48, "FastqRec is copied back as 48-byte records");

enum : uint8_t { kFastqNoAt = 1, kFastqNoPlus = 2 };

struct FastqNewline {
    const char* text;
    __host__ __device__ __forceinline__ bool operator()(uint32_t i) const { return text[i] == '\n'; }
};

struct FastqArgs {
    const char* text; uint64_t text_len;
    const uint32_t* nl; uint64_t n_nl;            // positions of the newlines (a text is shorter than 2^31 bytes)
    uint64_t n_records;                           // whole records (four lines each)
    double error_probability; uint64_t query_errors, seed_errors;
};

__device__ __forceinline__ uint8_t fastq_rank(uint8_t c) {
    c = (c >= 'a' && c <= 'z') ? uint8_t(c - 32) : c;
    return c == '$' ? 0 : c == 'A' ? 1 : c == 'C' ? 2 : c == 'G' ? 3 : c == 'T' ? 4 : 5;
}

// input.cpp:106-129 in that order: a length outside 1..FXG_MAX_QUERY_LENGTH, then fewer errors than a leaf's budget
__host__ __device__ __forceinline__ uint8_t fastq_read_status(uint64_t m, uint64_t k, uint64_t seed_errors) {
    if (m == 0 || m > FXG_MAX_QUERY_LENGTH) return FXG_READ_BAD_LENGTH;
    return k < seed_errors ? uint8_t(FXG_READ_TOO_FEW_ERRORS) : uint8_t(FXG_READ_KEPT);
}

// line j as [begin, end) without its newline and one '\r' before it
__device__ __forceinline__ void fastq_line(FastqArgs const& A, uint64_t j, uint64_t& b, uint64_t& e) {
    b = j == 0 ? 0 : A.nl[j - 1] + 1;
    e = j < A.n_nl ? A.nl[j] : A.text_len;
    if (e > b && A.text[e - 1] == '\r') --e;
}

__global__ void fastq_record_kernel(FastqArgs A, FastqRec* recs, uint64_t* kept_len, unsigned long long* first_bad) {
    uint64_t const r = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (r >= A.n_records) return;
    uint64_t hb, he, sb, se, pb, pe, qb, qe;
    fastq_line(A, 4 * r, hb, he);
    fastq_line(A, 4 * r + 1, sb, se);
    fastq_line(A, 4 * r + 2, pb, pe);
    fastq_line(A, 4 * r + 3, qb, qe);
    FastqRec R{};
    R.fault = he == hb || A.text[hb] != '@' ? kFastqNoAt : pe == pb || A.text[pb] != '+' ? kFastqNoPlus : 0;
    uint64_t ie = hb + 1;
    if (!R.fault) while (ie < he && A.text[ie] != ' ' && A.text[ie] != '\t') ++ie;
    R.id = hb + 1; R.l_id = R.fault ? 0u : uint32_t(ie - hb - 1);
    R.seq = sb; R.l_seq = uint32_t(min(se - sb, uint64_t(UINT32_MAX)));
    R.qual = qb; R.l_qual = uint32_t(min(qe - qb, uint64_t(UINT32_MAX)));
    uint64_t const m = se - sb;
    // floating_point_error_aware_ceil(m * p): the rounding steps spelled out, so that no contraction changes the result
    R.errors = A.query_errors != FXG_NULL_ID ? A.query_errors
                                             : uint64_t(ceil(__dadd_rn(__dmul_rn(double(m), A.error_probability), -0.000000001)));
    R.status = fastq_read_status(m, R.errors, A.seed_errors);
    recs[r] = R;
    kept_len[r] = !R.fault && R.status == FXG_READ_KEPT ? m : 0;
    if (R.fault) atomicMin(first_bad, (unsigned long long)r);
}

// kept_off: the exclusive scan of kept_len (n_records + 1 entries; the last is the pool's length)
__global__ void fastq_ranks_kernel(FastqArgs A, const FastqRec* recs, const uint64_t* kept_off, uint8_t* pool) {
    uint64_t const r = (uint64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    uint32_t const lane = threadIdx.x & 31;
    if (r >= A.n_records) return;
    uint64_t const off = kept_off[r], m = kept_off[r + 1] - off;
    if (m == 0) return;
    uint64_t const pool_len = kept_off[A.n_records];
    const uint8_t* const s = reinterpret_cast<const uint8_t*>(A.text) + recs[r].seq;
    uint8_t* const fwd = pool + off;
    uint8_t* const rc = pool + pool_len + off + m - 1;
    for (uint64_t i = lane; i < m; i += 32) {
        uint8_t const x = fastq_rank(s[i]);
        fwd[i] = x;
        rc[-int64_t(i)] = x >= 1 && x <= 4 ? uint8_t(5 - x) : x;
    }
}

}  // namespace fxg
