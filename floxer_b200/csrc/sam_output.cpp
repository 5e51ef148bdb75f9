// sam_output.cpp -- SAM records for the alignments of a verified job (row N3 of SURVEY 8f).
//
// Restates output::alignment_output::write_alignments_for_query (src/lib/output.cpp:49-108 of the reference) and the
// header set up by internal::create_seqan_alignment_output (src/lib/output.cpp:197-212): per query, the alignments
// reference by reference in insertion order; the first one whose number of errors equals the query's best is the primary
// alignment (flag 0 / 16, SEQ and QUAL written), every other one is secondary (flag | 256, SEQ and QUAL '*'); MAPQ 255
// ("not available"), tag NM = number of errors, POS = start_in_reference + 1 saturated to int32; a query without any
// alignment gets one unmapped record (flag 4).  SEQ is the query as it was read (forward), also for alignments of the
// reverse complement -- that is what the reference writes.
//
// The bytes themselves are SeqAn3's business in the reference (seqan3::sam_file_output, not on disk here): field order
// and '*' conventions follow the SAM specification, the header line is the one SeqAn3 writes by default as recalled
// ("@HD VN:1.6 SO:unknown GO:none"); byte-level parity of the text is unpinned, the record contents are pinned by
// test/floxer_whole_program_via_cli_test.cpp:38-93 (tests/test_sam_output.py).
//
// Host-only code: the array entry point fxg_write_sam needs neither a context nor a GPU (tests/test_sam_arrays.py);
// fxg_write_sam_device (floxer_gpu.cu, sam_kernels.cuh) writes the same text on the device.
#include "../../include/floxer_gpu.h"

#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <vector>

namespace {

constexpr char kRankToChar[6] = {'$', 'A', 'C', 'G', 'T', 'N'};     // ivs::d_dna5 ranks as used by src/lib/input.cpp:165-176

void append_uint(std::string& s, uint64_t v) {
    char buf[24]; int n = 0;
    do { buf[n++] = char('0' + v % 10); v /= 10; } while (v);
    while (n) s.push_back(buf[--n]);
}

void append_cigar(std::string& s, const uint32_t* ops, uint32_t n) {
    if (n == 0) { s.push_back('*'); return; }
    for (uint32_t i = 0; i < n; ++i) {
        append_uint(s, ops[i] >> 4);
        switch (ops[i] & 15u) {
            case FXG_CIGAR_I: s.push_back('I'); break;
            case FXG_CIGAR_D: s.push_back('D'); break;
            case FXG_CIGAR_EQ: s.push_back('='); break;
            case FXG_CIGAR_X: s.push_back('X'); break;
            default: s.push_back('?'); break;
        }
    }
}

}  // namespace

extern "C" {

int fxg_write_sam(const fxg_alignment* al, size_t n_al, const uint32_t* ops, size_t n_references, const char* const* reference_ids,
                  const uint64_t* reference_lengths, const fxg_read* reads, size_t n_reads, const uint8_t* forward_pool,
                  const fxg_sam_query* queries, int with_header, char** text, size_t* text_len) {
    if (!text || !text_len || (n_al && !al) || (n_reads && (!reads || !forward_pool || !queries)) || (n_references && (!reference_ids || !reference_lengths)))
        return FXG_ERR_INVALID_ARGUMENT;
    *text = nullptr; *text_len = 0;
    try {
    std::string out;
    out.reserve(size_t(1) << 20);
    if (with_header) {
        out += "@HD\tVN:1.6\tSO:unknown\tGO:none\n";
        for (size_t r = 0; r < n_references; ++r) {
            out += "@SQ\tSN:"; out += reference_ids[r]; out += "\tLN:"; append_uint(out, reference_lengths[r]); out.push_back('\n');
        }
    }
    std::vector<uint32_t> order;
    std::string seq;
    size_t a = 0;
    for (size_t ri = 0; ri < n_reads; ++ri) {
        // the job lists a read's alignments in insertion order (forward package, then reverse complement)
        size_t const a0 = a;
        while (a < n_al && al[a].read_index == ri) ++a;
        if (a < n_al && al[a].read_index < ri) return FXG_ERR_STATE;                 // alignments must be grouped by read
        const char* const qname = queries[ri].id ? queries[ri].id : "*";
        const char* const qual = (queries[ri].quality && queries[ri].quality[0]) ? queries[ri].quality : "*";
        seq.resize(reads[ri].query_len);
        for (uint32_t p = 0; p < reads[ri].query_len; ++p) {
            uint8_t const rk = forward_pool[reads[ri].query_offset + p];
            seq[p] = rk < 6 ? kRankToChar[rk] : 'N';
        }
        if (seq.empty()) seq = "*";
        if (a == a0) {
            // output.cpp:95-107: unmapped
            out += qname; out += "\t4\t*\t0\t255\t*\t*\t0\t0\t"; out += seq; out.push_back('\t'); out += qual; out.push_back('\n');
            continue;
        }
        // query_alignments::to_reference: per reference, insertion order (alignment.cpp:37-79) -- a stable sort by reference
        order.resize(a - a0);
        for (size_t k = 0; k < a - a0; ++k) order[k] = uint32_t(a0 + k);
        std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return al[x].reference_id < al[y].reference_id; });
        uint32_t best = std::numeric_limits<uint32_t>::max();
        for (size_t k = a0; k < a; ++k) best = std::min(best, al[k].num_errors);
        bool primary_written = false;
        for (uint32_t k : order) {
            fxg_alignment const& A = al[k];
            if (A.reference_id >= n_references || (A.cigar_len && !ops)) return FXG_ERR_INVALID_ARGUMENT;
            uint32_t flag = A.orientation == FXG_REVERSE_COMPLEMENT ? 16u : 0u;
            bool const primary = !primary_written && A.num_errors == best;
            if (primary) primary_written = true; else flag |= 256u;
            uint64_t const pos0 = std::min<uint64_t>(A.start_in_reference, uint64_t(std::numeric_limits<int32_t>::max()));   // math.hpp:10-16
            out += qname; out.push_back('\t'); append_uint(out, flag); out.push_back('\t'); out += reference_ids[A.reference_id]; out.push_back('\t');
            append_uint(out, pos0 + 1); out += "\t255\t";
            append_cigar(out, A.cigar_len ? ops + A.cigar_offset : nullptr, A.cigar_len);
            out += "\t*\t0\t0\t";
            if (primary) { out += seq; out.push_back('\t'); out += qual; } else out += "*\t*";
            out += "\tNM:i:"; append_uint(out, A.num_errors); out.push_back('\n');
        }
    }
    if (a != n_al) return FXG_ERR_STATE;
    char* buf = static_cast<char*>(std::malloc(out.size() + 1));
    if (!buf) return FXG_ERR_OUT_OF_MEMORY;
    std::memcpy(buf, out.data(), out.size());
    buf[out.size()] = 0;
    *text = buf; *text_len = out.size();
    return FXG_OK;
    } catch (...) { return FXG_ERR_OUT_OF_MEMORY; }              // (std::bad_alloc / length_error of the text buffer: nothing crosses the C ABI)
}

int fxg_job_write_sam(const fxg_job* job, size_t n_references, const char* const* reference_ids, const uint64_t* reference_lengths,
                      const fxg_read* reads, size_t n_reads, const uint8_t* forward_pool, const fxg_sam_query* queries,
                      int with_header, char** text, size_t* text_len) {
    if (!job) return FXG_ERR_INVALID_ARGUMENT;
    return fxg_write_sam(fxg_job_alignments(job), fxg_job_num_alignments(job), fxg_job_cigar_pool(job), n_references, reference_ids,
                         reference_lengths, reads, n_reads, forward_pool, queries, with_header, text, text_len);
}

void fxg_free(void* p) { std::free(p); }

}  // extern "C"
