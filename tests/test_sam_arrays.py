"""fxg_write_sam, the array form of the SAM writer, on the CPU: it is host-only code.  The records of random cases are
compared with the CPU restatement of src/lib/output.cpp:49-108 (oracle/sam_oracle.py); the corner cases of the text
(null and empty ids and qualities, a quality longer than the read, an empty read, ranks of 6 and more, unknown CIGAR
operations, a CIGAR of 70 001 operations, a 64-bit reference length, POS at and above 2^31) are pinned byte for byte;
every refusal is checked with its code.  tests/test_sam_device.py runs the same cases through fxg_write_sam_device."""
import ctypes as C

import numpy as np
import pytest

from floxer_b200 import abi
from floxer_b200.batch import ReadBatch
from oracle import oracle as o
from oracle import sam_oracle
from test_bam_output import random_case

REF_IDS = ["chr1", "second reference", "r3"]
REF_LENS = [1 << 21, 2**32 + 5, 77]
HD = "@HD\tVN:1.6\tSO:unknown\tGO:none\n"

INVALID_ARGUMENT, STATE = -1, -5


@pytest.fixture(scope="module")
def gpu():
    from floxer_b200 import build, gpu as g
    build.build_native()
    g.lib()
    return g


def batch_of(seqs):
    """A batch of the given forward reads (rank arrays, empty ones allowed); only its reads and forward pool are read."""
    reads = np.zeros(len(seqs), dtype=abi.READ_DTYPE)
    at = 0
    for i, s in enumerate(seqs):
        reads[i]["query_offset"], reads[i]["query_len"] = at, len(s)
        at += len(s)
    pool = np.concatenate([np.asarray(s, dtype=np.uint8) for s in seqs]) if seqs else np.zeros(0, np.uint8)
    return ReadBatch(reads, pool, np.zeros_like(pool), np.zeros(0, dtype=abi.PEX_NODE_DTYPE), np.zeros(0, dtype=abi.ANCHOR_DTYPE))


def alignments(*rows):
    """rows: (read_index, reference_id, start, num_errors, orientation, cigar_offset, cigar_len)."""
    al = np.zeros(len(rows), dtype=abi.ALIGNMENT_DTYPE)
    for i, (ri, ref, start, errors, orient, off, n) in enumerate(rows):
        al[i]["read_index"], al[i]["reference_id"], al[i]["start_in_reference"] = ri, ref, start
        al[i]["num_errors"], al[i]["orientation"], al[i]["cigar_offset"], al[i]["cigar_len"] = errors, orient, off, n
    return al


def c_arguments(gpu, al, cigars, batch, ref_ids, ref_lens, ids, quals):
    """The ctypes arguments of fxg_write_sam up to with_header, and what keeps them alive.  ids / quals entries may be
    None: a null pointer."""
    al = np.ascontiguousarray(al, dtype=abi.ALIGNMENT_DTYPE)
    cg = np.ascontiguousarray(cigars, dtype=np.uint32)
    n_ref, n = len(ref_ids), len(batch.reads)
    rids = (C.c_char_p * max(n_ref, 1))(*[r.encode() for r in ref_ids])
    rlens = (C.c_uint64 * max(n_ref, 1))(*[int(x) for x in ref_lens])
    qs = (gpu._SamQuery * max(n, 1))()
    for i in range(n):
        qs[i].id = None if ids[i] is None else ids[i].encode()
        qs[i].quality = None if quals[i] is None else quals[i].encode()
    args = [al.ctypes.data if len(al) else None, len(al), cg.ctypes.data if len(cg) else None, n_ref, rids, rlens,
            batch.reads.ctypes.data, n, batch.forward_pool.ctypes.data, qs]
    return args, (al, cg, rids, rlens, qs, batch)


def host_sam(gpu, args, header=True):
    """(return code, bytes) of fxg_write_sam."""
    L = gpu.lib()
    out, length = C.c_void_p(), C.c_size_t(0)
    rc = L.fxg_write_sam(*args, int(header), C.byref(out), C.byref(length))
    if rc != 0:
        return rc, None
    try:
        return rc, C.string_at(out, length.value)
    finally:
        L.fxg_free(out)


def long_cigar(m=70_001):
    return np.array([(1 << 4) | (7 if i % 2 == 0 else 8) for i in range(m)], dtype=np.uint32)


def corner_cases():
    """name -> (alignments, cigar pool, batch, reference ids, reference lengths, ids, qualities, with_header, the text)."""
    acgt = [1, 2, 3, 4]
    eq4 = np.array([(4 << 4) | 7], dtype=np.uint32)
    rec = "\t0\tchr\t11\t255\t4=\t*\t0\t0\t"
    cases = {
        "header_full_64_bit_length": (alignments(), [], batch_of([]), ["chr", "big one"], [10, 2**32 + 5], [], [], True,
                                      HD + "@SQ\tSN:chr\tLN:10\n@SQ\tSN:big one\tLN:4294967301\n"),
        "null_id": (alignments(), [], batch_of([acgt]), [], [], [None], ["IIII"], False, "*\t4\t*\t0\t255\t*\t*\t0\t0\tACGT\tIIII\n"),
        "null_and_empty_quality": (alignments((0, 0, 10, 0, 0, 0, 1)), eq4, batch_of([acgt, acgt]), ["chr"], [100], ["a", "b"],
                                   [None, ""], False,
                                   "a" + rec + "ACGT\t*\tNM:i:0\n" + "b\t4\t*\t0\t255\t*\t*\t0\t0\tACGT\t*\n"),
        "quality_longer_than_the_read": (alignments((0, 0, 10, 0, 0, 0, 1), (0, 0, 20, 1, 0, 0, 1)), eq4, batch_of([acgt]), ["chr"],
                                         [100], ["q"], ["ABCDEFGHIJ"], False,
                                         "q" + rec + "ACGT\tABCDEFGHIJ\tNM:i:0\n" + "q\t256\tchr\t21\t255\t4=\t*\t0\t0\t*\t*\tNM:i:1\n"),
        "empty_read": (alignments((1, 0, 0, 0, 1, 0, 0)), [], batch_of([[], []]), ["chr"], [100], ["e", "f"], ["", "!"], False,
                       "e\t4\t*\t0\t255\t*\t*\t0\t0\t*\t*\n" + "f\t16\tchr\t1\t255\t*\t*\t0\t0\t*\t!\tNM:i:0\n"),
        "ranks_of_six_and_more": (alignments(), [], batch_of([[0, 1, 2, 3, 4, 5, 6, 7, 200, 255]]), [], [], ["r"], [""], False,
                                  "r\t4\t*\t0\t255\t*\t*\t0\t0\t$ACGTNNNNN\t*\n"),
        "unknown_op_codes": (alignments((0, 0, 5, 3, 0, 0, 6)),
                             np.array([(3 << 4) | 0, (1 << 4) | 3, (12 << 4) | 4, (2 << 4) | 15, (7 << 4) | 1, (1 << 4) | 2], np.uint32),
                             batch_of([acgt]), ["chr"], [100], ["u"], [""], False,
                             "u\t0\tchr\t6\t255\t3?1?12?2?7I1D\t*\t0\t0\tACGT\t*\tNM:i:3\n"),
        "cigar_of_70001_operations": (alignments((0, 0, 1234, 70_000, 1, 0, 70_001)), long_cigar(), batch_of([acgt]), ["chr"], [1 << 20],
                                      ["long"], [""], False,
                                      "long\t16\tchr\t1235\t255\t" + "1=1X" * 35_000 + "1=\t*\t0\t0\tACGT\t*\tNM:i:70000\n"),
        "pos_at_and_above_2_to_the_31": (alignments((0, 1, 2**31 - 1, 2, 0, 0, 1), (0, 0, 2**33, 2, 0, 0, 1), (0, 0, 2**31 - 2, 2, 1, 0, 1)),
                                         eq4, batch_of([acgt]), ["a", "b"], [1, 2], ["p"], ["IIII"], False,
                                         "p\t0\ta\t2147483648\t255\t4=\t*\t0\t0\tACGT\tIIII\tNM:i:2\n"
                                         "p\t272\ta\t2147483647\t255\t4=\t*\t0\t0\t*\t*\tNM:i:2\n"
                                         "p\t256\tb\t2147483648\t255\t4=\t*\t0\t0\t*\t*\tNM:i:2\n"),
        "primary_in_reference_order": (alignments((0, 2, 0, 1, 0, 0, 1), (0, 0, 1, 3, 0, 0, 1), (0, 0, 2, 1, 1, 0, 1), (0, 1, 3, 1, 0, 0, 1)),
                                       eq4, batch_of([acgt]), ["x", "y", "z"], [9, 9, 9], ["o"], ["JJJJ"], False,
                                       "o\t256\tx\t2\t255\t4=\t*\t0\t0\t*\t*\tNM:i:3\n"
                                       "o\t16\tx\t3\t255\t4=\t*\t0\t0\tACGT\tJJJJ\tNM:i:1\n"
                                       "o\t256\ty\t4\t255\t4=\t*\t0\t0\t*\t*\tNM:i:1\n"
                                       "o\t256\tz\t1\t255\t4=\t*\t0\t0\t*\t*\tNM:i:1\n"),
    }
    return cases


def refusal_cases():
    """name -> (alignments, cigar pool, batch, reference ids, reference lengths, ids, qualities, the code)."""
    acgt = [1, 2, 3, 4]
    eq4 = np.array([(4 << 4) | 7], dtype=np.uint32)
    two = batch_of([acgt, acgt])
    return {
        "not_grouped_by_read": (alignments((1, 0, 0, 0, 0, 0, 1), (0, 0, 0, 0, 0, 0, 1)), eq4, two, ["c"], [9], ["a", "b"], ["", ""], STATE),
        "read_index_past_the_reads": (alignments((0, 0, 0, 0, 0, 0, 1), (5, 0, 0, 0, 0, 0, 1)), eq4, two, ["c"], [9], ["a", "b"], ["", ""], STATE),
        "reference_id_out_of_range": (alignments((0, 1, 0, 0, 0, 0, 1)), eq4, two, ["c"], [9], ["a", "b"], ["", ""], INVALID_ARGUMENT),
        "cigar_without_a_pool": (alignments((0, 0, 0, 0, 0, 0, 1)), [], two, ["c"], [9], ["a", "b"], ["", ""], INVALID_ARGUMENT),
        # the walk meets read 0's bad reference id before the misplaced alignment behind read 1
        "first_problem_decides": (alignments((0, 3, 0, 0, 0, 0, 1), (1, 0, 0, 0, 0, 0, 1), (0, 0, 0, 0, 0, 0, 1)), eq4, two, ["c"], [9],
                                  ["a", "b"], ["", ""], INVALID_ARGUMENT),
        "grouping_before_a_later_bad_reference": (alignments((1, 0, 0, 0, 0, 0, 1), (0, 0, 0, 0, 0, 0, 1), (1, 7, 0, 0, 0, 0, 1)), eq4, two,
                                                  ["c"], [9], ["a", "b"], ["", ""], STATE),
    }


# ----------------------------------------------------------------------------- records against the restatement

@pytest.mark.parametrize("seed", [1, 2, 3, 5])
def test_records_match_the_restatement_of_output_cpp(gpu, seed):
    rng = np.random.default_rng(seed)
    batch, al, cg, per_read = random_case(rng, 60, 3)      # every rank including '$', starts above 2^31, NM above 65 535
    assert (al["start_in_reference"] >= 2**31).any() and (al["num_errors"] > 65_535).any()
    names = [f"read/{i}" for i in range(len(batch.reads))]
    quals = ["".join(chr(33 + int(x)) for x in rng.integers(0, 42, size=int(R["query_len"]))) if i % 3 else "" for i, R in enumerate(batch.reads)]
    want = []
    for ri, R in enumerate(batch.reads):
        qo, ql = int(R["query_offset"]), int(R["query_len"])
        want += sam_oracle.sam_records(names[ri], batch.forward_pool[qo:qo + ql], quals[ri],
                                       [(ref, start, errors, orient, o.cigar_to_string(ops)) for ref, start, errors, orient, ops in per_read[ri]],
                                       REF_IDS)
    for header in (True, False):
        text = gpu.write_sam(al, cg, batch, REF_IDS, REF_LENS, names, quals, header=header)
        head, records = sam_oracle.parse_sam(text)
        assert head == ([HD.strip()] + [f"@SQ\tSN:{n}\tLN:{l}" for n, l in zip(REF_IDS, REF_LENS)] if header else [])
        assert records == want
        assert text.endswith("\n")


def test_job_form_is_the_array_form(gpu):
    """fxg_job_write_sam feeds a job's arrays to fxg_write_sam: its text for the job's own arrays is the same.  (Without a
    GPU no job can be made, so the array form is checked against what a job's arrays look like: the cigar pool with gaps.)"""
    rng = np.random.default_rng(11)
    batch, al, cg, _ = random_case(rng, 30, 3)
    gapped = np.concatenate([np.full(7, 0xdead, np.uint32), cg])
    shifted = al.copy()
    shifted["cigar_offset"] += 7
    names = [f"g{i}" for i in range(len(batch.reads))]
    assert gpu.write_sam(shifted, gapped, batch, REF_IDS, REF_LENS, names) == gpu.write_sam(al, cg, batch, REF_IDS, REF_LENS, names)


# ----------------------------------------------------------------------------- exact bytes

@pytest.mark.parametrize("name", sorted(corner_cases()))
def test_corner_case_bytes(gpu, name):
    al, cg, batch, rids, rlens, ids, quals, header, want = corner_cases()[name]
    args, _keep = c_arguments(gpu, al, cg, batch, rids, rlens, ids, quals)
    rc, text = host_sam(gpu, args, header)
    assert rc == 0
    assert text == want.encode()


def test_no_reads_without_header_is_empty(gpu):
    args, _keep = c_arguments(gpu, alignments(), [], batch_of([]), ["a"], [1], [], [])
    assert host_sam(gpu, args, False) == (0, b"")


# ----------------------------------------------------------------------------- refusals and what SAM does not refuse

@pytest.mark.parametrize("name", sorted(refusal_cases()))
def test_refusals(gpu, name):
    al, cg, batch, rids, rlens, ids, quals, code = refusal_cases()[name]
    args, _keep = c_arguments(gpu, al, cg, batch, rids, rlens, ids, quals)
    assert host_sam(gpu, args)[0] == code


def test_null_arguments_are_refused(gpu):
    al, cg, batch, rids, rlens, ids, quals, _, _ = corner_cases()["null_and_empty_quality"]
    args, _keep = c_arguments(gpu, al, cg, batch, rids, rlens, ids, quals)
    for i in (0, 4, 5, 6, 8, 9):                             # alignments, reference ids / lengths, reads, forward pool, queries
        bad = list(args)
        bad[i] = None
        assert host_sam(gpu, bad)[0] == INVALID_ARGUMENT, i
    L = gpu.lib()
    length = C.c_size_t(0)
    assert L.fxg_write_sam(*args, 1, None, C.byref(length)) == INVALID_ARGUMENT
    out = C.c_void_p()
    assert L.fxg_write_sam(*args, 1, C.byref(out), None) == INVALID_ARGUMENT


def test_long_name_and_long_cigar_spanning_2_to_the_28_are_written(gpu):
    """BAM's limits (a 254-character name, a CG-tag CIGAR spanning 2^28 bases) do not exist in SAM."""
    ops = np.full(70_000, (4096 << 4) | 2, dtype=np.uint32)         # deletions: more than 2^28 reference bases
    al = alignments((0, 0, 0, 1, 0, 0, len(ops)))
    name = "n" * 300
    text = gpu.write_sam(al, ops, batch_of([[1, 2]]), ["chr"], [10], [name], header=False)
    assert text == name + "\t0\tchr\t1\t255\t" + "4096D" * 70_000 + "\t*\t0\t0\tAC\t*\tNM:i:1\n"


def test_job_sam_bgzf_needs_the_device(gpu):
    job = gpu.Job(None, None, None)                          # (refused before the job is touched)
    with pytest.raises(ValueError):
        job.sam(batch_of([]), [], [], [], bgzf=True)
