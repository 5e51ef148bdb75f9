"""The FASTQ rules of fxg_parse_fastq as a test-only Python model, checked on hand-written cases, and the host side of
`python -m floxer_b200.map`: its FASTA reader, its chunk cutter and its argument mapping.  Runs on the CPU;
tests/test_fastq_device.py checks the device parser against the model."""
import gzip
import io
import re

import numpy as np
import pytest

from floxer_b200 import abi
from floxer_b200 import map as fmap
from floxer_b200.batch import ReadConfig
from floxer_b200.synthetic import ceil_eps
from harness import revcomp, to_ranks


class Malformed(ValueError):
    def __init__(self, record: int):
        super().__init__(f"record {record}")
        self.record = record


def parse_model(text: bytes, config: ReadConfig, pex_build, q: int | None = None) -> dict:
    """fxg_parse_fastq's rules in Python: four lines per record, lines at '\\n' less one '\\r', the last newline optional;
    id = header after '@' up to the first space or tab; ranks of input.cpp:165-176; k = query_errors or
    ceil_eps(m * p); status BAD_LENGTH (m = 0 or m > 100 000), then TOO_FEW_ERRORS (k < seed_errors); with q, also
    UNSEEDABLE for a leaf with m / (e + 1) < q or e > 8.  Raises Malformed with the first bad record's index."""
    raw = text.split(b"\n")
    if text.endswith(b"\n") or not text:
        raw.pop()
    starts = np.cumsum([0] + [len(x) + 1 for x in raw])
    lines = [x[:-1] if x.endswith(b"\r") else x for x in raw]
    n_full = len(lines) // 4
    for r in range(n_full):
        if not lines[4 * r].startswith(b"@") or not lines[4 * r + 2].startswith(b"+"):
            raise Malformed(r)
    if len(lines) % 4:
        raise Malformed(n_full)
    out = {"statuses": [], "reads": [], "spans": [], "forward": [], "reverse": [], "nodes": [], "ids": [], "qualities": []}
    pool = node = 0
    for r in range(n_full):
        head, seq, qual = lines[4 * r], lines[4 * r + 1], lines[4 * r + 3]
        ident = re.split(rb"[ \t]", head[1:], maxsplit=1)[0]
        m = len(seq)
        k = config.query_errors if config.query_errors is not None else ceil_eps(m * config.error_probability)
        status = (abi.READ_BAD_LENGTH if m == 0 or m > abi_max_query_length() else
                  abi.READ_TOO_FEW_ERRORS if k < config.seed_errors else abi.READ_KEPT)
        inner = leaves = None
        if status == abi.READ_KEPT:
            inner, leaves = pex_build(m, k, config.seed_errors, int(config.bottom_up))
            if q is not None and any(int(lv["num_errors"]) > 8 or
                                     (int(lv["query_index_to"]) - int(lv["query_index_from"]) + 1) // (int(lv["num_errors"]) + 1) < q
                                     for lv in leaves):
                status = abi.READ_UNSEEDABLE
        out["statuses"].append(status)
        if status != abi.READ_KEPT:
            continue
        fwd = to_ranks(seq.decode("latin-1"))
        out["forward"].append(fwd)
        out["reverse"].append(revcomp(fwd))
        out["reads"].append((pool, node, 0, m, len(inner), len(leaves), 0, 0, 0))
        out["nodes"] += [np.asarray(inner, dtype=abi.PEX_NODE_DTYPE), np.asarray(leaves, dtype=abi.PEX_NODE_DTYPE)]
        out["spans"].append((r, int(starts[4 * r]) + 1, int(starts[4 * r + 3]), len(ident), len(qual)))
        out["ids"].append(ident.decode("latin-1"))
        out["qualities"].append(qual.decode("latin-1"))
        pool += m
        node += len(inner) + len(leaves)
    cat = lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dtype=dt)
    out["statuses"] = np.array(out["statuses"], dtype=np.uint8)
    out["reads"] = np.array(out["reads"], dtype=abi.READ_DTYPE)
    out["spans"] = np.array(out["spans"], dtype=abi.READ_SPAN_DTYPE)
    out["forward"], out["reverse"] = cat(out["forward"], np.uint8), cat(out["reverse"], np.uint8)
    out["nodes"] = cat(out["nodes"], abi.PEX_NODE_DTYPE)
    return out


def abi_max_query_length() -> int:
    return 100_000                                       # FXG_MAX_QUERY_LENGTH, include/input.hpp:42


@pytest.fixture(scope="module")
def pex(oracle):
    return oracle.pex_build


# ---------------------------------------------------------------------------------------------------- the model

def test_records_ids_and_spans(pex):
    text = b"@r1 first read\nACGT\n+\nIIII\n@r2\tsecond\r\nacgtn\r\n+r2\r\n!!!!!\r\n@\nGATTACA\n+\n#######"
    P = parse_model(text, ReadConfig(query_errors=2, seed_errors=0), pex)
    assert P["ids"] == ["r1", "r2", ""]
    assert P["qualities"] == ["IIII", "!!!!!", "#######"]
    assert list(P["statuses"]) == [abi.READ_KEPT] * 3
    sp = P["spans"]
    assert [text[o:o + n] for o, n in zip(sp["id_offset"], sp["id_len"])] == [b"r1", b"r2", b""]
    assert [text[o:o + n] for o, n in zip(sp["quality_offset"], sp["quality_len"])] == [b"IIII", b"!!!!!", b"#######"]
    assert list(sp["record"]) == [0, 1, 2]
    assert list(P["reads"]["query_offset"]) == [0, 4, 9] and list(P["reads"]["query_len"]) == [4, 5, 7]


def test_ranks_and_reverse_complement(pex):
    seq = b"$AaCcGgTtNnRYKMSWBDHVn.-*"
    P = parse_model(b"@x\n" + seq + b"\n+\n" + b"I" * len(seq) + b"\n", ReadConfig(query_errors=3, seed_errors=0), pex)
    want = [0, 1, 1, 2, 2, 3, 3, 4, 4] + [5] * (len(seq) - 9)
    assert list(P["forward"]) == want
    comp = {0: 0, 1: 4, 2: 3, 3: 2, 4: 1, 5: 5}
    assert list(P["reverse"]) == [comp[x] for x in reversed(want)]


def test_error_budget_and_skip_statuses(pex):
    def record(i, m):
        return b"@r%d\n" % i + b"A" * m + b"\n+\n" + b"I" * m + b"\n"
    lengths = [0, 20, 40, 100, 100_001, 100_000]
    text = b"".join(record(i, m) for i, m in enumerate(lengths))
    P = parse_model(text, ReadConfig(error_probability=0.05, seed_errors=2), pex)
    # k = ceil_eps(m * 0.05): 0, 1, 2, 5, -, 5000
    assert list(P["statuses"]) == [abi.READ_BAD_LENGTH, abi.READ_TOO_FEW_ERRORS, abi.READ_KEPT, abi.READ_KEPT,
                                   abi.READ_BAD_LENGTH, abi.READ_KEPT]
    assert ceil_eps(40 * 0.05) == 2 and ceil_eps(20 * 0.05) == 1
    P = parse_model(text, ReadConfig(query_errors=1, seed_errors=2), pex)
    assert list(P["statuses"]) == [abi.READ_BAD_LENGTH, *[abi.READ_TOO_FEW_ERRORS] * 3, abi.READ_BAD_LENGTH, abi.READ_TOO_FEW_ERRORS]


def test_trees_follow_the_build_strategy(pex):
    text = b"@a\n" + b"ACGT" * 500 + b"\n+\n" + b"I" * 2000 + b"\n"
    for bottom_up in (False, True):
        P = parse_model(text, ReadConfig(error_probability=0.05, seed_errors=2, bottom_up=bottom_up), pex)
        inner, leaves = pex(2000, 100, 2, int(bottom_up))
        R = P["reads"][0]
        assert (int(R["num_inner"]), int(R["num_leaves"])) == (len(inner), len(leaves))
        assert P["nodes"].tobytes() == np.concatenate([inner, leaves]).astype(abi.PEX_NODE_DTYPE).tobytes()


def test_unseedable_leaves(pex):
    text = b"@short\n" + b"A" * 25 + b"\n+\n" + b"I" * 25 + b"\n@long\n" + b"A" * 30 + b"\n+\n" + b"I" * 30 + b"\n"
    P = parse_model(text, ReadConfig(error_probability=0.05, seed_errors=2), pex, q=10)
    assert list(P["statuses"]) == [abi.READ_UNSEEDABLE, abi.READ_KEPT]          # 25 // 3 = 8 < 10; 30 // 3 = 10


@pytest.mark.parametrize("text,bad", [
    (b"@a\nAC\n+\nII\nb\nAC\n+\nII\n", 1),                   # the header lacks '@'
    (b"@a\nAC\n-\nII\n", 0),                                  # the third line lacks '+'
    (b"@a\nAC\n+\nII\n@b\nAC\n+\n", 1),                      # cut short
    (b"@a\nAC\n+\nII\n\n", 1),                               # an empty line after the last record
    (b"@a\nAC\n+\nII\n@b\nAC\n", 1),
])
def test_malformed_texts(pex, text, bad):
    with pytest.raises(Malformed) as e:
        parse_model(text, ReadConfig(query_errors=2, seed_errors=0), pex)
    assert e.value.record == bad


def test_empty_text_and_missing_final_newline(pex):
    assert len(parse_model(b"", ReadConfig(query_errors=2, seed_errors=0), pex)["statuses"]) == 0
    a = parse_model(b"@a\nAC\n+\nII\n", ReadConfig(query_errors=2, seed_errors=0), pex)
    b = parse_model(b"@a\nAC\n+\nII", ReadConfig(query_errors=2, seed_errors=0), pex)
    assert a["qualities"] == b["qualities"] == ["II"]


# ---------------------------------------------------------------------------------------------------- the command line

def test_fasta_reader(tmp_path):
    text = b">chr1 the first\nACGTN\nacgt$\r\n>chr2\tdesc\n\nGGG\n>empty\n"
    for name, data in (("ref.fa", text), ("ref.fa.gz", gzip.compress(text))):
        p = tmp_path / name
        p.write_bytes(data)
        refs = fmap.read_fasta(str(p))
        assert [r[0] for r in refs] == ["chr1", "chr2", "empty"]
        assert list(refs[0][1]) == [1, 2, 3, 4, 5, 1, 2, 3, 4, 0]
        assert list(refs[1][1]) == [3, 3, 3] and len(refs[2][1]) == 0


def fastq_text(n: int, rng) -> bytes:
    out = []
    for i in range(n):
        m = int(rng.integers(0, 30))
        seq = bytes(rng.choice(list(b"ACGT"), size=m).astype(np.uint8))
        qual = b"@" + bytes(rng.integers(33, 74, size=max(m - 1, 0)).astype(np.uint8)) if m else b""    # starts with '@'
        out.append(b"@read%d x\n%s\n+\n%s\n" % (i, seq, qual))
    return b"".join(out)


@pytest.mark.parametrize("batch,block", [(1, 3), (3, 7), (5, 1 << 20), (100, 64)])
def test_chunks_end_on_whole_records(batch, block):
    rng = np.random.default_rng(batch)
    text = fastq_text(23, rng)
    for t in (text, text[:-1]):                                    # with and without the final newline
        chunks = list(fmap.fastq_chunks(io.BytesIO(t), batch, block=block))
        assert b"".join(chunks) == t
        for c in chunks[:-1]:
            assert c.count(b"\n") == 4 * batch and c.endswith(b"\n")
        assert chunks[-1].count(b"\n") + (0 if t.endswith(b"\n") else 1) == 4 * (23 - batch * (len(chunks) - 1))
        for c in chunks:
            assert c.startswith(b"@read")


def test_output_formats():
    assert fmap.output_format("x.bam") == "bam"
    assert fmap.output_format("x.sam") == "sam"
    assert fmap.output_format("dir/x.sam.gz") == "sam.gz"
    with pytest.raises(ValueError):
        fmap.output_format("x.cram")


def test_argument_mapping():
    base = ["--reference", "r.fa", "--queries", "q.fq", "--output", "o.bam"]
    a = fmap.parser().parse_args(base + ["--error-probability", "0.08"])
    rc, vc, seeding = fmap.configs_from_args(a)
    assert (rc.error_probability, rc.query_errors, rc.seed_errors, rc.bottom_up) == (0.08, None, 2, False)
    assert (vc.verification_kind, vc.interval_optimization, vc.extra_verification_ratio, vc.without_cigar) == (abi.KIND_HIERARCHICAL, False, 0.05, False)
    assert seeding == {"max_anchors_hard": 500, "max_anchors_soft": 50}
    assert (a.q, a.device) == (10, 0)
    a = fmap.parser().parse_args(base + ["--query-errors", "7", "--seed-errors", "1", "--pex-tree-build-strategy", "bottom-up",
                                         "--max-anchors-hard", "90", "--max-anchors-soft", "9", "--extra-verification-ratio", "2",
                                         "--interval-optimization", "--direct-full-verification", "--without-cigar",
                                         "--device", "3", "--q", "12", "--batch-reads", "64"])
    rc, vc, seeding = fmap.configs_from_args(a)
    assert (rc.query_errors, rc.seed_errors, rc.bottom_up) == (7, 1, True)
    c = rc.to_c()
    assert (c.query_errors, c.seed_errors, c.build_strategy) == (7, 1, 1)
    assert (vc.verification_kind, vc.interval_optimization, vc.extra_verification_ratio, vc.without_cigar) == (abi.KIND_DIRECT_FULL, True, 2.0, True)
    assert seeding == {"max_anchors_hard": 90, "max_anchors_soft": 9}
    assert (a.device, a.q, a.batch_reads) == (3, 12, 64)
    assert fmap.configs_from_args(fmap.parser().parse_args(base + ["--error-probability", "0.1"]))[0].to_c().query_errors == abi.NULL_ID
    for bad in ([], ["--query-errors", "2", "--error-probability", "0.1"]):
        with pytest.raises(SystemExit):
            fmap.parser().parse_args(base + bad)
