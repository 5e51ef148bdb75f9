"""fxg_parse_fastq against the Python model of tests/test_map_cli.py, field for field, and fxg_map_fastq against the calls
it composes (host parsing -> seed_verify_reads -> Job.sam / Job.bam), plus `python -m floxer_b200.map` against one
map_fastq call.  Needs a B200: run with -m gpu."""
import gzip
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

from floxer_b200 import abi, synthetic
from floxer_b200.batch import ReadBatch, ReadConfig, VerifyConfig
from test_bam_output import bgzf_blocks
from test_map_cli import parse_model

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LETTERS = np.frombuffer(b"$ACGTN", dtype=np.uint8)
REF_IDS = ["chrA", "chrB"]


@pytest.fixture(scope="module")
def gpu():
    from floxer_b200 import build, gpu as g
    build.build_native()
    g.lib()
    return g


@pytest.fixture(scope="module")
def ctx(gpu):
    c = gpu.Context(0)
    yield c
    c.close()


# ---------------------------------------------------------------------------------------------------- parsing

def awkward_fastq(seed: int) -> bytes:
    """Random records with lowercase, '$', N and IUPAC bytes, '\\r\\n' line ends, ids with spaces and tabs, '+id' third
    lines, an empty sequence, a read over 100 kbp and short reads whose k falls below the seed errors."""
    rng = np.random.default_rng(seed)
    alphabet = np.frombuffer(b"ACGTACGTACGTacgtN$nRYKMSWbdhv", dtype=np.uint8)
    lengths = [int(x) for x in rng.integers(1, 3000, size=60)] + [0, 120_000, 100_000, 5, 12, 19, 1]
    rng.shuffle(lengths)
    out = []
    for i, m in enumerate(lengths):
        nl = b"\r\n" if rng.random() < 0.3 else b"\n"
        sep = [b" ", b"\t", b""][int(rng.integers(0, 3))]
        head = b"@rd%d%s%s" % (i, sep, b"extra words\there" if sep else b"")
        plus = b"+" + (head[1:] if rng.random() < 0.4 else b"")
        seq = bytes(rng.choice(alphabet, size=m))
        qual = bytes(rng.integers(33, 75, size=m if rng.random() < 0.9 else max(m - 3, 0)).astype(np.uint8))
        out.append(head + nl + seq + nl + plus + nl + qual + nl)
    return b"".join(out)[:-1]                                      # the last record without its final newline


READ_CONFIGS = [ReadConfig(query_errors=3, seed_errors=1), ReadConfig(error_probability=0.05, seed_errors=2),
                ReadConfig(error_probability=0.08, seed_errors=1, bottom_up=True), ReadConfig(query_errors=6, seed_errors=2, bottom_up=True)]


@pytest.mark.parametrize("rc", READ_CONFIGS)
def test_parse_equals_the_model(ctx, oracle, rc):
    text = awkward_fastq(11)
    want = parse_model(text, rc, oracle.pex_build)
    got = ctx.parse_fastq(text, rc)
    assert got.statuses.tolist() == want["statuses"].tolist()
    assert set(want["statuses"].tolist()) >= {abi.READ_KEPT, abi.READ_BAD_LENGTH} and len(got.statuses) == 67
    assert got.batch.reads.tobytes() == want["reads"].tobytes()
    assert got.spans.tobytes() == want["spans"].tobytes()
    assert np.array_equal(got.batch.forward_pool, want["forward"])
    assert np.array_equal(got.batch.reverse_pool, want["reverse"])
    assert got.batch.nodes.tobytes() == want["nodes"].tobytes()
    assert got.ids == want["ids"] and got.qualities == want["qualities"]


def test_too_few_errors_are_skipped(ctx, oracle):
    text = awkward_fastq(12)
    rc = ReadConfig(error_probability=0.05, seed_errors=2)
    got = ctx.parse_fastq(text, rc)
    assert abi.READ_TOO_FEW_ERRORS in got.statuses.tolist()
    assert got.statuses.tolist() == parse_model(text, rc, oracle.pex_build)["statuses"].tolist()


@pytest.mark.parametrize("text,bad", [
    (b"@a\nACGT\n+\nIIII\n@b\nACGT\n+\nIIII\nc\nACGT\n+\nIIII\n", 2),      # a header without '@'
    (b"@a\nACGT\n+\nIIII\n@b\nACGT\n-\nIIII\n", 1),                        # a third line without '+'
    (b"@a\nACGT\n+\nIIII\n@b\nACGT\n+\nIIII\n@c\nACGT\n", 2),              # cut short
])
def test_malformed_texts_are_refused(ctx, gpu, text, bad):
    with pytest.raises(gpu.FloxerGpuError) as e:
        ctx.parse_fastq(text, ReadConfig(query_errors=2, seed_errors=0))
    assert e.value.code == abi.ERR_INVALID_ARGUMENT
    assert f"record {bad}" in str(e.value)


# ---------------------------------------------------------------------------------------------------- mapping

def fastq_of(reads, rng, names=None) -> bytes:
    out = []
    for i, r in enumerate(reads):
        seq = bytes(LETTERS[r])
        qual = bytes(rng.integers(33, 75, size=len(r)).astype(np.uint8))
        out.append(b"@%s sample=%d\n%s\n+\n%s\n" % ((names[i] if names else b"read%d" % i), i, seq, qual))
    return b"".join(out)


def simulated_reads(refs, n, base_len, rate, seed):
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        rid = int(rng.integers(0, len(refs)))
        start = int(rng.integers(0, len(refs[rid]) - base_len - 1))
        seq, _, _ = synthetic.simulate_read(rng, refs[rid], start, base_len, int(rate * base_len))
        out.append(synthetic.reverse_complement(seq) if i % 2 else seq)
    return out


@pytest.fixture(scope="module")
def dataset(ctx, gpu):
    """Config-2 shape: a 2 Mbp reference (and a second, shorter one), 240 reads of 5 kbp at 5 % with qualities, and among
    them reads that are skipped (k below the seed errors, empty) or that the q-gram seeder refuses (25 bases)."""
    refs = [synthetic.random_reference(2_000_000, 20240001), synthetic.random_reference(300_000, 20240011)]
    ctx.set_references(refs)
    seeder = gpu.GpuSeeder(ctx, 10)
    rng = np.random.default_rng(5)
    reads = simulated_reads(refs, 240, 5000, 0.05, 7)
    for at, r in ((17, refs[0][1000:1020]), (60, refs[0][5000:5025]), (61, refs[1][7000:7025]), (130, np.zeros(0, np.uint8)),
                  (200, refs[1][100:116])):
        reads.insert(at, r)
    text = fastq_of(reads, rng)
    yield refs, seeder, text
    seeder.close()


def composed(ctx, oracle, seeder, text, rc, vc, refs, fmt, header=True):
    """host parsing -> seed_verify_reads -> Job.sam / Job.bam, and the job's alignments"""
    P = parse_model(text, rc, oracle.pex_build, q=seeder.q)
    batch = ReadBatch(P["reads"], P["forward"], P["reverse"], P["nodes"], np.zeros(0, dtype=abi.ANCHOR_DTYPE))
    job, seeded, st = ctx.seed_verify_reads(seeder, batch, vc)
    lens = [len(r) for r in refs]
    try:
        args = (seeded, REF_IDS, lens, P["ids"], P["qualities"], header)
        if fmt == "sam":
            out = job.sam(*args).encode()
        elif fmt == "sam.gz":
            out = job.sam(*args, on_device=True, bgzf=True)
        else:
            out = job.bam(*args)
        return out, P, len(job.alignments()[0]), st
    finally:
        job.free()


def assert_same_output(fmt, got: bytes, want: bytes):
    if fmt == "sam":
        assert got == want
    else:
        assert bgzf_blocks(got) == bgzf_blocks(want)                  # the same stream cut into the same blocks


MAP_CONFIGS = [VerifyConfig(verification_kind=kind, interval_optimization=iv)
               for kind in (abi.KIND_HIERARCHICAL, abi.KIND_DIRECT_FULL) for iv in (False, True)]


@pytest.mark.parametrize("vc", MAP_CONFIGS, ids=lambda v: f"kind{v.verification_kind}-iv{int(v.interval_optimization)}")
def test_map_equals_composition(ctx, oracle, dataset, vc):
    refs, seeder, text = dataset
    rc = ReadConfig(error_probability=0.05, seed_errors=2)
    lens = [len(r) for r in refs]
    for fmt in ("sam", "bam", "sam.gz"):
        for header in (True, False):
            got, summary = ctx.map_fastq(seeder, text, rc, vc, REF_IDS, lens, fmt=fmt, header=header)
            want, P, n_al, st = composed(ctx, oracle, seeder, text, rc, vc, refs, fmt, header)
            assert_same_output(fmt, got, want)
            statuses = P["statuses"].tolist()
            assert summary["records"] == 245 and summary["alignments"] == n_al > 0
            assert (summary["kept"], summary["too_few_errors"], summary["bad_length"], summary["unseedable"]) == tuple(
                statuses.count(s) for s in (abi.READ_KEPT, abi.READ_TOO_FEW_ERRORS, abi.READ_BAD_LENGTH, abi.READ_UNSEEDABLE))
            assert summary["unseedable"] == 2 and summary["too_few_errors"] == 2 and summary["bad_length"] == 1
            assert summary["seed"] == st


def test_bam_name_limit_is_refused(ctx, gpu, dataset):
    refs, seeder, _ = dataset
    rng = np.random.default_rng(3)
    text = fastq_of(simulated_reads(refs, 3, 2000, 0.05, 9), rng, names=[b"a", b"n" * 255, b"c"])
    lens = [len(r) for r in refs]
    rc = ReadConfig(error_probability=0.05, seed_errors=2)
    with pytest.raises(gpu.FloxerGpuError) as e:
        ctx.map_fastq(seeder, text, rc, VerifyConfig(), REF_IDS, lens, fmt="bam")
    assert e.value.code == abi.ERR_INVALID_ARGUMENT
    sam, _ = ctx.map_fastq(seeder, text, rc, VerifyConfig(), REF_IDS, lens, fmt="sam")
    assert b"n" * 255 + b"\t" in sam


def test_empty_text(ctx, dataset):
    refs, seeder, _ = dataset
    lens = [len(r) for r in refs]
    rc = ReadConfig(error_probability=0.05, seed_errors=2)
    sam, summary = ctx.map_fastq(seeder, b"", rc, VerifyConfig(), REF_IDS, lens, fmt="sam")
    assert sam.startswith(b"@HD") and sam.count(b"\n") == 3 and summary["records"] == 0
    bam, _ = ctx.map_fastq(seeder, b"", rc, VerifyConfig(), REF_IDS, lens, fmt="bam", header=False)
    assert bgzf_blocks(bam) == [b""]


def test_threads_give_the_same_bytes(ctx, dataset):
    refs, seeder, text = dataset
    lens = [len(r) for r in refs]
    rc = ReadConfig(error_probability=0.05, seed_errors=2)
    # four texts of whole records
    lines = text.split(b"\n")[:-1]
    cut = [b"\n".join(lines[4 * a:4 * b]) + b"\n" for a, b in ((0, 60), (60, 125), (125, 190), (190, 245))]
    jobs = [(t, fmt) for t in cut for fmt in ("sam", "bam")]
    alone = [ctx.map_fastq(seeder, t, rc, VerifyConfig(), REF_IDS, lens, fmt=fmt)[0] for t, fmt in jobs]
    together, errors = [None] * len(jobs), []

    def run(i):
        try:
            together[i] = ctx.map_fastq(seeder, jobs[i][0], rc, VerifyConfig(), REF_IDS, lens, fmt=jobs[i][1])[0]
        except Exception as e:                                     # noqa: BLE001
            errors.append(e)
    threads = [threading.Thread(target=run, args=(i,)) for i in range(len(jobs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors
    for (_, fmt), a, b in zip(jobs, alone, together):
        assert_same_output(fmt, b, a)


def test_uploads_are_counted_and_not_repeated(ctx, oracle, dataset):
    refs, seeder, text = dataset
    lens = [len(r) for r in refs]
    rc, vc = ReadConfig(error_probability=0.05, seed_errors=2), VerifyConfig()
    ctx.reset_counters()
    out, summary = ctx.map_fastq(seeder, text, rc, vc, REF_IDS, lens, fmt="bam")
    h2d_map = ctx.counters()["h2d_bytes"]
    ctx.reset_counters()
    want, P, n_al, _ = composed(ctx, oracle, seeder, text, rc, vc, refs, "bam")
    batch = ReadBatch(P["reads"], P["forward"], P["reverse"], P["nodes"], np.zeros(0, dtype=abi.ANCHOR_DTYPE))
    job, seeded, _ = ctx.seed_verify_reads(seeder, batch, vc)
    al, cg = job.alignments()
    ctx.reset_counters()
    job.bam(seeded, REF_IDS, lens, P["ids"], P["qualities"], on_device=True)
    h2d_writer = ctx.counters()["h2d_bytes"]
    ctx.reset_counters()
    job.free()
    job, _, _ = ctx.seed_verify_reads(seeder, batch, vc)
    h2d_seed_verify = ctx.counters()["h2d_bytes"]
    job.free()
    n_reads, pool = len(P["reads"]), len(P["forward"])
    names = sum(len(x) + 1 for x in P["ids"])
    quals = sum(len(x) for x in P["qualities"])
    cigar_bytes = 4 * int(cg.size)
    # the text, per-read records, the nodes, the writer's alignments and CIGARs and a small constant -- a second upload of
    # the pools (2 x pool bytes), of SEQ (pool bytes) or of the qualities (pool bytes) does not fit
    bound = len(text) + 512 * n_reads + 32 * len(P["nodes"]) + 40 * len(al) + cigar_bytes + 65536
    detail = f"map {h2d_map}, bound {bound}, text {len(text)}, pool {pool}, seed+verify {h2d_seed_verify}, writer {h2d_writer}"
    assert h2d_map < bound, detail
    assert bound - (len(text) + h2d_seed_verify - 2 * pool + h2d_writer - pool - names - quals) < quals, detail
    # and what the composition uploads, less the pools, SEQ, names and qualities, plus the text (the writer's upload has
    # three empty segments fewer, so up to 3 x 255 bytes less padding)
    assert h2d_map <= h2d_seed_verify - 2 * pool + h2d_writer - pool - names - quals + len(text) + 1024, detail


# ---------------------------------------------------------------------------------------------------- the command line

@pytest.mark.parametrize("suffix", ["bam", "sam", "sam.gz"])
def test_command_line_equals_one_call(ctx, dataset, tmp_path, suffix):
    refs, seeder, _ = dataset
    rng = np.random.default_rng(21)
    reads = simulated_reads(refs, 70, 2000, 0.05, 23)
    reads.insert(30, refs[0][500:520])                              # skipped: k < seed errors
    text = fastq_of(reads, rng)
    fa = tmp_path / "ref.fa"
    with open(fa, "wb") as f:
        for name, r in zip(REF_IDS, refs):
            seq = bytes(LETTERS[r])
            f.write(b">%s description\n" % name.encode())
            for i in range(0, len(seq), 80):
                f.write(seq[i:i + 80] + b"\n")
    fq = tmp_path / "reads.fq"
    fq.write_bytes(text)
    out = tmp_path / f"out.{suffix}"
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-m", "floxer_b200.map", "--reference", str(fa), "--queries", str(fq), "--output", str(out),
                        "--error-probability", "0.05", "--batch-reads", "16"], cwd=ROOT, env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "records=71 kept=70 too_few_errors=1 bad_length=0 unseedable=0" in r.stdout
    want, _ = ctx.map_fastq(seeder, text, ReadConfig(error_probability=0.05, seed_errors=2), VerifyConfig(), REF_IDS,
                            [len(x) for x in refs], fmt=suffix)
    got = out.read_bytes()
    if suffix == "sam":
        assert got == want
    else:
        assert gzip.decompress(got) == gzip.decompress(want)
        assert got.endswith(want[-28:]) and got.count(want[-28:]) == 1
