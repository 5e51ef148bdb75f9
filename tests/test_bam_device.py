"""fxg_write_bam_device (Context.write_bam, Job.bam(on_device=True)) against the host writer fxg_write_bam: the same BGZF
blocks -- count, ISIZE, CRC32, inflated payload --, the same end-of-file block and records, the same refusals; encoder
shapes (empty batches, exact multiples of 0xff00 bytes, runs, incompressible chunks, a CIGAR in the CG tag, many blocks);
a config-2 job whose image stays within 1.15x of zlib level 1; determinism and concurrent callers.  Needs a B200: run
with -m gpu."""
import struct
import threading
import zlib

import numpy as np
import pytest

from floxer_b200 import abi, synthetic
from floxer_b200.batch import BatchBuilder, ReadBatch, VerifyConfig
from test_bam_output import bgzf_blocks, parse_bam, random_case

pytestmark = pytest.mark.gpu

EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
REF_IDS = ["chr1", "second reference", "r3"]
REF_LENS = [1 << 21, 2**32 + 5, 77]


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


def raw_blocks(data: bytes):
    """The BGZF blocks of an image as they are, with their (ISIZE, CRC32) trailers."""
    out, at = [], 0
    while at < len(data):
        size = struct.unpack_from("<H", data, at + 16)[0] + 1
        block = data[at:at + size]
        crc, isize = struct.unpack_from("<II", block, size - 8)
        out.append((block, isize, crc))
        at += size
    assert at == len(data)
    return out


def assert_same_blocks(host: bytes, dev: bytes, with_header=True):
    hb, db = raw_blocks(host), raw_blocks(dev)
    assert len(db) == len(hb)
    assert [(i, c) for _, i, c in db] == [(i, c) for _, i, c in hb]
    assert bgzf_blocks(dev) == bgzf_blocks(host)                  # (gzip checks every block's CRC32 and ISIZE as well)
    assert db[-1][0] == hb[-1][0] == EOF_BLOCK
    for block, isize, _ in db:
        assert len(block) <= 65536 and len(block) <= isize + 5 + 26 or isize == 0
    assert parse_bam(dev, with_header) == parse_bam(host, with_header)


def both(ctx, gpu, *args, **kw):
    return gpu.write_bam(*args, **kw), ctx.write_bam(*args, **kw)


def qualities_for(rng, batch, every=3):
    return ["".join(chr(33 + int(x)) for x in rng.integers(0, 42, size=int(R["query_len"]))) if i % every else ""
            for i, R in enumerate(batch.reads)]


def unmapped_batch(seqs):
    bb = BatchBuilder()
    node = np.zeros(1, dtype=abi.PEX_NODE_DTYPE)
    node["parent_id"] = abi.NULL_ID
    for fwd in seqs:
        node["query_index_to"] = len(fwd) - 1
        bb.add(fwd, fwd[::-1].copy(), node[:0], node, np.zeros(0, dtype=abi.ANCHOR_DTYPE), np.zeros(0, dtype=abi.ANCHOR_DTYPE))
    return bb.build()


NO_ALIGNMENTS = np.zeros(0, dtype=abi.ALIGNMENT_DTYPE)
NO_CIGARS = np.zeros(0, dtype=np.uint32)


# ----------------------------------------------------------------------------- block-for-block equality

@pytest.mark.parametrize("seed", [1, 2, 3])
def test_blocks_equal_the_host_writers(ctx, gpu, seed):
    rng = np.random.default_rng(seed)
    batch, al, cg, _ = random_case(rng, 40, 3)
    names = [f"read/{i}" for i in range(len(batch.reads))]
    quals = qualities_for(rng, batch)
    for header in (True, False):
        host, dev = both(ctx, gpu, al, cg, batch, REF_IDS, REF_LENS, names, quals, header=header)
        assert_same_blocks(host, dev, header)


# ----------------------------------------------------------------------------- shapes that stress the encoder

def test_zero_reads_and_reads_without_alignments(ctx, gpu):
    rng = np.random.default_rng(4)
    batch, _, _, _ = random_case(rng, 30, 2)
    empty = ReadBatch(batch.reads[:0], batch.forward_pool, batch.reverse_pool, batch.nodes, batch.anchors, dict(batch.meta))
    for header in (True, False):
        host, dev = both(ctx, gpu, NO_ALIGNMENTS, NO_CIGARS, empty, ["a", "b"], [10, 20], [], header=header)
        assert_same_blocks(host, dev, header)
        names = [f"u{i}" for i in range(len(batch.reads))]
        host, dev = both(ctx, gpu, NO_ALIGNMENTS, NO_CIGARS, batch, ["a", "b"], [10, 20], names, qualities_for(rng, batch, 2), header=header)
        assert_same_blocks(host, dev, header)
    assert ctx.write_bam(NO_ALIGNMENTS, NO_CIGARS, empty, [], [], [], header=False) == EOF_BLOCK


def test_stream_of_exactly_two_chunks(ctx, gpu):
    # 128 unmapped records of 1020 bytes: 36 fixed + 84 name (83 characters and NUL) + 300 SEQ + 600 QUAL = 2 * 0xff00
    rng = np.random.default_rng(5)
    batch = unmapped_batch([rng.integers(1, 5, size=600, dtype=np.uint8) for _ in range(128)])
    names = [f"{i:03d}" + "n" * 80 for i in range(128)]
    host, dev = both(ctx, gpu, NO_ALIGNMENTS, NO_CIGARS, batch, [], [], names, qualities_for(rng, batch, 1), header=False)
    assert [isize for _, isize, _ in raw_blocks(host)] == [0xff00, 0xff00, 0]
    assert_same_blocks(host, dev, False)


def test_chunk_of_one_repeated_byte(ctx, gpu):
    # one unmapped 200 kbp read of A without qualities: SEQ is 0x11 * 100 000, QUAL 0xff * 200 000
    batch = unmapped_batch([np.ones(200_000, dtype=np.uint8)])
    host, dev = both(ctx, gpu, NO_ALIGNMENTS, NO_CIGARS, batch, [], [], ["run"], header=False)
    payloads = bgzf_blocks(dev)
    assert set(payloads[2]) == {0xff} and len(payloads[2]) == 0xff00
    assert_same_blocks(host, dev, False)
    assert len(dev) < 3000                                          # long matches, not literals


def test_chunks_of_random_bytes(ctx, gpu):
    # a CIGAR of 40 000 random words: 160 kB that do not compress (stored blocks, or payloads that still fit)
    rng = np.random.default_rng(6)
    batch = unmapped_batch([rng.integers(1, 5, size=100, dtype=np.uint8)])
    ops = rng.integers(0, 2**32, size=40_000, dtype=np.uint64).astype(np.uint32)
    al = np.array([(5, 0, len(ops), 3, 0, 0, 0, (0,) * 7)], dtype=abi.ALIGNMENT_DTYPE)
    host = gpu.write_bam(al, ops, batch, ["chr"], [1 << 20], ["noise"], header=False)
    dev = ctx.write_bam(al, ops, batch, ["chr"], [1 << 20], ["noise"], header=False)
    hb, db = raw_blocks(host), raw_blocks(dev)
    assert [(i, c) for _, i, c in db] == [(i, c) for _, i, c in hb] and len(db) >= 3
    assert bgzf_blocks(dev) == bgzf_blocks(host) and db[-1][0] == EOF_BLOCK
    for block, isize, _ in db[1:-2]:                                # the blocks that hold nothing but random words
        assert len(block) <= isize + 5 + 26


def test_cigar_with_more_than_65535_operations(ctx, gpu):
    m = 70_001
    batch = unmapped_batch([(np.arange(m) % 4 + 1).astype(np.uint8)])
    ops = np.array([(1 << 4) | (7 if i % 2 == 0 else 8) for i in range(m)], dtype=np.uint32)
    al = np.array([(1234, 0, len(ops), m // 2, 0, 0, 0, (0,) * 7), (99, 0, 3, 5, 0, 0, 1, (0,) * 7)], dtype=abi.ALIGNMENT_DTYPE)
    host, dev = both(ctx, gpu, al, ops, batch, ["chr"], [1 << 20], ["long"])
    assert_same_blocks(host, dev)
    assert parse_bam(dev)[2][0]["span"] == m


def test_many_blocks_and_bad_input(ctx, gpu):
    rng = np.random.default_rng(9)
    batch, al, cg, _ = random_case(rng, 4000, 2)
    names = [f"q{i}" for i in range(len(batch.reads))]
    host, dev = both(ctx, gpu, al, cg, batch, ["a", "b"], [10, 20], names)
    assert len(raw_blocks(dev)) > 3
    assert_same_blocks(host, dev)
    bad = al.copy()
    bad["read_index"][0], bad["read_index"][-1] = bad["read_index"][-1], bad["read_index"][0]
    cases = [(bad, cg, batch, ["a", "b"], [10, 20], names),                  # not grouped by read
             (al, cg, batch, ["a"], [10], names),                            # an alignment names reference 1
             (al, cg, batch, ["a", "b"], [10, 20], ["x" * 300] + names[1:])]   # a name of 300 characters
    for args in cases:
        with pytest.raises(gpu.FloxerGpuError) as want:
            gpu.write_bam(*args)
        with pytest.raises(gpu.FloxerGpuError) as got:
            ctx.write_bam(*args)
        assert got.value.code == want.value.code


def test_long_cigar_spanning_2_to_the_28_is_refused_like_the_host(ctx, gpu):
    batch = unmapped_batch([np.ones(10, dtype=np.uint8)])
    ops = np.full(70_000, (4096 << 4) | 2, dtype=np.uint32)            # deletions: 2^28 + ... reference bases
    al = np.array([(0, 0, len(ops), 1, 0, 0, 0, (0,) * 7)], dtype=abi.ALIGNMENT_DTYPE)
    with pytest.raises(gpu.FloxerGpuError) as want:
        gpu.write_bam(al, ops, batch, ["chr"], [10], ["x"])
    with pytest.raises(gpu.FloxerGpuError) as got:
        ctx.write_bam(al, ops, batch, ["chr"], [10], ["x"])
    assert got.value.code == want.value.code == -4


# ----------------------------------------------------------------------------- a real job

def zlib_level1_size(image: bytes) -> int:
    """zlib level 1 (raw deflate) over the same 0xff00-byte chunks, plus 26 bytes of BGZF framing per block and the
    end-of-file block."""
    raw = b"".join(bgzf_blocks(image))
    total = 28
    for at in range(0, len(raw), 0xff00):
        z = zlib.compressobj(1, zlib.DEFLATED, -15)
        total += len(z.compress(raw[at:at + 0xff00]) + z.flush()) + 26
    return total


def test_config2_job(ctx, gpu):
    from floxer_b200 import workloads as W
    refs = [W.random_reference(10_000_000, 20240001)]
    ctx.set_references(refs)
    dev = gpu.GpuSeeder(ctx, 12)
    bare = W.make_reads_seeded(refs, 1000, 5000, 0.05, 20240003, gpu.pex_build, W._NoAnchors(), threads=16)
    job, seeded, _ = ctx.seed_verify_reads(dev, bare, VerifyConfig())
    rng = np.random.default_rng(7)
    ids = [f"r{i}" for i in range(len(seeded.reads))]
    quals = ["".join(chr(33 + int(x)) for x in rng.integers(2, 41, size=int(R["query_len"]))) for R in seeded.reads]
    host = job.bam(seeded, ["chr"], [10_000_000], ids, quals)
    on_dev = job.bam(seeded, ["chr"], [10_000_000], ids, quals, on_device=True)
    assert_same_blocks(host, on_dev)
    assert len(parse_bam(on_dev)[2]) >= 1000
    assert len(on_dev) <= 1.15 * zlib_level1_size(on_dev)
    job.free()
    dev.close()


# ----------------------------------------------------------------------------- determinism and concurrency

def test_deterministic_concurrent_and_counted(ctx, gpu):
    refs = [synthetic.random_reference(200_000, 5), synthetic.random_reference(50_000, 6)]
    ctx.set_references(refs)
    vbatch = synthetic.make_batch(refs, 8, 1500, 0.06, 17, gpu.pex_build, seed_errors=2, decoy_fraction=0.3)
    cases = []
    for seed in range(8):
        rng = np.random.default_rng(100 + seed)
        batch, al, cg, _ = random_case(rng, 300, 3)
        cases.append((al, cg, batch, REF_IDS, REF_LENS, [f"t{seed}/{i}" for i in range(len(batch.reads))], qualities_for(rng, batch)))
    want = [ctx.write_bam(*args) for args in cases]
    assert [ctx.write_bam(*args) for args in cases] == want        # the same bytes every time
    for args, image in zip(cases, want):
        assert_same_blocks(gpu.write_bam(*args), image)

    got, errors = [None] * len(cases), []

    def writer(i):
        try:
            got[i] = ctx.write_bam(*cases[i])
        except Exception as e:                                       # (reported below)
            errors.append(e)

    def verifier():
        try:
            for _ in range(3):
                ctx.verify_reads(vbatch, VerifyConfig()).free()
        except Exception as e:
            errors.append(e)
    threads = [threading.Thread(target=writer, args=(i,)) for i in range(len(cases))] + [threading.Thread(target=verifier)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors
    assert got == want

    al, cg, batch, ids, lens, names, quals = cases[0]
    before = ctx.counters()
    image = ctx.write_bam(*cases[0])
    after = ctx.counters()
    uploaded = al.nbytes + cg.nbytes + int(batch.reads["query_len"].sum()) + sum(len(n) + 1 for n in names)
    assert after["h2d_bytes"] - before["h2d_bytes"] >= uploaded
    assert after["d2h_bytes"] - before["d2h_bytes"] >= len(image)
