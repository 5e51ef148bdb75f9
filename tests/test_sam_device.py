"""fxg_write_sam_device (Context.write_sam, Job.sam(on_device=True)) against the host writer fxg_write_sam: the same text
byte for byte on random cases and on every corner case of tests/test_sam_arrays.py; zero reads, reads without alignments
and a single 400 KB record; the same refusals before any device work; the BGZF image (bgzf=True) block by block --
ISIZE, CRC32 of the matching chunk of the host text, the inflated text, the end-of-file block --; jobs from
verify_reads and seed_verify_reads; determinism, concurrent callers and the copy counters.  Needs a B200: run with
-m gpu."""
import ctypes as C
import gzip
import struct
import threading
import zlib

import numpy as np
import pytest

from floxer_b200 import abi, synthetic
from floxer_b200.batch import VerifyConfig
from test_bam_output import random_case
from test_sam_arrays import REF_IDS, REF_LENS, batch_of, c_arguments, corner_cases, host_sam, refusal_cases

pytestmark = pytest.mark.gpu

EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
CHUNK = 0xff00


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


def device_sam(ctx, gpu, args, header=True, bgzf=False):
    """(return code, bytes) of fxg_write_sam_device."""
    L = gpu.lib()
    out, length = C.c_void_p(), C.c_size_t(0)
    rc = L.fxg_write_sam_device(ctx._h, *args, int(header), int(bgzf), C.byref(out), C.byref(length))
    if rc != 0:
        return rc, None
    try:
        data = C.string_at(out, length.value + (0 if bgzf else 1))
        if not bgzf:
            assert data[-1] == 0                                     # NUL-terminated, not counted
            data = data[:-1]
        return rc, data
    finally:
        L.fxg_free(out)


def raw_blocks(image: bytes):
    """The BGZF blocks of an image: (block, ISIZE, CRC32)."""
    out, at = [], 0
    while at < len(image):
        assert image[at:at + 4] == b"\x1f\x8b\x08\x04" and image[at + 12:at + 16] == b"BC\x02\x00"
        size = struct.unpack_from("<H", image, at + 16)[0] + 1
        block = image[at:at + size]
        crc, isize = struct.unpack_from("<II", block, size - 8)
        out.append((block, isize, crc))
        at += size
    assert at == len(image)
    return out


def assert_image_of(image: bytes, text: bytes):
    """image is text cut at 0xff00-byte boundaries, one BGZF block per chunk, then the end-of-file block."""
    blocks = raw_blocks(image)
    chunks = [text[at:at + CHUNK] for at in range(0, len(text), CHUNK)]
    assert len(blocks) == len(chunks) + 1
    for (block, isize, crc), chunk in zip(blocks, chunks):
        assert isize == len(chunk) and crc == zlib.crc32(chunk)
        assert zlib.decompress(block[18:-8], -15) == chunk
        assert len(block) <= 65536
    assert blocks[-1][0] == EOF_BLOCK
    assert gzip.decompress(image) == text


def assert_same(ctx, gpu, args, header=True):
    """Device text == host text, and the device's BGZF image holds the host text; returns the text."""
    rc, want = host_sam(gpu, args, header)
    assert rc == 0
    rc, got = device_sam(ctx, gpu, args, header)
    assert rc == 0 and got == want
    rc, image = device_sam(ctx, gpu, args, header, bgzf=True)
    assert rc == 0
    assert_image_of(image, want)
    return want


def qualities_for(rng, batch, every=3):
    return ["".join(chr(33 + int(x)) for x in rng.integers(2, 41, size=int(R["query_len"]))) if i % every else ""
            for i, R in enumerate(batch.reads)]


NO_ALIGNMENTS = np.zeros(0, dtype=abi.ALIGNMENT_DTYPE)


# ----------------------------------------------------------------------------- the same text

@pytest.mark.parametrize("seed", [1, 2, 3])
def test_text_equals_the_host_writers(ctx, gpu, seed):
    rng = np.random.default_rng(seed)
    batch, al, cg, _ = random_case(rng, 40, 3)
    names = [f"read/{i}" for i in range(len(batch.reads))]
    args, _keep = c_arguments(gpu, al, cg, batch, REF_IDS, REF_LENS, names, qualities_for(rng, batch))
    for header in (True, False):
        assert_same(ctx, gpu, args, header)
    assert ctx.write_sam(al, cg, batch, REF_IDS, REF_LENS, names) == gpu.write_sam(al, cg, batch, REF_IDS, REF_LENS, names)


@pytest.mark.parametrize("name", sorted(corner_cases()))
def test_corner_cases(ctx, gpu, name):
    al, cg, batch, rids, rlens, ids, quals, header, want = corner_cases()[name]
    args, _keep = c_arguments(gpu, al, cg, batch, rids, rlens, ids, quals)
    assert assert_same(ctx, gpu, args, header) == want.encode()


def test_long_name_and_long_cigar_spanning_2_to_the_28(ctx, gpu):
    ops = np.full(70_000, (4096 << 4) | 2, dtype=np.uint32)
    al = np.zeros(1, dtype=abi.ALIGNMENT_DTYPE)
    al["cigar_len"], al["num_errors"] = len(ops), 1
    args, _keep = c_arguments(gpu, al, ops, batch_of([[1, 2]]), ["chr"], [10], ["n" * 300], [""])
    assert_same(ctx, gpu, args, False)


def test_zero_reads_and_reads_without_alignments(ctx, gpu):
    rng = np.random.default_rng(4)
    batch, _, _, _ = random_case(rng, 30, 2)
    empty = batch_of([])
    for header in (True, False):
        args, _keep = c_arguments(gpu, NO_ALIGNMENTS, [], empty, ["a", "b"], [10, 20], [], [])
        assert assert_same(ctx, gpu, args, header) == (b"" if not header else b"@HD\tVN:1.6\tSO:unknown\tGO:none\n@SQ\tSN:a\tLN:10\n@SQ\tSN:b\tLN:20\n")
        names = [f"u{i}" for i in range(len(batch.reads))]
        args, _keep = c_arguments(gpu, NO_ALIGNMENTS, [], batch, ["a", "b"], [10, 20], names, qualities_for(rng, batch, 2))
        assert_same(ctx, gpu, args, header)
    args, _keep = c_arguments(gpu, NO_ALIGNMENTS, [], empty, [], [], [], [])
    assert device_sam(ctx, gpu, args, False, bgzf=True) == (0, EOF_BLOCK)       # an empty stream: the end-of-file block only
    assert device_sam(ctx, gpu, args, False) == (0, b"")


def test_one_record_of_400_kb(ctx, gpu):
    rng = np.random.default_rng(5)
    seq = rng.integers(1, 6, size=200_000, dtype=np.uint8)
    qual = "".join(chr(33 + int(x)) for x in rng.integers(2, 41, size=200_000))
    args, _keep = c_arguments(gpu, NO_ALIGNMENTS, [], batch_of([seq]), [], [], ["big"], [qual])
    text = assert_same(ctx, gpu, args, False)
    assert len(text) > 400_000 and text.count(b"\n") == 1


# ----------------------------------------------------------------------------- refusals

@pytest.mark.parametrize("name", sorted(refusal_cases()))
def test_refusals_match_the_host_and_do_no_device_work(ctx, gpu, name):
    al, cg, batch, rids, rlens, ids, quals, code = refusal_cases()[name]
    args, _keep = c_arguments(gpu, al, cg, batch, rids, rlens, ids, quals)
    assert host_sam(gpu, args)[0] == code
    for bgzf in (False, True):
        before = ctx.counters()
        assert device_sam(ctx, gpu, args, bgzf=bgzf)[0] == code
        after = ctx.counters()
        assert gpu.lib().fxg_last_error(ctx._h)
        for k in ("h2d_bytes", "d2h_bytes", "kernel_launches"):
            assert after[k] == before[k], k


# ----------------------------------------------------------------------------- BGZF

def test_bgzf_blocks_of_many_records(ctx, gpu):
    rng = np.random.default_rng(9)
    batch, al, cg, _ = random_case(rng, 4000, 2)
    names = [f"q{i}" for i in range(len(batch.reads))]
    quals = qualities_for(rng, batch)
    args, _keep = c_arguments(gpu, al, cg, batch, ["a", "b"], [10, 20], names, quals)
    text = assert_same(ctx, gpu, args)
    image = ctx.write_sam(al, cg, batch, ["a", "b"], [10, 20], names, quals, bgzf=True)
    assert_image_of(image, text)
    blocks = raw_blocks(image)
    assert len(blocks) > 3
    assert all(isize == CHUNK for _, isize, _ in blocks[:-2]) and 0 < blocks[-2][1] <= CHUNK and blocks[-1][1] == 0
    assert len(text) > 3 * CHUNK


def test_text_of_exactly_two_chunks(ctx, gpu):
    # 128 unmapped records of 1020 bytes: 399-character name + 19 fixed + 300 SEQ + tab + 300 QUAL + newline = 2 * 0xff00
    rng = np.random.default_rng(6)
    seqs = [rng.integers(1, 5, size=300, dtype=np.uint8) for _ in range(128)]
    names = [f"{i:03d}" + "n" * 396 for i in range(128)]
    quals = ["".join(chr(33 + int(x)) for x in rng.integers(2, 41, size=300)) for _ in range(128)]
    args, _keep = c_arguments(gpu, NO_ALIGNMENTS, [], batch_of(seqs), [], [], names, quals)
    text = assert_same(ctx, gpu, args, False)
    assert len(text) == 2 * CHUNK
    rc, image = device_sam(ctx, gpu, args, False, bgzf=True)
    assert [isize for _, isize, _ in raw_blocks(image)] == [CHUNK, CHUNK, 0]


# ----------------------------------------------------------------------------- jobs

def test_jobs_from_verify_reads(ctx, gpu):
    refs = [synthetic.random_reference(90_000, 71), synthetic.random_reference(40_000, 72)]
    ctx.set_references(refs)
    batch = synthetic.make_batch(refs, 9, 800, 0.06, 19, gpu.pex_build, seed_errors=1, decoy_fraction=0.3)
    names = [f"read{i}" for i in range(len(batch))]
    quals = ["" if i % 3 == 0 else "F" * int(batch.reads[i]["query_len"]) for i in range(len(batch))]
    ref_ids, ref_lens = ["chrA", "chrB"], [len(r) for r in refs]
    for cfg in (VerifyConfig(), VerifyConfig(interval_optimization=True), VerifyConfig(without_cigar=True)):
        job = ctx.verify_reads(batch, cfg)
        for header in (True, False):
            host = job.sam(batch, ref_ids, ref_lens, names, quals, header=header)
            assert job.sam(batch, ref_ids, ref_lens, names, quals, header=header, on_device=True) == host
            image = job.sam(batch, ref_ids, ref_lens, names, quals, header=header, on_device=True, bgzf=True)
            assert_image_of(image, host.encode())
        if cfg.without_cigar:
            assert "\t255\t*\t*\t0\t0\t" in host
        job.free()


def zlib_level1_size(text: bytes) -> int:
    total = 28
    for at in range(0, len(text), CHUNK):
        z = zlib.compressobj(1, zlib.DEFLATED, -15)
        total += len(z.compress(text[at:at + CHUNK]) + z.flush()) + 26
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
    host = job.sam(seeded, ["chr"], [10_000_000], ids, quals)
    assert job.sam(seeded, ["chr"], [10_000_000], ids, quals, on_device=True) == host
    image = job.sam(seeded, ["chr"], [10_000_000], ids, quals, on_device=True, bgzf=True)
    assert_image_of(image, host.encode())
    assert host.count("\n") >= 1000
    assert len(image) <= 1.15 * zlib_level1_size(host.encode())
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
    kinds = ["text", "bgzf", "bam", "text", "bgzf", "bam", "text", "bgzf"]

    def write(i):
        if kinds[i] == "bam":
            return ctx.write_bam(*cases[i])
        return ctx.write_sam(*cases[i], bgzf=kinds[i] == "bgzf")

    want = [write(i) for i in range(len(cases))]
    assert [write(i) for i in range(len(cases))] == want                   # the same bytes every time
    for i, args in enumerate(cases):
        host = gpu.write_sam(*args)
        if kinds[i] == "text":
            assert want[i] == host
        elif kinds[i] == "bgzf":
            assert_image_of(want[i], host.encode())

    got, errors = [None] * len(cases), []

    def writer(i):
        try:
            got[i] = write(i)
        except Exception as e:                                               # (reported below)
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
    uploaded = al.nbytes + cg.nbytes + int(batch.reads["query_len"].sum()) + sum(len(n) for n in names) + sum(len(q) for q in quals)
    for bgzf in (False, True):
        before = ctx.counters()
        out = ctx.write_sam(*cases[0], bgzf=bgzf)
        after = ctx.counters()
        assert after["h2d_bytes"] - before["h2d_bytes"] >= uploaded
        assert after["d2h_bytes"] - before["d2h_bytes"] >= len(out)
