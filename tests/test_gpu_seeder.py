"""The device seeder (fxg_gpu_seeder_create / fxg_seed_reads) against the host seeder (fxg_seeder_search) on the same
references, reads and trees: every anchor, in order, and the updated read records.  Needs a B200: run with -m gpu."""
import os
import threading

import numpy as np
import pytest

from floxer_b200 import abi, synthetic
from floxer_b200.batch import BatchBuilder, ReadBatch, VerifyConfig, alignment_records
from harness import oracle_verify_batch

pytestmark = pytest.mark.gpu


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


def host_seed(seeder, batch: ReadBatch, hard=500, soft=50, erase=True):
    """What fxg_seed_reads must return: the host seeder on both orientations of every read, as (anchors, reads)."""
    reads = batch.reads.copy()
    parts, at = [], 0
    for i, r in enumerate(batch.reads):
        q0, n = int(r["query_offset"]), int(r["query_len"])
        lo = int(r["node_offset"]) + int(r["num_inner"])
        leaves = batch.nodes[lo: lo + int(r["num_leaves"])]
        af = seeder.search(batch.forward_pool[q0:q0 + n], leaves, hard, soft, erase) if len(leaves) else np.zeros(0, abi.ANCHOR_DTYPE)
        ar = seeder.search(batch.reverse_pool[q0:q0 + n], leaves, hard, soft, erase) if len(leaves) else np.zeros(0, abi.ANCHOR_DTYPE)
        reads[i]["anchor_offset"], reads[i]["num_anchors_forward"], reads[i]["num_anchors_reverse"] = at, len(af), len(ar)
        parts += [af, ar]
        at += len(af) + len(ar)
    return (np.concatenate(parts) if parts else np.zeros(0, abi.ANCHOR_DTYPE)), reads


def assert_same(got: ReadBatch, want_anchors, want_reads):
    assert np.array_equal(got.reads, want_reads)
    assert len(got.anchors) == len(want_anchors)
    assert np.array_equal(got.anchors, want_anchors)


def awkward_references(seed):
    """Several records: one shorter than any q used here, lengths that are not multiples of 32, runs of rank 5 and rank 0,
    a planted repeat (a leaf hits several loci)."""
    rng = np.random.default_rng(seed)
    refs = [rng.integers(1, 5, size=n, dtype=np.uint8) for n in (6001, 3, 2333, 4097, 50)]
    refs[0][3000:3600] = refs[0][500:1100]
    refs[3][100:700] = refs[0][500:1100]
    for r in (refs[0], refs[2], refs[3]):
        for at in rng.integers(0, len(r) - 20, size=8):
            r[at:at + int(rng.integers(1, 15))] = 5
        r[rng.integers(0, len(r), size=6)] = 0
    return refs


def awkward_batch(gpu, refs, seed, n_reads, q, leaf_errors, strategy):
    """Reads simulated from the records, a few with rank 5 / rank 0 inside, with trees whose leaves the index admits."""
    rng = np.random.default_rng(seed)
    bb = BatchBuilder()
    src = [r for r in refs if len(r) > 600]
    while len(bb._reads) < n_reads:
        ref = src[int(rng.integers(0, len(src)))]
        length = int(rng.integers(200, 500))
        read, _, _ = synthetic.simulate_read(rng, ref, int(rng.integers(0, len(ref) - length - 1)), length, int(rng.integers(0, 8)))
        if rng.random() < 0.2:
            at = int(rng.integers(0, len(read) - 10))
            read[at:at + int(rng.integers(1, 8))] = 5 if rng.random() < 0.5 else 0
        k = max(1, len(read) // (q * (leaf_errors + 1) * 2))
        inner, leaves = gpu.pex_build(len(read), k, leaf_errors, strategy)
        m = leaves["query_index_to"] - leaves["query_index_from"] + 1
        assert (m // (leaves["num_errors"] + 1) >= q).all()
        bb.add(read, synthetic.reverse_complement(read), inner, leaves, np.zeros(0, abi.ANCHOR_DTYPE), np.zeros(0, abi.ANCHOR_DTYPE))
    return bb.build()


# ----------------------------------------------------------------------------- 1. small, awkward references

@pytest.mark.parametrize("q", [4, 6, 8])
@pytest.mark.parametrize("strategy", [0, 1])
def test_awkward_references(ctx, gpu, q, strategy):
    refs = awkward_references(100 + q)
    ctx.set_references(refs)
    host = gpu.Seeder(refs, q=q)
    dev = gpu.GpuSeeder(ctx, q)
    for leaf_errors in range(4):
        batch = awkward_batch(gpu, refs, 1000 * q + 10 * strategy + leaf_errors, 50, q, leaf_errors, strategy)
        for erase in (True, False):
            got, stats = ctx.seed_reads(dev, batch, erase_useless=erase)
            assert_same(got, *host_seed(host, batch, erase=erase))
            assert stats["hits"] > 0
    dev.close()
    host.close()


# ----------------------------------------------------------------------------- 2. caps

def test_caps_device(ctx, gpu):
    """test_seeder.py's test_caps on the device: the soft cap binds, then the hard cap excludes the seed."""
    ref = np.tile(np.array([1, 2, 3, 4, 1, 1, 2, 2, 3, 3, 4, 4], dtype=np.uint8), 100)
    ctx.set_references([ref])
    host, dev = gpu.Seeder([ref], q=6), gpu.GpuSeeder(ctx, 6)
    leaves = np.array([(abi.NULL_ID, 0, 11, 0), (abi.NULL_ID, 12, 23, 0)], dtype=abi.PEX_NODE_DTYPE)
    query = np.concatenate([ref[:12], np.array([4, 4, 4, 4, 3, 3, 3, 3, 2, 2, 2, 1], dtype=np.uint8)])
    bb = BatchBuilder()
    bb.add(query, synthetic.reverse_complement(query), np.zeros(0, abi.PEX_NODE_DTYPE), leaves, [], [])
    batch = bb.build()
    got, _ = ctx.seed_reads(dev, batch, 500, 50)
    assert got.reads[0]["num_anchors_forward"] == 50
    assert_same(got, *host_seed(host, batch, 500, 50))
    got, stats = ctx.seed_reads(dev, batch, 90, 50)
    assert got.reads[0]["num_anchors_forward"] == 0 and stats["dropped_hard"] >= 99
    assert_same(got, *host_seed(host, batch, 90, 50))


def test_caps_seeds_on_both_sides(ctx, gpu):
    """Units tiled 30, 60 and 120 times: with soft cap 40 and hard cap 100 the seeds of one batch fall under both caps,
    between them and over both; ties in errors are broken by position."""
    rng = np.random.default_rng(31)
    units = [rng.integers(1, 5, size=12, dtype=np.uint8) for _ in range(3)]
    ref = np.concatenate([np.tile(u, n) for u, n in zip(units, (30, 60, 120))] + [rng.integers(1, 5, size=3000, dtype=np.uint8)])
    ctx.set_references([ref])
    host, dev = gpu.Seeder([ref], q=6), gpu.GpuSeeder(ctx, 6)
    bb = BatchBuilder()
    for i in range(24):
        pieces = [units[int(rng.integers(0, 3))] if rng.random() < 0.7 else ref[int(rng.integers(1500, 4800)):][:12] for _ in range(4)]
        query = np.concatenate(pieces).astype(np.uint8)
        if i % 3 == 0:
            query[int(rng.integers(0, 48))] = 1 + int(rng.integers(0, 4))
        e = i % 2
        leaves = np.array([(abi.NULL_ID, 12 * k, 12 * k + 11, e if 12 // (e + 1) >= 6 else 0) for k in range(4)], dtype=abi.PEX_NODE_DTYPE)
        bb.add(query, synthetic.reverse_complement(query), np.zeros(0, abi.PEX_NODE_DTYPE), leaves, [], [])
    batch = bb.build()
    for erase in (True, False):
        got, stats = ctx.seed_reads(dev, batch, 100, 40, erase)
        assert_same(got, *host_seed(host, batch, 100, 40, erase))
        assert stats["dropped_hard"] > 0 and stats["cut_soft"] > 0


# ----------------------------------------------------------------------------- 3. chunking

def test_chunking_gives_the_same_result(ctx, gpu):
    """FXG_SEED_CANDIDATES set very small on a second context: every seed (many of them above the budget) is sorted in a
    chunk of its own or with few others; the result is identical."""
    refs = awkward_references(7)
    batch = awkward_batch(gpu, refs, 77, 50, 4, 1, 0)
    ctx.set_references(refs)
    dev = gpu.GpuSeeder(ctx, 4)
    want, want_stats = ctx.seed_reads(dev, batch)
    os.environ["FXG_SEED_CANDIDATES"] = "40"
    try:
        c2 = gpu.Context(0)
        c2.set_references(refs)
        small = gpu.GpuSeeder(c2, 4)
    finally:
        del os.environ["FXG_SEED_CANDIDATES"]
    got, got_stats = c2.seed_reads(small, batch)
    assert np.array_equal(got.reads, want.reads) and np.array_equal(got.anchors, want.anchors)
    assert got_stats == want_stats
    assert_same(got, *host_seed(gpu.Seeder(refs, q=4), batch))
    small.close()
    c2.close()
    dev.close()


# ----------------------------------------------------------------------------- 4. config-2 and config-3 scale

def test_config2_scale(ctx, gpu):
    from floxer_b200 import workloads as W
    refs = [W.random_reference(10_000_000, 20240001)]
    ctx.set_references(refs)
    host, dev = gpu.Seeder(refs, q=12), gpu.GpuSeeder(ctx, 12)
    want = W.make_reads_seeded(refs, 1000, 5000, 0.05, 20240003, gpu.pex_build, host, threads=16)
    got = W.make_reads_device_seeded(refs, 1000, 5000, 0.05, 20240003, gpu.pex_build, ctx, dev, threads=16)
    assert np.array_equal(got.forward_pool, want.forward_pool) and np.array_equal(got.nodes, want.nodes)
    assert_same(got, want.anchors, want.reads)
    assert len(got.anchors) > 20_000
    dev.close()
    host.close()


def test_config3_scale_sample(ctx, gpu):
    from floxer_b200 import workloads as W
    refs, _ = W.build_references("config3")
    cfg = W.CONFIGS["config3"]
    inner, leaves = gpu.pex_build(cfg["read_len"], synthetic.ceil_eps(cfg["read_len"] * cfg["error"]), 2, 0)
    m = leaves["query_index_to"] - leaves["query_index_from"] + 1
    q = int(min(8, (m // (leaves["num_errors"] + 1)).min()))
    ctx.set_references(refs)
    host, dev = gpu.Seeder(refs, q=q), gpu.GpuSeeder(ctx, q)
    want = W.make_reads_seeded(refs, 3, cfg["read_len"], cfg["error"], cfg["read_seed"], gpu.pex_build, host, threads=16)
    got, stats = ctx.seed_reads(dev, want)
    assert_same(got, want.anchors, want.reads)
    assert stats["checked"] > 1_000_000
    dev.close()
    host.close()


# ----------------------------------------------------------------------------- 5. seed -> verify

def test_seed_then_verify(ctx, gpu, oracle):
    from floxer_b200 import workloads as W
    refs = [synthetic.random_reference(90_000, 71), synthetic.plant_repeats(synthetic.random_reference(50_000, 72), 73, families=4, unit=(300, 900), copies=(3, 5))]
    ctx.set_references(refs)
    host, dev = gpu.Seeder(refs, q=8), gpu.GpuSeeder(ctx, 8)
    want = W.make_reads_seeded(refs, 10, 800, 0.06, 74, gpu.pex_build, host, seed_errors=1, threads=2)
    got = W.make_reads_device_seeded(refs, 10, 800, 0.06, 74, gpu.pex_build, ctx, dev, seed_errors=1, threads=2)
    assert_same(got, want.anchors, want.reads)
    for cfg in (VerifyConfig(), VerifyConfig(interval_optimization=True)):
        jobs = [ctx.verify_reads(b, cfg) for b in (got, want)]
        (a1, c1), (a2, c2) = jobs[0].alignments(), jobs[1].alignments()
        assert alignment_records(a1, c1) == alignment_records(a2, c2) and jobs[0].stats() == jobs[1].stats()
        o, o_stats = oracle_verify_batch(oracle, refs, got, cfg)
        assert alignment_records(a1, c1) == o and jobs[0].stats() == o_stats and len(o) > 0
        for j in jobs:
            j.free()


def test_seed_then_verify_config2_shape(ctx, gpu):
    """Config-2 reads seeded on the device and on the host: the same alignments, CIGARs and statistics."""
    from floxer_b200 import workloads as W
    refs = [W.random_reference(10_000_000, 20240001)]
    ctx.set_references(refs)
    host, dev = gpu.Seeder(refs, q=12), gpu.GpuSeeder(ctx, 12)
    want = W.make_reads_seeded(refs, 200, 5000, 0.05, 99, gpu.pex_build, host, threads=16)
    got, _ = ctx.seed_reads(dev, want)
    for cfg in (VerifyConfig(), VerifyConfig(interval_optimization=True)):
        j1, j2 = ctx.verify_reads(got, cfg), ctx.verify_reads(want, cfg)
        (a1, c1), (a2, c2) = j1.alignments(), j2.alignments()
        assert alignment_records(a1, c1) == alignment_records(a2, c2) and j1.stats() == j2.stats()
        assert len(a1) >= 150
        j1.free(); j2.free()


# ----------------------------------------------------------------------------- 6. errors and state

def one_read_batch(query, leaves):
    bb = BatchBuilder()
    bb.add(query, synthetic.reverse_complement(query), np.zeros(0, abi.PEX_NODE_DTYPE), np.asarray(leaves, dtype=abi.PEX_NODE_DTYPE), [], [])
    return bb.build()


def test_refused_leaves_and_state(ctx, gpu):
    rng = np.random.default_rng(3)
    ref = rng.integers(1, 5, size=5000, dtype=np.uint8)
    ctx.set_references([ref])
    host, dev = gpu.Seeder([ref], q=6), gpu.GpuSeeder(ctx, 6)
    query = ref[100:160].copy()
    good = (abi.NULL_ID, 0, 29, 1)
    for bad in [(abi.NULL_ID, 20, 10, 0),          # to < from
                (abi.NULL_ID, 30, 60, 0),          # to >= query length
                (abi.NULL_ID, 0, 59, 9),           # more than 8 errors
                (abi.NULL_ID, 0, 10, 1)]:          # pieces shorter than q (11 // 2 < 6)
        with pytest.raises(gpu.FloxerGpuError) as h:
            host.search(query, np.array([good, bad], dtype=abi.PEX_NODE_DTYPE))
        with pytest.raises(gpu.FloxerGpuError) as d:
            ctx.seed_reads(dev, one_read_batch(query, [good, bad]))
        assert d.value.code == h.value.code == abi.ERR_INVALID_ARGUMENT
        assert "leaf 1" in str(d.value)
    for q in (3, 15):
        with pytest.raises(gpu.FloxerGpuError) as d:
            gpu.GpuSeeder(ctx, q)
        assert d.value.code == abi.ERR_INVALID_ARGUMENT
    # an empty batch, reads without leaves, reads whose pieces hold no A/C/G/T-only q-gram
    empty = BatchBuilder().build()
    got, stats = ctx.seed_reads(dev, empty)
    assert len(got.anchors) == 0 and len(got.reads) == 0 and stats["seeds"] == 0
    bb = BatchBuilder()
    bb.add(query, synthetic.reverse_complement(query), [], [], [], [])
    nn = np.full(60, 5, dtype=np.uint8)
    bb.add(nn, nn, [], np.array([good], dtype=abi.PEX_NODE_DTYPE), [], [])
    bb.add(query, synthetic.reverse_complement(query), [], np.array([good], dtype=abi.PEX_NODE_DTYPE), [], [])
    batch = bb.build()
    got, stats = ctx.seed_reads(dev, batch)
    assert_same(got, *host_seed(host, batch))
    assert got.reads[0]["num_anchors_forward"] == got.reads[1]["num_anchors_forward"] == 0 and got.reads[2]["num_anchors_forward"] > 0
    # the references replaced: the seeder no longer describes them
    ctx.set_references([ref[:4000]])
    with pytest.raises(gpu.FloxerGpuError) as d:
        ctx.seed_reads(dev, batch)
    assert d.value.code == abi.ERR_STATE
    dev.close()
    host.close()


# ----------------------------------------------------------------------------- 7. concurrency

def test_concurrent_seeding_beside_verification(ctx, gpu):
    from floxer_b200 import workloads as W
    refs = [W.random_reference(2_000_000, 5)]
    ctx.set_references(refs)
    host, dev = gpu.Seeder(refs, q=11), gpu.GpuSeeder(ctx, 11)
    batches = [W.make_reads_seeded(refs, 40, 3000, 0.05, 600 + i, gpu.pex_build, host, threads=8) for i in range(8)]
    single = [ctx.seed_reads(dev, b)[0] for b in batches]
    verify_want = [alignment_records(*ctx.verify_reads(b, VerifyConfig()).alignments()) for b in batches[:2]]
    results, errors = [None] * 8, []

    def seed(i):
        try:
            for _ in range(3):
                got, _ = ctx.seed_reads(dev, batches[i])
                assert np.array_equal(got.anchors, single[i].anchors) and np.array_equal(got.reads, single[i].reads)
            results[i] = True
        except Exception as e:           # reported below
            errors.append(e)

    def verify(i):
        try:
            for _ in range(3):
                assert alignment_records(*ctx.verify_reads(batches[i], VerifyConfig()).alignments()) == verify_want[i]
        except Exception as e:
            errors.append(e)
    threads = [threading.Thread(target=seed, args=(i,)) for i in range(8)] + [threading.Thread(target=verify, args=(i,)) for i in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    assert all(results)
    for i in range(8):
        assert np.array_equal(single[i].anchors, batches[i].anchors) and np.array_equal(single[i].reads, batches[i].reads)
    dev.close()
    host.close()


# ----------------------------------------------------------------------------- 8. statistics

def numpy_recount(refs, q, batch):
    """candidates (starts >= 0 before de-duplication) and checked (distinct starts inside a reference) as seeder.cpp
    defines them, from a numpy q-gram table."""
    lens = np.array([len(r) for r in refs], dtype=np.int64)
    base = np.concatenate([[0], np.cumsum(lens)])[:-1]
    occ = {}
    for r, ref in enumerate(refs):
        for p in range(len(ref) - q + 1):
            g = ref[p:p + q]
            if ((g >= 1) & (g <= 4)).all():
                occ.setdefault(bytes(g), []).append(int(base[r] + p))
    cand = checked = 0
    for rd in batch.reads:
        q0, n = int(rd["query_offset"]), int(rd["query_len"])
        lo = int(rd["node_offset"]) + int(rd["num_inner"])
        for pool in (batch.forward_pool, batch.reverse_pool):
            query = pool[q0:q0 + n]
            for leaf in batch.nodes[lo: lo + int(rd["num_leaves"])]:
                f, m, e = int(leaf["query_index_from"]), int(leaf["query_index_to"] - leaf["query_index_from"] + 1), int(leaf["num_errors"])
                starts = []
                for k in range(e + 1):
                    off = m * k // (e + 1)
                    for p in occ.get(bytes(query[f + off: f + off + q]), []):
                        starts += [p - off + d for d in range(-e, e + 1) if p - off + d >= 0]
                cand += len(starts)
                for g in set(starts):
                    r = int(np.searchsorted(base, g, side="right") - 1)
                    checked += int(g - base[r] < lens[r])
    return cand, checked


def test_statistics(ctx, gpu):
    refs = awkward_references(11)
    ctx.set_references(refs)
    dev = gpu.GpuSeeder(ctx, 6)
    batch = awkward_batch(gpu, refs, 12, 12, 6, 2, 1)
    for hard, soft, erase in ((500, 50, True), (8, 3, True), (10**9, 10**9, False)):
        got, st = ctx.seed_reads(dev, batch, hard, soft, erase)
        assert len(got.anchors) == st["hits"] - st["dropped_hard"] - st["cut_soft"] - st["erased"]
        assert st["seeds"] == 2 * int(batch.reads["num_leaves"].sum())
    assert (st["candidates"], st["checked"]) == numpy_recount(refs, 6, batch)
    dev.close()
