"""fxg_seed_verify_reads (Context.seed_verify_reads) against fxg_seed_reads + fxg_verify_reads on the same context and
batch: the alignments in order with their CIGARs, the job's statistics, the updated read records and the seed statistics.
Needs a B200: run with -m gpu."""
import os
import threading

import numpy as np
import pytest

from floxer_b200 import abi, synthetic
from floxer_b200.batch import BatchBuilder, VerifyConfig, alignment_records
from harness import oracle_verify_batch
from test_gpu_seeder import awkward_batch, awkward_references, one_read_batch

pytestmark = pytest.mark.gpu

CONFIGS = [VerifyConfig(verification_kind=kind, interval_optimization=iv, without_cigar=nc)
           for kind in (abi.KIND_HIERARCHICAL, abi.KIND_DIRECT_FULL) for iv in (False, True) for nc in (False, True)]


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


def context_with(gpu, refs, q, **env):
    """A second context and its seeder, both made with the given environment (restored afterwards)."""
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        c = gpu.Context(0)
        c.set_references(refs)
        return c, gpu.GpuSeeder(c, q)
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


def result_of(job):
    out = alignment_records(*job.alignments()), job.stats()
    job.free()
    return out


def two_calls(ctx, dev, batch, cfg, hard=500, soft=50, erase=True):
    """(records, stats), the seeded batch and the seed statistics of seed_reads + verify_reads."""
    seeded, st = ctx.seed_reads(dev, batch, hard, soft, erase)
    return result_of(ctx.verify_reads(seeded, cfg)), seeded, st


def fused(ctx, dev, batch, cfg, hard=500, soft=50, erase=True):
    job, seeded, st = ctx.seed_verify_reads(dev, batch, cfg, hard, soft, erase)
    assert len(seeded.anchors) == 0
    return result_of(job), seeded, st


def check_same(ctx, dev, batch, cfg, **kw):
    want, w_batch, w_st = two_calls(ctx, dev, batch, cfg, **kw)
    got, g_batch, g_st = fused(ctx, dev, batch, cfg, **kw)
    assert got[0] == want[0]
    assert got[1] == want[1]
    assert np.array_equal(g_batch.reads, w_batch.reads)
    assert g_st == w_st
    return got, w_batch


# ----------------------------------------------------------------------------- 1. small, awkward references

@pytest.mark.parametrize("q", [4, 6, 8])
@pytest.mark.parametrize("strategy", [0, 1])
def test_awkward_references(ctx, gpu, q, strategy):
    refs = awkward_references(100 + q)
    ctx.set_references(refs)
    dev = gpu.GpuSeeder(ctx, q)
    batch = awkward_batch(gpu, refs, 2000 * q + 10 * strategy, 40, q, (q + strategy) % 3, strategy)
    n_alignments = 0
    for cfg in CONFIGS:
        (records, _), _ = check_same(ctx, dev, batch, cfg)
        n_alignments += len(records)
    assert n_alignments > 0
    dev.close()


def test_repeats_against_the_oracle(ctx, gpu, oracle):
    from floxer_b200 import workloads as W
    refs = [synthetic.random_reference(90_000, 71), synthetic.plant_repeats(synthetic.random_reference(50_000, 72), 73, families=4, unit=(300, 900), copies=(3, 5))]
    ctx.set_references(refs)
    dev = gpu.GpuSeeder(ctx, 8)
    bare = W.make_reads_seeded(refs, 10, 800, 0.06, 74, gpu.pex_build, W._NoAnchors(), seed_errors=1, threads=2)
    for cfg in (VerifyConfig(), VerifyConfig(interval_optimization=True)):
        (records, stats), seeded = check_same(ctx, dev, bare, cfg)
        want, want_stats = oracle_verify_batch(oracle, refs, seeded, cfg)
        assert records == want and stats == want_stats and len(want) > 0
    dev.close()


# ----------------------------------------------------------------------------- 2. config-2 scale, 7. no anchor round trip

def test_config2_scale(ctx, gpu):
    from floxer_b200 import workloads as W
    refs = [W.random_reference(10_000_000, 20240001)]
    ctx.set_references(refs)
    dev = gpu.GpuSeeder(ctx, 12)
    bare = W.make_reads_seeded(refs, 1000, 5000, 0.05, 20240003, gpu.pex_build, W._NoAnchors(), threads=16)
    ids = [f"r{i}" for i in range(len(bare.reads))]
    for cfg in (VerifyConfig(), VerifyConfig(interval_optimization=True)):
        seeded, _ = ctx.seed_reads(dev, bare)
        assert len(seeded.anchors) > 20_000
        j2 = ctx.verify_reads(seeded, cfg)
        j1, g_batch, _ = ctx.seed_verify_reads(dev, bare, cfg)
        assert np.array_equal(g_batch.reads, seeded.reads)
        assert alignment_records(*j1.alignments()) == alignment_records(*j2.alignments()) and j1.stats() == j2.stats()
        sam1 = j1.sam(g_batch, ["chr1"], [len(refs[0])], ids)
        assert sam1 == j2.sam(seeded, ["chr1"], [len(refs[0])], ids)
        assert sam1.count("\n") > 1000
        j1.free(); j2.free()
    # the anchors do not cross PCIe: beyond what verification reads back, only the counts per read (8 bytes) and a few counters
    cfg = VerifyConfig()
    ctx.reset_counters()
    job, g_batch, _ = ctx.seed_verify_reads(dev, bare, cfg)
    fused_ctr = ctx.counters()
    job.free()
    seeded, _ = ctx.seed_reads(dev, bare)
    ctx.reset_counters()
    ctx.verify_reads(seeded, cfg).free()
    two_ctr = ctx.counters()
    assert fused_ctr["d2h_bytes"] - two_ctr["d2h_bytes"] <= 8 * len(bare.reads) + 4096
    assert fused_ctr["d2h_bytes"] > 0 and fused_ctr["h2d_bytes"] > 2 * len(bare.forward_pool)
    dev.close()


# ----------------------------------------------------------------------------- 3. config-3 sample

def test_config3_scale_sample(ctx, gpu):
    from floxer_b200 import workloads as W
    refs, _ = W.build_references("config3")
    c = W.CONFIGS["config3"]
    _, leaves = gpu.pex_build(c["read_len"], synthetic.ceil_eps(c["read_len"] * c["error"]), 2, 0)
    m = leaves["query_index_to"] - leaves["query_index_from"] + 1
    q = int(min(8, (m // (leaves["num_errors"] + 1)).min()))
    ctx.set_references(refs)
    dev = gpu.GpuSeeder(ctx, q)
    bare = W.make_reads_seeded(refs, 3, c["read_len"], c["error"], c["read_seed"], gpu.pex_build, W._NoAnchors(), threads=16)
    (records, _), _ = check_same(ctx, dev, bare, VerifyConfig())
    assert len(records) > 0
    dev.close()


# ----------------------------------------------------------------------------- 4. chunking

def test_chunking_gives_the_same_result(ctx, gpu):
    refs = awkward_references(7)
    batch = awkward_batch(gpu, refs, 77, 50, 4, 1, 0)
    ctx.set_references(refs)
    dev = gpu.GpuSeeder(ctx, 4)
    c2, small = context_with(gpu, refs, 4, FXG_SEED_CANDIDATES=40)
    for cfg in (VerifyConfig(), VerifyConfig(interval_optimization=True)):
        want = fused(ctx, dev, batch, cfg)
        got = fused(c2, small, batch, cfg)
        assert got[0] == want[0] and np.array_equal(got[1].reads, want[1].reads) and got[2] == want[2]
        assert len(got[0][0]) > 0
    check_same(c2, small, batch, VerifyConfig())
    small.close()
    c2.close()
    dev.close()


# ----------------------------------------------------------------------------- 5. a job of several parts

def repeat_references(seed, copies=150, unit_len=1500, spacer=3000, divergence=0.005):
    """One record: `copies` copies of one unit, each with a few substitutions, between random spacers."""
    rng = np.random.default_rng(seed)
    unit = rng.integers(1, 5, size=unit_len, dtype=np.uint8)
    parts = []
    for _ in range(copies):
        u = unit.copy()
        at = rng.random(unit_len) < divergence
        u[at] = 1 + (u[at] + rng.integers(0, 3, size=int(at.sum()), dtype=np.uint8)) % 4
        parts += [rng.integers(1, 5, size=spacer, dtype=np.uint8), u]
    return [np.concatenate(parts)]


def test_job_in_parts(ctx, gpu):
    """Reads from a unit with 150 copies, soft cap 200: more than 512 Ki anchors, so the run splits the job into parts."""
    refs = repeat_references(41)
    rng = np.random.default_rng(42)
    bb = BatchBuilder()
    inner, leaves = gpu.pex_build(1200, synthetic.ceil_eps(1200 * 0.05), 2, 0)
    for _ in range(200):
        start = int(rng.integers(0, 150)) * 4500 + 3000 + int(rng.integers(0, 250))
        read, _, _ = synthetic.simulate_read(rng, refs[0], start, 1200, 20)
        read = read[:1200] if len(read) >= 1200 else np.concatenate([read, refs[0][start + len(read): start + 1200]])
        bb.add(read, synthetic.reverse_complement(read), inner, leaves, [], [])
    batch = bb.build()
    ctx.set_references(refs)
    dev = gpu.GpuSeeder(ctx, 12)
    (records, _), seeded = check_same(ctx, dev, batch, VerifyConfig(), hard=1000, soft=200)
    assert len(seeded.anchors) > 512 * 1024
    assert len(records) > 0
    dev.close()


# ----------------------------------------------------------------------------- 6. host-driven levels

def test_host_fallback(ctx, gpu):
    refs = awkward_references(106)
    batch = awkward_batch(gpu, refs, 606, 40, 6, 1, 0)
    ctx.set_references(refs)
    dev = gpu.GpuSeeder(ctx, 6)
    c2, dev2 = context_with(gpu, refs, 6, FXG_DEVICE_LEVELS=0)
    for cfg in (VerifyConfig(), VerifyConfig(interval_optimization=True), VerifyConfig(verification_kind=abi.KIND_DIRECT_FULL)):
        got, _ = check_same(c2, dev2, batch, cfg)
        want = fused(ctx, dev, batch, cfg)[0]
        assert got == want and len(got[0]) > 0
    dev2.close()
    c2.close()
    dev.close()


# ----------------------------------------------------------------------------- 8. errors and state

def test_errors_and_state(ctx, gpu):
    rng = np.random.default_rng(3)
    ref = rng.integers(1, 5, size=5000, dtype=np.uint8)
    ctx.set_references([ref])
    dev = gpu.GpuSeeder(ctx, 6)
    cfg = VerifyConfig()
    query = ref[100:160].copy()
    good_leaf = (abi.NULL_ID, 0, 29, 1)
    good = one_read_batch(query, [good_leaf, (abi.NULL_ID, 30, 59, 1)])
    want = two_calls(ctx, dev, good, cfg)[0]
    assert len(want[0]) > 0

    def refused(batch):
        with pytest.raises(gpu.FloxerGpuError) as e:
            ctx.seed_verify_reads(dev, batch, cfg)
        assert fused(ctx, dev, good, cfg)[0] == want              # the context serves the next call
        return e.value

    # leaves the seeder refuses
    for bad in [(abi.NULL_ID, 20, 10, 0), (abi.NULL_ID, 30, 60, 0), (abi.NULL_ID, 0, 59, 9), (abi.NULL_ID, 0, 10, 1)]:
        batch = one_read_batch(query, [good_leaf, bad])
        with pytest.raises(gpu.FloxerGpuError) as d:
            ctx.seed_reads(dev, batch)
        e = refused(batch)
        assert e.code == d.value.code == abi.ERR_INVALID_ARGUMENT and "leaf 1" in str(e)
    # what only verification refuses: a read without leaves, a tree whose root has a parent, a rank above 5
    bb = BatchBuilder()
    bb.add(query, synthetic.reverse_complement(query), [], [good_leaf], [], [])
    bb.add(query, synthetic.reverse_complement(query), [], [], [], [])
    no_leaves = bb.build()
    bb = BatchBuilder()
    bb.add(query, synthetic.reverse_complement(query), np.array([(0, 0, 59, 2)], dtype=abi.PEX_NODE_DTYPE),
           np.array([(0, 0, 29, 1), (0, 30, 59, 1)], dtype=abi.PEX_NODE_DTYPE), [], [])
    broken = bb.build()
    rank6 = query.copy()
    rank6[40] = 6
    bb = BatchBuilder()
    bb.add(rank6, synthetic.reverse_complement(query), [], [good_leaf], [], [])
    bad_rank = bb.build()
    for batch, text in ((no_leaves, "read 1: bad node range"), (broken, "inner node 0 is not the root"), (bad_rank, "rank above 5")):
        seeded, _ = ctx.seed_reads(dev, batch)
        with pytest.raises(gpu.FloxerGpuError) as v:
            ctx.verify_reads(seeded, cfg)
        e = refused(batch)
        assert e.code == v.value.code == abi.ERR_INVALID_ARGUMENT
        assert text in str(e) and str(e) == str(v.value)
    # an empty batch
    job, seeded, st = ctx.seed_verify_reads(dev, BatchBuilder().build(), cfg)
    assert job.alignments()[0].size == 0 and all(v == 0 for v in job.stats().values()) and all(v == 0 for v in st.values())
    assert len(seeded.reads) == 0
    job.free()
    # the references replaced: the seeder no longer describes them
    ctx.set_references([ref[:4000]])
    with pytest.raises(gpu.FloxerGpuError) as e:
        ctx.seed_verify_reads(dev, good, cfg)
    assert e.value.code == abi.ERR_STATE
    dev.close()
    dev = gpu.GpuSeeder(ctx, 6)
    assert fused(ctx, dev, good, cfg)[0] == two_calls(ctx, dev, good, cfg)[0]
    dev.close()


# ----------------------------------------------------------------------------- 9. concurrency

def test_concurrent_calls(ctx, gpu):
    """Fused calls on 8 threads beside verify_reads on 4 and seed_reads on 2, three rounds each: every result equals the
    result of the same call made alone."""
    from floxer_b200 import workloads as W
    refs = [W.random_reference(2_000_000, 5)]
    ctx.set_references(refs)
    dev = gpu.GpuSeeder(ctx, 11)
    bare = [W.make_reads_seeded(refs, 40, 3000, 0.05, 600 + i, gpu.pex_build, W._NoAnchors(), threads=8) for i in range(8)]
    cfg = VerifyConfig()
    fused_want = [fused(ctx, dev, b, cfg) for b in bare]
    seeded = [ctx.seed_reads(dev, b)[0] for b in bare]
    verify_want = [result_of(ctx.verify_reads(seeded[i], cfg)) for i in range(4)]
    errors = []

    def run(fn, i):
        try:
            for _ in range(3):
                fn(i)
        except Exception as e:           # reported below
            errors.append(e)

    def fused_call(i):
        got = fused(ctx, dev, bare[i], cfg)
        assert got[0] == fused_want[i][0] and np.array_equal(got[1].reads, fused_want[i][1].reads) and got[2] == fused_want[i][2]

    def verify_call(i):
        assert result_of(ctx.verify_reads(seeded[i], cfg)) == verify_want[i]

    def seed_call(i):
        got, _ = ctx.seed_reads(dev, bare[i])
        assert np.array_equal(got.anchors, seeded[i].anchors) and np.array_equal(got.reads, seeded[i].reads)

    threads = ([threading.Thread(target=run, args=(fused_call, i)) for i in range(8)] +
               [threading.Thread(target=run, args=(verify_call, i)) for i in range(4)] +
               [threading.Thread(target=run, args=(seed_call, i)) for i in range(2)])
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for i in range(8):
        assert fused_want[i][0] == result_of(ctx.verify_reads(seeded[i], cfg))
    dev.close()
