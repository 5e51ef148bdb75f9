"""Device seeding (fxg_seed_reads) against the host seeder on all host cores, on config 2 and a config-3 sample.

For each config: index build time, device seeding rate over repeated passes (reads/s, checked candidates/s, with the
spread), the host seeder on all cores on the same reads, every anchor and read record compared, end-to-end
seed + verify_reads both ways, and the per-kernel device time of one seeding pass (torch.profiler, a pass of its own).
Host clocks around calls that end in a synchronise (fxg_seed_reads and verify_reads return after their device work).
Prints one JSON line and writes it to OUT/seed_bench.json.

    python scripts/seed_bench.py --out DIR [--reps 5] [--config2-reads 32000] [--config3-reads 64]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from floxer_b200 import abi, gpu, synthetic, workloads as W  # noqa: E402
from floxer_b200.batch import ReadBatch, VerifyConfig  # noqa: E402


def gpu_identity():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    name, power = [x.strip() for x in out.stdout.strip().splitlines()[0].split(",")]
    return name, power


def host_seed(seeder, batch, threads):
    """The host seeder on both orientations of every read, reads spread over `threads` threads (the ctypes calls release
    the GIL).  Returns (anchors, read records) in fxg_seed_reads's layout."""
    def one(i):
        r = batch.reads[i]
        q0, n = int(r["query_offset"]), int(r["query_len"])
        lo = int(r["node_offset"]) + int(r["num_inner"])
        leaves = batch.nodes[lo: lo + int(r["num_leaves"])]
        return seeder.search(batch.forward_pool[q0:q0 + n], leaves), seeder.search(batch.reverse_pool[q0:q0 + n], leaves)
    with ThreadPoolExecutor(max_workers=threads) as ex:
        parts = list(ex.map(one, range(len(batch.reads))))
    reads = batch.reads.copy()
    counts = np.array([[len(a), len(b)] for a, b in parts], dtype=np.int64).reshape(-1, 2)
    reads["num_anchors_forward"], reads["num_anchors_reverse"] = counts[:, 0], counts[:, 1]
    reads["anchor_offset"] = np.concatenate([[0], np.cumsum(counts.sum(axis=1))])[:-1]
    flat = [x for ab in parts for x in ab]
    return (np.concatenate(flat) if flat else np.zeros(0, abi.ANCHOR_DTYPE)), reads


def spread(xs):
    xs = sorted(xs)
    return dict(median=xs[len(xs) // 2], min=xs[0], max=xs[-1], n=len(xs))


def kernel_times(ctx, seeder, batch, out_dir, tag):
    """Device time per kernel name over one seeding pass, from torch.profiler (a pass of its own)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        ctx.seed_reads(seeder, batch)
        torch.cuda.synchronize()
    acc = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            key = ev.name if len(ev.name) < 80 else ev.name[:77] + "..."
            acc[key] = acc.get(key, 0.0) + ev.device_time / 1000.0
    ranked = dict(sorted(((k, round(v, 3)) for k, v in acc.items()), key=lambda kv: -kv[1])[:14])
    with open(os.path.join(out_dir, f"seed_kernels_{tag}.json"), "w") as f:
        json.dump(ranked, f, indent=1)
    return ranked


def run_config(ctx, tag, refs, q, bare, reps, threads, out_dir):
    r = dict(q=q, reads=len(bare.reads), leaves_per_read=float(bare.reads["num_leaves"].mean()))
    ctx.set_references(refs)
    # index: build time (the first build also loads the kernels; reported apart)
    t = []
    for _ in range(3):
        t0 = time.perf_counter()
        s = gpu.GpuSeeder(ctx, q)
        t.append(time.perf_counter() - t0)
        s.close()
    r["index_build_s_first"], r["index_build_s"] = round(t[0], 4), spread([round(x, 4) for x in t[1:]])
    dev = gpu.GpuSeeder(ctx, q)
    ctx.seed_reads(dev, bare)                                   # warm-up
    times, stats = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        got, stats = ctx.seed_reads(dev, bare)
        times.append(time.perf_counter() - t0)
    n = len(bare.reads)
    r["device_s"] = spread([round(x, 4) for x in times])
    r["device_reads_per_s"] = spread([round(n / x) for x in times])
    r["device_checked_per_s"] = spread([round(stats["checked"] / x) for x in times])
    r["stats"] = stats
    r["anchors_per_read"] = round(len(got.anchors) / max(n, 1), 2)
    # the host seeder on all cores, the same reads
    host = gpu.Seeder(refs, q=q)
    t0 = time.perf_counter()
    h_anchors, h_reads = host_seed(host, bare, threads)
    host_s = time.perf_counter() - t0
    host.close()
    r["host_threads"], r["host_s"], r["host_reads_per_s"] = threads, round(host_s, 3), round(n / host_s)
    r["speedup_vs_host_all_cores"] = round(r["device_reads_per_s"]["median"] / r["host_reads_per_s"], 1)
    r["parity"] = dict(anchors=int(len(got.anchors)), equal=bool(np.array_equal(got.anchors, h_anchors) and np.array_equal(got.reads, h_reads)))
    # end to end: seed + verify_reads, device seeding against host seeding
    cfg = VerifyConfig()
    hb = ReadBatch(h_reads, bare.forward_pool, bare.reverse_pool, bare.nodes, h_anchors)
    ctx.verify_reads(got, cfg).free()                            # warm-up
    e2e_dev, e2e_host = [], []
    for _ in range(max(1, reps // 2)):
        t0 = time.perf_counter()
        b, _ = ctx.seed_reads(dev, bare)
        job = ctx.verify_reads(b, cfg)
        al_d = job.alignments()
        e2e_dev.append(time.perf_counter() - t0)
        job.free()
        t0 = time.perf_counter()
        job = ctx.verify_reads(hb, cfg)
        al_h = job.alignments()
        e2e_host.append(time.perf_counter() - t0 + host_s)      # + the host seeding time measured above
        job.free()
    r["e2e_device_seed_verify_reads_per_s"] = spread([round(n / x) for x in e2e_dev])
    r["e2e_host_seed_verify_reads_per_s"] = spread([round(n / x) for x in e2e_host])
    r["e2e_alignments_equal"] = bool(np.array_equal(al_d[0], al_h[0]) and np.array_equal(al_d[1], al_h[1]))
    r["kernel_ms_one_pass"] = kernel_times(ctx, dev, bare, out_dir, tag)
    dev.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--config2-reads", type=int, default=32_000)
    ap.add_argument("--config3-reads", type=int, default=64)
    ap.add_argument("--threads", type=int, default=len(os.sched_getaffinity(0)), help="host seeder threads (default: every core)")
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    name, power = gpu_identity()
    res = dict(gpu=name, power_limit=power, host_cores=len(os.sched_getaffinity(0)))
    ctx = gpu.Context(0)
    # config 2: 10 Mbp uniform reference, q = 12, distinct 5 kbp reads at 5 % (recursive trees, leaf errors 2)
    c = W.CONFIGS["config2"]
    refs = [W.random_reference(c["ref_lens"][0], c["ref_seed"])]
    bare = W.make_reads_seeded(refs, a.config2_reads, c["read_len"], c["error"], c["read_seed"], gpu.pex_build, W._NoAnchors(), threads=a.threads)
    res["config2"] = run_config(ctx, "config2", refs, 12, bare, a.reps, a.threads, a.out)
    # config 3: 100 Mbp repeat-seeded reference, 15 kbp reads at 8 %: q = 8 or the largest q every leaf admits
    c = W.CONFIGS["config3"]
    refs, _ = W.build_references("config3")
    _, leaves = gpu.pex_build(c["read_len"], synthetic.ceil_eps(c["read_len"] * c["error"]), 2, 0)
    m = leaves["query_index_to"] - leaves["query_index_from"] + 1
    q3 = int(min(8, (m // (leaves["num_errors"] + 1)).min()))
    bare = W.make_reads_seeded(refs, a.config3_reads, c["read_len"], c["error"], c["read_seed"], gpu.pex_build, W._NoAnchors(), threads=a.threads)
    res["config3_sample"] = run_config(ctx, "config3", refs, q3, bare, max(2, a.reps // 2), a.threads, a.out)
    ctx.close()
    line = json.dumps(res)
    with open(os.path.join(a.out, "seed_bench.json"), "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
