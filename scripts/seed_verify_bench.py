"""Seeding and verification of read batches in one call (fxg_seed_verify_reads) against two calls (fxg_seed_reads, then
fxg_verify_reads), on config 2 and a config-3 sample.

N caller threads each seed and verify a batch of their own at the same time (config 2: 1 000-read batches, default 32
callers; config 3: 4 callers).  The two arms run in alternating repetitions in the same process, and the results of
every batch are compared record for record (alignments, CIGARs, statistics, read records, seed statistics) in every
repetition.  Reported per arm: reads/s with its spread over the repetitions, wall time per call (seen by the caller,
queueing included), process CPU time per batch, and the h2d / d2h bytes per batch from the context's counters.  Host
clocks around calls that return after their device work.  Prints one JSON line and writes it to OUT/seed_verify_bench.json.

    python scripts/seed_verify_bench.py --out DIR [--reps 5] [--callers 32] [--config3-reads 8]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from floxer_b200 import gpu, synthetic, workloads as W  # noqa: E402
from floxer_b200.batch import VerifyConfig, alignment_records  # noqa: E402


def gpu_identity():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, check=True)
    name, power = [x.strip() for x in out.stdout.strip().splitlines()[0].split(",")]
    return name, power


T0 = time.perf_counter()


def log(msg):
    print(f"[{time.perf_counter() - T0:7.1f} s] {msg}", file=sys.stderr, flush=True)


def spread(xs):
    xs = sorted(xs)
    return dict(median=xs[len(xs) // 2], min=xs[0], max=xs[-1], n=len(xs))


def two_calls(ctx, dev, batch, cfg):
    seeded, st = ctx.seed_reads(dev, batch)
    job = ctx.verify_reads(seeded, cfg)
    out = job.alignments(), job.stats(), seeded.reads, st
    job.free()
    return out


def one_call(ctx, dev, batch, cfg):
    job, seeded, st = ctx.seed_verify_reads(dev, batch, cfg)
    out = job.alignments(), job.stats(), seeded.reads, st
    job.free()
    return out


def run_arm(ctx, fn, dev, batches, cfg):
    """Every batch on a caller thread of its own, at once; returns (wall s, CPU s, per-call wall s, results, counters)."""
    results, call_s, errors = [None] * len(batches), [0.0] * len(batches), []

    def caller(i):
        try:
            t0 = time.perf_counter()
            results[i] = fn(ctx, dev, batches[i], cfg)
            call_s[i] = time.perf_counter() - t0
        except Exception as e:           # re-raised below
            errors.append(e)
    threads = [threading.Thread(target=caller, args=(i,)) for i in range(len(batches))]
    ctx.reset_counters()
    c0, t0 = time.process_time(), time.perf_counter()
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    wall, cpu = time.perf_counter() - t0, time.process_time() - c0
    if errors:
        raise errors[0]
    return wall, cpu, call_s, results, ctx.counters()


def same(a, b):
    (al_a, cg_a), st_a, reads_a, seed_a = a
    (al_b, cg_b), st_b, reads_b, seed_b = b
    return alignment_records(al_a, cg_a) == alignment_records(al_b, cg_b) and st_a == st_b and np.array_equal(reads_a, reads_b) and seed_a == seed_b


def run_config(ctx, refs, q, batches, reps):
    ctx.set_references(refs)
    dev = gpu.GpuSeeder(ctx, q)
    cfg = VerifyConfig()
    arms = dict(two_calls=two_calls, seed_verify_reads=one_call)
    n_reads = sum(len(b.reads) for b in batches)
    for name, fn in arms.items():                               # warm-up: kernels loaded, buffers grown
        run_arm(ctx, fn, dev, batches, cfg)
        log(f"warm-up {name} done")
    acc = {k: dict(rate=[], call_ms=[], cpu_ms_per_batch=[], h2d=[], d2h=[]) for k in arms}
    agree = True
    n_alignments = 0
    for rep in range(reps):
        order = list(arms) if rep % 2 == 0 else list(arms)[::-1]
        out = {}
        for name in order:
            wall, cpu, call_s, results, ctr = run_arm(ctx, arms[name], dev, batches, cfg)
            a = acc[name]
            a["rate"].append(round(n_reads / wall))
            a["call_ms"] += [round(x * 1e3, 2) for x in call_s]
            a["cpu_ms_per_batch"].append(round(cpu * 1e3 / len(batches), 2))
            a["h2d"].append(ctr["h2d_bytes"] // len(batches))
            a["d2h"].append(ctr["d2h_bytes"] // len(batches))
            out[name] = results
            log(f"rep {rep} {name}: {n_reads / wall:.0f} reads/s")
        agree = agree and all(same(x, y) for x, y in zip(out["two_calls"], out["seed_verify_reads"]))
        n_alignments = sum(len(x[0][0]) for x in out["seed_verify_reads"])
    dev.close()
    res = dict(q=q, callers=len(batches), reads=n_reads, alignments=n_alignments, reps=reps, results_equal_every_rep=bool(agree))
    for name, a in acc.items():
        res[name] = dict(reads_per_s=spread(a["rate"]), call_ms=spread(a["call_ms"]), cpu_ms_per_batch=spread(a["cpu_ms_per_batch"]),
                         h2d_bytes_per_batch=spread(a["h2d"]), d2h_bytes_per_batch=spread(a["d2h"]))
    res["rate_ratio_one_call_over_two"] = round(res["seed_verify_reads"]["reads_per_s"]["median"] / res["two_calls"]["reads_per_s"]["median"], 3)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--callers", type=int, default=32, help="config-2 caller threads, one 1 000-read batch each")
    ap.add_argument("--config3-reads", type=int, default=8, help="reads per config-3 batch (4 callers)")
    ap.add_argument("--threads", type=int, default=16, help="host threads that simulate the reads")
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    name, power = gpu_identity()
    res = dict(gpu=name, power_limit=power, host_cores=len(os.sched_getaffinity(0)))
    ctx = gpu.Context(0)
    log(f"{name}, power limit {power}")
    # config 2: 10 Mbp uniform reference, q = 12, 5 kbp reads at 5 % (recursive trees, leaf errors 2), distinct reads per caller
    c = W.CONFIGS["config2"]
    refs = [W.random_reference(c["ref_lens"][0], c["ref_seed"])]
    batches = [W.make_reads_seeded(refs, c["reads"], c["read_len"], c["error"], c["read_seed"] + i, gpu.pex_build, W._NoAnchors(), threads=a.threads)
               for i in range(a.callers)]
    log("config 2 reads made")
    res["config2"] = run_config(ctx, refs, 12, batches, a.reps)
    # config 3: 100 Mbp repeat-seeded reference, 15 kbp reads at 8 %: q = 8 or the largest q every leaf admits
    c = W.CONFIGS["config3"]
    refs, _ = W.build_references("config3")
    _, leaves = gpu.pex_build(c["read_len"], synthetic.ceil_eps(c["read_len"] * c["error"]), 2, 0)
    m = leaves["query_index_to"] - leaves["query_index_from"] + 1
    q3 = int(min(8, (m // (leaves["num_errors"] + 1)).min()))
    batches = [W.make_reads_seeded(refs, a.config3_reads, c["read_len"], c["error"], c["read_seed"] + i, gpu.pex_build, W._NoAnchors(), threads=a.threads)
               for i in range(4)]
    log("config 3 references and reads made")
    res["config3_sample"] = run_config(ctx, refs, q3, batches, max(2, a.reps // 2 + 1))
    ctx.close()
    line = json.dumps(res)
    with open(os.path.join(a.out, "seed_verify_bench.json"), "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
