#!/usr/bin/env python
"""bench.py -- PEX hierarchical verification throughput (BASELINE.json metric) on N B200s of one node.

Headline workload: config 2 of BASELINE.json (10 Mbp random reference, 1 000 simulated 5 kbp reads at 5 % error, floxer
defaults) per GPU.  The library serves many callers at once and merges the jobs that wait into batches, so the bench
drives it the way floxer's thread pool would: `--lanes` host threads (default 32), each verifying the 1 000-read batch
over and over.  One STEP = one pass of every lane over its batch (lanes x 1 000 reads per GPU); the timed region is
exactly K steps, i.e. K back-to-back batches per lane.  Reads shard across ranks with no data-path collective (weak
scaling: every rank runs its own lanes on its own reads).

The one JSON line also carries, under "sub", the other configs of BASELINE.json on this GPU, each with its own
device-resident value, end-to-end value, CPU baseline and roofline: config 2 with --interval-optimization, config 3
(100 Mbp repeat-seeded reference, 10 k reads x 15 kbp at 8 %), a sample of one GPU's shard of config 4 (3.1 Gbp in 24
records, 20 kbp reads at 10 %; reads sharded over 8 GPUs) -- both settings of the interval optimisation each -- and the
config-5 microbenchmark (batched edit distance, 2^20 tasks per cell).  `--only config2` runs the headline alone.

  python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (CUDA path through the C ABI)
  python bench.py --impl reference [...]                         CPU arm: the multithreaded CPU port of the reference path
                                                                 (the reference binary cannot be built offline, DESIGN.md)
  python bench.py [...] --dump-outputs bench_outputs             also writes the headline's result of its last timed step
                                                                 as .npy files to that directory (dump_outputs); the inputs
                                                                 are seeded, so two builds compare file by file

Prints ONE JSON line on rank 0.  Runs from the tree as build() left it and writes nothing into it: the tree may be
read-only.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # no __pycache__ in the tree from a benchmark run

# the library asks for 32 hardware work queues when it is loaded (floxer_gpu.cu, fxg_on_load); torch may create the CUDA
# context before that, so the same default is set here, before torch is imported
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

import numpy as np  # noqa: E402

MYERS_INSTR_PER_WORD_STEP = 11          # SURVEY 8(d): minimal LOP3/IADD3/SHF sequence of one 32-cell word-step
ROUND1_ANCHORS = dict(seed_errors=2, decoy_fraction=0.25)       # the stand-in seeder of round 1 (kept for the headline's continuity)


def describe(name: str, ivopt: bool, n_reads: int, anchors: str) -> str:
    from floxer_b200 import workloads as W
    c = W.CONFIGS[name.replace("_seeded", "")]
    ref = f"{sum(c['ref_lens'])} bp in {len(c['ref_lens'])} record(s)" + (f", {c['families']} repeat families" if c.get("families") else ", uniform random")
    return (f"{name}: reference {ref}; {n_reads} simulated reads x {c['read_len']} bp at {int(c['error'] * 100)} % error per GPU; "
            f"recursive PEX tree, seed errors 2, hierarchical verification, interval optimization {'on' if ivopt else 'off'}, "
            f"extra verification ratio 0.05, CIGAR output; anchors: {anchors}")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed regions (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.windows = index, [], None, []

    def window(self, t0: float, t1: float):
        self.windows.append((t0, t1))

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self) -> dict:
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        inside = [r for t, r in self.rows if any(a <= t <= b + 0.1 for a, b in self.windows)]
        rows = inside if inside else [r for _, r in self.rows]
        sm = [float(r[0]) for r in rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------- workloads

def build_workload(name: str, rank: int, pex_build, n_reads: int | None, threads: int):
    """(references, batch, anchors description) of a named config for this rank."""
    from floxer_b200 import synthetic, workloads as W
    refs, table = W.build_references(name, threads=threads)
    if name == "config2":
        # the headline keeps round 1's read set and anchors (ground-truth anchors + 25 % random decoys per leaf)
        c = W.CONFIGS[name]
        batch = synthetic.make_batch(refs, n_reads or c["reads"], c["read_len"], c["error"], c["read_seed"] + 1000 * rank, pex_build, **ROUND1_ANCHORS)
        return refs, batch, "ground-truth stand-in seeder of round 1 (true loci at the origin position, 25 % random decoys per leaf)"
    batch = W.build_reads(name, refs, table, pex_build, n_reads=n_reads, rank=rank, procs=threads)
    return refs, batch, ("stand-in seeder (floxer_b200/workloads.py): true loci with position jitter, hits at the other copies of "
                         "overlapped repeats, Poisson false positives at the rate of a uniform text of the references' length, "
                         "hard cap 500 / soft cap 50 per seed")


def digest(al, cg, with_cigars: bool) -> int:
    """Order-sensitive checksum of a job's alignment records (and, if asked, of every cigar's operations)."""
    fields = np.stack([al["start_in_reference"].astype(np.uint64), al["num_errors"].astype(np.uint64), al["read_index"].astype(np.uint64),
                       al["reference_id"].astype(np.uint64), al["orientation"].astype(np.uint64), al["cigar_len"].astype(np.uint64)], axis=1)
    h = zlib.crc32(np.ascontiguousarray(fields).tobytes())
    if with_cigars and len(al):
        off = al["cigar_offset"].astype(np.int64)
        ln = al["cigar_len"].astype(np.int64)
        # weighted sums of every cigar's operations (shared cigars are read through every alignment that points at them)
        csum = np.concatenate([np.zeros(1, dtype=np.uint64), np.cumsum((cg.astype(np.uint64) * np.uint64(2654435761)) & np.uint64(0xffffffff), dtype=np.uint64)])
        per = csum[off + ln] - csum[off]
        h = zlib.crc32(per.tobytes(), h)
    return h


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(out_dir: str, al, cg, stats: dict):
    """Writes what one verification job hands its caller, so that two builds can be compared output for output:

      alignments.npy  float64 [n, 7]: alignment index, read_index, reference_id, orientation, start_in_reference,
                      num_errors, cigar_len -- in the job's output order
      cigars.npy      float32: the cigars of those alignments one after the other, every operation as count << 4 | code
                      (exact in float32: a count stays far below 2^20)
      stats.npy       float64 [8]: the job's statistics in abi.Stats order

    cigar_offset and the gaps of the cigar pool are layout, not result, and are left out.  Where the files would pass
    DUMP_LIMIT_BYTES, a fixed, seeded sample of the alignments (kept in output order) is written instead."""
    n = len(al)
    ln = al["cigar_len"].astype(np.int64)
    row_bytes = 7 * 8 + 4 * ln
    keep = np.arange(n)
    budget = DUMP_LIMIT_BYTES - 8 * 8 - 3 * 4096            # stats and the three .npy headers
    if int(row_bytes.sum()) > budget:
        order = np.random.default_rng(20240000).permutation(n)
        keep = np.sort(order[np.cumsum(row_bytes[order]) <= budget])
    sel, ln = al[keep], ln[keep]
    rows = np.stack([keep, sel["read_index"], sel["reference_id"], sel["orientation"], sel["start_in_reference"],
                     sel["num_errors"], ln], axis=1).astype(np.float64)
    first = np.cumsum(ln) - ln
    at = np.repeat(sel["cigar_offset"].astype(np.int64) - first, ln) + np.arange(int(ln.sum()))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "alignments.npy"), rows)
    np.save(os.path.join(out_dir, "cigars.npy"), cg[at].astype(np.float32))
    np.save(os.path.join(out_dir, "stats.npy"), np.array(list(stats.values()), dtype=np.float64))


def cpu_arm(refs, batch, cfg, threads: int, target_s: float):
    """Times the multithreaded CPU port on a bounded sample (first reads of the batch); returns a cpu_baseline object.
    A probe of one read per thread gives the rate; the sample is sized for about target_s seconds of wall time on all
    threads (the probe itself is the sample where it already took half of that: config 4 without the interval optimisation)."""
    from oracle import cpu_baseline
    n = min(len(batch), max(2, threads))
    sample = batch.slice(0, n)
    t0 = time.perf_counter()
    _, _, stats = cpu_baseline.verify_reads(refs, sample, cfg, threads=threads)
    dt = time.perf_counter() - t0
    if dt < 0.5 * target_s and n < len(batch):
        n = int(max(min(len(batch), n / max(dt, 1e-6) * target_s), n))
        sample = batch.slice(0, n)
        t0 = time.perf_counter()
        _, _, stats = cpu_baseline.verify_reads(refs, sample, cfg, threads=threads)
        dt = time.perf_counter() - t0
    cells = stats["cells_inner"] + stats["cells_root"]
    return {"value": cells / dt / 1e9, "unit": "GCUPS", "cores": threads, "kind": "port", "reads_per_s": n / dt,
            "sample": f"first {n} reads of the batch, all anchors, both strands, CIGARs ({dt:.1f} s on {threads} threads)"}


def run_lanes(step_fns, n_each: int):
    """Every lane (host thread) runs its step function n_each times; returns (wall seconds, per-lane completion times)."""
    errors = []
    done = [[0.0] * n_each for _ in step_fns]
    t0_box = [0.0]
    start = threading.Barrier(len(step_fns) + 1)

    def lane(i):
        try:
            start.wait()
            for s in range(n_each):
                step_fns[i]()
                done[i][s] = time.perf_counter() - t0_box[0]
        except Exception as e:                           # noqa: BLE001 -- re-raised by the main thread
            errors.append(e)
            try:
                start.abort()
            except Exception:                            # noqa: BLE001
                pass
    threads = [threading.Thread(target=lane, args=(i,)) for i in range(len(step_fns))]
    for t in threads:
        t.start()
    t0_box[0] = time.perf_counter()
    start.wait()
    for t in threads:
        t.join()
    dt = time.perf_counter() - t0_box[0]
    if errors:
        raise errors[0]
    return dt, done


def step_spread(done, n_each):
    """Per-step times: step s ends when the last lane has finished its s-th batch."""
    ends = [max(d[s] for d in done) for s in range(n_each)]
    per = [ends[0]] + [ends[s] - ends[s - 1] for s in range(1, n_each)]
    per_ms = sorted(x * 1e3 for x in per)
    return {"min": round(per_ms[0], 3), "median": round(per_ms[len(per_ms) // 2], 3), "max": round(per_ms[-1], 3)}


def measure(ctx, g, torch, dist, refs, batch, cfg, lanes: int, steps: int, warmup: int, int32_peak: float, sampler, pageable: bool,
            cpu_threads: int, cpu_target_s: float, rank: int, dump_dir: str | None = None):
    """Device-resident arm, end-to-end arm (page-locked inputs; pageable as well if asked), result check, roofline and CPU
    baseline of one workload.  Returns (record for rank 0, [ms_total, e2e_ms_total], [cells, reads]).  With dump_dir, rank 0
    writes the result of the device-resident arm's last timed step there (dump_outputs)."""
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- device-resident arm: one staged copy of the batch per lane, each step = fxg_verify_run ----
    jobs = [ctx.stage_verify(batch, cfg) for _ in range(lanes)]

    def resident_step(j):
        def f():
            flush.fill_(1)                               # 256 MiB written between steps (queued on torch's stream, no host sync)
            j.run()
        return f
    # warm-up: the W steps asked for, and on until two seconds have passed -- the queue's workers size their buffers for
    # the batches they meet, and the first batches of every size pay for that (page-locking memory takes tens of ms)
    def warm_up(step_fns, first: int, at_least_s: float, at_most_s: float = 10.0):
        # ... and on while the library still allocates (its counter of allocations moved during the last round), bounded
        t_warm = time.perf_counter()
        run_lanes(step_fns, first)
        calls = ctx.counters()["alloc_calls"]
        while True:
            spent = time.perf_counter() - t_warm
            if spent >= at_most_s:
                break
            run_lanes(step_fns, 2)
            now = ctx.counters()["alloc_calls"]
            if now == calls and time.perf_counter() - t_warm >= at_least_s:
                break
            calls = now
    warm_up([resident_step(j) for j in jobs], max(warmup, 3), 2.0)
    # one batch at a time first: its latency, and its device time between the run's first and last operation
    lat_ms = []
    for it in range(3):
        flush.fill_(it & 0xff)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        jobs[0].run()
        lat_ms.append((time.perf_counter() - t0) * 1e3)
    al0, cg0 = jobs[0].alignments()
    want = digest(al0, cg0, True)
    want_fields = digest(al0, cg0, False)
    stats = jobs[0].stats()
    n_alignments = len(al0)
    barrier()
    ctx.reset_counters()
    t_region = time.perf_counter()
    total_s, done = run_lanes([resident_step(j) for j in jobs], steps)
    barrier()
    sampler.window(t_region, time.perf_counter())
    ctr = ctx.counters()
    # every lane's last result is the staged batch's result
    bad = 0
    for j in jobs:
        a, c = j.alignments(copy=False)
        bad += digest(a, c, True) != want
    if bad:
        raise RuntimeError(f"{bad} of {lanes} lanes of the device-resident arm ended with results that differ from a batch run alone")
    if dump_dir and rank == 0:
        # every lane ran the same batch and, as checked above, ended with the same result: lane 0's stands for the step
        a, c = jobs[0].alignments(copy=False)
        dump_outputs(dump_dir, a, c, jobs[0].stats())
        del a, c
    spread = step_spread(done, steps)
    for j in jobs:
        j.free()

    # ---- end-to-end arm: host buffers in, alignments + CIGARs out, every step; every job's records are checked ----
    want_quick = (len(al0), int(al0["start_in_reference"].sum()), int(al0["num_errors"].sum()), int(al0["cigar_len"].sum()))

    def e2e_arm(b):
        mismatches = [0]
        last = [None] * lanes

        def e2e_step(i):
            def f():
                flush.fill_(2)
                j2 = ctx.verify_reads(b, cfg)            # host buffers in: H2D, all waves, tracebacks, D2H of alignments + CIGARs
                a2, c2 = j2.alignments(copy=False)       # what a C caller reads: the job's own result arrays
                # every job is checked where it costs microseconds (the interpreter lock serialises the lanes' Python code);
                # the last job of every lane is kept, and its records and cigars are compared in full after the region
                if (len(a2), int(a2["start_in_reference"].sum()), int(a2["num_errors"].sum()), int(a2["cigar_len"].sum())) != want_quick:
                    mismatches[0] += 1
                del a2, c2
                if last[i] is not None:
                    last[i].free()
                last[i] = j2
            return f

        def check_and_free():
            for i, j2 in enumerate(last):
                if j2 is not None:
                    a2, c2 = j2.alignments(copy=False)
                    if digest(a2, c2, True) != want:
                        mismatches[0] += 1
                    del a2, c2
                    j2.free()
                    last[i] = None
        warm_up([e2e_step(i) for i in range(lanes)], 3, 1.0)     # (page-locked pools are allocated once)
        check_and_free()
        barrier()
        ctx.reset_counters()
        t_reg = time.perf_counter()
        s, d = run_lanes([e2e_step(i) for i in range(lanes)], steps)
        barrier()
        sampler.window(t_reg, time.perf_counter())
        check_and_free()
        if mismatches[0]:
            raise RuntimeError(f"{mismatches[0]} end-to-end jobs returned records that differ from the staged batch's")
        return s, ctx.counters(), step_spread(d, steps)

    pinned = [torch.from_numpy(a).pin_memory() for a in (batch.forward_pool, batch.reverse_pool)]
    from floxer_b200.batch import ReadBatch
    pinned_batch = ReadBatch(batch.reads, pinned[0].numpy(), pinned[1].numpy(), batch.nodes, batch.anchors, dict(batch.meta))
    e2e_s, e2e_ctr, e2e_spread = e2e_arm(pinned_batch)
    pageable_s = None
    if pageable:
        pageable_s, _, _ = e2e_arm(batch)                # the caller's buffers as floxer has them: ordinary std::vector memory

    # max over ranks of the times, sum of the units
    t = torch.tensor([total_s, e2e_s, pageable_s or 0.0, ctr["alloc_ms"], e2e_ctr["alloc_ms"]], dtype=torch.float64, device="cuda")
    cells_batch = stats["cells_inner"] + stats["cells_root"]
    u = torch.tensor([cells_batch * lanes, len(batch) * lanes], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(u, op=dist.ReduceOp.SUM)
    total_s, e2e_s, pageable_s, alloc_ms_worst, e2e_alloc_ms_worst = [float(x) for x in t.cpu()]
    cells_step, reads_step = [float(x) for x in u.cpu()]
    if rank != 0:
        return None
    ms_per_step = total_s * 1e3 / steps
    e2e_ms = e2e_s * 1e3 / steps
    n_batches = lanes * steps
    # roofline of the dominant kernel (the bit-vector DP engine, integer-ALU bound, SURVEY 8d) over the TIMED REGION of
    # the device-resident arm: every word-step the engine's launches issued in it x 11 instructions / the region's time.
    ws_region = ctr["dp_word_steps"]
    achieved = ws_region * MYERS_INSTR_PER_WORD_STEP / total_s
    rec = {
        "value": cells_step / (ms_per_step * 1e-3) / 1e9, "unit": "GCUPS", "reads_per_s": reads_step / (ms_per_step * 1e-3),
        "ms_per_step": ms_per_step, "ms_per_batch": ms_per_step / lanes, "step_ms_spread": spread,
        "lanes": lanes, "reads_per_step_per_gpu": len(batch) * lanes,
        "e2e": {"value": cells_step / (e2e_ms * 1e-3) / 1e9, "unit": "GCUPS", "reads_per_s": reads_step / (e2e_ms * 1e-3), "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": e2e_ctr["h2d_bytes"] // steps, "d2h_bytes_per_step": e2e_ctr["d2h_bytes"] // steps,
                "step_ms_spread": e2e_spread, "inputs": "page-locked host memory",
                "checked": f"every one of the {n_batches} timed jobs: number of alignments and the sums of their positions, errors and cigar lengths against the "
                           f"staged batch's; the last job of every lane: checksum of every record and every cigar's operations"},
        "gpu_launches": int(ctr["kernel_launches"]),
        "roofline": {
            "bound": "int32_alu", "achieved": achieved / 1e9, "peak": int32_peak / 1e9, "unit": "Ginstr/s",
            "frac": achieved / int32_peak if int32_peak else None,
            "traffic": (_captured_traffic() or {}).get("bytes_per_launch"),
            "traffic_source": _captured_traffic(),
            "hbm_view": _hbm_view(ctr, n_batches, total_s),
            "kernel": "fxg::dp_kernel<W, CKPT> -- every launch of the engine in the timed region (inner tree levels and root level)",
            "how": "algorithmic 11 int32 instructions per 32-cell word-step x the word-steps the engine's launches issued inside the timed "
                   "region of the device-resident arm (band-limited; counted per task from the band geometry, on the device for the inner "
                   "levels) / the wall time of that region (barrier + synchronize on both sides, so launches that overlap are not counted "
                   "twice); peak = LOP3/IADD3/SHF 8:1:2 issue-rate microbenchmark on this GPU in this run.  Everything else of a step "
                   "(tree-level kernels, tracebacks, copies, host scheduling) is inside the denominator.",
            "word_steps_per_batch": ws_region / n_batches,
            "cells_computed_per_batch": ws_region * 32 / n_batches, "cells_full_matrix_per_batch": cells_batch,
            "launch_event_ms_per_batch": {"engine_waves": ctr["dp_kernel_ms"] / n_batches, "tracebacks": ctr["trace_kernel_ms"] / n_batches,
                                          "root_launch": ctr["root_launch_ms"] / n_batches,
                                          "note": "CUDA-event times on the launching streams, summed over workers; launches of different batches overlap"},
            # the dominant launch (the root level's largest class, a checkpointed score pass) with its own CUDA-event pair on its
            # stream, measured live in the timed region: algorithmic instructions per launch / its average duration
            "dominant_launch": {
                "kernel": "fxg::dp_kernel<W, true> -- the root level's largest launch of every batch",
                "launches": int(ctr["root_launches"]),
                "ms_per_launch": ctr["root_launch_ms"] / max(ctr["root_launches"], 1),
                "word_steps_per_launch": ctr["root_launch_word_steps"] / max(ctr["root_launches"], 1),
                "achieved": (ctr["root_launch_word_steps"] * MYERS_INSTR_PER_WORD_STEP / (ctr["root_launch_ms"] * 1e-3) / 1e9) if ctr["root_launch_ms"] > 0 else None,
                "frac": (ctr["root_launch_word_steps"] * MYERS_INSTR_PER_WORD_STEP / (ctr["root_launch_ms"] * 1e-3) / int32_peak)
                if int32_peak and ctr["root_launch_ms"] > 0 else None,
                "note": "launches of other batches run beside it: its duration includes what it waits for them"},
            "checkpoint_bytes_per_batch": ctr["trace_bytes"] / n_batches},
        "queue": {"batches": int(ctr["batches"]), "jobs": int(ctr["batch_jobs"]), "jobs_per_batch": ctr["batch_jobs"] / max(ctr["batches"], 1),
                  "launches_per_job": ctr["kernel_launches"] / max(ctr["batch_jobs"], 1),
                  "alloc_ms_in_region": ctr["alloc_ms"], "alloc_calls_in_region": int(ctr["alloc_calls"]),
                  "alloc_ms_in_region_worst_rank": alloc_ms_worst, "alloc_ms_in_e2e_region_worst_rank": e2e_alloc_ms_worst},
        "shortcuts_per_batch": {k: ctr[k] / n_batches for k in ("shared_score_passes", "rescored_roots", "inferred_inner", "shared_tracebacks")},
        "batch_latency_alone_ms": [round(x, 3) for x in lat_ms],
        "alignments_per_batch": n_alignments, "stats_per_batch": stats,
    }
    if pageable_s:
        pms = pageable_s * 1e3 / steps
        rec["e2e_pageable"] = {"value": cells_step / (pms * 1e-3) / 1e9, "unit": "GCUPS", "reads_per_s": reads_step / (pms * 1e-3), "ms_per_step": pms,
                               "inputs": "ordinary (pageable) host memory, as floxer's std::vector pools"}
    rec["cpu_baseline"] = cpu_arm(refs, batch, cfg, cpu_threads, cpu_target_s)
    return rec


def _hbm_view(ctr, n_batches, region_s):
    """The same path seen from HBM: the bytes the engine's checkpoint records take in the timed region (counter trace_bytes:
    the dominant algorithmic traffic, written once and read by the tracebacks) over the region's wall time, and the captured
    launch's DRAM bytes over its duration, against the measured copy bandwidth -- far from the bound, which is why the
    roofline above is the integer issue rate."""
    peak = _measured_peak("hbm_gbs") or 6500.0           # fallback: the recipe's B200 copy bandwidth
    cap = _captured_traffic() or {}
    out = {"peak_gbs": peak, "peak_source": "MEASURED_PEAKS.json" if _measured_peak("hbm_gbs") else "fallback of B200_PROFILING.md",
           "region_checkpoint_gbs": ctr["trace_bytes"] / region_s / 1e9 if region_s > 0 else None}
    if out["region_checkpoint_gbs"] is not None:
        out["region_frac"] = out["region_checkpoint_gbs"] / peak
    if cap.get("bytes_per_launch") and cap.get("launch_ms_under_ncu"):
        out["captured_launch_gbs"] = cap["bytes_per_launch"] / (cap["launch_ms_under_ncu"] * 1e-3) / 1e9
        out["captured_launch_frac"] = out["captured_launch_gbs"] / peak
    return out


def _captured_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the engine's dominant launch, from the committed
    `ncu --set full` capture summary of this round (profiles/r02_traffic.json); null when there is none."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            return json.load(f)
    except (OSError, ValueError):
        return None


def microbench(ctx, g, torch, int32_peak: float, cpu_threads: int, tasks_per_cell: int, distinct: int, cells=None):
    """Config 5: batched edit distance, query 100..2000 bp x window m + 2k + 1, error 2..15 %, modes exists and CIGAR."""
    from floxer_b200 import abi, synthetic
    from oracle import cpu_baseline
    ref = synthetic.random_reference(10_000_000, 20240006)
    ctx.set_references([ref])
    out = []
    for m in (100, 200, 500, 1000, 2000):
        for e in (0.02, 0.05, 0.10, 0.15):
            if cells and (m, e) not in cells:
                continue
            base, pool = synthetic.microbench_tasks(ref, [m], [e], distinct, 20240006 + m + int(e * 100), abi.MODE_EXISTS)
            reps = max(1, tasks_per_cell // distinct)
            row = {"m": m, "error": e, "k": int(base["max_errors"][0]), "tasks": len(base) * reps}
            for mode, key in ((abi.MODE_EXISTS, "exists"), (abi.MODE_CIGAR, "cigar")):
                tasks = np.tile(base, reps)
                tasks["mode"] = mode
                b = ctx.stage_align_batch(tasks, pool)
                b.run()
                ctx.reset_counters()
                t0 = time.perf_counter()
                b.run()
                dt = time.perf_counter() - t0
                c = ctx.counters()
                cells_full = float((tasks["ref_len"].astype(np.float64) * tasks["query_len"]).sum())
                res, cig = b.fetch()
                b.free()
                # parity of the distinct tasks with the CPU port, and its speed on the same
                one = base.copy()
                one["mode"] = mode
                t0 = time.perf_counter()
                cres, ccig = cpu_baseline.align_batch([ref], one, pool, threads=cpu_threads)
                cdt = time.perf_counter() - t0
                same = bool((res["exists"][:distinct] == cres["exists"]).all() and (res["num_errors"][:distinct] == cres["num_errors"]).all()
                            and (res["start_in_reference"][:distinct] == cres["start_in_reference"]).all())
                if not same:
                    raise RuntimeError(f"config 5 cell m={m} e={e} mode={key}: results differ from the CPU port")
                dev_s = (c["dp_kernel_ms"] + c["trace_kernel_ms"]) * 1e-3
                row[key] = {"gcups": cells_full / dt / 1e9, "tasks_per_s": len(tasks) / dt, "ms": dt * 1e3,
                            "roofline_frac": c["dp_word_steps"] * MYERS_INSTR_PER_WORD_STEP / dt / int32_peak if int32_peak else None,
                            # the same over the CUDA-event time of the call's kernels (the wall time of a call with a million small
                            # tasks is mostly the host's: one pass, one sort key and one 32-byte result record per task)
                            "device_ms": dev_s * 1e3, "gcups_device": cells_full / dev_s / 1e9 if dev_s > 0 else None,
                            "roofline_frac_device": c["dp_word_steps"] * MYERS_INSTR_PER_WORD_STEP / dev_s / int32_peak if int32_peak and dev_s > 0 else None,
                            "cpu_gcups": float((one["ref_len"].astype(np.float64) * one["query_len"]).sum()) / cdt / 1e9}
            out.append(row)
    return {"workload": f"config5: batched edit distance against a 10 Mbp random reference, {tasks_per_cell} tasks per cell ({distinct} distinct "
                        f"query/window pairs, repeated), 50 % positives; wall time of one fxg_align_batch_run on staged inputs",
            "cells": out, "cpu_cores": cpu_threads,
            "parity": "results of the distinct tasks of every cell equal the CPU port's (exists, errors, start)"}


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--only", default="", help="comma-separated subset of: config2,config2_ivopt,config2_seeded,config3,config4_shard,config5")
    ap.add_argument("--lanes", type=int, default=32, help="host threads that submit batches concurrently (config 2)")
    ap.add_argument("--config3-reads", type=int, default=10_000)
    ap.add_argument("--config4-reads", type=int, default=2_500, help="reads of the 12 500-read shard that are generated and verified")
    ap.add_argument("--cpu-seconds", type=float, default=2.0, help="wall time of every CPU baseline sample on all host threads (about 30 core-seconds on 16 cores)")
    ap.add_argument("--big-lanes", type=int, default=4, help="host threads that submit batches concurrently (configs 3 and 4: one batch fills the machine; "
                    "the others keep it fed while a caller stages its next batch -- measured 2 -> 4: config-4 shard end to end 18 k -> 25 k reads/s)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline's result of its last timed step (with --impl reference: the CPU port's) to "
                         "DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    threads = max(1, len(os.sched_getaffinity(0)) // max(local_world, 1)) if args.impl == "ours" else (os.cpu_count() or 1)
    only = set(x for x in args.only.split(",") if x)
    want = lambda name: not only or name in only

    from floxer_b200.batch import VerifyConfig

    # ------------------------------------------------------------------ CPU arm ("reference")
    if args.impl == "reference":
        if rank != 0:
            return 0
        from oracle import cpu_baseline, oracle
        threads = os.cpu_count() or 1
        cfg = VerifyConfig()
        refs, batch, anchors = build_workload("config2", 0, oracle.pex_build, None, threads)
        # every step is a sample of the workload sized so that the K steps together take two to three minutes
        probe = batch.slice(0, max(4, threads // 2))
        t0 = time.perf_counter()
        cpu_baseline.verify_reads(refs, probe, cfg, threads=threads)
        rate = len(probe) / max(time.perf_counter() - t0, 1e-6)
        n_sample = int(max(min(len(batch), rate * min(10.0, max(0.3, 150.0 / max(args.steps, 1)))), min(len(batch), threads)))
        sample = batch.slice(0, n_sample)
        times, stats = [], None
        for _ in range(max(args.steps, 1)):
            t0 = time.perf_counter()
            al, cg, stats = cpu_baseline.verify_reads(refs, sample, cfg, threads=threads)
            times.append(time.perf_counter() - t0)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, al, cg, stats)
        sec = sum(times) / len(times)
        gcups = (stats["cells_inner"] + stats["cells_root"]) / sec / 1e9
        line = {"impl": "reference", "metric": "pex_verification_gcups", "value": gcups, "unit": "GCUPS",
                "reads_per_s": n_sample / sec, "n_gpus": args.gpus, "steps": len(times), "warmup": args.warmup,
                "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u64", "data": "synthetic",
                "config": {"workload": describe("config2", False, len(batch), anchors), "lanes": args.lanes},
                "cpu_baseline": {"value": gcups, "unit": "GCUPS", "cores": threads, "kind": "port", "reads_per_s": n_sample / sec,
                                 "sample": f"first {n_sample} reads of the workload per step, all anchors, both strands, CIGARs"},
                "e2e": {"value": gcups, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": "CPU port of floxer 0.2.0 + SeqAn3 edit-distance path (oracle/cpu_baseline.c) on all host cores; the reference "
                        "binary cannot be built offline (DESIGN.md section 2)"}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm
    # all inputs first: the read generator forks worker processes, and CUDA must not be up by then
    from floxer_b200 import build
    from floxer_b200 import gpu as g
    build.build_native()
    t_gen = time.perf_counter()
    made = {}
    if want("config2") or want("config2_ivopt"):
        made["config2"] = build_workload("config2", rank, g.pex_build, None, threads)
    if want("config2_seeded"):
        # the same reference and read model, anchors from the q-gram seeder (row N2) instead of the ground truth
        from floxer_b200 import workloads as W
        refs2 = made["config2"][0] if "config2" in made else W.build_references("config2", threads=threads)[0]
        seeder = g.Seeder(refs2, q=12)
        c2 = W.CONFIGS["config2"]
        made["config2_seeded"] = (refs2, W.make_reads_seeded(refs2, c2["reads"], c2["read_len"], c2["error"], c2["read_seed"] + 1000 * rank, g.pex_build, seeder,
                                                             threads=threads),
                                  "q-gram seeder (floxer_b200/csrc/seeder.cpp): every position where a leaf matches within its error budget, both "
                                  "orientations, hard cap 500 / soft cap 50, erase_useless_anchors")
        seeder.close()
    if want("config3"):
        made["config3"] = build_workload("config3", rank, g.pex_build, args.config3_reads, threads)
    if want("config4_shard"):
        made["config4_shard"] = build_workload("config4_shard", rank, g.pex_build, args.config4_reads, threads)
    gen_s = time.perf_counter() - t_gen

    import torch
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the product path has no CPU fallback"}))
        return 1
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL announces its version on stdout when it initialises: keep stdout for the one JSON line
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    ctx = g.Context(local_rank)
    sampler = ClockSampler(local_rank)
    if rank == 0 and os.environ.get("BENCH_NO_SAMPLER") != "1":      # rank 0 reports its GPU's clocks (one nvidia-smi, not one per rank)
        sampler.start()
    head, sub = None, {}
    int32_peak = None
    plan = [("config2", False, args.lanes, args.steps, True), ("config2", True, args.lanes, args.steps, False),
            ("config2_seeded", False, args.lanes, max(3, args.steps // 2), False),
            ("config3", False, args.big_lanes, max(3, args.steps // 4), False), ("config3", True, args.big_lanes, max(3, args.steps // 4), False),
            ("config4_shard", False, args.big_lanes, max(3, args.steps // 5), False), ("config4_shard", True, args.big_lanes, max(3, args.steps // 5), False)]
    current, measured = None, False
    for name, ivopt, lanes, steps, is_head in plan:
        key = name + ("_ivopt" if ivopt else "")
        if name not in made or not (want(key) or (ivopt and want(name) and name != "config2")):
            continue
        refs, batch, anchors = made[name]
        if current != name:
            ctx.set_references(refs)
            current = name
            if int32_peak is None:
                int32_peak = ctx.measure_int32_peak()
        cfg = VerifyConfig(interval_optimization=ivopt, without_cigar=os.environ.get("BENCH_WITHOUT_CIGAR") == "1")      # (development: the path without tracebacks)
        # the first workload measured is the headline, or what stands in for it under --only
        rec = measure(ctx, g, torch, dist, refs, batch, cfg, lanes, steps, args.warmup, int32_peak, sampler, pageable=is_head,
                      cpu_threads=threads, cpu_target_s=args.cpu_seconds, rank=rank, dump_dir=None if measured else args.dump_outputs)
        measured = True
        if rec is not None:
            rec["config"] = {"workload": describe(name, ivopt, len(batch), anchors), "lanes": lanes, "steps": steps,
                             "l2": "256 MiB written to HBM between batches (twice the 126 MB L2); the lanes run concurrently, so a batch never finds its own data in L2"}
            if is_head:
                head = rec
            else:
                sub[key] = rec
    if want("config5") and rank == 0:
        if int32_peak is None:
            ctx.set_references([np.ones(64, dtype=np.uint8)])
            int32_peak = ctx.measure_int32_peak()
        sub["config5"] = microbench(ctx, g, torch, int32_peak, threads, 1 << 20, 1 << 12)
    clocks = sampler.stop()
    line = None
    if rank == 0:
        if head is None:                                 # --only without the headline: the first record stands in
            key = next(iter(sub))
            head = sub.pop(key)
        cfg_obj = head.pop("config")
        line = {"metric": "pex_verification_gcups", "value": head.pop("value"), "unit": "GCUPS", "reads_per_s": head.pop("reads_per_s"),
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": head.pop("ms_per_step"),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
                "config": cfg_obj,
                "clocks": {"sm_mhz": clocks["sm_mhz"], "sm_max_mhz": clocks["sm_max_mhz"], "reasons": clocks["reasons"]},
                "e2e": head.pop("e2e"), "gpu_launches": head.pop("gpu_launches"), "roofline": head.pop("roofline"),
                "cpu_baseline": head.pop("cpu_baseline")}
        line.update(head)
        line["host_cores"] = len(os.sched_getaffinity(0))
        line["generation_s"] = round(gen_s, 1)
        line["sub"] = sub
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()
    return 0


def _measured_peak(key: str):
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f).get(key)
    except (OSError, ValueError):
        return None


if __name__ == "__main__":
    sys.exit(main())
