"""Reads per second and PCIe bytes per read of two ways to map a FASTQ text on the config-2 and config-3 shapes:

  map_fastq   Context.map_fastq: the text goes up once, parsing, seeding, verification and BAM output on the device;
  composed    the FASTQ parsed on the host (ranks, reverse complements, PEX trees), then Context.seed_verify_reads and
              Job.bam(on_device=True): the pools go up for seeding and the forward pool, names and qualities again for
              the writer.

Both paths write the same BAM records (checked on the inflated streams).  Repetitions alternate between the paths; the
medians are printed with the GPU's name and power limit.  Copies are fxg_counters h2d_bytes + d2h_bytes.

    python scripts/map_bench.py [--reps 3] [--config3-reads 1000]
"""
from __future__ import annotations

import argparse
import gzip
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from floxer_b200 import abi, gpu, synthetic  # noqa: E402
from floxer_b200.batch import BatchBuilder, ReadConfig, VerifyConfig  # noqa: E402
from floxer_b200.map import RANKS  # noqa: E402

LETTERS = np.frombuffer(b"$ACGTN", dtype=np.uint8)


def gpu_name_and_power() -> tuple[str, str]:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return out[0], out[1]
    except Exception:                                      # noqa: BLE001
        return "unknown", "unknown"


def dataset(config: int, n_reads: int):
    if config == 2:
        refs = [synthetic.random_reference(10_000_000, 20240001)]
        base_len, rate, seed = 5000, 0.05, 20240001
    else:
        refs = [synthetic.plant_repeats(synthetic.random_reference(100_000_000, 20240002), 20240002, 2000)]
        base_len, rate, seed = 15000, 0.08, 20240003
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n_reads):
        start = int(rng.integers(0, len(refs[0]) - base_len - 1))
        seq, _, _ = synthetic.simulate_read(rng, refs[0], start, base_len, int(rate * base_len))
        seq = synthetic.reverse_complement(seq) if i % 2 else seq
        qual = rng.integers(33, 75, size=len(seq)).astype(np.uint8)
        out.append(b"@read%d\n%s\n+\n%s\n" % (i, bytes(LETTERS[seq]), bytes(qual)))
    return refs, b"".join(out), rate


def host_parse(text: bytes, rc: ReadConfig):
    """The composed path's host parser (four-line records, all kept): the batch, ids and qualities."""
    lines = text.split(b"\n")
    bb, ids, quals = BatchBuilder(), [], []
    for r in range(len(lines) // 4):
        head, seq, qual = lines[4 * r], lines[4 * r + 1], lines[4 * r + 3]
        fwd = RANKS[np.frombuffer(seq, dtype=np.uint8)]
        k = synthetic.ceil_eps(len(fwd) * rc.error_probability)
        inner, leaves = gpu.pex_build(len(fwd), k, rc.seed_errors, int(rc.bottom_up))
        bb.add(fwd, synthetic.reverse_complement(fwd), inner, leaves, np.zeros(0, abi.ANCHOR_DTYPE), np.zeros(0, abi.ANCHOR_DTYPE))
        ids.append(head[1:].split()[0].decode())
        quals.append(qual.decode())
    return bb.build(), ids, quals


def copies(ctx) -> int:
    c = ctx.counters()
    return int(c["h2d_bytes"] + c["d2h_bytes"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--config2-reads", type=int, default=1000)
    ap.add_argument("--config3-reads", type=int, default=1000)
    args = ap.parse_args()
    name, power = gpu_name_and_power()
    ctx = gpu.Context(0)
    for config, n in ((2, args.config2_reads), (3, args.config3_reads)):
        refs, text, rate = dataset(config, n)
        ctx.set_references(refs)
        seeder = gpu.GpuSeeder(ctx, 10)
        ids_ref, lens = ["ref"], [len(refs[0])]
        rc, vc = ReadConfig(error_probability=rate, seed_errors=2), VerifyConfig()

        def one_call():
            return ctx.map_fastq(seeder, text, rc, vc, ids_ref, lens, fmt="bam")[0]

        def composed():
            batch, ids, quals = host_parse(text, rc)
            job, seeded, _ = ctx.seed_verify_reads(seeder, batch, vc)
            try:
                return job.bam(seeded, ids_ref, lens, ids, quals, on_device=True)
            finally:
                job.free()
        paths = {"map_fastq": one_call, "composed": composed}
        outputs = {k: f() for k, f in paths.items()}                 # warm-up, and the outputs compared
        assert gzip.decompress(outputs["map_fastq"]) == gzip.decompress(outputs["composed"]), "the two paths differ"
        times, moved = {k: [] for k in paths}, {}
        for _ in range(args.reps):
            for k, f in paths.items():
                ctx.reset_counters()
                t0 = time.perf_counter()
                f()
                times[k].append(time.perf_counter() - t0)
                moved[k] = copies(ctx)
        for k in paths:
            sec = float(np.median(times[k]))
            print(json.dumps({"config": config, "path": k, "reads": n, "text_bytes": len(text), "median_s": round(sec, 4),
                              "min_s": round(min(times[k]), 4), "max_s": round(max(times[k]), 4), "reads_per_s": round(n / sec, 1),
                              "pcie_bytes_per_read": round(moved[k] / n, 1), "gpu": name, "power_limit": power}))
        seeder.close()
    ctx.close()


if __name__ == "__main__":
    main()
