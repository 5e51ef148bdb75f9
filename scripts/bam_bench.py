"""BAM output on the host (fxg_write_bam) against BAM output on the device (fxg_write_bam_device), on a config-2 job.

One 1 000-read config-2 batch is seeded and verified on the device (fxg_seed_verify_reads); its alignments get random
Phred 2..40 qualities.  The two writers then turn the job's output into a BAM image in alternating repetitions, and
every device image is checked against the host image of the same repetition (same block count, ISIZE and CRC32 per
block, equal inflated payloads).  Host clocks around calls that return after their device work.  Reported per writer:
ms per 1 000-read batch with its spread, raw MB/s (uncompressed BAM bytes over the call time); and the compressed size
as a share of the raw stream and of zlib level 1 / level 6 over the same 0xff00-byte chunks (plus the same BGZF
framing).  Prints one JSON line and writes it to OUT/bam_bench.json.

    python scripts/bam_bench.py --out DIR [--reps 10]
"""
from __future__ import annotations

import argparse
import json
import os
import struct
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from floxer_b200 import gpu, workloads as W  # noqa: E402
from floxer_b200.batch import VerifyConfig  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from seed_verify_bench import gpu_identity, log, spread  # noqa: E402


def blocks(image: bytes):
    """(ISIZE, CRC32, inflated payload) per BGZF block."""
    out, at = [], 0
    while at < len(image):
        size = struct.unpack_from("<H", image, at + 16)[0] + 1
        crc, isize = struct.unpack_from("<II", image, at + size - 8)
        out.append((isize, crc, zlib.decompress(image[at + 18:at + size - 8], -15)))
        at += size
    assert at == len(image)
    return out


def zlib_size(raw: bytes, level: int) -> int:
    total = 28
    for at in range(0, len(raw), 0xff00):
        z = zlib.compressobj(level, zlib.DEFLATED, -15)
        total += len(z.compress(raw[at:at + 0xff00]) + z.flush()) + 26
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--threads", type=int, default=16, help="host threads that simulate the reads")
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    name, power = gpu_identity()
    ctx = gpu.Context(0)
    log(f"{name}, power limit {power}")
    c = W.CONFIGS["config2"]
    refs = [W.random_reference(c["ref_lens"][0], c["ref_seed"])]
    ctx.set_references(refs)
    dev = gpu.GpuSeeder(ctx, 12)
    batch = W.make_reads_seeded(refs, c["reads"], c["read_len"], c["error"], c["read_seed"], gpu.pex_build, W._NoAnchors(), threads=a.threads)
    job, seeded, _ = ctx.seed_verify_reads(dev, batch, VerifyConfig())
    al, cg = job.alignments()
    rng = np.random.default_rng(11)
    ids = [f"read_{i}" for i in range(len(seeded.reads))]
    quals = ["".join(chr(33 + int(x)) for x in rng.integers(2, 41, size=int(R["query_len"]))) for R in seeded.reads]
    args = (al, cg, seeded, ["chr"], [c["ref_lens"][0]], ids, quals)
    log(f"job: {len(seeded.reads)} reads, {len(al)} alignments, {len(cg)} CIGAR operations")
    writers = dict(host=lambda: gpu.write_bam(*args), device=lambda: ctx.write_bam(*args))
    for w in writers.values():                                 # warm-up: kernels loaded, buffers grown
        w()
    ms = {k: [] for k in writers}
    agree, images = True, {}
    for rep in range(a.reps):
        order = list(writers) if rep % 2 == 0 else list(writers)[::-1]
        for k in order:
            t0 = time.perf_counter()
            images[k] = writers[k]()
            ms[k].append((time.perf_counter() - t0) * 1e3)
        hb, db = blocks(images["host"]), blocks(images["device"])
        agree = agree and len(hb) == len(db) and all(x == y for x, y in zip(hb, db))
        log(f"rep {rep}: host {ms['host'][-1]:.1f} ms, device {ms['device'][-1]:.1f} ms")
    raw = b"".join(p for _, _, p in blocks(images["host"]))
    per_batch = 1000 / len(seeded.reads)
    res = dict(gpu=name, power_limit=power, host_cores=len(os.sched_getaffinity(0)), reads=len(seeded.reads), alignments=len(al),
               raw_bytes=len(raw), reps=a.reps, images_equal_every_rep=bool(agree))
    z1, z6 = zlib_size(raw, 1), zlib_size(raw, 6)
    for k in writers:
        med = spread(ms[k])["median"]
        res[k] = dict(ms_per_1000_reads=spread([round(x * per_batch, 2) for x in ms[k]]), raw_mb_per_s=round(len(raw) / med / 1e3, 1),
                      bytes=len(images[k]), share_of_raw=round(len(images[k]) / len(raw), 4),
                      share_of_zlib1=round(len(images[k]) / z1, 4), share_of_zlib6=round(len(images[k]) / z6, 4))
    res["speedup_device_over_host"] = round(spread(ms["host"])["median"] / spread(ms["device"])["median"], 1)
    job.free()
    dev.close()
    ctx.close()
    line = json.dumps(res)
    with open(os.path.join(a.out, "bam_bench.json"), "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
