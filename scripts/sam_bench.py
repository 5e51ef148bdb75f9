"""SAM output on the host (fxg_write_sam) against SAM output on the device (fxg_write_sam_device, as text and as its BGZF
image), on a config-2 job.

One 1 000-read config-2 batch is seeded and verified on the device (fxg_seed_verify_reads); its alignments get random
Phred 2..40 qualities.  The three writers then turn the job's output into SAM in alternating repetitions, and every
repetition checks the device text against the host text and the inflated BGZF image (block by block: ISIZE, CRC32,
payload) against the host text.  Host clocks around calls that return after their device work.  Reported per writer:
ms per 1 000-read batch with its spread and text MB/s (SAM text bytes over the call time); for the BGZF image also its
size as a share of the text and of zlib level 1 / level 6 over the same 0xff00-byte chunks (plus the same BGZF framing).
Prints one JSON line and writes it to OUT/sam_bench.json.

    python scripts/sam_bench.py --out DIR [--reps 10]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from floxer_b200 import gpu, workloads as W  # noqa: E402
from floxer_b200.batch import VerifyConfig  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bam_bench import blocks, zlib_size  # noqa: E402
from seed_verify_bench import gpu_identity, log, spread  # noqa: E402


def image_holds(image: bytes, text: bytes) -> bool:
    """The BGZF image is the text cut at 0xff00-byte boundaries (one block per chunk) plus the end-of-file block."""
    chunks = [text[at:at + 0xff00] for at in range(0, len(text), 0xff00)] + [b""]
    got = blocks(image)
    return len(got) == len(chunks) and all(isize == len(c) and crc == zlib.crc32(c) and payload == c
                                           for (isize, crc, payload), c in zip(got, chunks))


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
    writers = dict(host=lambda: gpu.write_sam(*args), device_text=lambda: ctx.write_sam(*args),
                   device_bgzf=lambda: ctx.write_sam(*args, bgzf=True))
    for w in writers.values():                                 # warm-up: kernels loaded, buffers grown
        w()
    ms = {k: [] for k in writers}
    agree, out = True, {}
    for rep in range(a.reps):
        order = list(writers) if rep % 2 == 0 else list(writers)[::-1]
        for k in order:
            t0 = time.perf_counter()
            out[k] = writers[k]()
            ms[k].append((time.perf_counter() - t0) * 1e3)
        text = out["host"].encode()
        agree = agree and out["device_text"] == out["host"] and image_holds(out["device_bgzf"], text)
        log(f"rep {rep}: " + ", ".join(f"{k} {ms[k][-1]:.1f} ms" for k in writers))
    text = out["host"].encode()
    per_batch = 1000 / len(seeded.reads)
    res = dict(gpu=name, power_limit=power, host_cores=len(os.sched_getaffinity(0)), reads=len(seeded.reads), alignments=len(al),
               text_bytes=len(text), reps=a.reps, images_equal_every_rep=bool(agree))
    for k in writers:
        med = spread(ms[k])["median"]
        res[k] = dict(ms_per_1000_reads=spread([round(x * per_batch, 2) for x in ms[k]]), text_mb_per_s=round(len(text) / med / 1e3, 1))
    image = out["device_bgzf"]
    z1, z6 = zlib_size(text, 1), zlib_size(text, 6)
    res["device_bgzf"].update(bytes=len(image), share_of_text=round(len(image) / len(text), 4), share_of_zlib1=round(len(image) / z1, 4),
                              share_of_zlib6=round(len(image) / z6, 4))
    res["speedup_device_text_over_host"] = round(spread(ms["host"])["median"] / spread(ms["device_text"])["median"], 1)
    res["speedup_device_bgzf_over_host"] = round(spread(ms["host"])["median"] / spread(ms["device_bgzf"])["median"], 1)
    job.free()
    dev.close()
    ctx.close()
    line = json.dumps(res)
    with open(os.path.join(a.out, "sam_bench.json"), "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
