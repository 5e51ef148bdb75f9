"""Command line: map a FASTQ file against a FASTA reference on one GPU and write BAM, SAM or BGZF-compressed SAM.

    python -m floxer_b200.map --reference ref.fa --queries reads.fq[.gz] --output out.bam --error-probability 0.05

It takes floxer's flags (include/floxer_cli.hpp) and two of its own: --q, the q-gram length of the device seeder that
stands in for floxer's FM-index search, and --batch-reads, the number of FASTQ records per call of Context.map_fastq.
The reference is read on the host and kept on the GPU; the FASTQ is streamed in chunks of whole records, each parsed,
seeded, verified and written on the device.  The output file is what one map_fastq call over the whole FASTQ writes:
the header comes with the first chunk only and, for BGZF outputs, the chunks' end-of-file blocks are dropped and one
is written at the end.  A read whose PEX leaves the q-gram seeder refuses (fewer than q * (errors + 1) bases, or more
than 8 errors) is counted as unseedable and not written.
"""
from __future__ import annotations

import argparse
import gzip
import sys

import numpy as np

from .batch import ReadConfig, VerifyConfig

BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")

# input::internal::chars_to_rank_sequence (src/lib/input.cpp:165-176): '$' -> 0, ACGT in either case -> 1..4, else 5
RANKS = np.full(256, 5, dtype=np.uint8)
RANKS[ord("$")] = 0
for _i, _c in enumerate("ACGT"):
    RANKS[ord(_c)] = RANKS[ord(_c.lower())] = _i + 1


def output_format(path: str) -> str:
    """The format an output path asks for: "bam", "sam" or "sam.gz"."""
    for suffix, fmt in ((".sam.gz", "sam.gz"), (".bam", "bam"), (".sam", "sam")):
        if path.endswith(suffix):
            return fmt
    raise ValueError(f"{path}: the output must end in .bam, .sam or .sam.gz")


def _open(path: str):
    return gzip.open(path, "rb") if path.endswith(".gz") else open(path, "rb")


def read_fasta(path: str):
    """[(id, ranks)] of a FASTA file (plain or .gz): the id is the header up to the first whitespace, the sequence lines
    are joined and turned into ranks."""
    out, name, parts = [], None, []

    def flush():
        if name is not None:
            seq = b"".join(parts).translate(None, b" \t\r\n")
            out.append((name, RANKS[np.frombuffer(seq, dtype=np.uint8)] if seq else np.zeros(0, np.uint8)))

    with _open(path) as f:
        for line in f:
            if line.startswith(b">"):
                flush()
                head = line[1:].split(None, 1)
                name, parts = (head[0] if head else b"").decode(), []
            elif name is not None:
                parts.append(line)
    flush()
    return out


def fastq_chunks(stream, batch_reads: int, block: int = 1 << 24):
    """Chunks of whole FASTQ records (4 * batch_reads lines each; the last one may be shorter) from a binary stream.
    Chunks are cut by counting newlines, so a quality line that starts with '@' cannot move a cut."""
    want = 4 * batch_reads
    buf, n, pos = bytearray(), 0, 0         # n: newlines in buf[:pos]
    eof = False
    while not eof:
        data = stream.read(block)
        eof = not data
        buf += data
        while True:
            while n < want:
                at = buf.find(b"\n", pos)
                if at < 0:
                    break
                n, pos = n + 1, at + 1
            if n < want:
                break
            yield bytes(buf[:pos])
            del buf[:pos]
            n = pos = 0
    if buf:
        yield bytes(buf)


def configs_from_args(args):
    """(ReadConfig, VerifyConfig, seeding keywords) of parsed command-line arguments."""
    rc = ReadConfig(error_probability=args.error_probability if args.error_probability is not None else 0.0,
                    query_errors=args.query_errors, seed_errors=args.seed_errors,
                    bottom_up=args.pex_tree_build_strategy == "bottom-up")
    vc = VerifyConfig(verification_kind=0 if args.direct_full_verification else 1,
                      interval_optimization=args.interval_optimization,
                      extra_verification_ratio=args.extra_verification_ratio, without_cigar=args.without_cigar)
    seeding = dict(max_anchors_hard=args.max_anchors_hard, max_anchors_soft=args.max_anchors_soft)
    return rc, vc, seeding


def parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser(prog="python -m floxer_b200.map", description=__doc__.split("\n\n")[0])
    p.add_argument("--reference", required=True, help="FASTA file (plain or .gz)")
    p.add_argument("--queries", required=True, help="FASTQ file (plain or .gz), four lines per record")
    p.add_argument("--output", required=True, help=".bam, .sam or .sam.gz (BGZF-compressed SAM)")
    errors = p.add_mutually_exclusive_group(required=True)
    errors.add_argument("--query-errors", type=int, help="errors allowed in every read")
    errors.add_argument("--error-probability", type=float, help="errors allowed per base: k = ceil(m * p)")
    p.add_argument("--seed-errors", type=int, default=2, help="errors allowed in a PEX leaf (default 2)")
    p.add_argument("--pex-tree-build-strategy", choices=["recursive", "bottom-up"], default="recursive")
    p.add_argument("--max-anchors-hard", type=int, default=500, help="a seed with more raw anchors is dropped (default 500)")
    p.add_argument("--max-anchors-soft", type=int, default=50, help="anchors kept per seed, fewest errors first (default 50)")
    p.add_argument("--extra-verification-ratio", type=float, default=0.05)
    p.add_argument("--interval-optimization", action="store_true")
    p.add_argument("--direct-full-verification", action="store_true")
    p.add_argument("--without-cigar", action="store_true")
    p.add_argument("--device", type=int, default=0, help="CUDA device")
    p.add_argument("--q", type=int, default=10, help="q-gram length of the device seeder (4..14, default 10)")
    p.add_argument("--batch-reads", type=int, default=20000, help="FASTQ records per device call (default 20000)")
    return p


def main(argv=None) -> int:
    args = parser().parse_args(argv)
    fmt = output_format(args.output)
    if args.batch_reads < 1:
        raise SystemExit("--batch-reads must be at least 1")
    from . import gpu
    read_config, verify_config, seeding = configs_from_args(args)
    refs = read_fasta(args.reference)
    ids, ranks = [r[0] for r in refs], [r[1] for r in refs]
    ctx = gpu.Context(args.device)
    ctx.set_references(ranks)
    seeder = gpu.GpuSeeder(ctx, args.q)
    lengths = [len(r) for r in ranks]
    total = {"records": 0, "kept": 0, "too_few_errors": 0, "bad_length": 0, "unseedable": 0, "alignments": 0}
    first = True
    try:
        with _open(args.queries) as queries, open(args.output, "wb") as out:
            chunks = fastq_chunks(queries, args.batch_reads)
            for text in _at_least_one(chunks):
                data, summary = ctx.map_fastq(seeder, text, read_config, verify_config, ids, lengths, fmt=fmt, header=first, **seeding)
                if fmt != "sam":
                    assert data.endswith(BGZF_EOF)
                    data = data[:-len(BGZF_EOF)]
                out.write(data)
                first = False
                for k in total:
                    total[k] += summary[k]
            if fmt != "sam":
                out.write(BGZF_EOF)
    finally:
        seeder.close()
        ctx.close()
    print(" ".join(f"{k}={v}" for k, v in total.items()))
    return 0


def _at_least_one(chunks):
    """The chunks, or one empty text when there are none (an empty FASTQ still gets its header)."""
    any_chunk = False
    for c in chunks:
        any_chunk = True
        yield c
    if not any_chunk:
        yield b""


if __name__ == "__main__":
    sys.exit(main())
