"""Host-side containers for one batch of reads in the layout of include/floxer_gpu.h (fxg_read et al.)."""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from . import abi


@dataclass
class VerifyConfig:
    """pex::pex_verification_config (include/pex.hpp:47-53) + --without-cigar (include/floxer_cli.hpp:67)."""
    verification_kind: int = abi.KIND_HIERARCHICAL
    interval_optimization: bool = False          # include/floxer_cli.hpp:60, off by default
    extra_verification_ratio: float = 0.05       # include/floxer_cli.hpp:61
    without_cigar: bool = False

    def to_c(self) -> abi.VerifyConfig:
        return abi.VerifyConfig(float(self.extra_verification_ratio), int(self.verification_kind),
                                int(bool(self.interval_optimization)), int(bool(self.without_cigar)))


@dataclass
class ReadConfig:
    """How reads are taken from a FASTQ text (--query-errors / --error-probability, --seed-errors,
    --pex-tree-build-strategy): k is query_errors when given, else ceil(m * error_probability); a read with
    k < seed_errors is skipped (src/lib/input.cpp:26-34,114-129)."""
    error_probability: float = 0.05
    query_errors: int | None = None
    seed_errors: int = 2                         # include/floxer_cli.hpp, default 2
    bottom_up: bool = False                      # pex tree build strategy: recursive (0) or bottom_up (1)

    def to_c(self) -> abi.ReadConfig:
        qe = abi.NULL_ID if self.query_errors is None else int(self.query_errors)
        return abi.ReadConfig(float(self.error_probability), qe, int(self.seed_errors), int(bool(self.bottom_up)), 0)


@dataclass
class ReadBatch:
    reads: np.ndarray                     # abi.READ_DTYPE
    forward_pool: np.ndarray              # uint8 ranks
    reverse_pool: np.ndarray              # uint8 ranks, same offsets as forward_pool
    nodes: np.ndarray                     # abi.PEX_NODE_DTYPE
    anchors: np.ndarray                   # abi.ANCHOR_DTYPE
    meta: dict = field(default_factory=dict)

    def __post_init__(self):
        self.reads = np.ascontiguousarray(self.reads, dtype=abi.READ_DTYPE)
        self.forward_pool = np.ascontiguousarray(self.forward_pool, dtype=np.uint8)
        self.reverse_pool = np.ascontiguousarray(self.reverse_pool, dtype=np.uint8)
        self.nodes = np.ascontiguousarray(self.nodes, dtype=abi.PEX_NODE_DTYPE)
        self.anchors = np.ascontiguousarray(self.anchors, dtype=abi.ANCHOR_DTYPE)
        assert len(self.forward_pool) == len(self.reverse_pool)

    def __len__(self):
        return len(self.reads)

    def slice(self, lo: int, hi: int) -> "ReadBatch":
        """A batch holding reads [lo, hi) that shares the pools (offsets stay valid)."""
        return ReadBatch(self.reads[lo:hi].copy(), self.forward_pool, self.reverse_pool, self.nodes, self.anchors,
                         dict(self.meta))


class BatchBuilder:
    """Accumulates reads one by one: forward / reverse-complement ranks, tree, anchors per orientation."""

    def __init__(self):
        self._reads, self._fwd, self._rc, self._nodes, self._anchors = [], [], [], [], []
        self._q = self._n = self._a = 0

    def add(self, forward, reverse_complement, inner, leaves, anchors_forward, anchors_reverse):
        f = np.asarray(forward, dtype=np.uint8)
        r = np.asarray(reverse_complement, dtype=np.uint8)
        assert len(f) == len(r)
        inner = np.asarray(inner, dtype=abi.PEX_NODE_DTYPE)
        leaves = np.asarray(leaves, dtype=abi.PEX_NODE_DTYPE)
        af = np.asarray(anchors_forward, dtype=abi.ANCHOR_DTYPE).reshape(-1)
        ar = np.asarray(anchors_reverse, dtype=abi.ANCHOR_DTYPE).reshape(-1)
        self._reads.append((self._q, self._n, self._a, len(f), len(inner), len(leaves), len(af), len(ar), 0))
        self._fwd.append(f)
        self._rc.append(r)
        self._nodes += [inner, leaves]
        self._anchors += [af, ar]
        self._q += len(f)
        self._n += len(inner) + len(leaves)
        self._a += len(af) + len(ar)

    def build(self, **meta) -> ReadBatch:
        cat = lambda xs, dt: np.concatenate(xs).astype(dt, copy=False) if xs else np.zeros(0, dtype=dt)
        return ReadBatch(np.array(self._reads, dtype=abi.READ_DTYPE), cat(self._fwd, np.uint8), cat(self._rc, np.uint8),
                         cat(self._nodes, abi.PEX_NODE_DTYPE), cat(self._anchors, abi.ANCHOR_DTYPE), meta)


def alignment_records(alignments: np.ndarray, cigar_pool: np.ndarray):
    """[(read_index, reference_id, start_in_reference, num_errors, orientation, cigar_string)] in output order."""
    out = []
    for a in alignments:
        ops = cigar_pool[int(a["cigar_offset"]): int(a["cigar_offset"]) + int(a["cigar_len"])]
        out.append((int(a["read_index"]), int(a["reference_id"]), int(a["start_in_reference"]),
                    int(a["num_errors"]), int(a["orientation"]), abi.cigar_to_string(ops)))
    return out
