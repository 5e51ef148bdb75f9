"""ctypes / numpy mirrors of the structs declared in include/floxer_gpu.h (layouts must stay identical)."""
from __future__ import annotations

import ctypes as C

import numpy as np

NULL_ID = 2**64 - 1
REF_INLINE = 2**32 - 1
MAX_RANK = 5

MODE_EXISTS, MODE_NO_CIGAR, MODE_CIGAR = 0, 1, 2
FORWARD, REVERSE_COMPLEMENT = 0, 1
KIND_DIRECT_FULL, KIND_HIERARCHICAL = 0, 1
CIGAR_CHARS = {1: "I", 2: "D", 7: "=", 8: "X"}

OK, ERR_INVALID_ARGUMENT, ERR_CUDA, ERR_OUT_OF_MEMORY, ERR_OVERFLOW, ERR_STATE = 0, -1, -2, -3, -4, -5

PEX_NODE_DTYPE = np.dtype([("parent_id", "<u8"), ("query_index_from", "<u8"),
                           ("query_index_to", "<u8"), ("num_errors", "<u8")])
ANCHOR_DTYPE = np.dtype([("pex_leaf_index", "<u8"), ("reference_id", "<u8"),
                         ("reference_position", "<u8"), ("num_errors", "<u8")])
ALIGN_TASK_DTYPE = np.dtype([("ref_offset", "<u8"), ("reference_span_offset", "<u8"), ("query_offset", "<u8"),
                             ("ref_len", "<u4"), ("query_len", "<u4"), ("ref_id", "<u4"), ("max_errors", "<u4"),
                             ("mode", "u1"), ("orientation", "u1"), ("reserved", "u1", (6,))])
ALIGN_RESULT_DTYPE = np.dtype([("start_in_reference", "<u8"), ("cigar_offset", "<u8"), ("cigar_len", "<u4"),
                               ("num_errors", "<u4"), ("exists", "u1"), ("orientation", "u1"),
                               ("reserved", "u1", (6,))])
READ_DTYPE = np.dtype([("query_offset", "<u8"), ("node_offset", "<u8"), ("anchor_offset", "<u8"),
                       ("query_len", "<u4"), ("num_inner", "<u4"), ("num_leaves", "<u4"),
                       ("num_anchors_forward", "<u4"), ("num_anchors_reverse", "<u4"), ("reserved", "<u4")])
ALIGNMENT_DTYPE = np.dtype([("start_in_reference", "<u8"), ("cigar_offset", "<u8"), ("cigar_len", "<u4"),
                            ("num_errors", "<u4"), ("read_index", "<u4"), ("reference_id", "<u4"),
                            ("orientation", "u1"), ("reserved", "u1", (7,))])

assert ALIGN_TASK_DTYPE.itemsize == 48 and ALIGN_RESULT_DTYPE.itemsize == 32
assert READ_DTYPE.itemsize == 48 and ALIGNMENT_DTYPE.itemsize == 40


class VerifyConfig(C.Structure):
    _fields_ = [("extra_verification_ratio", C.c_double), ("verification_kind", C.c_uint8),
                ("interval_optimization", C.c_uint8), ("without_cigar", C.c_uint8), ("reserved", C.c_uint8 * 5)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "n_aligned_inner", "sum_aligned_inner", "n_aligned_root", "sum_aligned_root",
        "n_avoided_root", "sum_avoided_root", "cells_inner", "cells_root")]

    def as_dict(self) -> dict:
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class Counters(C.Structure):
    _fields_ = [("kernel_launches", C.c_uint64), ("dp_tasks", C.c_uint64), ("dp_word_steps", C.c_uint64),
                ("dp_cells_full", C.c_uint64), ("trace_bytes", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("dp_kernel_ms", C.c_double), ("trace_kernel_ms", C.c_double), ("waves", C.c_uint64),
                ("run_ms", C.c_double), ("trace_word_steps", C.c_uint64),
                ("root_launch_ms", C.c_double), ("root_launch_word_steps", C.c_uint64), ("shared_tracebacks", C.c_uint64), ("inferred_inner", C.c_uint64),
                ("shared_score_passes", C.c_uint64), ("rescored_roots", C.c_uint64),
                ("batches", C.c_uint64), ("batch_jobs", C.c_uint64), ("alloc_ms", C.c_double), ("alloc_calls", C.c_uint64), ("root_launches", C.c_uint64)]

    def as_dict(self) -> dict:
        return {n: getattr(self, n) for n, _ in self._fields_}


class SeedStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "seeds", "candidates", "checked", "hits", "dropped_hard", "cut_soft", "erased", "reserved")]

    def as_dict(self) -> dict:
        return {n: int(getattr(self, n)) for n, _ in self._fields_ if n != "reserved"}


def cigar_to_string(ops) -> str:
    return "".join(f"{int(o) >> 4}{CIGAR_CHARS[int(o) & 15]}" for o in ops)


def ptr(a: np.ndarray, ctype=C.c_void_p):
    return a.ctypes.data_as(ctype) if ctype is not C.c_void_p else C.c_void_p(a.ctypes.data)
