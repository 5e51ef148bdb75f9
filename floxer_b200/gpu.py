"""ctypes binding of the C ABI in include/floxer_gpu.h (floxer_b200/libfloxer_gpu.so).

This is the only way the Python side reaches the GPU path; there is no CPU fallback.  Loading fails
loudly when the library has not been built (run `python __graft_entry__.py` or floxer_b200.build)."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import abi
from .batch import ReadBatch, VerifyConfig

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfloxer_gpu.so")

EXPORTS = [
    "fxg_create", "fxg_destroy", "fxg_last_error", "fxg_version", "fxg_set_references",
    "fxg_align_batch", "fxg_align_batch_stage", "fxg_align_batch_run", "fxg_align_batch_fetch", "fxg_batch_free",
    "fxg_verify_stage", "fxg_verify_run", "fxg_job_num_alignments", "fxg_job_alignments", "fxg_job_cigar_len",
    "fxg_job_cigar_pool", "fxg_job_stats", "fxg_job_free", "fxg_verify_reads",
    "fxg_get_counters", "fxg_reset_counters", "fxg_measure_int32_peak", "fxg_engine_shape",
    "fxg_pex_build", "fxg_pex_free", "fxg_job_write_sam", "fxg_free", "fxg_write_bam", "fxg_job_write_bam",
    "fxg_seeder_create", "fxg_seeder_free", "fxg_seeder_search",
    "fxg_gpu_seeder_create", "fxg_gpu_seeder_free", "fxg_seed_reads", "fxg_seed_verify_reads",
    "fxg_write_bam_device", "fxg_job_write_bam_device", "fxg_write_sam", "fxg_write_sam_device", "fxg_job_write_sam_device",
]

_lib = None


class FloxerGpuError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"floxer_gpu error {code}: {message}")
        self.code = code


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: the CUDA library has not been built (no CPU fallback exists)")
    L = C.CDLL(LIB_PATH)
    vp, sz = C.c_void_p, C.c_size_t
    L.fxg_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.fxg_destroy.argtypes = [vp]
    L.fxg_destroy.restype = None
    L.fxg_last_error.argtypes = [vp]
    L.fxg_last_error.restype = C.c_char_p
    L.fxg_version.restype = C.c_char_p
    L.fxg_set_references.argtypes = [vp, sz, vp, vp]
    L.fxg_align_batch.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp, vp, sz, C.POINTER(sz)]
    L.fxg_align_batch_stage.argtypes = [vp, vp, sz, vp, sz, vp, sz, C.POINTER(vp)]
    L.fxg_align_batch_run.argtypes = [vp, vp]
    L.fxg_align_batch_fetch.argtypes = [vp, vp, vp, vp, sz, C.POINTER(sz)]
    L.fxg_batch_free.argtypes = [vp, vp]
    L.fxg_batch_free.restype = None
    L.fxg_verify_stage.argtypes = [vp, vp, vp, sz, vp, vp, sz, vp, sz, vp, sz, C.POINTER(vp)]
    L.fxg_verify_reads.argtypes = L.fxg_verify_stage.argtypes
    L.fxg_verify_run.argtypes = [vp, vp]
    L.fxg_job_num_alignments.argtypes = [vp]
    L.fxg_job_num_alignments.restype = sz
    L.fxg_job_alignments.argtypes = [vp]
    L.fxg_job_alignments.restype = vp
    L.fxg_job_cigar_len.argtypes = [vp]
    L.fxg_job_cigar_len.restype = sz
    L.fxg_job_cigar_pool.argtypes = [vp]
    L.fxg_job_cigar_pool.restype = vp
    L.fxg_job_stats.argtypes = [vp]
    L.fxg_job_stats.restype = C.POINTER(abi.Stats)
    L.fxg_job_free.argtypes = [vp, vp]
    L.fxg_job_free.restype = None
    L.fxg_get_counters.argtypes = [vp, C.POINTER(abi.Counters)]
    L.fxg_reset_counters.argtypes = [vp]
    L.fxg_measure_int32_peak.argtypes = [vp, C.POINTER(C.c_double)]
    L.fxg_engine_shape.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32),
                                   C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]
    L.fxg_pex_build.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.POINTER(vp), C.POINTER(sz),
                                C.POINTER(vp), C.POINTER(sz)]
    L.fxg_pex_free.argtypes = [vp]
    L.fxg_pex_free.restype = None
    L.fxg_job_write_sam.argtypes = [vp, sz, vp, vp, vp, sz, vp, vp, C.c_int, C.POINTER(vp), C.POINTER(sz)]
    L.fxg_free.argtypes = [vp]
    L.fxg_free.restype = None
    L.fxg_write_bam.argtypes = [vp, sz, vp, sz, vp, vp, vp, sz, vp, vp, C.c_int, C.POINTER(vp), C.POINTER(sz)]
    L.fxg_job_write_bam.argtypes = [vp, sz, vp, vp, vp, sz, vp, vp, C.c_int, C.POINTER(vp), C.POINTER(sz)]
    L.fxg_write_bam_device.argtypes = [vp, *L.fxg_write_bam.argtypes]
    L.fxg_job_write_bam_device.argtypes = [vp, *L.fxg_job_write_bam.argtypes]
    L.fxg_write_sam.argtypes = [vp, sz, vp, sz, vp, vp, vp, sz, vp, vp, C.c_int, C.POINTER(vp), C.POINTER(sz)]
    L.fxg_write_sam_device.argtypes = [vp, vp, sz, vp, sz, vp, vp, vp, sz, vp, vp, C.c_int, C.c_int, C.POINTER(vp), C.POINTER(sz)]
    L.fxg_job_write_sam_device.argtypes = [vp, vp, sz, vp, vp, vp, sz, vp, vp, C.c_int, C.c_int, C.POINTER(vp), C.POINTER(sz)]
    L.fxg_seeder_create.argtypes = [sz, vp, vp, C.c_uint32, C.POINTER(vp)]
    L.fxg_seeder_free.argtypes = [vp]
    L.fxg_seeder_free.restype = None
    L.fxg_seeder_search.argtypes = [vp, vp, sz, vp, sz, C.c_uint64, C.c_uint64, C.c_int, C.POINTER(vp), C.POINTER(sz)]
    L.fxg_gpu_seeder_create.argtypes = [vp, C.c_uint32, C.POINTER(vp)]
    L.fxg_gpu_seeder_free.argtypes = [vp, vp]
    L.fxg_gpu_seeder_free.restype = None
    L.fxg_seed_reads.argtypes = [vp, vp, vp, sz, vp, vp, sz, vp, sz, C.c_uint64, C.c_uint64, C.c_int, C.POINTER(vp), C.POINTER(sz),
                                 C.POINTER(abi.SeedStats)]
    L.fxg_seed_verify_reads.argtypes = [vp, vp, vp, vp, sz, vp, vp, sz, vp, sz, C.c_uint64, C.c_uint64, C.c_int,
                                        C.POINTER(abi.SeedStats), C.POINTER(vp)]
    _lib = L
    return L


class _SamQuery(C.Structure):
    _fields_ = [("id", C.c_char_p), ("quality", C.c_char_p)]


def _output_arguments(batch, reference_ids, reference_lengths, query_ids, qualities):
    n_ref, n = len(reference_ids), len(batch.reads)
    ref_ids = (C.c_char_p * max(n_ref, 1))(*[r.encode() for r in reference_ids])
    ref_lens = (C.c_uint64 * max(n_ref, 1))(*[int(x) for x in reference_lengths])
    qs = (_SamQuery * max(n, 1))()
    for i in range(n):
        qs[i].id = query_ids[i].encode()
        qs[i].quality = (qualities[i] if qualities is not None else "").encode()
    return n_ref, ref_ids, ref_lens, n, qs


def write_bam(alignments, cigars, batch, reference_ids, reference_lengths, query_ids, qualities=None, header: bool = True) -> bytes:
    """BAM file image (BGZF) of alignment records given as arrays (abi.ALIGNMENT_DTYPE, grouped by read in read order, and
    their cigar pool): fxg_write_bam, host only -- no context, no GPU."""
    L = lib()
    al = np.ascontiguousarray(alignments, dtype=abi.ALIGNMENT_DTYPE)
    cg = np.ascontiguousarray(cigars, dtype=np.uint32)
    n_ref, ref_ids, ref_lens, n, qs = _output_arguments(batch, reference_ids, reference_lengths, query_ids, qualities)
    out, length = C.c_void_p(), C.c_size_t(0)
    rc = L.fxg_write_bam(al.ctypes.data if len(al) else None, len(al), cg.ctypes.data if len(cg) else None, n_ref, ref_ids, ref_lens,
                         batch.reads.ctypes.data, n, batch.forward_pool.ctypes.data, qs, int(header), C.byref(out), C.byref(length))
    if rc != 0:
        raise FloxerGpuError(rc, "fxg_write_bam failed")
    try:
        return C.string_at(out, length.value)
    finally:
        L.fxg_free(out)


def write_sam(alignments, cigars, batch, reference_ids, reference_lengths, query_ids, qualities=None, header: bool = True) -> str:
    """SAM text of alignment records given as arrays (abi.ALIGNMENT_DTYPE, grouped by read in read order, and their cigar
    pool): fxg_write_sam, host only -- no context, no GPU."""
    L = lib()
    al = np.ascontiguousarray(alignments, dtype=abi.ALIGNMENT_DTYPE)
    cg = np.ascontiguousarray(cigars, dtype=np.uint32)
    n_ref, ref_ids, ref_lens, n, qs = _output_arguments(batch, reference_ids, reference_lengths, query_ids, qualities)
    out, length = C.c_void_p(), C.c_size_t(0)
    rc = L.fxg_write_sam(al.ctypes.data if len(al) else None, len(al), cg.ctypes.data if len(cg) else None, n_ref, ref_ids, ref_lens,
                         batch.reads.ctypes.data, n, batch.forward_pool.ctypes.data, qs, int(header), C.byref(out), C.byref(length))
    if rc != 0:
        raise FloxerGpuError(rc, "fxg_write_sam failed")
    try:
        return C.string_at(out, length.value).decode()
    finally:
        L.fxg_free(out)


def pex_build(total_len: int, num_errors: int, leaf_max_errors: int, strategy: int = 0):
    """pex::pex_tree construction (src/lib/pex.cpp:84-256) by the native host library.
    Returns (inner, leaves) as arrays of abi.PEX_NODE_DTYPE; inner[0] is the root."""
    L = lib()
    pi, pl = C.c_void_p(), C.c_void_p()
    ni, nl = C.c_size_t(0), C.c_size_t(0)
    rc = L.fxg_pex_build(total_len, num_errors, leaf_max_errors, strategy, C.byref(pi), C.byref(ni), C.byref(pl), C.byref(nl))
    if rc != 0:
        raise FloxerGpuError(rc, "pex tree construction failed")

    def grab(p, n):
        if n == 0:
            return np.zeros(0, dtype=abi.PEX_NODE_DTYPE)
        return np.frombuffer(C.string_at(p, n * abi.PEX_NODE_DTYPE.itemsize), dtype=abi.PEX_NODE_DTYPE).copy()
    inner, leaves = grab(pi, ni.value), grab(pl, nl.value)
    L.fxg_pex_free(pi)
    L.fxg_pex_free(pl)
    return inner, leaves


def engine_shape(n: int, m: int, k: int, with_traceback: bool = False):
    """(words per lane, lanes per ring, blocks, band-limited word-steps) the engine picks for one align call (with_traceback:
    a pass whose CIGAR is wanted); None when no alignment is possible.  Host arithmetic only (fxg_engine_shape)."""
    w, g, nb, ws = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0), C.c_uint64(0)
    rc = lib().fxg_engine_shape(n, m, k, int(with_traceback), C.byref(w), C.byref(g), C.byref(nb), C.byref(ws))
    return None if rc != 0 else (w.value, g.value, nb.value, ws.value)


class Seeder:
    """fxg_seeder: the q-gram seeder that stands in for search::searcher::search_seeds (host only)."""

    def __init__(self, references, q: int = 10):
        refs = [np.ascontiguousarray(r, dtype=np.uint8) for r in references]
        n = len(refs)
        ptrs = (C.c_void_p * max(n, 1))(*[r.ctypes.data for r in refs])
        lens = (C.c_uint64 * max(n, 1))(*[len(r) for r in refs])
        self._h = C.c_void_p()
        rc = lib().fxg_seeder_create(n, ptrs, lens, q, C.byref(self._h))
        if rc != 0:
            raise FloxerGpuError(rc, "fxg_seeder_create failed")

    def search(self, query, leaves, max_anchors_hard: int = 500, max_anchors_soft: int = 50, erase_useless: bool = True) -> np.ndarray:
        """Anchors (abi.ANCHOR_DTYPE) of one query orientation, in seed -> reference -> position order."""
        qy = np.ascontiguousarray(query, dtype=np.uint8)
        lv = np.ascontiguousarray(leaves, dtype=abi.PEX_NODE_DTYPE)
        out, n = C.c_void_p(), C.c_size_t(0)
        rc = lib().fxg_seeder_search(self._h, qy.ctypes.data, len(qy), lv.ctypes.data, len(lv), max_anchors_hard, max_anchors_soft,
                                     int(erase_useless), C.byref(out), C.byref(n))
        if rc != 0:
            raise FloxerGpuError(rc, "fxg_seeder_search failed (a leaf shorter than q * (errors + 1)?)")
        if n.value == 0:
            return np.zeros(0, dtype=abi.ANCHOR_DTYPE)
        try:
            return np.frombuffer(C.string_at(out, n.value * abi.ANCHOR_DTYPE.itemsize), dtype=abi.ANCHOR_DTYPE).copy()
        finally:
            lib().fxg_free(out)

    def close(self):
        if self._h:
            lib().fxg_seeder_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class GpuSeeder:
    """fxg_gpu_seeder: the q-gram index of the references resident in `ctx`, built on the device; Context.seed_reads
    searches whole read batches with it.  Invalid once ctx.set_references replaces the references."""

    def __init__(self, ctx: "Context", q: int = 10):
        self._ctx, self.q = ctx, q
        self._h = C.c_void_p()
        ctx._check(lib().fxg_gpu_seeder_create(ctx._h, q, C.byref(self._h)))

    def close(self):
        if self._h:
            lib().fxg_gpu_seeder_free(self._ctx._h, self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Job:
    """A staged fxg_verify_* job (inputs resident in HBM)."""

    def __init__(self, ctx: "Context", handle, keepalive):
        self._ctx, self._h, self._keep = ctx, handle, keepalive

    def run(self):
        self._ctx._check(lib().fxg_verify_run(self._ctx._h, self._h))
        return self

    def alignments(self, copy: bool = True):
        """(alignments[abi.ALIGNMENT_DTYPE], cigar_pool[uint32]).

        cigar_offset indexes cigar_pool; the pool may hold unused gaps between cigars.  With copy=False the arrays are
        views of the job's own (page-locked) memory -- what a C caller reads through fxg_job_alignments /
        fxg_job_cigar_pool -- and are valid until free()."""
        L = lib()
        n = L.fxg_job_num_alignments(self._h)
        nc = L.fxg_job_cigar_len(self._h)
        if n:
            buf = (C.c_char * (n * abi.ALIGNMENT_DTYPE.itemsize)).from_address(L.fxg_job_alignments(self._h))
            al = np.frombuffer(buf, dtype=abi.ALIGNMENT_DTYPE)
        else:
            al = np.empty(0, dtype=abi.ALIGNMENT_DTYPE)
        if nc:
            cg = np.frombuffer((C.c_uint32 * nc).from_address(L.fxg_job_cigar_pool(self._h)), dtype=np.uint32)
        else:
            cg = np.empty(0, dtype=np.uint32)
        return (al.copy(), cg.copy()) if copy else (al, cg)

    def stats(self) -> dict:
        return lib().fxg_job_stats(self._h).contents.as_dict()

    def sam(self, batch: ReadBatch, reference_ids, reference_lengths, query_ids, qualities=None, header: bool = True,
            on_device: bool = False, bgzf: bool = False):
        """SAM text of the job's alignments (output::alignment_output::write_alignments_for_query, src/lib/output.cpp:49-108):
        fxg_job_write_sam, or with on_device=True fxg_job_write_sam_device on the job's context (the same text, formatted on
        the GPU).  bgzf=True (device only) returns the BGZF-compressed text as bytes instead of a str."""
        L = lib()
        if bgzf and not on_device:
            raise ValueError("bgzf=True needs on_device=True")
        if on_device:
            n_ref, ref_ids, ref_lens, n, qs = _output_arguments(batch, reference_ids, reference_lengths, query_ids, qualities)
            out, length = C.c_void_p(), C.c_size_t(0)
            self._ctx._check(L.fxg_job_write_sam_device(self._ctx._h, self._h, n_ref, ref_ids, ref_lens, batch.reads.ctypes.data, n,
                                                        batch.forward_pool.ctypes.data, qs, int(header), int(bgzf), C.byref(out),
                                                        C.byref(length)))
            try:
                data = C.string_at(out, length.value)
            finally:
                L.fxg_free(out)
            return data if bgzf else data.decode()
        n_ref, n = len(reference_ids), len(batch.reads)
        ref_ids = (C.c_char_p * max(n_ref, 1))(*[r.encode() for r in reference_ids])
        ref_lens = (C.c_uint64 * max(n_ref, 1))(*[int(x) for x in reference_lengths])

        class SamQuery(C.Structure):
            _fields_ = [("id", C.c_char_p), ("quality", C.c_char_p)]
        qs = (SamQuery * max(n, 1))()
        for i in range(n):
            qs[i].id = query_ids[i].encode()
            qs[i].quality = (qualities[i] if qualities is not None else "").encode()
        text, length = C.c_void_p(), C.c_size_t(0)
        rc = L.fxg_job_write_sam(self._h, n_ref, ref_ids, ref_lens, batch.reads.ctypes.data, n, batch.forward_pool.ctypes.data,
                                 qs, int(header), C.byref(text), C.byref(length))
        if rc != 0:
            raise FloxerGpuError(rc, "fxg_job_write_sam failed")
        try:
            return C.string_at(text, length.value).decode()
        finally:
            L.fxg_free(text)

    def bam(self, batch: ReadBatch, reference_ids, reference_lengths, query_ids, qualities=None, header: bool = True,
            on_device: bool = False) -> bytes:
        """The same records as a BAM file image (BGZF blocks incl. the end-of-file block): fxg_job_write_bam, or with
        on_device=True fxg_job_write_bam_device on the job's context (the same records and blocks, compressed on the GPU)."""
        L = lib()
        n_ref, ref_ids, ref_lens, n, qs = _output_arguments(batch, reference_ids, reference_lengths, query_ids, qualities)
        out, length = C.c_void_p(), C.c_size_t(0)
        args = (self._h, n_ref, ref_ids, ref_lens, batch.reads.ctypes.data, n, batch.forward_pool.ctypes.data, qs, int(header),
                C.byref(out), C.byref(length))
        if on_device:
            self._ctx._check(L.fxg_job_write_bam_device(self._ctx._h, *args))
        else:
            rc = L.fxg_job_write_bam(*args)
            if rc != 0:
                raise FloxerGpuError(rc, "fxg_job_write_bam failed")
        try:
            return C.string_at(out, length.value)
        finally:
            L.fxg_free(out)

    def free(self):
        if self._h:
            lib().fxg_job_free(self._ctx._h, self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class AlignBatch:
    """A staged fxg_align_batch (inputs resident in HBM)."""

    def __init__(self, ctx: "Context", handle, tasks, keepalive):
        self._ctx, self._h, self._tasks, self._keep = ctx, handle, tasks, keepalive

    def run(self):
        self._ctx._check(lib().fxg_align_batch_run(self._ctx._h, self._h))
        return self

    def fetch(self, cigar_capacity: int | None = None):
        t = self._tasks
        if cigar_capacity is None:
            cig = t["mode"] == abi.MODE_CIGAR
            cigar_capacity = int((2 * t["max_errors"][cig].astype(np.int64) + 3).sum()) + 1
        res = np.zeros(len(t), dtype=abi.ALIGN_RESULT_DTYPE)
        pool = np.zeros(max(cigar_capacity, 1), dtype=np.uint32)
        used = C.c_size_t(0)
        self._ctx._check(lib().fxg_align_batch_fetch(self._ctx._h, self._h, res.ctypes.data, pool.ctypes.data,
                                                     cigar_capacity, C.byref(used)))
        return res, pool[: used.value]

    def free(self):
        if self._h:
            lib().fxg_batch_free(self._ctx._h, self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    """fxg_ctx: one CUDA device with the packed references resident in HBM."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        rc = lib().fxg_create(device, C.byref(self._h))
        if rc != 0:
            raise FloxerGpuError(rc, "fxg_create failed (no usable CUDA device?)")
        self._refs = None

    def close(self):
        if self._h:
            lib().fxg_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise FloxerGpuError(rc, lib().fxg_last_error(self._h).decode(errors="replace"))

    def set_references(self, references):
        refs = [np.ascontiguousarray(r, dtype=np.uint8) for r in references]
        n = len(refs)
        ptrs = (C.c_void_p * max(n, 1))(*[r.ctypes.data for r in refs])
        lens = (C.c_uint64 * max(n, 1))(*[len(r) for r in refs])
        self._check(lib().fxg_set_references(self._h, n, ptrs, lens))
        self._refs = refs

    # ---- alignment::align, batched ----
    def stage_align_batch(self, tasks, query_pool, inline_ref_pool=None) -> AlignBatch:
        tasks = np.ascontiguousarray(tasks, dtype=abi.ALIGN_TASK_DTYPE)
        qp = np.ascontiguousarray(query_pool, dtype=np.uint8)
        ip = np.ascontiguousarray(inline_ref_pool, dtype=np.uint8) if inline_ref_pool is not None else np.zeros(0, np.uint8)
        h = C.c_void_p()
        self._check(lib().fxg_align_batch_stage(self._h, tasks.ctypes.data, len(tasks), qp.ctypes.data, len(qp),
                                                ip.ctypes.data if len(ip) else None, len(ip), C.byref(h)))
        return AlignBatch(self, h, tasks, (qp, ip))

    def align_batch(self, tasks, query_pool, inline_ref_pool=None):
        """One call of fxg_align_batch with host buffers; returns (results, cigar_pool)."""
        tasks = np.ascontiguousarray(tasks, dtype=abi.ALIGN_TASK_DTYPE)
        qp = np.ascontiguousarray(query_pool, dtype=np.uint8)
        ip = np.ascontiguousarray(inline_ref_pool, dtype=np.uint8) if inline_ref_pool is not None else np.zeros(0, np.uint8)
        cig = tasks["mode"] == abi.MODE_CIGAR
        cap = int((2 * tasks["max_errors"][cig].astype(np.int64) + 3).sum()) + 1
        res = np.zeros(len(tasks), dtype=abi.ALIGN_RESULT_DTYPE)
        pool = np.zeros(cap, dtype=np.uint32)
        used = C.c_size_t(0)
        self._check(lib().fxg_align_batch(self._h, tasks.ctypes.data, len(tasks), qp.ctypes.data, len(qp),
                                          ip.ctypes.data if len(ip) else None, len(ip),
                                          res.ctypes.data, pool.ctypes.data, cap, C.byref(used)))
        return res, pool[: used.value]

    # ---- query_verifier::verify over whole reads ----
    def _verify_args(self, batch: ReadBatch, config: VerifyConfig):
        cfg = config.to_c()
        return cfg, [C.byref(cfg), batch.reads.ctypes.data, len(batch.reads), batch.forward_pool.ctypes.data,
                     batch.reverse_pool.ctypes.data, len(batch.forward_pool), batch.nodes.ctypes.data, len(batch.nodes),
                     batch.anchors.ctypes.data, len(batch.anchors)]

    def stage_verify(self, batch: ReadBatch, config: VerifyConfig) -> Job:
        cfg, args = self._verify_args(batch, config)
        h = C.c_void_p()
        self._check(lib().fxg_verify_stage(self._h, *args, C.byref(h)))
        return Job(self, h, (batch, cfg))

    def verify_reads(self, batch: ReadBatch, config: VerifyConfig) -> Job:
        cfg, args = self._verify_args(batch, config)
        h = C.c_void_p()
        self._check(lib().fxg_verify_reads(self._h, *args, C.byref(h)))
        return Job(self, h, (batch, cfg))

    # ---- seeding on the device ----
    def seed_reads(self, seeder: GpuSeeder, batch: ReadBatch, max_anchors_hard: int = 500, max_anchors_soft: int = 50,
                   erase_useless: bool = True):
        """fxg_seed_reads: both orientations of every read of `batch` (its pools, trees and read records; its anchors are
        ignored).  Returns (a new ReadBatch with the anchors and the updated read records, stats dict); `batch` is not
        modified.  The anchors of read i and orientation o equal Seeder.search(pool_o[i], leaves of i, ...)."""
        reads = batch.reads.copy()
        out, n, st = C.c_void_p(), C.c_size_t(0), abi.SeedStats()
        self._check(lib().fxg_seed_reads(self._h, seeder._h, reads.ctypes.data, len(reads), batch.forward_pool.ctypes.data,
                                         batch.reverse_pool.ctypes.data, len(batch.forward_pool), batch.nodes.ctypes.data,
                                         len(batch.nodes), max_anchors_hard, max_anchors_soft, int(erase_useless),
                                         C.byref(out), C.byref(n), C.byref(st)))
        if n.value:
            try:
                anchors = np.frombuffer(C.string_at(out, n.value * abi.ANCHOR_DTYPE.itemsize), dtype=abi.ANCHOR_DTYPE).copy()
            finally:
                lib().fxg_free(out)
        else:
            anchors = np.zeros(0, dtype=abi.ANCHOR_DTYPE)
        return ReadBatch(reads, batch.forward_pool, batch.reverse_pool, batch.nodes, anchors, dict(batch.meta)), st.as_dict()

    def seed_verify_reads(self, seeder: GpuSeeder, batch: ReadBatch, config: VerifyConfig, max_anchors_hard: int = 500,
                          max_anchors_soft: int = 50, erase_useless: bool = True):
        """fxg_seed_verify_reads: seed_reads then verify_reads in one call, the anchors kept in device memory.  Returns
        (Job, a new ReadBatch with the updated read records and no anchors -- what Job.sam / Job.bam take --, stats dict);
        `batch` is not modified.  The results equal those of verify_reads on seed_reads's batch."""
        reads = batch.reads.copy()
        cfg = config.to_c()
        h, st = C.c_void_p(), abi.SeedStats()
        self._check(lib().fxg_seed_verify_reads(self._h, seeder._h, C.byref(cfg), reads.ctypes.data, len(reads),
                                                batch.forward_pool.ctypes.data, batch.reverse_pool.ctypes.data,
                                                len(batch.forward_pool), batch.nodes.ctypes.data, len(batch.nodes),
                                                max_anchors_hard, max_anchors_soft, int(erase_useless), C.byref(st), C.byref(h)))
        seeded = ReadBatch(reads, batch.forward_pool, batch.reverse_pool, batch.nodes, np.zeros(0, dtype=abi.ANCHOR_DTYPE), dict(batch.meta))
        return Job(self, h, (seeded, cfg)), seeded, st.as_dict()

    # ---- BAM output on the device ----
    def write_bam(self, alignments, cigars, batch, reference_ids, reference_lengths, query_ids, qualities=None,
                  header: bool = True) -> bytes:
        """gpu.write_bam with the work on this context's device (fxg_write_bam_device): the same records and BGZF blocks,
        deflated on the GPU."""
        L = lib()
        al = np.ascontiguousarray(alignments, dtype=abi.ALIGNMENT_DTYPE)
        cg = np.ascontiguousarray(cigars, dtype=np.uint32)
        n_ref, ref_ids, ref_lens, n, qs = _output_arguments(batch, reference_ids, reference_lengths, query_ids, qualities)
        out, length = C.c_void_p(), C.c_size_t(0)
        self._check(L.fxg_write_bam_device(self._h, al.ctypes.data if len(al) else None, len(al), cg.ctypes.data if len(cg) else None,
                                           n_ref, ref_ids, ref_lens, batch.reads.ctypes.data, n, batch.forward_pool.ctypes.data, qs,
                                           int(header), C.byref(out), C.byref(length)))
        try:
            return C.string_at(out, length.value)
        finally:
            L.fxg_free(out)

    # ---- SAM output on the device ----
    def write_sam(self, alignments, cigars, batch, reference_ids, reference_lengths, query_ids, qualities=None,
                  header: bool = True, bgzf: bool = False):
        """gpu.write_sam with the work on this context's device (fxg_write_sam_device): the same text as a str, or with
        bgzf=True its BGZF image (.sam.gz) as bytes."""
        L = lib()
        al = np.ascontiguousarray(alignments, dtype=abi.ALIGNMENT_DTYPE)
        cg = np.ascontiguousarray(cigars, dtype=np.uint32)
        n_ref, ref_ids, ref_lens, n, qs = _output_arguments(batch, reference_ids, reference_lengths, query_ids, qualities)
        out, length = C.c_void_p(), C.c_size_t(0)
        self._check(L.fxg_write_sam_device(self._h, al.ctypes.data if len(al) else None, len(al), cg.ctypes.data if len(cg) else None,
                                           n_ref, ref_ids, ref_lens, batch.reads.ctypes.data, n, batch.forward_pool.ctypes.data, qs,
                                           int(header), int(bgzf), C.byref(out), C.byref(length)))
        try:
            data = C.string_at(out, length.value)
        finally:
            L.fxg_free(out)
        return data if bgzf else data.decode()

    # ---- accounting ----
    def counters(self) -> dict:
        ctr = abi.Counters()
        self._check(lib().fxg_get_counters(self._h, C.byref(ctr)))
        return ctr.as_dict()

    def reset_counters(self):
        self._check(lib().fxg_reset_counters(self._h))

    def measure_int32_peak(self) -> float:
        v = C.c_double(0)
        self._check(lib().fxg_measure_int32_peak(self._h, C.byref(v)))
        return float(v.value)
