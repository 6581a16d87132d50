"""hifir_b200 -- B200 (sm_100a) device backend for HIFIR's preconditioner-application hot path.

The product is the C-ABI shared library ``hifir_b200/_lib/libhifir_b200.so``
(``include/hifir_b200.h``), built from the hand-written CUDA in ``hifir_b200/csrc``.
This module is only the ctypes harness the Python tests / bench use to reach that
C-ABI; it contains no numerical code and NO fallback: if the library is missing
every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

__version__ = "0.1.0"

_HERE = os.path.dirname(os.path.abspath(__file__))
# HIFIR_B200_LIB: developer override (A/B of differently built libraries); the default is the in-tree build
LIB_PATH = os.environ.get("HIFIR_B200_LIB") or os.path.join(_HERE, "_lib", "libhifir_b200.so")

LHF_SUCCESS, LHF_NULL_OBJ, LHF_MISMATCHED_SIZES, LHF_BAD_PREC, LHF_HIFIR_ERROR = range(5)
LHF_S, LHF_SH, LHF_M, LHF_MH = range(4)
LHF_DEFAULT_RANK = -2
FULL_RANK = (1 << 64) - 1  # size_t(-1)

STAT_NAMES = ("levels", "n", "nnz", "dense_n", "dense_rank", "bytes_factors", "bytes_vec_per_rhs",
              "bytes_dense", "device_bytes", "kernels_per_apply", "depth_total", "launch_count", "depth_merged",
              "sweep_bytes", "sweep_entries")


class LhfdGpuCcs(C.Structure):
    _fields_ = [("nrows", C.c_size_t), ("ncols", C.c_size_t), ("col_start", C.c_void_p),
                ("row_ind", C.c_void_p), ("vals", C.c_void_p)]


class LhfdGpuLevel(C.Structure):
    _fields_ = [("m", C.c_size_t), ("n", C.c_size_t), ("L_B", LhfdGpuCcs), ("d_B", C.c_void_p),
                ("U_B", LhfdGpuCcs), ("E", LhfdGpuCcs), ("F", LhfdGpuCcs), ("s", C.c_void_p),
                ("t", C.c_void_p), ("p", C.c_void_p), ("p_inv", C.c_void_p), ("q", C.c_void_p),
                ("q_inv", C.c_void_p), ("dense_n", C.c_size_t), ("dense_rank", C.c_size_t),
                ("qr_mat", C.c_void_p), ("qr_tau", C.c_void_p), ("qr_jpvt", C.c_void_p),
                ("has_symm_dense", C.c_int)]


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None and a.size else None


def levels_dtype(levels):
    """float32 if the factor values of `levels` are single precision (hif::HIF<float>), else float64"""
    return np.dtype(np.float32) if np.asarray(levels[0]["s"]).dtype == np.float32 else np.dtype(np.float64)


def make_level_structs(levels, dtype=np.float64):
    """Describe per-level factors (list of dicts, the layout produced by the factor producer:
    CCS blocks 'L','U','E','F' = (nrows, ncols, col_start[int64], row_ind[int32], vals[f64]),
    'd','s','t','p','p_inv','q','q_inv', optional 'qr_mat','qr_tau','qr_jpvt','dense_n',
    'dense_rank') as a ctypes LhfdGpuLevel array (dtype=float32: LhfsGpuLevel, same field layout
    with float value arrays).  Returns (array, keepalive)."""
    arr = (LhfdGpuLevel * len(levels))()
    keep = []

    def ccs(block):
        nr, nc, cs, ri, va = block
        cs = np.ascontiguousarray(cs, dtype=np.int64)
        ri = np.ascontiguousarray(ri, dtype=np.int32)
        va = np.ascontiguousarray(va, dtype=dtype)
        keep.extend((cs, ri, va))
        return LhfdGpuCcs(nr, nc, _ptr(cs), _ptr(ri), _ptr(va))

    def vec(a, dt):
        a = np.ascontiguousarray(a, dtype=dtype if dt is np.float64 else dt)
        keep.append(a)
        return _ptr(a)

    for k, L in enumerate(levels):
        s = arr[k]
        s.m, s.n = L["m"], L["n"]
        s.L_B, s.U_B, s.E, s.F = ccs(L["L"]), ccs(L["U"]), ccs(L["E"]), ccs(L["F"])
        s.d_B = vec(L["d"], np.float64)
        s.s, s.t = vec(L["s"], np.float64), vec(L["t"], np.float64)
        for nm in ("p", "p_inv", "q", "q_inv"):
            setattr(s, nm, vec(L[nm], np.int32) if L.get(nm) is not None else None)
        s.dense_n = int(L.get("dense_n", 0))
        s.dense_rank = int(L.get("dense_rank", 0))
        if s.dense_n:
            s.qr_mat = vec(L["qr_mat"], np.float64)
            s.qr_tau = vec(L["qr_tau"], np.float64)
            s.qr_jpvt = vec(L["qr_jpvt"], np.int32)
        s.has_symm_dense = int(L.get("has_symm_dense", 0))
    return arr, keep


_lib = None


def lib():
    """The C-ABI library.  Raises if it has not been built -- there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'`"
                               " (the product has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        vp, sz, i, d = C.c_void_p, C.c_size_t, C.c_int, C.c_double
        sig = {
            "lhfdGpuAttachLevels": [i, sz, vp, vp],
            "lhfdGpuDestroy": [vp],
            "lhfdGpuSetMatrix": [vp, i, sz, vp, vp, vp],
            "lhfdGpuSetNspConst": [vp, sz, sz],
            "lhfdGpuSetNspTranConst": [vp, sz, sz],
            "lhfdGpuClearNsp": [vp],
            "lhfdGpuSetStream": [vp, vp, i],
            "lhfdGpuSynchronize": [vp],
            "lhfdGpuSolve": [vp, vp, vp],
            "lhfdGpuSolveAsync": [vp, vp, vp],
            "lhfdGpuApply": [vp, i, vp, i, vp, i, vp, vp],
            "lhfdGpuSolveMrhs": [vp, sz, vp, vp],
            "lhfdGpuFgmres": [vp, vp, i, d, i, i, vp, vp, vp, vp],
            "lhfdGpuGmres": [vp, vp, i, d, i, vp, vp, vp],
            "lhfdGpuFgmresMrhs": [vp, sz, vp, i, d, i, i, vp, vp, vp, vp],
            "lhfdGpuGmresMrhs": [vp, sz, vp, i, d, i, vp, vp, vp],
            "lhfdGpuApplyDev": [vp, i, vp, i, i, vp],
            "lhfdGpuSolveDev": [vp, vp, vp, sz],
            "lhfdGpuSolveMrhsDev": [vp, sz, vp, vp, sz],
            "lhfdGpuHifirDev": [vp, vp, sz, vp, sz],
            "lhfdGpuHifirMrhsDev": [vp, sz, vp, sz, vp, sz],
            "lhfdGpuSpmvDev": [vp, vp, vp],
            "lhfdGpuProfileSolveDev": [vp, vp, vp, sz, sz, vp, vp, vp, sz],
            "lhfdGpuDebugSweepHost": [vp, i, vp, vp, vp, vp, i],
            "lhfdGpuDebugSweepDev": [vp, i, sz, i, vp, vp, vp, vp, sz, vp, vp, vp],
            "lhfdGpuDebugPlanLab": [vp, i, vp, vp, vp],
            "lhfdGpuDebugMergePlan": [vp, i, vp],
            "lhfdGpuDebugExportInts": [vp, sz, i, vp, sz, vp],
            "lhfdGpuDebugTraceSweep": [vp, vp, vp, i, i, vp, sz, vp],
            "lhfdGpuDebugSegmentGraph": [vp, i, sz, sz, vp, vp, vp],
            "lhfdGpuDebugNorm2Dev": [vp, vp, sz, vp],
            "lhfdGpuGetStats": [vp, vp],
            "lhfdGpuGetDepths": [vp, sz, vp],
            "lhfsGpuAttachLevels": [i, sz, vp, vp],
            "lhfsGpuDestroy": [vp],
            "lhfsGpuSetMatrix": [vp, i, sz, vp, vp, vp],
            "lhfsdGpuUpdate": [vp, i, sz, vp, vp, vp],
            "lhfsGpuSolve": [vp, vp, vp],
            "lhfsGpuApply": [vp, i, vp, i, vp, i, vp, vp],
            "lhfsdGpuSolve": [vp, vp, vp],
            "lhfsdGpuApply": [vp, i, vp, i, vp, i, vp, vp],
            "lhfsGpuDebugSweepHost": [vp, i, vp, vp, vp, vp, i],
            "lhfdGpuSaveLevels": [sz, vp, i, C.c_char_p],
            "lhfsGpuSaveLevels": [sz, vp, i, C.c_char_p],
            "lhfdGpuAttachFile": [i, C.c_char_p, vp],
            "lhfsGpuAttachFile": [i, C.c_char_p, vp],
            "lhfGpuFileInfo": [C.c_char_p, vp],
            "lhfGpuDebugFileSweepHost": [C.c_char_p, sz, i, vp, vp, vp],
        }
        for name, argt in sig.items():
            f = getattr(L, name)
            f.argtypes = argt
            f.restype = C.c_int
        L.lhfsGpuAsDouble.argtypes = [vp]
        L.lhfsGpuAsDouble.restype = vp
        L.lhfGpuGetErrorMsg.restype = C.c_char_p
        L.lhfGpuVersion.restype = C.c_char_p
        _lib = L
    return _lib


EXPORTED_SYMBOLS = (
    "lhfdGpuAttachLevels", "lhfdGpuDestroy", "lhfdGpuSetMatrix", "lhfdGpuSetNspConst", "lhfdGpuSetNspTranConst", "lhfdGpuClearNsp",
    "lhfdGpuSetStream", "lhfdGpuSynchronize", "lhfdGpuSolve", "lhfdGpuSolveAsync", "lhfdGpuApply", "lhfdGpuSolveMrhs",
    "lhfdGpuFgmres", "lhfdGpuGmres", "lhfdGpuFgmresMrhs", "lhfdGpuGmresMrhs",
    "lhfdGpuApplyDev", "lhfdGpuSolveDev", "lhfdGpuSolveMrhsDev", "lhfdGpuHifirDev", "lhfdGpuHifirMrhsDev",
    "lhfdGpuSpmvDev", "lhfdGpuProfileSolveDev",
    "lhfdGpuGetStats", "lhfdGpuGetDepths", "lhfGpuGetErrorMsg", "lhfGpuVersion",
    "lhfsGpuAttachLevels", "lhfsGpuDestroy", "lhfsGpuAsDouble", "lhfsGpuSetMatrix", "lhfsdGpuUpdate", "lhfsGpuSolve",
    "lhfsGpuApply", "lhfsdGpuSolve", "lhfsdGpuApply",
    "lhfdGpuSaveLevels", "lhfsGpuSaveLevels", "lhfdGpuAttachFile", "lhfsGpuAttachFile", "lhfGpuFileInfo")
# developer / test hooks declared in hifir_b200/csrc/debug_api.h (not part of the drop-in boundary)
DEBUG_SYMBOLS = ("lhfdGpuDebugSweepHost", "lhfsGpuDebugSweepHost", "lhfGpuDebugFileSweepHost", "lhfdGpuDebugPlanLab",
                 "lhfdGpuDebugMergePlan",
                 "lhfdGpuDebugExportInts", "lhfdGpuDebugTraceSweep", "lhfdGpuDebugSegmentGraph",
                 "lhfdGpuDebugNorm2Dev", "lhfdGpuDebugSweepDev")


class LhfError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"LhfStatus {status}: {msg}")
        self.status = status


def _chk(st):
    if st != LHF_SUCCESS:
        raise LhfError(st, (lib().lhfGpuGetErrorMsg() or b"").decode())


def debug_sweep_host(block, upper, rhs, diag=None, parity=None):
    """Host-only hook (lhfdGpuDebugSweepHost): merge and pack the triangular CCS block as attach
    does and solve with the packed data on the CPU.  parity 0 / 1: every published value carries the
    device's readiness tag.  Returns (x, stats dict)."""
    nr, nc, cs, ri, va = block
    single = np.asarray(va).dtype == np.float32  # float block -> lhfsGpuDebugSweepHost (values stored as float)
    cs = np.ascontiguousarray(cs, dtype=np.int64)
    ri = np.ascontiguousarray(ri, dtype=np.int32)
    va = np.ascontiguousarray(va, dtype=np.float32 if single else np.float64)
    c = LhfdGpuCcs(nr, nc, _ptr(cs), _ptr(ri), _ptr(va))
    rhs = np.ascontiguousarray(rhs, dtype=np.float64)
    x = np.zeros_like(rhs)
    st = np.zeros(4, dtype=np.uint64)
    d = None if diag is None else np.ascontiguousarray(diag, dtype=np.float64)
    f = lib().lhfsGpuDebugSweepHost if single else lib().lhfdGpuDebugSweepHost
    _chk(f(C.byref(c), int(upper), _ptr(rhs), _ptr(d) if d is not None else None, _ptr(x), _ptr(st),
           -1 if parity is None else int(parity)))
    return x, dict(zip(("slices", "padded", "bytes", "depth"), (int(v) for v in st)))


MERGE_PLAN_KEYS = ("rows", "entries", "depth", "merged_rows", "merged_entries", "steps", "super_levels", "predicted_us")


def debug_merge_plan(block, upper):
    """Host-only hook (lhfdGpuDebugMergePlan): the attach-time merge plan of the triangular CCS block
    under the current settings, with its predicted sweep time under the library's cost model."""
    nr, nc, cs, ri, va = block
    cs = np.ascontiguousarray(cs, dtype=np.int64)
    ri = np.ascontiguousarray(ri, dtype=np.int32)
    va = np.ascontiguousarray(va, dtype=np.float64)
    c = LhfdGpuCcs(nr, nc, _ptr(cs), _ptr(ri), _ptr(va))
    out = np.zeros(8)
    _chk(lib().lhfdGpuDebugMergePlan(C.byref(c), int(upper), _ptr(out)))
    return {k: (float(v) if k == "predicted_us" else int(v)) for k, v in zip(MERGE_PLAN_KEYS, out)}


def debug_segment_graph(block, upper, max_segs=1 << 19, max_deps=1 << 26):
    """lhfdGpuDebugSegmentGraph: (dep_ptr, dep_idx) of the packed warp streams, trace numbering"""
    nr, nc, cs, ri, va = block
    cs = np.ascontiguousarray(cs, dtype=np.int64)
    ri = np.ascontiguousarray(ri, dtype=np.int32)
    va = np.ascontiguousarray(va, dtype=np.float64)
    c = LhfdGpuCcs(nr, nc, _ptr(cs), _ptr(ri), _ptr(va))
    dp = np.zeros(max_segs + 1, dtype=np.uint32)
    di = np.zeros(max_deps, dtype=np.uint32)
    ns = C.c_size_t()
    _chk(lib().lhfdGpuDebugSegmentGraph(C.byref(c), int(upper), max_segs, max_deps, _ptr(dp), _ptr(di), C.byref(ns)))
    n = ns.value
    return dp[: n + 1], di[: dp[n]]


FILE_INFO_NAMES = ("version", "single", "levels", "n", "nnz", "has_plans", "plan_entries", "plan_depth")


def save_arena(path, levels, with_plans=True):
    """lhf?GpuSaveLevels: write the level description (and the attach-time plans) to an arena file.
    Host only -- needs no GPU."""
    dt = levels_dtype(levels)
    arr, keep = make_level_structs(levels, dt)
    f = lib().lhfsGpuSaveLevels if dt == np.float32 else lib().lhfdGpuSaveLevels
    _chk(f(len(levels), C.cast(arr, C.c_void_p), int(bool(with_plans)), os.fsencode(path)))


def arena_info(path):
    """lhfGpuFileInfo: reads and verifies the whole file (host only)"""
    info = np.zeros(8, dtype=np.uint64)
    _chk(lib().lhfGpuFileInfo(os.fsencode(path), _ptr(info)))
    return {k: int(v) for k, v in zip(FILE_INFO_NAMES, info)}


def attach_arena(path, device=0):
    """lhf?GpuAttachFile -> GpuHif (single or double precision as the file says)"""
    single = bool(arena_info(path)["single"])
    h = C.c_void_p()
    f = lib().lhfsGpuAttachFile if single else lib().lhfdGpuAttachFile
    _chk(f(device, os.fsencode(path), C.byref(h)))
    return GpuHif(raw_handle=h.value, single=single)


def debug_file_sweep_host(path, level, upper, rhs):
    """lhfGpuDebugFileSweepHost: host emulation of one sweep from an arena file (its stored plan)"""
    rhs = np.ascontiguousarray(rhs, dtype=np.float64)
    x = np.zeros_like(rhs)
    st = np.zeros(4, dtype=np.uint64)
    _chk(lib().lhfGpuDebugFileSweepHost(os.fsencode(path), level, int(upper), _ptr(rhs), _ptr(x), _ptr(st)))
    return x, dict(zip(("slices", "padded", "bytes", "depth"), (int(v) for v in st)))


class GpuHif:
    """Thin handle wrapper: one attached preconditioner on one device.

    Mirrors the libhifir calling pattern (lhfdCreate/Setup -> lhfdSolve/lhfdApply ->
    lhfdDestroy); every method is one C-ABI call."""

    def __init__(self, levels=None, device=0, raw_handle=None, single=False):
        """levels with float32 factor values (or raw_handle + single=True: an LhfsGpuHdl) attach a
        single-precision preconditioner: solve/apply then go through lhfsdGpu* (double vectors) and
        solve_f32/apply_f32 through lhfsGpu* (float vectors); every other method reaches the handle
        through lhfsGpuAsDouble."""
        self._h = None
        self.single = bool(single)
        if raw_handle is not None:
            self._h = C.c_void_p(raw_handle)
        else:
            self.single = levels_dtype(levels) == np.float32
            arr, keep = make_level_structs(levels, np.float32 if self.single else np.float64)
            h = C.c_void_p()
            f = lib().lhfsGpuAttachLevels if self.single else lib().lhfdGpuAttachLevels
            _chk(f(device, len(levels), C.cast(arr, C.c_void_p), C.byref(h)))
            self._h = h
        if self.single:
            assert lib().lhfsGpuAsDouble(self._h) == self._h.value
        self.n = self.stats()["n"]

    def close(self):
        if self._h is not None and _lib is not None:
            (_lib.lhfsGpuDestroy if self.single else _lib.lhfdGpuDestroy)(self._h)
        self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def stats(self):
        s = np.zeros(len(STAT_NAMES), dtype=np.uint64)
        _chk(lib().lhfdGpuGetStats(self._h, _ptr(s)))
        return {k: int(v) for k, v in zip(STAT_NAMES, s)}

    def depths(self):
        nl = self.stats()["levels"]
        d = np.zeros(2 * nl, dtype=np.uint64)
        _chk(lib().lhfdGpuGetDepths(self._h, nl, _ptr(d)))
        return d.reshape(nl, 2).astype(np.int64)

    def set_matrix(self, A, rowmajor=True):
        n, indptr, indices, vals = A
        ip = np.ascontiguousarray(indptr, dtype=np.int64)
        ix = np.ascontiguousarray(indices, dtype=np.int32)
        va = np.ascontiguousarray(vals, dtype=np.float64)
        f = lib().lhfsdGpuUpdate if self.single else lib().lhfdGpuSetMatrix
        _chk(f(self._h, int(bool(rowmajor)), n, _ptr(ip), _ptr(ix), _ptr(va)))

    def set_matrix_f32(self, A, rowmajor=True):
        """lhfsGpuSetMatrix: a single-precision user matrix (widened at upload)"""
        assert self.single
        n, indptr, indices, vals = A
        ip = np.ascontiguousarray(indptr, dtype=np.int64)
        ix = np.ascontiguousarray(indices, dtype=np.int32)
        va = np.ascontiguousarray(vals, dtype=np.float32)
        _chk(lib().lhfsGpuSetMatrix(self._h, int(bool(rowmajor)), n, _ptr(ip), _ptr(ix), _ptr(va)))

    def set_nsp_const(self, start=0, end=FULL_RANK):
        _chk(lib().lhfdGpuSetNspConst(self._h, start, end))

    def set_nsp_tran_const(self, start=0, end=FULL_RANK):
        """hif::HIF::nsp_tran: the filter of the transposed solve (LHF_SH)"""
        _chk(lib().lhfdGpuSetNspTranConst(self._h, start, end))

    def norm2_dev(self, d_v, n):
        """lhfdGpuDebugNorm2Dev: the device 2-norm of the refinement / Krylov loops"""
        out = C.c_double()
        _chk(lib().lhfdGpuDebugNorm2Dev(self._h, C.c_void_p(d_v), n, C.byref(out)))
        return out.value

    def clear_nsp(self):
        _chk(lib().lhfdGpuClearNsp(self._h))

    def set_stream(self, stream_ptr=None):
        """stream_ptr: raw cudaStream_t (0 = legacy default stream); None = the handle's own stream"""
        if stream_ptr is None:
            _chk(lib().lhfdGpuSetStream(self._h, None, 1))
        else:
            _chk(lib().lhfdGpuSetStream(self._h, C.c_void_p(stream_ptr), 0))

    def synchronize(self):
        _chk(lib().lhfdGpuSynchronize(self._h))

    # ---- host-buffer entry points (numpy in, numpy out) ----
    def solve(self, b, out=None):
        b = np.ascontiguousarray(b, dtype=np.float64)
        x = np.empty_like(b) if out is None else out
        _chk((lib().lhfsdGpuSolve if self.single else lib().lhfdGpuSolve)(self._h, _ptr(b), _ptr(x)))
        return x

    def solve_async(self, b, out):
        """lhfdGpuSolveAsync: enqueue x = M^-1 b for host arrays (contiguous float64, ideally pinned);
        `out` must not be read before synchronize().  b and out must stay alive until then."""
        assert b.dtype == np.float64 and out.dtype == np.float64 and b.flags.c_contiguous and out.flags.c_contiguous
        _chk(lib().lhfdGpuSolveAsync(self._h, _ptr(b), _ptr(out)))

    def solve_f32(self, b):
        """lhfsGpuSolve: float vectors (single-precision handles only)"""
        assert self.single
        b = np.ascontiguousarray(b, dtype=np.float32)
        x = np.empty_like(b)
        _chk(lib().lhfsGpuSolve(self._h, _ptr(b), _ptr(x)))
        return x

    def apply_f32(self, b, op=LHF_S, nirs=1, betas=None, rank=LHF_DEFAULT_RANK):
        """lhfsGpuApply: float vectors (single-precision handles only)"""
        assert self.single
        b = np.ascontiguousarray(b, dtype=np.float32)
        x = np.empty_like(b)
        bt = None if betas is None else np.asarray(betas, dtype=np.float64)
        irs = np.zeros(2, dtype=np.int32)
        _chk(lib().lhfsGpuApply(self._h, op, _ptr(b), nirs, _ptr(bt) if bt is not None else None, rank,
                                _ptr(x), _ptr(irs)))
        return x, (int(irs[0]), int(irs[1]))

    def apply(self, b, op=LHF_S, nirs=1, betas=None, rank=LHF_DEFAULT_RANK):
        b = np.ascontiguousarray(b, dtype=np.float64)
        x = np.empty_like(b)
        bt = None if betas is None else np.asarray(betas, dtype=np.float64)
        irs = np.zeros(2, dtype=np.int32)
        f = lib().lhfsdGpuApply if self.single else lib().lhfdGpuApply
        _chk(f(self._h, op, _ptr(b), nirs, _ptr(bt) if bt is not None else None, rank, _ptr(x), _ptr(irs)))
        return x, (int(irs[0]), int(irs[1]))

    def solve_mrhs(self, B):
        B = np.ascontiguousarray(B, dtype=np.float64)
        assert B.ndim == 2 and B.shape[0] == self.n
        X = np.empty_like(B)
        _chk(lib().lhfdGpuSolveMrhs(self._h, B.shape[1], _ptr(B), _ptr(X)))
        return X

    def fgmres(self, b, restart=30, rtol=1e-6, maxit=500, full_rank=False):
        b = np.ascontiguousarray(b, dtype=np.float64)
        x = np.empty_like(b)
        flag, iters, nmv = C.c_int(), C.c_int(), C.c_int()
        _chk(lib().lhfdGpuFgmres(self._h, _ptr(b), restart, rtol, maxit, int(full_rank), _ptr(x),
                                 C.byref(flag), C.byref(iters), C.byref(nmv)))
        return x, flag.value, iters.value, nmv.value

    def gmres(self, b, restart=30, rtol=1e-6, maxit=500):
        b = np.ascontiguousarray(b, dtype=np.float64)
        x = np.empty_like(b)
        flag, iters = C.c_int(), C.c_int()
        _chk(lib().lhfdGpuGmres(self._h, _ptr(b), restart, rtol, maxit, _ptr(x), C.byref(flag),
                                C.byref(iters)))
        return x, flag.value, iters.value

    def _block(self, B):
        B = np.ascontiguousarray(B, dtype=np.float64)
        assert B.ndim == 2 and B.shape[0] == self.n
        k = B.shape[1]
        return B, np.empty_like(B), np.zeros(k, dtype=np.int32), np.zeros(k, dtype=np.int32), np.zeros(k, dtype=np.int32)

    def fgmres_mrhs(self, B, restart=30, rtol=1e-6, maxit=500, full_rank=False):
        """lhfdGpuFgmresMrhs: one fgmres per column of the (n, nrhs) block B, run together on the batched
        apply.  Returns (X, flags, iters, num_mv), the last three arrays of nrhs entries."""
        B, X, flags, iters, nmv = self._block(B)
        if B.shape[1]:
            _chk(lib().lhfdGpuFgmresMrhs(self._h, B.shape[1], _ptr(B), restart, rtol, maxit, int(full_rank), _ptr(X),
                                         _ptr(flags), _ptr(iters), _ptr(nmv)))
        return X, flags, iters, nmv

    def gmres_mrhs(self, B, restart=30, rtol=1e-6, maxit=500):
        """lhfdGpuGmresMrhs: one gmres per column of the (n, nrhs) block B.  Returns (X, flags, iters)."""
        B, X, flags, iters, _ = self._block(B)
        if B.shape[1]:
            _chk(lib().lhfdGpuGmresMrhs(self._h, B.shape[1], _ptr(B), restart, rtol, maxit, _ptr(X), _ptr(flags),
                                        _ptr(iters)))
        return X, flags, iters

    # ---- device-pointer entry points (ints = raw device addresses, e.g. tensor.data_ptr()) ----
    def solve_dev(self, d_b, d_x, rank=0):
        _chk(lib().lhfdGpuSolveDev(self._h, C.c_void_p(d_b), C.c_void_p(d_x), rank))

    def apply_dev(self, d_b, d_x, op=LHF_S, nirs=1, rank=LHF_DEFAULT_RANK):
        _chk(lib().lhfdGpuApplyDev(self._h, op, C.c_void_p(d_b), nirs, rank, C.c_void_p(d_x)))

    def solve_mrhs_dev(self, nrhs, d_B, d_X, rank=0):
        _chk(lib().lhfdGpuSolveMrhsDev(self._h, nrhs, C.c_void_p(d_B), C.c_void_p(d_X), rank))

    def hifir_dev(self, d_b, nirs, d_x, rank=FULL_RANK):
        _chk(lib().lhfdGpuHifirDev(self._h, C.c_void_p(d_b), nirs, C.c_void_p(d_x), rank))

    def hifir_mrhs_dev(self, nrhs, d_B, nirs, d_X, rank=FULL_RANK):
        """lhfdGpuHifirMrhsDev: hifir_dev on a row-interleaved (n, nrhs) device block"""
        _chk(lib().lhfdGpuHifirMrhsDev(self._h, nrhs, C.c_void_p(d_B), nirs, C.c_void_p(d_X), rank))

    def profile_solve_dev(self, d_b, d_x, rank=0):
        """Instrumented apply: [(label, milliseconds)] for every kernel of the schedule."""
        ms = np.zeros(256, dtype=np.float32)
        cnt = C.c_size_t()
        names = C.create_string_buffer(8192)
        _chk(lib().lhfdGpuProfileSolveDev(self._h, C.c_void_p(d_b), C.c_void_p(d_x), rank, 256, _ptr(ms),
                                          C.byref(cnt), names, 8192))
        labels = names.value.decode().split("\n")
        return [(labels[k], float(ms[k])) for k in range(cnt.value)]

    def trace_sweep(self, d_b, d_x, level, which, max_segs=1 << 20):
        """per-segment trace of one warp-stream sweep: array [nsegs, 4] (see lhfdGpuDebugTraceSweep)"""
        out = np.zeros(max_segs * 4, dtype=np.uint64)
        ns = C.c_size_t()
        _chk(lib().lhfdGpuDebugTraceSweep(self._h, C.c_void_p(d_b), C.c_void_p(d_x), level, which, _ptr(out),
                                          max_segs, C.byref(ns)))
        return out[: ns.value * 4].reshape(-1, 4)

    SWEEP_FACTORS = ("L", "U", "LU")

    def debug_sweep_dev(self, level, factor, rhs, transposed=False):
        """lhfdGpuDebugSweepDev: one sweep of factor 'L', 'U' or 'LU' (the fused plan) of a level on the device,
        next to the tag-exact host emulation of the plan the device holds.  rhs in original row order (m).
        Returns dict(x, words, emul, slot_of, slot_of_l, parity): x (m) = the result rows as the apply reads
        them, words / emul = the device's and the emulation's tagged words (uint64, slot order), slot_of = word
        of every result row, slot_of_l = word of every row of the L part of a fused plan (else None)."""
        rhs = np.ascontiguousarray(rhs, dtype=np.float64)
        m = rhs.size
        x = np.zeros(m)
        words = np.zeros(4 * m, dtype=np.uint64)
        emul = np.zeros(4 * m, dtype=np.uint64)
        slot_of = np.zeros(2 * m, dtype=np.uint32)
        nw, par = C.c_size_t(), C.c_uint()
        _chk(lib().lhfdGpuDebugSweepDev(self._h, int(bool(transposed)), level, self.SWEEP_FACTORS.index(factor), _ptr(rhs),
                                        _ptr(x), _ptr(words), _ptr(emul), words.size, C.byref(nw), _ptr(slot_of),
                                        C.byref(par)))
        return dict(x=x, words=words[: nw.value], emul=emul[: nw.value], slot_of=slot_of[:m],
                    slot_of_l=slot_of[m:] if factor == "LU" else None, parity=par.value)

    def export_ints(self, level, which):
        """lhfdGpuDebugExportInts: a device-resident index array of one level, copied back
        (which: 'p', 'q_inv', 'E_ptr', 'E_col', 'F_ptr', 'F_col', 'jpvt')"""
        sel = ("p", "q_inv", "E_ptr", "E_col", "F_ptr", "F_col", "jpvt").index(which)
        cnt = C.c_size_t()
        dummy = np.zeros(1, dtype=np.int32)
        _chk(lib().lhfdGpuDebugExportInts(self._h, level, sel, _ptr(dummy), 0, C.byref(cnt)))
        out = np.zeros(max(1, cnt.value), dtype=np.int32)
        _chk(lib().lhfdGpuDebugExportInts(self._h, level, sel, _ptr(out), out.size, C.byref(cnt)))
        return out[: cnt.value]

    def spmv_dev(self, d_x, d_y):
        _chk(lib().lhfdGpuSpmvDev(self._h, C.c_void_p(d_x), C.c_void_p(d_y)))
