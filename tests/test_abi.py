"""CPU-side checks of the drop-in boundary: the C-ABI library builds, loads and exports every
symbol include/hifir_b200.h declares; argument validation works without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import hifir_b200 as hb
from conftest import ROOT, gpu_available, load_golden


@pytest.fixture(scope="module")
def lib():
    from hifir_b200 import build
    build.build()
    return hb.lib()


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "hifir_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(lhf\w*Gpu\w*)\s*\(", src)))


def test_header_symbols_are_exported(lib):
    names = _declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/hifir_b200.h but not exported"
    assert set(names) == set(hb.EXPORTED_SYMBOLS)


def test_debug_header_symbols_are_exported(lib):
    """the developer / test hooks live in a private header (hifir_b200/csrc/debug_api.h), not in the
    drop-in boundary; they must be exported too and must not leak into the public header"""
    src = open(os.path.join(ROOT, "hifir_b200", "csrc", "debug_api.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = sorted(set(re.findall(r"\b(lhf\w*Gpu\w*)\s*\(", src)))
    assert set(names) == set(hb.DEBUG_SYMBOLS)
    for n in names:
        assert hasattr(lib, n), f"{n} declared in debug_api.h but not exported"
    assert not [n for n in _declared_symbols() if "Debug" in n]


def test_plan_validation_refuses_inconsistent_sweep_forms(lib, tmp_path):
    """ADVICE r1: a stored plan is checked before it can become an out-of-bounds device access --
    every sweep row must reference earlier rows only (the arena loader runs the same check on the
    plans of a file; here a CCS block that is not strictly triangular is refused by the packer's
    front door)."""
    import scipy.sparse as sp
    A = sp.csc_matrix(np.array([[0.0, 0.5, 0.0], [0.3, 0.0, 0.0], [0.0, 0.2, 0.0]]))  # entry above the diagonal
    blk = (3, 3, A.indptr.astype(np.int64), A.indices.astype(np.int32), A.data)
    with pytest.raises(hb.LhfError) as e:
        hb.debug_sweep_host(blk, False, np.ones(3))
    assert e.value.status == hb.LHF_BAD_PREC
    bad = (3, 3, np.array([1, 1, 2, 2], dtype=np.int64), np.array([1, 2], dtype=np.int32), np.array([0.3, 0.2]))
    with pytest.raises(hb.LhfError):
        hb.debug_sweep_host(bad, False, np.ones(3))  # col_start[0] != 0


def test_version_and_enums(lib):
    assert b"sm_100a" in lib.lhfGpuVersion()
    assert (hb.LHF_SUCCESS, hb.LHF_NULL_OBJ, hb.LHF_MISMATCHED_SIZES, hb.LHF_BAD_PREC, hb.LHF_HIFIR_ERROR) == (
        0, 1, 2, 3, 4)  # libhifir.h:148-154
    assert (hb.LHF_S, hb.LHF_SH, hb.LHF_M, hb.LHF_MH) == (0, 1, 2, 3)  # libhifir.h:160-165
    assert hb.LHF_DEFAULT_RANK == -2  # libhifir.h:167


def test_null_handle_is_refused(lib):
    x = np.zeros(4)
    p = x.ctypes.data_as(C.c_void_p)
    assert lib.lhfdGpuSolve(None, p, p) == hb.LHF_NULL_OBJ
    assert lib.lhfdGpuApply(None, hb.LHF_S, p, 1, None, hb.LHF_DEFAULT_RANK, p, None) == hb.LHF_NULL_OBJ
    assert lib.lhfdGpuDestroy(None) == hb.LHF_NULL_OBJ
    assert lib.lhfdGpuSolveMrhs(None, 2, p, p) == hb.LHF_NULL_OBJ
    assert lib.lhfdGpuFgmres(None, p, 30, 1e-6, 500, 0, p, None, None, None) == hb.LHF_NULL_OBJ
    assert b"NULL" in lib.lhfGpuGetErrorMsg()
    out = C.c_void_p()
    assert lib.lhfdGpuAttachLevels(0, 0, None, C.byref(out)) == hb.LHF_NULL_OBJ
    # the single / mixed precision family and the arena entry points follow the same rule
    assert lib.lhfsGpuAttachLevels(0, 0, None, C.byref(out)) == hb.LHF_NULL_OBJ
    assert lib.lhfsGpuSolve(None, p, p) == hb.LHF_NULL_OBJ
    assert lib.lhfsdGpuSolve(None, p, p) == hb.LHF_NULL_OBJ
    assert lib.lhfsGpuApply(None, hb.LHF_S, p, 1, None, hb.LHF_DEFAULT_RANK, p, None) == hb.LHF_NULL_OBJ
    assert lib.lhfsdGpuApply(None, hb.LHF_S, p, 1, None, hb.LHF_DEFAULT_RANK, p, None) == hb.LHF_NULL_OBJ
    assert lib.lhfsGpuDestroy(None) == hb.LHF_NULL_OBJ
    assert lib.lhfsGpuAsDouble(None) is None
    assert lib.lhfdGpuAttachFile(0, None, C.byref(out)) == hb.LHF_NULL_OBJ
    assert lib.lhfdGpuSaveLevels(1, None, 1, b"/tmp/x.hifb") == hb.LHF_NULL_OBJ


def test_level_struct_layout_matches_header():
    """ctypes mirror of LhfdGpuLevel: field order/size must follow include/hifir_b200.h."""
    assert C.sizeof(hb.LhfdGpuCcs) == 5 * 8
    assert C.sizeof(hb.LhfdGpuLevel) == 2 * 8 + 4 * 40 + 7 * 8 + 2 * 8 + 3 * 8 + 8
    arr, keep = hb.make_level_structs(load_golden("poisson14_ml").levels)
    assert arr[0].m == 2544 and arr[0].n == 2744 and arr[1].dense_n == 1
    assert arr[0].L_B.nrows == 2544 and arr[0].E.nrows == 200 and arr[0].F.ncols == 200


@pytest.mark.skipif(gpu_available(), reason="checks the no-GPU failure mode")
def test_attach_without_gpu_fails_loudly(lib):
    """No CPU fallback: without a CUDA device attach must fail with a message, not emulate."""
    with pytest.raises(hb.LhfError) as e:
        hb.GpuHif(load_golden("poisson14_ml").levels)
    assert e.value.status == hb.LHF_HIFIR_ERROR
    assert "cuda" in str(e.value).lower()


SWEEP_MODES = [("ws", "1"), ("ws", "0"), ("stream", "1"), ("stream", "0")]


@pytest.mark.parametrize("mode", SWEEP_MODES, ids=lambda m: f"{m[0]}-merge{m[1]}")
@pytest.mark.parametrize("case", ["demo_A", "poisson14_ml", "stokes28_ml"])
def test_sweep_packing_host_emulation(lib, case, mode, monkeypatch):
    """Host logic of the triangular sweeps: transform each L_B / U_B of the fixtures the way
    attach does (algebraic level merging, merge.cu; packing into per-warp segment streams,
    wsweep.cu; or round 1's level-major sliced ELL, stream.cu) and solve with the packed data on the CPU -- must equal
    plain substitution up to rounding (merging is an exact reformulation; the packed layouts
    list a row's entries by the dependency depth of their producers)."""
    import scipy.sparse as sp
    monkeypatch.setenv("HIFIR_B200_SWEEP", mode[0])
    monkeypatch.setenv("HIFIR_B200_MERGE", mode[1])
    g = load_golden(case)
    rng = np.random.default_rng(1)
    for L in g.levels:
        m = L["m"]
        if not m:
            continue
        rhs = rng.uniform(-1, 1, m)
        for name, upper in (("L", False), ("U", True)):
            nr, nc, cs, ri, va = L[name]
            x, st = hb.debug_sweep_host(L[name], upper, rhs, L["d"] if upper else None)
            T = sp.csc_matrix((va, ri, cs), shape=(m, m)).tocsr()
            T.sort_indices()
            ref = np.array(rhs / L["d"] if upper else rhs)
            order = range(m - 1, -1, -1) if upper else range(m)
            for i in order:  # same per-row update order as the reference's column sweeps
                cols = T.indices[T.indptr[i]:T.indptr[i + 1]]
                vals = T.data[T.indptr[i]:T.indptr[i + 1]]
                seq = zip(cols[::-1], vals[::-1]) if upper else zip(cols, vals)
                acc = ref[i]
                for j, v in seq:
                    acc -= v * ref[j]
                ref[i] = acc
            assert np.linalg.norm(x - ref) <= 1e-13 * np.linalg.norm(ref), (case, name)
            assert st["slices"] >= 1 and st["bytes"] >= 10 * len(va)


@pytest.mark.parametrize("merge", ["1", "0"])
def test_float_sweep_packing_host_emulation(lib, merge, monkeypatch):
    """Single-precision factors (lhfsGpuAttachLevels): the streamed values are the merged values
    rounded to float.  Emulated on the host, the packed sweep must agree with plain substitution on
    the float factor to float rounding -- far inside the 1e-5 gate."""
    import scipy.sparse as sp
    import scipy.sparse.linalg as spl
    # default sweep kernel (warp streams)
    monkeypatch.setenv("HIFIR_B200_MERGE", merge)
    g = load_golden("stokes28_ml_f32")
    rng = np.random.default_rng(2)
    for L in g.levels:
        m = L["m"]
        rhs = rng.uniform(-1, 1, m)
        for name, upper in (("L", False), ("U", True)):
            nr, nc, cs, ri, va = L[name]
            assert va.dtype == np.float32
            d = L["d"].astype(np.float64)
            x, st = hb.debug_sweep_host(L[name], upper, rhs, d if upper else None)
            T = sp.csc_matrix((va.astype(np.float64), ri, cs), shape=(m, m)) + sp.identity(m, format="csc")
            ref = spl.spsolve_triangular(T.tocsr(), rhs / d if upper else rhs, lower=not upper)
            err = np.linalg.norm(x - ref) / np.linalg.norm(ref)
            assert err <= (2e-6 if merge == "1" else 1e-13), (name, err)
            if merge == "1" and len(va) > 100:
                assert err > 0.0  # the merged values really were rounded


@pytest.mark.parametrize("case", ["stokes28_ml", "neumann12_nsp", "poisson14_ml_f32"])
def test_arena_file_roundtrip_on_host(lib, case, tmp_path):
    """Factor arena files (csrc/arena.cu): written without a GPU from the plain level description;
    the stored plans (sweep form + level merging of every L_B / U_B) must reproduce, bit for bit,
    what the attach-time analysis computes from the factors read back."""
    g = load_golden(case)
    single = case.endswith("_f32")
    with_plans, without = str(tmp_path / "a.hifb"), str(tmp_path / "b.hifb")
    hb.save_arena(with_plans, g.levels, True)
    hb.save_arena(without, g.levels, False)
    nnz = sum(len(L[k][3]) for L in g.levels for k in "LUEF")
    ia, ib = hb.arena_info(with_plans), hb.arena_info(without)
    assert (ia["version"], ia["single"], ia["levels"], ia["n"], ia["nnz"]) == (1, int(single), len(g.levels), g.n, nnz)
    assert ia["has_plans"] == 1 and ia["plan_entries"] > 0 and ib["has_plans"] == 0 and ib["nnz"] == nnz
    assert os.path.getsize(without) < os.path.getsize(with_plans)
    rng = np.random.default_rng(5)
    for lvl, L in enumerate(g.levels):
        if not L["m"]:
            continue
        rhs = rng.uniform(-1, 1, L["m"])
        for name, upper in (("L", False), ("U", True)):
            x0, s0 = hb.debug_sweep_host(L[name], upper, rhs, L["d"].astype(np.float64) if upper else None)
            for path in (with_plans, without):
                x1, s1 = hb.debug_file_sweep_host(path, lvl, upper, rhs)
                assert np.array_equal(x0, x1) and s0 == s1, (case, lvl, name, path)


def test_arena_file_corruption_is_refused(lib, tmp_path):
    g = load_golden("poisson14_ml")
    good = str(tmp_path / "good.hifb")
    hb.save_arena(good, g.levels, True)
    raw = bytearray(open(good, "rb").read())
    bad = str(tmp_path / "bad.hifb")
    flipped = bytearray(raw)
    flipped[len(raw) // 2] ^= 0x40  # one bit somewhere in the middle
    open(bad, "wb").write(flipped)
    with pytest.raises(hb.LhfError) as e:
        hb.arena_info(bad)
    assert "arena file" in str(e.value)
    open(bad, "wb").write(raw[: len(raw) // 3])  # truncated
    with pytest.raises(hb.LhfError):
        hb.arena_info(bad)
    open(bad, "wb").write(b"%%MatrixMarket matrix coordinate real general\n" * 4)  # some other file
    with pytest.raises(hb.LhfError) as e:
        hb.arena_info(bad)
    assert e.value.status == hb.LHF_BAD_PREC
    with pytest.raises(hb.LhfError):
        hb.arena_info(str(tmp_path / "does_not_exist.hifb"))


def test_level_merging_shortens_the_dependency_chain(lib, monkeypatch):
    """merge.cu: the merged factor (the one the streaming sweep runs) must be much shallower than
    the reference's factor, at a bounded cost in entries."""
    import scipy.sparse as sp
    g = load_golden("poisson14_ml")
    L = g.levels[0]
    m = L["m"]
    rhs = np.random.default_rng(3).uniform(-1, 1, m)
    depth = {}
    for merge in ("0", "1"):
        monkeypatch.setenv("HIFIR_B200_MERGE", merge)
        for name, upper in (("L", False), ("U", True)):
            x, st = hb.debug_sweep_host(L[name], upper, rhs, L["d"] if upper else None)
            depth[(merge, name)] = st["depth"]  # dependency depth of the packed factor
            depth[(merge, name, "bytes")] = st["bytes"]
    for name in ("L", "U"):
        assert depth[("1", name)] * 3 <= depth[("0", name)], depth
        # tiny factor: no cap but gain / row_cap binds; a thin level set is spread over many lanes
        # (few entries per lane), which costs segment headers
        assert depth[("1", name, "bytes")] <= 8 * depth[("0", name, "bytes")], depth


REF_SRC = "/root/reference/src"


@pytest.mark.skipif(not os.path.exists(os.path.join(REF_SRC, "hifir.hpp")), reason="needs the reference HIFIR headers, which this repository does not contain")
def test_cxx_adapter_compiles_against_the_reference_headers(tmp_path):
    """include/hifir_b200.hpp next to the reference's own <hifir.hpp>: the link-time attach overloads for
    hif::HIF<double,int> and hif::HIF<float,int>, the entry-point-table form and describe() + SaveLevels
    must compile as C++11 (the reference's language level) -- INTEGRATION.md sections 1, 1b, 1c."""
    import subprocess
    src = tmp_path / "adapter_check.cpp"
    src.write_text('''
#include <hifir.hpp>
#include <hifir_b200.hpp>
int use_double(const hif::HIF<double, int> &M, LhfdGpuHdl *out) { return hifir_b200::attach(M, 0, out); }
int use_single(const hif::HIF<float, int> &M, LhfsGpuHdl *out) { return hifir_b200::attach(M, 0, out); }
int use_table(const hif::HIF<float, int> &M, const hifir_b200::AttachApi &api, void **out) {
  return hifir_b200::attach(M, api, 0, out);
}
int save(const hif::HIF<double, int> &M) {
  std::vector<std::vector<LhfInt>> scratch;
  auto lv = hifir_b200::describe(M, scratch);
  return lhfdGpuSaveLevels(lv.size(), lv.data(), 1, "M.hifb");
}
''')
    r = subprocess.run(["g++", "-std=c++11", "-fsyntax-only", "-w", "-I" + REF_SRC, "-I" + os.path.join(ROOT, "include"),
                        str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]


def test_header_is_plain_c(tmp_path):
    """include/hifir_b200.h is a C header (extern "C", plain pointers and sizes): it must compile as C99."""
    import subprocess
    src = tmp_path / "c_check.c"
    src.write_text('#include <hifir_b200.h>\nint main(void) { LhfdGpuLevel l; LhfsGpuLevel s; (void)l; (void)s; '
                   'return (int)LHF_GPU_NUMBER_STATS - 15; }\n')
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-I" + os.path.join(ROOT, "include"),
                        str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]


def test_product_never_imports_oracle():
    """The package must not reach into oracle/ (only tests, bench cpu legs and smoke may)."""
    pkg = os.path.join(ROOT, "hifir_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in txt.replace("the parity oracle", ""), f"{f} mentions oracle"
