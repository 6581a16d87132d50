"""GPU parity tests proper (-m gpu): the CUDA path, called through the C-ABI, against
  * the committed golden vectors of the unmodified reference,
  * the plain-C oracle on the same seeded inputs,
  * the reference itself, live, on the very object the device backend was attached to
    (through the header-only C++ adapter), when oracle/_ref travelled to this box,
  * size-independent properties at larger sizes (linearity, M (M^-1 b) = b round trip).
Tolerance (north_star): ||x_gpu - x_ref|| / ||x_ref|| <= 1e-12 in double; iteration counts +-1."""
import ctypes as C

import numpy as np
import pytest

import hifir_b200 as hb
from conftest import TOL_F64, have_reference, load_golden, relerr
from hifir_b200 import problems as P
from oracle import port as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _built():
    from hifir_b200 import build
    build.build()
    assert b"sm_100a" in hb.lib().lhfGpuVersion()


def _gpu(g):
    G = hb.GpuHif(g.levels)
    G.set_matrix(g.A)
    if g.nsp:
        G.set_nsp_const()
    return G


def test_solve_matches_golden_and_oracle(golden):
    Oh = O.OracleHif(golden.levels, golden.A)
    if golden.nsp:
        Oh.set_nsp_const()
    with _gpu(golden) as G:
        st = G.stats()
        assert st["n"] == golden.n and st["levels"] == len(golden.levels)
        for k in range(golden["B"].shape[1]):
            b = np.ascontiguousarray(golden["B"][:, k])
            x = G.solve(b)
            assert relerr(x, golden["X"][:, k]) <= TOL_F64, "vs reference golden"
            assert relerr(x, Oh.solve(b)) <= TOL_F64, "vs C oracle"
        # repeated applies flip the ready-bit parity: results must not depend on it
        b = np.ascontiguousarray(golden["B"][:, 0])
        x1, x2, x3 = G.solve(b), G.solve(b), G.solve(b)
        assert np.array_equal(x1, x3) and relerr(x2, x1) <= 1e-14


@pytest.mark.parametrize("mode", [("ws", "0"), ("stream", "1"), ("stream", "0")], ids=lambda m: f"{m[0]}-merge{m[1]}")
def test_solve_other_sweep_kernels(golden, mode, monkeypatch):
    """The non-default sweep configurations (HIFIR_B200_SWEEP / HIFIR_B200_MERGE are read at attach):
    unmerged factors on the warp-stream kernel, merged and unmerged factors on round 1's streaming
    kernel -- single and multi right-hand side."""
    monkeypatch.setenv("HIFIR_B200_SWEEP", mode[0])
    monkeypatch.setenv("HIFIR_B200_MERGE", mode[1])
    with _gpu(golden) as G:
        for k in range(2):
            b = np.ascontiguousarray(golden["B"][:, k])
            assert relerr(G.solve(b), golden["X"][:, k]) <= TOL_F64
        if not golden.nsp:
            X = G.solve_mrhs(np.ascontiguousarray(golden["B"]))
            for k in range(golden["B"].shape[1]):
                assert relerr(X[:, k], golden["X"][:, k]) <= TOL_F64


def test_apply_semantics_follow_libhifir(golden):
    """lhfdApply (libhifir.cpp:447-472): op, nirs, betas, rank and ir_status."""
    with _gpu(golden) as G:
        b = np.ascontiguousarray(golden["B"][:, 0])
        x, _ = G.apply(b)  # LHF_S, nirs=1 -> plain solve, rank ignored
        assert relerr(x, golden["X"][:, 0]) <= TOL_F64
        x, _ = G.apply(b, rank=5)  # plain solve ignores rank (libhifir.cpp:461)
        assert relerr(x, golden["X"][:, 0]) <= TOL_F64
        x, _ = G.apply(b, nirs=3)  # hifir, default rank -> full (libhifir.cpp:453-455)
        assert relerr(x, golden["x_hifir3"]) <= TOL_F64
        x, (iters, flag) = G.apply(golden["b_krylov"], nirs=16, betas=[1e-8, 1e10])
        riters, rflag = (int(v) for v in golden["hifir_betas_status"])
        assert flag == rflag and abs(iters - riters) <= 1
        assert relerr(x, golden["x_hifir_betas"]) <= 1e-8
        with pytest.raises(hb.LhfError) as e:
            G.apply(b, op=7)
        assert e.value.status == hb.LHF_BAD_PREC


def test_other_operations_match_golden_and_oracle(golden):
    """LHF_SH / LHF_M / LHF_MH on the device (prec_solve.hpp:541-612, prec_prod.hpp:54-230) against the
    reference's golden vectors and the C oracle; then the on-device round trips M (M^-1 b) = b and
    M^H (M^-H b) = b (libhifir/tests/test_real.c:146)."""
    import torch
    if golden.nsp:
        pytest.skip("fixture made with the null-space filter")
    Oh = O.OracleHif(golden.levels, golden.A)
    with _gpu(golden) as G:
        b = np.ascontiguousarray(golden["B"][:, 0])
        for op, key in ((hb.LHF_SH, "x_SH"), (hb.LHF_M, "x_M"), (hb.LHF_MH, "x_MH")):
            x, _ = G.apply(b, op=op)
            assert relerr(x, golden[key]) <= TOL_F64, key
            assert relerr(x, Oh.apply_op(int(op), b)) <= TOL_F64, key
        x, _ = G.apply(b)  # the primary orientation still works after the twin was built
        assert relerr(x, golden["X"][:, 0]) <= TOL_F64
        db = torch.from_numpy(b).cuda()
        dx, dy = torch.empty_like(db), torch.empty_like(db)
        for s_op, m_op in ((hb.LHF_S, hb.LHF_M), (hb.LHF_SH, hb.LHF_MH)):
            G.apply_dev(db.data_ptr(), dx.data_ptr(), op=s_op)
            G.apply_dev(dx.data_ptr(), dy.data_ptr(), op=m_op)
            G.synchronize()
            assert relerr(dy.cpu().numpy(), b) <= 1e-10


def test_full_rank_device_solve(golden):
    import torch
    with _gpu(golden) as G:
        b = torch.from_numpy(np.ascontiguousarray(golden["B"][:, 1])).cuda()
        x = torch.empty_like(b)
        if golden.nsp:
            G.clear_nsp()
        G.solve_dev(b.data_ptr(), x.data_ptr(), hb.FULL_RANK)
        G.synchronize()
        if not golden.nsp:
            assert relerr(x.cpu().numpy(), golden["X_full"][:, 1]) <= TOL_F64
        # truncated last-level rank (QRCP.hpp:376-377) vs the C oracle
        dn = golden.levels[-1]["dense_n"]
        if dn > 2:
            Oh = O.OracleHif(golden.levels)
            G.solve_dev(b.data_ptr(), x.data_ptr(), dn - 1)
            G.synchronize()
            assert relerr(x.cpu().numpy(), Oh.solve(b.cpu().numpy(), dn - 1)) <= TOL_F64


@pytest.mark.parametrize("which", ["fgmres", "gmres"])
def test_krylov_iteration_parity(golden, which):
    with _gpu(golden) as G:
        if which == "fgmres":
            x, flag, iters, nmv = G.fgmres(golden["b_krylov"], restart=golden.restart)
        else:
            x, flag, iters = G.gmres(golden["b_krylov"], restart=golden.restart)
            nmv = iters
        rflag, riters, rnmv = (int(v) for v in golden[which + "_status"])
        assert flag == rflag
        assert abs(iters - riters) <= 1, (iters, riters)
        assert abs(nmv - rnmv) <= max(1, rnmv // max(riters, 1))
        # both satisfy ||b - A x|| <= rtol ||b||; the iterates agree far below rtol
        r = golden["b_krylov"] - P.csr_matvec(golden.A, x)
        assert np.linalg.norm(r) <= 2e-6 * np.linalg.norm(golden["b_krylov"])
        assert relerr(x, golden["x_" + which]) <= 1e-5


def test_mrhs_is_column_loop_of_solves(golden):
    """Row-interleaved B[i*nrhs+k] (builder.hpp:433-445); semantics = nrhs HIF::solve calls."""
    with _gpu(golden) as G:
        if golden.nsp:
            with pytest.raises(hb.LhfError):  # builder.hpp:440
                G.solve_mrhs(golden["B"])
            G.clear_nsp()
            Oh = O.OracleHif(golden.levels)
            ref = Oh.solve_mrhs(golden["B"])
        else:
            ref = golden["X"]
        X = G.solve_mrhs(golden["B"])
        for k in range(ref.shape[1]):
            assert relerr(X[:, k], ref[:, k]) <= TOL_F64
        B3 = np.ascontiguousarray(golden["B"][:, :3])  # ragged width
        X3 = G.solve_mrhs(B3)
        assert relerr(X3, ref[:, :3]) <= TOL_F64


@pytest.mark.parametrize("nrhs", [8, 11, 16, 20, 33, 64, 70])
def test_mrhs_batched_widths(nrhs):
    """Batched kernel (passes of 16 / 32 / 64 columns, lanes across the columns): full, ragged and several
    passes vs the C oracle."""
    g = load_golden("stokes28_ml")
    B = P.seeded_rhs(g.n, 100, nrhs=nrhs)
    ref = O.OracleHif(g.levels).solve_mrhs(B)
    with hb.GpuHif(g.levels) as G:
        X = G.solve_mrhs(B)
        for k in range(nrhs):
            assert relerr(X[:, k], ref[:, k]) <= TOL_F64, k
        # the single-rhs path afterwards still works on the same handle (shared tickets / epochs)
        assert relerr(G.solve(np.ascontiguousarray(B[:, 0])), ref[:, 0]) <= TOL_F64


def test_mrhs_width_changes_on_one_handle():
    """The tagged multi-rhs work vectors are laid out for one pass width: a handle that is given blocks of
    different widths (64 -> 16 -> 32 -> 64 columns per pass) must re-zero them (stale tags of an older layout)."""
    g = load_golden("stokes28_ml")
    Oh = O.OracleHif(g.levels)
    with hb.GpuHif(g.levels) as G:
        for rep, nrhs in enumerate([70, 5, 70, 24, 64, 3, 3, 64]):
            B = P.seeded_rhs(g.n, 200 + rep, nrhs=nrhs)
            X = G.solve_mrhs(B)
            ref = Oh.solve_mrhs(B)
            for k in range(nrhs):
                assert relerr(X[:, k], ref[:, k]) <= TOL_F64, (rep, nrhs, k)


def test_spmv_and_errors(golden):
    import torch
    with _gpu(golden) as G:
        x = torch.from_numpy(P.seeded_rhs(golden.n, 5)).cuda()
        y = torch.empty_like(x)
        G.spmv_dev(x.data_ptr(), y.data_ptr())
        G.synchronize()
        assert relerr(y.cpu().numpy(), P.csr_matvec(golden.A, x.cpu().numpy())) <= 1e-14
    with hb.GpuHif(golden.levels) as G2:  # no matrix attached
        with pytest.raises(hb.LhfError) as e:
            G2.apply(golden["B"][:, 0].copy(), nirs=2)
        assert e.value.status == hb.LHF_BAD_PREC
        bad = (4, np.zeros(5, dtype=np.int64), np.zeros(0, dtype=np.int32), np.zeros(0))
        with pytest.raises(hb.LhfError) as e:
            G2.set_matrix(bad)
        assert e.value.status == hb.LHF_MISMATCHED_SIZES


def test_attach_rejects_bad_input():
    g = load_golden("poisson14_ml")
    lv = [dict(L) for L in g.levels]
    lv[0]["has_symm_dense"] = 1
    with pytest.raises(hb.LhfError) as e:
        hb.GpuHif(lv)
    assert e.value.status == hb.LHF_BAD_PREC
    lv = [dict(L) for L in g.levels]
    p = lv[0]["p"].copy()
    p[0] = g.n + 3
    lv[0]["p"] = p
    with pytest.raises(hb.LhfError):
        hb.GpuHif(lv)


def test_linearity_and_zero_rhs():
    """size-independent properties: M^-1 is linear; M^-1 0 = 0."""
    g = load_golden("stokes28_ml")
    with _gpu(g) as G:
        b1, b2 = P.seeded_rhs(g.n, 11), P.seeded_rhs(g.n, 12)
        x1, x2, x12 = G.solve(b1), G.solve(b2), G.solve(2.0 * b1 - 3.0 * b2)
        assert relerr(x12, 2.0 * x1 - 3.0 * x2) <= 1e-11
        assert np.all(G.solve(np.zeros(g.n)) == 0.0)


# ------------------------------------------------------------------ live reference
needs_ref = pytest.mark.skipif(not have_reference(), reason="needs oracle/_ref/libhifir_ref.so, built from the reference HIFIR sources, which this repository does not contain")


def _attach_through_cxx_adapter(M):
    """hifir_b200::attach(hif::HIF&) of include/hifir_b200.hpp, compiled into the reference bridge."""
    fn = C.cast(hb.lib().lhfdGpuAttachLevels, C.c_void_p).value
    return hb.GpuHif(raw_handle=M.gpu_attach(fn))


@needs_ref
@pytest.mark.parametrize("case,N", [("poisson", 40), ("convdiff", 36), ("stokes", 96), ("neumann", 32)])
def test_against_live_reference_same_object(case, N):
    from oracle import refhost as R
    gen = {"poisson": P.poisson3d, "convdiff": P.convdiff3d, "stokes": P.stokes2d_mac, "neumann": P.neumann3d}[case]
    A = gen(N)
    M = R.RefHif(A, P.PDE_PARAMS, dense_thres=300 if case != "stokes" else 0)
    with _attach_through_cxx_adapter(M) as G:
        G.set_matrix(A)
        if case == "neumann":
            M.set_nsp_const()
            G.set_nsp_const()
        assert G.stats()["levels"] == M.num_precs
        for j in range(3):
            b = P.seeded_rhs(A[0], j)
            assert relerr(G.solve(b), M.solve(b)) <= TOL_F64
        b = P.seeded_rhs(A[0], 0)
        x, _ = G.apply(b, nirs=4)
        assert relerr(x, M.hifir(b, 4)) <= TOL_F64
        if case != "neumann":  # libhifir/tests/test_real.c:146 round trip through the reference's M x
            assert relerr(M.mmultiply(G.solve(b)), b) <= 1e-10
        bk = P.csr_matvec(A, np.ones(A[0]) if case != "neumann" else np.sin(0.37 * np.arange(A[0])))
        xr, fr, ir, nr = M.krylov(bk, "fgmres")
        xg, fg, ig, ng = G.fgmres(bk)
        assert fg == fr and abs(ig - ir) <= 1, (ig, ir)
        assert relerr(xg, xr) <= 1e-5


@needs_ref
def test_large_size_properties_and_merged_structure():
    """A BASELINE-scale factor (Poisson 96^3, n = 884 736, 3 levels; the 128^3 run itself is gated inside
    bench.py): parity against the reference's own apply on the same object, the size-independent
    properties (on-device round trip M (M^-1 b) = b, linearity, repeatability across ready-bit parities),
    and what the attach-time merging did to the dependency chain."""
    import torch
    from oracle import refhost as R
    A = P.poisson3d(96)
    M = R.RefHif(A, P.PDE_PARAMS)
    with _attach_through_cxx_adapter(M) as G:
        st = G.stats()
        assert st["levels"] == M.num_precs and st["n"] == A[0]
        assert st["depth_merged"] * 5 <= st["depth_total"], st        # 700-900-deep chains -> well under 100
        assert st["sweep_entries"] <= 2.5 * 2 * st["nnz"], st           # at a bounded cost in entries
        b1, b2 = P.seeded_rhs(A[0], 1), P.seeded_rhs(A[0], 2)
        x1 = G.solve(b1)
        assert relerr(x1, M.solve(b1)) <= TOL_F64
        x2, x12 = G.solve(b2), G.solve(2.0 * b1 - 3.0 * b2)
        assert relerr(x12, 2.0 * x1 - 3.0 * x2) <= 1e-11
        assert np.array_equal(G.solve(b1), G.solve(b1)) or relerr(G.solve(b1), x1) <= 1e-14
        db = torch.from_numpy(b1).cuda()
        dx, dy = torch.empty_like(db), torch.empty_like(db)
        G.apply_dev(db.data_ptr(), dx.data_ptr(), op=hb.LHF_S)
        G.apply_dev(dx.data_ptr(), dy.data_ptr(), op=hb.LHF_M)
        G.synchronize()
        assert relerr(dy.cpu().numpy(), b1) <= 1e-10
        X = G.solve_mrhs(np.stack([b1, b2, b1 - b2], axis=1))
        assert relerr(X[:, 2], x1 - x2) <= 1e-11


# ------------------------------------------------------------------ single / mixed precision
def _widened(levels):
    """the same factors with every value array widened to double (exact)"""
    out = []
    for L in levels:
        W = dict(L)
        for k in "LUEF":
            nr, nc, cs, ri, va = L[k]
            W[k] = (nr, nc, cs, ri, va.astype(np.float64))
        for k in ("d", "s", "t", "qr_mat", "qr_tau"):
            if k in L:
                W[k] = L[k].astype(np.float64)
        out.append(W)
    return out


def test_single_precision_preconditioner_matches_float_reference(golden_f32):
    """hif::HIF<float,int> (lhfs* and the mixed lhfsd* family, libhifir.h:775-872, 1231-1280): the
    device stores the sweep values as float and computes in double.  Gate (north_star): 1e-5 relative
    against the reference's single-precision apply; against the double restatement on the same float
    factors only the float rounding of the merged values remains."""
    from conftest import TOL_F32
    g = golden_f32
    Oh = O.OracleHif(g.levels, g.A)
    if g.nsp:
        Oh.set_nsp_const()
    with _gpu(g) as G:
        assert G.single
        for k in range(g["B"].shape[1]):
            b = np.ascontiguousarray(g["B"][:, k])
            x = G.solve(b)  # lhfsdGpuSolve: float factors, double vectors
            assert x.dtype == np.float64
            assert relerr(x, g["X"][:, k]) <= TOL_F32, "vs the reference's float apply"
            assert relerr(x, Oh.solve(b)) <= 2e-6, "vs the double restatement on the float factors"
            x32 = G.solve_f32(b)  # lhfsGpuSolve: float vectors
            assert x32.dtype == np.float32
            assert relerr(x32, g["X32"][:, k]) <= TOL_F32
            assert relerr(x32, x) <= 5e-7  # = rounding of b and x to float
        b = np.ascontiguousarray(g["B"][:, 0])
        x, _ = G.apply(b, nirs=3)  # lhfsdGpuApply: refinement with the double matrix (lhfsdUpdate)
        assert relerr(x, g["x_hifir3"]) <= TOL_F32
        x, _ = G.apply_f32(b)
        assert relerr(x, g["X32"][:, 0]) <= TOL_F32
        G.set_matrix_f32(g.A)  # lhfsGpuSetMatrix: single-precision user matrix (lhfsSetup / lhfsUpdate)
        x, _ = G.apply_f32(b, nirs=3)
        assert x.dtype == np.float32 and relerr(x, g["x_hifir3"]) <= TOL_F32
        G.set_matrix(g.A)
        if not g.nsp:
            for op, key in ((hb.LHF_SH, "x_SH"), (hb.LHF_M, "x_M"), (hb.LHF_MH, "x_MH")):
                x, _ = G.apply(b, op=op)
                assert relerr(x, g[key]) <= TOL_F32, key
            X = G.solve_mrhs(np.ascontiguousarray(g["B"]))  # through lhfsGpuAsDouble
            for k in range(g["B"].shape[1]):
                assert relerr(X[:, k], g["X"][:, k]) <= TOL_F32
        # what single precision buys: 8 instead of 12 bytes per streamed sweep entry
        st = G.stats()
        with hb.GpuHif(_widened(g.levels)) as Gd:
            std = Gd.stats()
            if g.nsp:
                Gd.set_nsp_const()
            assert not Gd.single and relerr(G.solve(b), Gd.solve(b)) <= 2e-6
        assert st["sweep_entries"] == std["sweep_entries"]
        assert st["sweep_bytes"] < 0.8 * std["sweep_bytes"], (st["sweep_bytes"], std["sweep_bytes"])
        assert st["bytes_factors"] < 0.8 * std["bytes_factors"]


@pytest.mark.parametrize("mode", [("ws", "0"), ("stream", "1")], ids=lambda m: f"{m[0]}-merge{m[1]}")
def test_single_precision_other_sweep_kernels(mode, monkeypatch):
    """unmerged warp streams (no rounding beyond the float factors themselves) and round 1's streaming
    kernel serve a single-precision preconditioner too"""
    from conftest import TOL_F32
    monkeypatch.setenv("HIFIR_B200_SWEEP", mode[0])
    monkeypatch.setenv("HIFIR_B200_MERGE", mode[1])
    g = load_golden("stokes28_ml_f32")
    Oh = O.OracleHif(g.levels, g.A)
    with _gpu(g) as G:
        b = np.ascontiguousarray(g["B"][:, 1])
        x = G.solve(b)
        assert relerr(x, g["X"][:, 1]) <= TOL_F32
        assert relerr(x, Oh.solve(b)) <= (1e-12 if mode[1] == "0" else 2e-6)


@needs_ref
def test_single_precision_against_live_reference_same_object():
    """attach through the C++ adapter to a live hif::HIF<float,int> (include/hifir_b200.hpp)"""
    from conftest import TOL_F32
    from oracle import refhost as R
    A = P.convdiff3d(32)
    M = R.RefHif(A, P.PDE_PARAMS, dense_thres=300, dtype=np.float32)
    fd = C.cast(hb.lib().lhfdGpuAttachLevels, C.c_void_p).value
    fs = C.cast(hb.lib().lhfsGpuAttachLevels, C.c_void_p).value
    with hb.GpuHif(raw_handle=M.gpu_attach(fd, attach_levels_s_fnptr=fs), single=True) as G:
        G.set_matrix(A)
        assert G.stats()["levels"] == M.num_precs
        for j in range(2):
            b = P.seeded_rhs(A[0], j)
            assert relerr(G.solve(b), M.solve(b)) <= TOL_F32
            assert relerr(G.solve_f32(b), M.solve_f32(b)) <= TOL_F32
        b = P.seeded_rhs(A[0], 0)
        x, _ = G.apply(b, nirs=4)
        assert relerr(x, M.hifir(b, 4)) <= TOL_F32
        # mixed-precision FGMRES-HIFIR: float preconditioner inside a double Krylov loop reaches rtol
        bk = P.csr_matvec(A, np.ones(A[0]))
        xg, fg, ig, ng = G.fgmres(bk)
        assert fg == 0 and relerr(P.csr_matvec(A, xg), bk) <= 1e-6


# ------------------------------------------------------------------ factor arena files
@pytest.mark.parametrize("case", ["demo_A", "stokes28_ml", "neumann12_nsp", "stokes28_ml_f32"])
@pytest.mark.parametrize("with_plans", [True, False], ids=["plans", "noplans"])
def test_attach_from_arena_file(case, with_plans, tmp_path):
    """lhf?GpuSaveLevels -> lhf?GpuAttachFile (csrc/arena.cu): the handle attached from the file must
    give bit-identical results to the handle attached to the live description, with or without the
    stored plans, and must pass the same gates against the reference's golden vectors."""
    from conftest import TOL_F32
    g = load_golden(case)
    single = case.endswith("_f32")
    tol = TOL_F32 if single else TOL_F64
    path = str(tmp_path / "arena.hifb")
    hb.save_arena(path, g.levels, with_plans)
    with _gpu(g) as G, hb.attach_arena(path) as F:
        assert F.single == single
        F.set_matrix(g.A)
        if g.nsp:
            F.set_nsp_const()
        sg, sf = G.stats(), F.stats()
        for k in ("levels", "n", "nnz", "depth_total", "depth_merged", "sweep_entries", "sweep_bytes", "bytes_factors"):
            assert sg[k] == sf[k], k
        for k in range(2):
            b = np.ascontiguousarray(g["B"][:, k])
            xf = F.solve(b)
            assert np.array_equal(xf, G.solve(b))
            assert relerr(xf, g["X"][:, k]) <= tol
        b = np.ascontiguousarray(g["B"][:, 0])
        assert np.array_equal(F.apply(b, nirs=3)[0], G.apply(b, nirs=3)[0])
        if not g.nsp:  # the transposed twin is built later, from the handle's own copies (no stored plan)
            for op, key in ((hb.LHF_SH, "x_SH"), (hb.LHF_M, "x_M")):
                x, _ = F.apply(b, op=op)
                assert relerr(x, g[key]) <= tol, key
            assert np.array_equal(F.solve_mrhs(np.ascontiguousarray(g["B"])), G.solve_mrhs(np.ascontiguousarray(g["B"])))
    # a file of the other precision is refused by the typed entry point
    h = C.c_void_p()
    wrong = hb.lib().lhfdGpuAttachFile if single else hb.lib().lhfsGpuAttachFile
    assert wrong(0, path.encode(), C.byref(h)) == hb.LHF_BAD_PREC and not h.value


def _ccs(dense):
    """dense 2-D array -> (nrows, ncols, col_start, row_ind, vals) as the level dicts hold them"""
    import scipy.sparse as sp
    A = sp.csc_matrix(dense)
    A.sort_indices()
    return (dense.shape[0], dense.shape[1], A.indptr.astype(np.int64), A.indices.astype(np.int32),
            A.data.astype(np.float64))


def _tiny_level(rng, n, m, dense=False):
    import scipy.linalg as sl
    nm = n - m
    L = np.tril(rng.uniform(-0.5, 0.5, (m, m)) * (rng.uniform(size=(m, m)) < 0.6), -1)
    U = np.triu(rng.uniform(-0.5, 0.5, (m, m)) * (rng.uniform(size=(m, m)) < 0.6), 1)
    lev = dict(m=m, n=n, dense_n=0, dense_rank=0, has_symm_dense=0, L=_ccs(L), U=_ccs(U),
               E=_ccs(rng.uniform(-1, 1, (nm, m))), F=_ccs(rng.uniform(-1, 1, (m, nm))),
               d=rng.uniform(1, 2, m), s=rng.uniform(0.5, 2, n), t=rng.uniform(0.5, 2, n))
    p, q = rng.permutation(n).astype(np.int32), rng.permutation(n).astype(np.int32)
    lev.update(p=p, q=q, p_inv=np.argsort(p).astype(np.int32), q_inv=np.argsort(q).astype(np.int32))
    if dense:
        (qr, tau), _, piv = sl.qr(rng.uniform(-1, 1, (nm, nm)) + 3 * np.eye(nm), mode="raw", pivoting=True)
        lev.update(dense_n=nm, dense_rank=nm, qr_mat=np.asfortranarray(qr).ravel(order="F"), qr_tau=tau,
                   qr_jpvt=(piv + 1).astype(np.int32))
    return lev


@pytest.mark.parametrize("shape", [(5, 5, False), (3, 1, True), (4, 0, True), (1, 1, False), (40, 33, True)],
                         ids=lambda s: f"n{s[0]}m{s[1]}")
def test_degenerate_levels(shape):
    """SURVEY.md App. B-4: levels with m = 0, m = 1, n = m (no Schur block), a dense level only --
    hand-made factors, checked against the C oracle (single and multi right-hand side)."""
    n, m, dense = shape
    rng = np.random.default_rng(100 * n + m)
    levels = [_tiny_level(rng, n, m, dense)]
    Oh = O.OracleHif(levels)
    with hb.GpuHif(levels) as G:
        for k in range(3):
            b = rng.uniform(-1, 1, n)
            assert relerr(G.solve(b), Oh.solve(b)) <= TOL_F64
        B = rng.uniform(-1, 1, (n, 3))
        X = G.solve_mrhs(B)
        for k in range(3):
            assert relerr(X[:, k], Oh.solve(np.ascontiguousarray(B[:, k]))) <= TOL_F64


@pytest.mark.parametrize("merge", ["1", "0"], ids=["merged", "unmerged"])
def test_rows_longer_than_one_segment(merge, monkeypatch):
    """Rows of L_B / U_B with more than 256 entries span several segments of a warp stream (32 lanes x 8
    entries each): the partial sums are carried from segment to segment (single-rhs sweep: in a register;
    multi-rhs sweep: parked in the row's own slot under the other tag).  Dense-ish hand-made factors, rows up to
    ~560 entries, checked against the C oracle for one right-hand side and for blocks of every pass width
    (16 / 32 / 64 columns: 4, 2, 1 rows per gather instruction, long rows shared by 4, 2, 1 lane groups)."""
    monkeypatch.setenv("HIFIR_B200_MERGE", merge)
    n, m = 860, 800
    rng = np.random.default_rng(4242)
    lev = _tiny_level(rng, n, m, dense=True)
    L = np.tril(rng.uniform(-1, 1, (m, m)) * (rng.uniform(size=(m, m)) < 0.7), -1) * (2.0 / m)
    U = np.triu(rng.uniform(-1, 1, (m, m)) * (rng.uniform(size=(m, m)) < 0.7), 1) * (2.0 / m)
    lev.update(L=_ccs(L), U=_ccs(U))
    assert (np.count_nonzero(L, axis=1).max() > 256) and (np.count_nonzero(U, axis=1).max() > 256)
    Oh = O.OracleHif([lev])
    with hb.GpuHif([lev]) as G:
        for k in range(2):
            b = rng.uniform(-1, 1, n)
            assert relerr(G.solve(b), Oh.solve(b)) <= TOL_F64
        for nrhs in (5, 20, 70):
            B = rng.uniform(-1, 1, (n, nrhs))
            X = G.solve_mrhs(B)
            for k in range(nrhs):
                assert relerr(X[:, k], Oh.solve(np.ascontiguousarray(B[:, k]))) <= TOL_F64, (nrhs, k)


def test_device_integer_arrays_are_bit_exact(golden):
    """north_star: index and permutation handling must be bit-exact.  The device-resident p, q_inv, jpvt
    and the CSR form of E and F (attach.cu: ccs_to_csr) are copied back and compared with the host
    arrays / with scipy's own CSC -> CSR conversion (= the reference's hif::CRS(const CCS&),
    CompressedStorage.hpp:861-890, ascending columns inside a row)."""
    import scipy.sparse as sp
    with _gpu(golden) as G:
        for l, L in enumerate(golden.levels):
            assert np.array_equal(G.export_ints(l, "p"), np.asarray(L["p"], dtype=np.int32))
            assert np.array_equal(G.export_ints(l, "q_inv"), np.asarray(L["q_inv"], dtype=np.int32))
            for name in ("E", "F"):
                nr, nc, cs, ri, va = L[name]
                if nr == 0 or nc == 0 or len(ri) == 0:
                    continue
                R = sp.csc_matrix((np.arange(1, len(ri) + 1, dtype=np.float64), ri, cs), shape=(nr, nc)).tocsr()
                R.sort_indices()
                assert np.array_equal(G.export_ints(l, name + "_ptr"), R.indptr.astype(np.int32))
                assert np.array_equal(G.export_ints(l, name + "_col"), R.indices.astype(np.int32))
        if golden.levels[-1].get("dense_n", 0):
            assert np.array_equal(G.export_ints(0, "jpvt"), np.asarray(golden.levels[-1]["qr_jpvt"], dtype=np.int32))


def test_norm2_on_device_matches_the_reference_scaling():
    """a13: norm2 is max-scaled (utils/math.hpp:112-137) -- finite for inputs whose squares overflow or
    underflow -- and deterministic (fixed two-stage reduction)."""
    import torch
    g = load_golden("poisson14_ml")
    rng = np.random.default_rng(7)
    with _gpu(g) as G:
        for n in (1, 31, 1000, 100003):
            for scale in (1.0, 1e200, 1e-200):
                v = rng.uniform(-1, 1, n) * scale
                d = torch.from_numpy(v).cuda()
                got = G.norm2_dev(d.data_ptr(), n)
                ref = float(np.linalg.norm(v / scale) * scale)
                assert np.isfinite(got) and abs(got - ref) <= 1e-13 * ref, (n, scale, got, ref)
                assert got == G.norm2_dev(d.data_ptr(), n)
        z = torch.zeros(100, dtype=torch.float64, device="cuda")
        assert G.norm2_dev(z.data_ptr(), 100) == 0.0


def _dense_only_level(R, Qraw_tau_piv, rank):
    (qr, tau), piv = Qraw_tau_piv
    nm = qr.shape[0]
    return dict(m=0, n=nm, dense_n=nm, dense_rank=rank, has_symm_dense=0, L=_ccs(np.zeros((0, 0))),
                U=_ccs(np.zeros((0, 0))), E=_ccs(np.zeros((nm, 0))), F=_ccs(np.zeros((0, nm))), d=np.zeros(0),
                s=np.ones(nm), t=np.ones(nm), p=np.arange(nm, dtype=np.int32), q=np.arange(nm, dtype=np.int32),
                p_inv=np.arange(nm, dtype=np.int32), q_inv=np.arange(nm, dtype=np.int32),
                qr_mat=np.asfortranarray(qr).ravel(order="F"), qr_tau=tau, qr_jpvt=(piv + 1).astype(np.int32))


@pytest.mark.parametrize("nm,rank", [(70, 45), (100, 33), (64, 64), (215, 215)], ids=lambda v: str(v))
def test_dense_level_rank_deficient_and_ill_conditioned(nm, rank):
    """QRCP.hpp:370-411 at the edges the suite did not cover: (i) an EXACTLY rank-deficient Schur block
    (zero columns beyond the numerical rank, rank not a multiple of the 32 x 32 tiles) solved with the
    numerical rank -- the inverted diagonal tiles then hold non-finite entries beyond the rank, which
    must never reach the arithmetic; (ii) a full-rank, badly conditioned block (cond ~ 1e12) solved with
    the full rank as hif::HIF::hifir does (builder.hpp:461).  Checked against the C oracle (unblocked
    dorm2r + dtrsv)."""
    import scipy.linalg as sl
    rng = np.random.default_rng(nm * 1000 + rank)
    if rank < nm:
        B = rng.uniform(-1, 1, (nm, rank)) @ rng.uniform(-1, 1, (rank, nm))
        (qr, tau), _, piv = sl.qr(B, mode="raw", pivoting=True)
        qr = np.array(qr)
        for j in range(rank, nm):  # what an exactly singular block leaves behind: zero trailing rows of R
            qr[rank:j + 1, j] = 0.0
    else:
        U_, _ = np.linalg.qr(rng.uniform(-1, 1, (nm, nm)))
        V_, _ = np.linalg.qr(rng.uniform(-1, 1, (nm, nm)))
        B = U_ @ np.diag(np.logspace(0, -12, nm)) @ V_.T
        (qr, tau), _, piv = sl.qr(B, mode="raw", pivoting=True)
    lev = _dense_only_level(None, ((qr, tau), piv), rank)
    Oh = O.OracleHif([lev])
    with hb.GpuHif([lev]) as G:
        for k in range(3):
            b = rng.uniform(-1, 1, nm)
            for r in ((0,) if rank < nm else (0, hb.FULL_RANK)):
                import torch
                db = torch.from_numpy(b).cuda()
                dx = torch.empty_like(db)
                G.solve_dev(db.data_ptr(), dx.data_ptr(), r)
                G.synchronize()
                x = dx.cpu().numpy()
                assert np.all(np.isfinite(x))
                ref = Oh.solve(b, 0 if r == 0 else nm)
                # a cond ~ 1e12 triangular solve amplifies the rounding of the two (equally valid) arithmetic orders
                assert relerr(x, ref) <= (TOL_F64 if rank < nm else 1e-6), (nm, rank, r, relerr(x, ref))


def test_transposed_solve_uses_nsp_tran_only():
    """hif::HIF::solve(b, x, true) filters with nsp_tran, never with nsp (builder.hpp:419-422)."""
    g = load_golden("poisson14_ml")
    b = np.ascontiguousarray(g["B"][:, 0])
    with _gpu(g) as G:
        x_sh, _ = G.apply(b, op=hb.LHF_SH)
        assert relerr(x_sh, g["x_SH"]) <= TOL_F64
        G.set_nsp_const()  # the filter of the plain solve does not touch the transposed one
        x2, _ = G.apply(b, op=hb.LHF_SH)
        assert np.array_equal(x2 != x2, np.zeros_like(x2, dtype=bool)) and relerr(x2, g["x_SH"]) <= TOL_F64
        xs, _ = G.apply(b)
        assert abs(xs.mean()) <= 1e-14 * np.abs(xs).max() + 1e-300
        G.set_nsp_tran_const()
        x3, _ = G.apply(b, op=hb.LHF_SH)
        assert relerr(x3, g["x_SH"] - g["x_SH"].mean()) <= 1e-12
        G.clear_nsp()
        x4, _ = G.apply(b, op=hb.LHF_SH)
        assert relerr(x4, g["x_SH"]) <= TOL_F64


def test_pipelined_host_solves_equal_synchronous_ones(golden):
    """lhfdGpuSolveAsync: same result as lhfdGpuSolve for a stream of right-hand sides over two slots."""
    import torch
    with _gpu(golden) as G:
        B = golden["B"]
        nb = B.shape[1]
        bs = [torch.from_numpy(np.ascontiguousarray(B[:, k])).pin_memory() for k in range(nb)]
        xs = [torch.empty(golden.n, dtype=torch.float64).pin_memory() for _ in range(3 * nb)]
        for rep in range(3):
            for k in range(nb):
                G.solve_async(bs[k].numpy(), xs[rep * nb + k].numpy())
        G.synchronize()
        for rep in range(3):
            for k in range(nb):
                assert relerr(xs[rep * nb + k].numpy(), golden["X"][:, k]) <= TOL_F64
