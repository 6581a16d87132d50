"""Block FGMRES / GMRES / fixed-count refinement over many right-hand sides (lhfdGpuFgmresMrhs,
lhfdGpuGmresMrhs, lhfdGpuHifirMrhsDev).  Semantics: nrhs independent fgmres_hifir / gmres_hif / hifir
runs, one per column -- checked column by column against the C oracle, the golden vectors and the
single-rhs device solver."""
import ctypes as C

import numpy as np
import pytest

import hifir_b200 as hb
from conftest import TOL_F64, load_golden, relerr
from hifir_b200 import problems as P

NSP_FREE = ("demo_A", "poisson14_ml", "convdiff14_ml", "stokes28_ml")
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def built():
    from hifir_b200 import build
    build.build()
    return hb.lib()


def _gpu(g):
    G = hb.GpuHif(g.levels)
    G.set_matrix(g.A)
    return G


def _oracle(g):
    from oracle import port as O
    return O.OracleHif(g.levels, g.A)


def _block(g):
    """b_krylov plus 4 seeded columns"""
    return np.ascontiguousarray(np.column_stack([g["b_krylov"], P.seeded_rhs(g.n, 0, nrhs=4)]))


def _col(B, k):
    return np.ascontiguousarray(B[:, k])


def _nmv_tol(riters, rnmv):  # as test_krylov_iteration_parity
    return max(1, rnmv // max(riters, 1))


def test_null_handle_is_refused(built):
    lib = built
    x = np.zeros(4)
    p = x.ctypes.data_as(C.c_void_p)
    assert lib.lhfdGpuFgmresMrhs(None, 2, p, 30, 1e-6, 500, 0, p, None, None, None) == hb.LHF_NULL_OBJ
    assert lib.lhfdGpuGmresMrhs(None, 2, p, 30, 1e-6, 500, p, None, None) == hb.LHF_NULL_OBJ
    assert lib.lhfdGpuHifirMrhsDev(None, 2, p, 2, p, 0) == hb.LHF_NULL_OBJ
    assert b"NULL" in lib.lhfGpuGetErrorMsg()
    for name in ("lhfdGpuFgmresMrhs", "lhfdGpuGmresMrhs", "lhfdGpuHifirMrhsDev"):
        assert name in hb.EXPORTED_SYMBOLS


@gpu
@pytest.mark.parametrize("which", ["fgmres", "gmres"])
@pytest.mark.parametrize("case", NSP_FREE)
def test_block_krylov_matches_oracle_per_column(built, case, which):
    g = load_golden(case)
    Oh = _oracle(g)
    B = _block(g)
    with _gpu(g) as G:
        if which == "fgmres":
            X, flags, iters, nmv = G.fgmres_mrhs(B, restart=g.restart)
        else:
            X, flags, iters = G.gmres_mrhs(B, restart=g.restart)
            nmv = iters
    for k in range(B.shape[1]):
        b = _col(B, k)
        xr, rflag, riters, rnmv = Oh.krylov(b, which, restart=g.restart)
        assert flags[k] == rflag, (k, flags[k], rflag)
        assert abs(iters[k] - riters) <= 1, (k, iters[k], riters)
        assert abs(nmv[k] - rnmv) <= _nmv_tol(riters, rnmv), (k, nmv[k], rnmv)
        assert np.linalg.norm(b - P.csr_matvec(g.A, X[:, k])) <= 2e-6 * np.linalg.norm(b), k
        assert relerr(X[:, k], xr) <= 1e-5, k
    rflag, riters, rnmv = (int(v) for v in g[which + "_status"])
    assert flags[0] == rflag and abs(iters[0] - riters) <= 1
    assert relerr(X[:, 0], g["x_" + which]) <= 1e-5


@gpu
@pytest.mark.parametrize("case", ["poisson14_ml", "stokes28_ml"])
def test_block_fgmres_matches_single_rhs_device_solver(built, case):
    g = load_golden(case)
    B = _block(g)
    with _gpu(g) as G:
        X, flags, iters, nmv = G.fgmres_mrhs(B, restart=g.restart)
        for k in range(B.shape[1]):
            x, f, it, _ = G.fgmres(_col(B, k), restart=g.restart)
            assert flags[k] == f and abs(iters[k] - it) <= 1, (k, flags[k], f, iters[k], it)
            assert relerr(X[:, k], x) <= 1e-6, k
        # one column: the single-rhs solver itself, bit for bit
        b = _col(B, 1)
        x, f, it, nm = G.fgmres(b, restart=g.restart)
        X1, f1, it1, nm1 = G.fgmres_mrhs(b[:, None], restart=g.restart)
        assert np.array_equal(X1[:, 0], x) and (f1[0], it1[0], nm1[0]) == (f, it, nm)
        # no columns: nothing to do
        X0, f0, _, _ = G.fgmres_mrhs(np.zeros((g.n, 0)))
        assert X0.shape == (g.n, 0) and f0.size == 0
        p = b.ctypes.data_as(C.c_void_p)
        assert hb.lib().lhfdGpuFgmresMrhs(G._h, 0, p, 30, 1e-6, 500, 0, p, None, None, None) == hb.LHF_SUCCESS


@gpu
def test_retired_columns_and_lockstep(built):
    """[b, 0, b, b', b] on Stokes: the zero column is inactive from the start, the copies of b retire together
    and see bit-identical arithmetic, b' runs on past them and past restart boundaries."""
    g = load_golden("stokes28_ml")
    Oh = _oracle(g)
    b = np.ascontiguousarray(g["b_krylov"])
    b2 = P.seeded_rhs(g.n, 0)
    B = np.ascontiguousarray(np.column_stack([b, np.zeros(g.n), b, b2, b]))
    with _gpu(g) as G:
        for which in ("fgmres", "gmres"):
            if which == "fgmres":
                X, flags, iters, nmv = G.fgmres_mrhs(B, restart=g.restart)
            else:
                X, flags, iters = G.gmres_mrhs(B, restart=g.restart)
                nmv = iters
            assert np.all(X[:, 1] == 0.0) and (flags[1], iters[1], nmv[1]) == (0, 0, 0)
            for k in (2, 4):
                assert (flags[k], iters[k], nmv[k]) == (flags[0], iters[0], nmv[0])
                assert relerr(X[:, k], X[:, 0]) <= 1e-14
            # the columns really finish at different counts, and past a restart boundary
            assert iters[3] != iters[0] and max(iters[0], iters[3]) > g.restart, (which, iters)
            for k in (0, 3):
                xr, rflag, riters, rnmv = Oh.krylov(_col(B, k), which, restart=g.restart)
                assert flags[k] == rflag and abs(iters[k] - riters) <= 1, (which, k, iters[k], riters)
                assert abs(nmv[k] - rnmv) <= _nmv_tol(riters, rnmv)
                assert relerr(X[:, k], xr) <= 1e-5
        # every column stops on the iteration limit (flag 2) inside the third cycle
        X, flags, iters, nmv = G.fgmres_mrhs(B, restart=3, maxit=7)
        for k in (0, 2, 3, 4):
            xr, rflag, riters, rnmv = Oh.krylov(_col(B, k), "fgmres", restart=3, maxit=7)
            assert rflag == 2 and flags[k] == 2 and iters[k] == riters and nmv[k] == rnmv, (k, flags[k], iters[k])
            assert relerr(X[:, k], xr) <= 1e-6, k
        assert np.all(X[:, 1] == 0.0) and (flags[1], iters[1], nmv[1]) == (0, 0, 0)


@gpu
@pytest.mark.parametrize("nrhs", [2, 17, 64, 70])
def test_block_widths(built, nrhs):
    """one pass, ragged passes and several passes of the batched apply; the handle keeps serving other widths"""
    g = load_golden("stokes28_ml")
    Oh = _oracle(g)
    B = P.seeded_rhs(g.n, 300, nrhs=nrhs)
    with _gpu(g) as G:
        X, flags, iters, nmv = G.fgmres_mrhs(B, restart=g.restart, maxit=12)
        for k in range(nrhs):
            xr, rflag, riters, rnmv = Oh.krylov(_col(B, k), "fgmres", restart=g.restart, maxit=12)
            assert flags[k] == rflag and abs(iters[k] - riters) <= 1, (k, flags[k], rflag, iters[k], riters)
            assert abs(nmv[k] - rnmv) <= _nmv_tol(riters, rnmv)
            assert relerr(X[:, k], xr) <= 1e-5, k
        b = _col(B, 0)
        assert relerr(G.solve(b), Oh.solve(b)) <= TOL_F64
        B5 = P.seeded_rhs(g.n, 400, nrhs=5)
        Y = G.solve_mrhs(B5)
        for k in range(5):
            assert relerr(Y[:, k], Oh.solve(_col(B5, k))) <= TOL_F64


@gpu
@pytest.mark.parametrize("case", ["poisson14_ml", "stokes28_ml"])
def test_block_refinement_matches_oracle(built, case):
    import torch
    g = load_golden(case)
    Oh = _oracle(g)
    B = P.seeded_rhs(g.n, 500, nrhs=6)
    with _gpu(g) as G:
        dB = torch.from_numpy(B).cuda()
        dX = torch.empty_like(dB)
        for nirs in (1, 2, 3):
            for rank in (hb.FULL_RANK, 0):
                G.hifir_mrhs_dev(B.shape[1], dB.data_ptr(), nirs, dX.data_ptr(), rank)
                G.synchronize()
                X = dX.cpu().numpy()
                for k in range(B.shape[1]):
                    assert relerr(X[:, k], Oh.hifir(_col(B, k), nirs, rank)) <= TOL_F64, (nirs, rank, k)


@gpu
def test_single_precision_block_fgmres(built):
    g = load_golden("poisson14_ml_f32")
    B = np.ascontiguousarray(np.column_stack([P.csr_matvec(g.A, np.ones(g.n)), P.seeded_rhs(g.n, 0, nrhs=4)]))
    with _gpu(g) as G:
        assert G.single
        X, flags, iters, _ = G.fgmres_mrhs(B, restart=g.restart)
        for k in range(B.shape[1]):
            x, f, it, _ = G.fgmres(_col(B, k), restart=g.restart)
            assert flags[k] == f and abs(iters[k] - it) <= 1, (k, flags[k], f, iters[k], it)


@gpu
def test_refusals(built):
    g = load_golden("neumann12_nsp")
    B = _block(g)
    with _gpu(g) as G:
        G.set_nsp_const()
        for call in (lambda: G.fgmres_mrhs(B), lambda: G.gmres_mrhs(B)):
            with pytest.raises(hb.LhfError) as e:
                call()
            assert e.value.status == hb.LHF_BAD_PREC and "null space" in str(e.value)
        import torch
        dB = torch.from_numpy(B).cuda()
        with pytest.raises(hb.LhfError) as e:
            G.hifir_mrhs_dev(B.shape[1], dB.data_ptr(), 2, dB.data_ptr())
        assert e.value.status == hb.LHF_BAD_PREC
        G.clear_nsp()
        for restart in (0, 97):
            with pytest.raises(hb.LhfError) as e:
                G.fgmres_mrhs(B, restart=restart)
            assert e.value.status == hb.LHF_BAD_PREC
        # n * nrhs beyond 2^32: refused before any device memory is touched
        huge = (1 << 32) // g.n + 1
        with pytest.raises(hb.LhfError) as e:
            G.hifir_mrhs_dev(huge, dB.data_ptr(), 2, dB.data_ptr())
        assert e.value.status == hb.LHF_MISMATCHED_SIZES
    g = load_golden("stokes28_ml")
    with hb.GpuHif(g.levels) as G:  # no matrix attached
        B = _block(g)
        for call in (lambda: G.fgmres_mrhs(B), lambda: G.gmres_mrhs(B)):
            with pytest.raises(hb.LhfError) as e:
                call()
            assert e.value.status == hb.LHF_BAD_PREC
