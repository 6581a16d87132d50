"""Pin the plain-C oracle (oracle/hif_oracle.c) before anything trusts it:
(a) against the committed golden vectors produced by the unmodified reference,
(b) against the reference itself, live, on the same factorized object (when oracle/_ref is present),
(c) against the reference's known-answer test of the dense level (tests/test_sss_qrcp.cpp)."""
import numpy as np
import pytest

from conftest import GOLDEN_DIR, have_reference, load_golden, relerr
from hifir_b200 import problems as P
from oracle import port as O

PORT_TOL = 1e-13  # port vs reference: same loop order, only -ffast-math contraction differs


def _oracle(g):
    Oh = O.OracleHif(g.levels, g.A)
    if g.nsp:
        Oh.set_nsp_const()
    return Oh


def test_port_solve_matches_golden(golden):
    Oh = _oracle(golden)
    for k in range(golden["B"].shape[1]):
        b = np.ascontiguousarray(golden["B"][:, k])
        assert relerr(Oh.solve(b), golden["X"][:, k]) <= PORT_TOL
        assert relerr(Oh.solve(b, O.FULL_RANK), golden["X_full"][:, k]) <= PORT_TOL


def test_port_hifir_matches_golden(golden):
    Oh = _oracle(golden)
    b = np.ascontiguousarray(golden["B"][:, 0])
    assert relerr(Oh.hifir(b, 3), golden["x_hifir3"]) <= PORT_TOL
    x, iters, flag = Oh.hifir_betas(golden["b_krylov"], 16, [1e-8, 1e10])
    assert (iters, flag) == tuple(int(v) for v in golden["hifir_betas_status"])
    assert relerr(x, golden["x_hifir_betas"]) <= 1e-10


def test_port_other_operations_match_golden(golden):
    """lhf?Apply's other operations (libhifir.cpp:447-472): S^H = prec_solve_tran (prec_solve.hpp:541-612),
    M / M^H = prec_prod / prec_prod_tran (prec_prod.hpp:54-230), numerical and full last-level rank."""
    if golden.nsp:
        pytest.skip("fixture made with the null-space filter; the reference has no transposed filter set")
    Oh = _oracle(golden)
    b = np.ascontiguousarray(golden["B"][:, 0])
    for op, key in ((1, "x_SH"), (2, "x_M"), (3, "x_MH")):
        assert relerr(Oh.apply_op(op, b), golden[key]) <= PORT_TOL
        assert relerr(Oh.apply_op(op, b, O.FULL_RANK), golden[key + "_full"]) <= PORT_TOL


@pytest.mark.parametrize("which", ["fgmres", "gmres"])
def test_port_krylov_matches_golden(golden, which):
    if which == "gmres" and golden.name == "stokes28_ml":
        pytest.skip("230-iteration GMRES: covered by fgmres on this case")
    Oh = _oracle(golden)
    x, flag, iters, nmv = Oh.krylov(golden["b_krylov"], which, restart=golden.restart)
    rflag, riters, rnmv = (int(v) for v in golden[which + "_status"])
    assert flag == rflag
    assert abs(iters - riters) <= 1 and abs(nmv - rnmv) <= max(1, rnmv // max(riters, 1))
    assert relerr(x, golden["x_" + which]) <= 1e-6


def test_port_roundtrip_invariant(golden):
    """libhifir/tests/test_real.c:146 -- ||M (M^-1 b) - b|| / ||b|| <= 1e-10 (reference's M x stored)."""
    if golden.nsp:
        pytest.skip("filtered solve is not the inverse of M")
    b = golden["B"][:, 0]
    assert relerr(golden["Mx"], b) <= 1e-10


def test_qrcp_known_answer():
    """reference tests/test_sss_qrcp.cpp:16-197: 20x20 system, |x - x_ref| <= 1e-10."""
    z = np.load(f"{GOLDEN_DIR}/qrcp_kat.npz")
    x = O.qrcp_solve(z["mat"], z["tau"], z["jpvt"], int(z["rank"]), z["b"])
    assert np.abs(x - z["x_ref"]).max() <= 1e-10
    assert np.abs(x - z["x_lapack"]).max() <= 1e-13
    # truncated rank: entries of the dropped pivots are exactly zero (QRCP.hpp:404-405)
    xt = O.qrcp_solve(z["mat"], z["tau"], z["jpvt"], int(z["rank"]), z["b"], rank=15)
    assert np.count_nonzero(xt) == 15 and all(xt[z["jpvt"][15:] - 1] == 0.0)


def test_norm2_restatement():
    v = P.seeded_rhs(1000, 3) * 1e200
    assert np.isclose(O.norm2(v), np.linalg.norm(v / 1e200) * 1e200, rtol=1e-14)
    assert O.norm2(np.zeros(5)) == 0.0


def test_ccs_to_crs_restatement(golden):
    import scipy.sparse as sp
    for L in golden.levels:
        for name in ("L", "U", "E", "F"):
            nr, nc, cs, ri, va = L[name]
            rs, ci, v = O.ccs_to_crs(L[name])
            if len(cs) < nc + 1:
                assert rs[-1] == 0
                continue
            ref = sp.csc_matrix((va, ri, cs), shape=(nr, nc)).tocsr()
            ref.sort_indices()
            assert np.array_equal(rs, ref.indptr) and np.array_equal(ci, ref.indices) and np.array_equal(v, ref.data)


# ---------------------------------------------------------------- single precision
# The oracle for hif::HIF<float,int> is the same C restatement run in double on the widened float
# factors; it is pinned here against the reference's own single-precision outputs (float work
# vectors, builder.hpp:125-131): they differ by the reference's float rounding only.
F32_PORT_TOL = 2e-6


def test_port_on_float_factors_matches_float_reference(golden_f32):
    from conftest import TOL_F32
    g = golden_f32
    assert g.levels[0]["L"][4].dtype == np.float32 and g.levels[0]["s"].dtype == np.float32
    Oh = _oracle(g)
    for k in range(g["B"].shape[1]):
        b = np.ascontiguousarray(g["B"][:, k])
        assert relerr(Oh.solve(b), g["X"][:, k]) <= F32_PORT_TOL          # lhfsdSolve
        assert relerr(Oh.solve(b, O.FULL_RANK), g["X_full"][:, k]) <= F32_PORT_TOL
        assert relerr(Oh.solve(b), g["X32"][:, k]) <= F32_PORT_TOL        # lhfsSolve (float vectors)
    b = np.ascontiguousarray(g["B"][:, 0])
    assert relerr(Oh.hifir(b, 3), g["x_hifir3"]) <= TOL_F32               # refinement with the double matrix
    if not g.nsp:
        for op, key in ((1, "x_SH"), (2, "x_M"), (3, "x_MH")):
            assert relerr(Oh.apply_op(op, b), g[key]) <= F32_PORT_TOL, key


# ---------------------------------------------------------------- live reference
needs_ref = pytest.mark.skipif(not have_reference(), reason="needs oracle/_ref/libhifir_ref.so, built from the reference HIFIR sources, which this repository does not contain")


@needs_ref
@pytest.mark.parametrize("case", ["poisson", "convdiff", "stokes", "neumann"])
def test_port_vs_live_reference(case):
    from oracle import refhost as R
    gen, N, dt = {"poisson": (P.poisson3d, 20, 100), "convdiff": (P.convdiff3d, 18, 100),
                  "stokes": (P.stokes2d_mac, 40, 100), "neumann": (P.neumann3d, 16, 100)}[case]
    A = gen(N)
    M = R.RefHif(A, P.PDE_PARAMS, dense_thres=dt)
    Oh = O.OracleHif(M.levels(), A)
    if case == "neumann":
        M.set_nsp_const()
        Oh.set_nsp_const()
    b = P.seeded_rhs(A[0], 7)
    assert relerr(Oh.solve(b), M.solve(b)) <= PORT_TOL
    assert relerr(Oh.solve(b, O.FULL_RANK), M.solve(b, R.FULL_RANK)) <= PORT_TOL
    assert relerr(Oh.hifir(b, 4), M.hifir(b, 4)) <= PORT_TOL
    bk = P.csr_matvec(A, np.sin(0.37 * np.arange(A[0])))
    xo, fo, io, no = Oh.krylov(bk, "fgmres", restart=10)
    xr, fr, ir, nr = M.krylov(bk, "fgmres", restart=10)
    assert (fo, io, no) == (fr, ir, nr)
    assert relerr(xo, xr) <= 1e-8
    assert np.isclose(O.norm2(b), R.norm2(b), rtol=1e-14)


@needs_ref
def test_port_vs_live_float_reference():
    """hif::HIF<float,int> factorized here from the double matrix (demo_mixedprecision.cpp)"""
    from oracle import refhost as R
    A = P.convdiff3d(16)
    M = R.RefHif(A, P.PDE_PARAMS, dense_thres=100, dtype=np.float32)
    lv = M.levels()
    assert all(L[k][4].dtype == np.float32 for L in lv for k in "LUEF")
    Oh = O.OracleHif(lv, A)
    b = P.seeded_rhs(A[0], 7)
    assert relerr(Oh.solve(b), M.solve(b)) <= F32_PORT_TOL
    assert relerr(Oh.solve(b), M.solve_f32(b)) <= F32_PORT_TOL
    assert relerr(Oh.hifir(b, 4), M.hifir(b, 4)) <= 1e-5


@needs_ref
def test_reference_crs_conversion_is_what_the_port_restates():
    from oracle import refhost as R
    A = P.poisson3d(10)
    M = R.RefHif(A, P.PDE_PARAMS, dense_thres=40)
    for lvl, L in enumerate(M.levels()):
        for which, name in enumerate(("L", "U", "E", "F")):
            nr, nc, cs, ri, va = L[name]
            if len(ri) == 0:
                continue
            rs, ci, v = O.ccs_to_crs(L[name])
            rrs, rci, rv = R.export_crs(M, lvl, which, nr, len(ri))
            assert np.array_equal(rs, rrs) and np.array_equal(ci, rci) and np.array_equal(v, rv)


@needs_ref
def test_goldens_are_reproducible_here():
    """The committed demo_A golden equals what the reference produces in this container."""
    from oracle import refhost as R
    g = load_golden("demo_A")
    M = R.RefHif(g.A)
    assert relerr(M.solve(np.ascontiguousarray(g["B"][:, 0])), g["X"][:, 0]) <= 1e-14
