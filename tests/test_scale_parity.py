"""The device path at the sizes the benchmark runs, against the C oracle on the same levels.

The golden fixtures (n <= 2 744) leave every size-dependent structure in its trivial case: under one warp-stream
segment per warp, one grid-stride pass of the reductions, one element per thread of the persistent Gram-Schmidt
slice, one row per thread of the block Krylov kernels, dense last levels of at most 215 rows.  The factors here
come from oracle/factor.py, as the benchmark's do, and reach all of them:

  P64   Poisson 64^3       n =   262 144, 3 levels, dense last level nm = 483
  C96   conv-diff 96^3     n =   884 736, 4 levels (the benchmark's multi-rhs workload)
  S400  Stokes MAC 400     n =   479 200, 4 levels, zero-diagonal rows deferred
  N48   Neumann 48^3       n =   110 592, constant null-space filter
  P64f  P64 with float factors (single-precision handle)
  P156  Poisson 156^3      n = 3 796 416: a Gram-Schmidt slice of ceil(n / 148) entries no longer fits the
        200 KB of the persistent kernel, the Krylov loop runs the per-step kernels (Krylov test only)

Krylov solves are compared after a FIXED number of steps (flag 2): two correct GMRES runs agree far more tightly
there than after convergence, so a reduction that is off in the 9th digit fails the gate.  The switches that the
library caches in function-local statics on first use run in a fresh interpreter."""
import json
import math
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

import hifir_b200 as hb
from conftest import ROOT, TOL_F64, relerr
from hifir_b200 import problems as P

gpu = pytest.mark.gpu
TOL_SINGLE = 2e-6  # float factors against the double oracle on the same float factors (worst observed 3.9e-9)
# Device against oracle, relative error of the iterate after a fixed number of (F)GMRES steps.  Worst observed on
# a B200 (1000 W power limit): 5.3e-14 single-rhs (P156), 1.0e-13 block (P64, 70 columns); with float factors
# 5.3e-11 (P64f: the merged sweep values are rounded to float, the oracle's are not).
KRYLOV_GATE = 1e-10
KRYLOV_GATE_SINGLE = 1e-8

FIXTURES = {
    "P64": (P.poisson3d, 64, np.float64, False),
    "C96": (P.convdiff3d, 96, np.float64, False),
    "S400": (P.stokes2d_mac, 400, np.float64, False),
    "N48": (P.neumann3d, 48, np.float64, True),
    "P64f": (P.poisson3d, 64, np.float32, False),
    "P156": (P.poisson3d, 156, np.float64, False),
}
APPLY_CASES = ("P64", "C96", "S400", "N48", "P64f")

# Regime floors, about half of what the factors give today (L0 / U0 of level 0, host packing for 148 SMs x 24
# warps = 3 552 warps): slices of the warp streams (>> 2 per warp: the TMA rings wrap, level sets go "wide"),
# packed bytes (HBM-streamed, beyond the 126 MB L2 for the fused L+U stream of C96 / S400), merged entries.
REGIME_FLOORS = {  # name: (slices, bytes, merged entries)
    "P64": (25_000, 56e6, 3.5e6),      # today: 50 551 / 49 564 slices, 112 / 115 MB, 7.2 / 7.4 M entries
    "C96": (52_000, 120e6, 7.5e6),     # 105 702 / 103 443, 241 / 244 MB, 15.2 / 15.5 M
    "S400": (38_000, 79e6, 5.0e6),     # 77 300 / 77 168, 160 / 158 MB, 10.0 / 10.0 M
    "N48": (14_000, 31e6, 2.0e6),      # 28 793 / 29 430, 64 / 65 MB, 4.0 / 4.1 M
    "P64f": (25_000, 40e6, 3.5e6),     # 50 551 / 49 564, 80 / 82 MB (8 bytes per entry), 7.2 / 7.4 M
}
PERSIST_LIMIT = 148 * 25_600  # krylov.cu: n beyond this, the persistent Gram-Schmidt slice exceeds 200 KB


class Case:
    def __init__(self, name):
        from oracle import factor as F
        gen, size, dtype, nsp = FIXTURES[name]
        self.name, self.nsp, self.single = name, nsp, dtype == np.float32
        self.A = gen(size)
        self.n = self.A[0]
        self.levels = F.multilevel_levels(self.A, dtype)
        self.tol = TOL_SINGLE if self.single else TOL_F64
        self.kgate = KRYLOV_GATE_SINGLE if self.single else KRYLOV_GATE
        self._oracle, self._memo, self._handle = None, {}, None

    @property
    def oracle(self):
        """the C oracle on the same levels (float factors: in double on the float values)"""
        if self._oracle is None:
            from oracle import port as O
            self._oracle = O.OracleHif(self.levels, self.A)
            if self.nsp:
                self._oracle.set_nsp_const()
        return self._oracle

    def ref(self, key, fn):
        """oracle results are shared between the tests of the module"""
        if key not in self._memo:
            self._memo[key] = fn()
        return self._memo[key]

    def solve_ref(self, j):
        return self.ref(("solve", j), lambda: self.oracle.solve(P.seeded_rhs(self.n, j)))

    def krylov_ref(self, j, which, restart, maxit, rtol=1e-6):
        b = self.rhs(j)
        return self.ref(("krylov", j, which, restart, maxit, rtol),
                        lambda: self.oracle.krylov(b, which, restart=restart, rtol=rtol, maxit=maxit))

    def rhs(self, j):
        return P.seeded_rhs(self.n, j)

    def attach(self):
        G = hb.GpuHif(self.levels)
        G.set_matrix(self.A)
        if self.nsp:
            G.set_nsp_const()
        return G

    def handle(self):
        """one handle per fixture, attached with the default configuration, shared by the module"""
        if self._handle is None:
            self._handle = self.attach()
        return self._handle

    def close(self):
        if self._handle is not None:
            self._handle.close()
            self._handle = None


_cases = {}


def case(name):
    if name not in _cases:
        _cases[name] = Case(name)
    return _cases[name]


@pytest.fixture(scope="module")
def built():
    from hifir_b200 import build
    build.build()
    yield hb.lib()
    for c in _cases.values():
        c.close()


def _col(B, k):
    return np.ascontiguousarray(B[:, k])


def _nmv_tol(riters, rnmv):  # as test_krylov_iteration_parity
    return max(1, rnmv // max(riters, 1))


# ------------------------------------------------------------------ 1. regime guard (host only)
@pytest.mark.parametrize("name", list(REGIME_FLOORS))
def test_factors_reach_the_benchmark_regime(built, name):
    """Without this guard a change to factor.py or to the packing could shrink the module back into the
    trivial case of the goldens unnoticed."""
    c = case(name)
    floor_slices, floor_bytes, floor_merged = REGIME_FLOORS[name]
    L0 = c.levels[0]
    rhs = np.random.default_rng(0).uniform(-1, 1, L0["m"])
    d = np.asarray(L0["d"], dtype=np.float64)
    for blk, upper in (("L", False), ("U", True)):
        _, st = hb.debug_sweep_host(L0[blk], upper, rhs, d if upper else None)
        plan = hb.debug_merge_plan(L0[blk], upper)
        assert st["slices"] >= floor_slices and st["slices"] > 2 * 1776, (name, blk, st)
        assert st["bytes"] >= floor_bytes, (name, blk, st)
        assert plan["merged_entries"] >= floor_merged, (name, blk, plan)
    if name == "P64":
        assert c.n > 151_552 and c.levels[-1]["dense_n"] > 256, "past one reduction pass, past 256 dense rows"
    assert FIXTURES["P156"][1] ** 3 > PERSIST_LIMIT


# ------------------------------------------------------------------ 2. apply parity at scale
@gpu
@pytest.mark.parametrize("name", APPLY_CASES)
def test_apply_parity_at_scale(built, name, record_property):
    import torch
    c = case(name)
    G, Oh = c.handle(), c.oracle
    errs = []
    for j in range(3):
        errs.append(relerr(G.solve(c.rhs(j)), c.solve_ref(j)))
    assert max(errs) <= c.tol, errs
    # repeated applies flip the ready-bit parity
    b = c.rhs(0)
    x1, x2, x3 = G.solve(b), G.solve(b), G.solve(b)
    assert np.array_equal(x1, x3) and relerr(x2, x1) <= 1e-14, relerr(x2, x1)
    x, _ = G.apply(b, nirs=3)
    e = relerr(x, c.ref(("hifir", 0, 3), lambda: Oh.hifir(b, 3)))
    errs.append(e)
    assert e <= c.tol, e
    if not c.nsp:
        for op in (hb.LHF_SH, hb.LHF_M, hb.LHF_MH):
            x, _ = G.apply(b, op=op)
            e = relerr(x, Oh.apply_op(int(op), b))
            errs.append(e)
            assert e <= c.tol, (op, e)
        if not c.single:  # float factors: M^-1 streams float-rounded merged values, M does not
            db = torch.from_numpy(b).cuda()
            dx, dy = torch.empty_like(db), torch.empty_like(db)
            G.apply_dev(db.data_ptr(), dx.data_ptr(), op=hb.LHF_S)
            G.apply_dev(dx.data_ptr(), dy.data_ptr(), op=hb.LHF_M)
            G.synchronize()
            assert relerr(dy.cpu().numpy(), b) <= 1e-10
    b2 = c.rhs(1)
    x1, x2, x12 = G.solve(b), G.solve(b2), G.solve(2.0 * b - 3.0 * b2)
    assert relerr(x12, 2.0 * x1 - 3.0 * x2) <= 1e-11
    # truncated rank of the dense last level through the device-pointer entry point
    rank = c.levels[-1]["dense_rank"] - 1
    db = torch.from_numpy(b).cuda()
    dx = torch.empty_like(db)
    if c.nsp:
        G.clear_nsp()
        Oh.clear_nsp()
    try:
        G.solve_dev(db.data_ptr(), dx.data_ptr(), rank)
        G.synchronize()
        e = relerr(dx.cpu().numpy(), Oh.solve(b, rank))
    finally:
        if c.nsp:
            G.set_nsp_const()
            Oh.set_nsp_const()
    errs.append(e)
    assert e <= c.tol, e
    record_property("worst_relerr", max(errs))


def _dense_level(nm, rank):
    import scipy.linalg as sl
    from test_gpu_parity import _dense_only_level
    rng = np.random.default_rng(nm * 7 + rank)
    if rank < nm:  # exactly rank-deficient, the trailing rows of R zero (as an exactly singular Schur block)
        B = rng.uniform(-1, 1, (nm, rank)) @ rng.uniform(-1, 1, (rank, nm))
        (qr, tau), _, piv = sl.qr(B, mode="raw", pivoting=True)
        qr = np.array(qr)
        for j in range(rank, nm):
            qr[rank:j + 1, j] = 0.0
    else:  # well conditioned: the two arithmetic orders agree to the double gate
        B = rng.uniform(-1, 1, (nm, nm)) / math.sqrt(nm) + 2.0 * np.eye(nm)
        (qr, tau), _, piv = sl.qr(B, mode="raw", pivoting=True)
    return _dense_only_level(None, ((qr, tau), piv), rank), rng


@gpu
@pytest.mark.parametrize("nm,rank", [(65, 65), (1000, 1000), (1500, 1111)], ids=lambda v: str(v))
def test_dense_only_level_at_scale(built, nm, rank, record_property):
    """dense levels past the one-launch path (nm > 64) and past 256 rows: the Q^T product, the transposed
    solve, both products and the multi-column triangular solve against the C oracle"""
    from oracle import port as O
    lev, rng = _dense_level(nm, rank)
    Oh = O.OracleHif([lev])
    worst = 0.0
    with hb.GpuHif([lev]) as G:
        for k in range(2):
            b = rng.uniform(-1, 1, nm)
            e = relerr(G.solve(b), Oh.solve(b))
            worst = max(worst, e)
            assert e <= TOL_F64, (k, e)
            for op in (hb.LHF_SH, hb.LHF_M, hb.LHF_MH):
                x, _ = G.apply(b, op=op)
                e = relerr(x, Oh.apply_op(int(op), b))
                worst = max(worst, e)
                assert e <= TOL_F64, (op, e)
        for nrhs in (5, 20, 70):
            B = rng.uniform(-1, 1, (nm, nrhs))
            X = G.solve_mrhs(B)
            for k in range(nrhs):
                e = relerr(X[:, k], Oh.solve(_col(B, k)))
                worst = max(worst, e)
                assert e <= TOL_F64, (nrhs, k, e)
    record_property("worst_relerr", worst)


# ------------------------------------------------------------------ 3. multi-rhs at scale
MRHS_SEED = 100


def _mrhs_block(c, nrhs=70):
    return P.seeded_rhs(c.n, MRHS_SEED, nrhs=nrhs)


@gpu
@pytest.mark.parametrize("name", ["C96", "P64f"])
def test_mrhs_at_scale(built, name, record_property):
    import torch
    c = case(name)
    G, Oh = c.handle(), c.oracle
    B = _mrhs_block(c)
    ref = [c.solve_ref(MRHS_SEED + k) for k in range(B.shape[1])]
    worst = 0.0
    # widths: one narrow pass, one pass of 32, one of 64, a pass of 64 and a ragged one; then the width
    # sequence 70 -> 5 -> 64 -> 3 on other column ranges of the same handle
    for lo, hi in ((0, 5), (0, 20), (0, 64), (0, 70), (0, 70), (65, 70), (6, 70), (1, 4)):
        X = G.solve_mrhs(np.ascontiguousarray(B[:, lo:hi]))
        for k in range(hi - lo):
            e = relerr(X[:, k], ref[lo + k])
            worst = max(worst, e)
            assert e <= c.tol, (lo, hi, k, e)
    Bk = np.ascontiguousarray(B[:, :6])
    dB = torch.from_numpy(Bk).cuda()
    dX = torch.empty_like(dB)
    for nirs in (2, 3):
        G.hifir_mrhs_dev(Bk.shape[1], dB.data_ptr(), nirs, dX.data_ptr())
        G.synchronize()
        X = dX.cpu().numpy()
        for k in range(Bk.shape[1]):
            r = c.ref(("hifir", MRHS_SEED + k, nirs), lambda: Oh.hifir(_col(Bk, k), nirs))
            e = relerr(X[:, k], r)
            worst = max(worst, e)
            assert e <= c.tol, (nirs, k, e)
    record_property("worst_relerr", worst)


# ------------------------------------------------------------------ 4. sweep configurations
SWEEP_CONFIGS = [
    *({"HIFIR_B200_WS_WARPS": str(w), "HIFIR_B200_WS_STAGES": str(s)}
      for w, s in ((16, 2), (16, 3), (16, 4), (20, 3), (24, 2), (28, 2), (32, 2))),
    {"HIFIR_B200_WS_PIPE": "1"},
    {"HIFIR_B200_WS_UMIN": "8"},
    {"HIFIR_B200_WS_GROUPS": "1"},
    {"HIFIR_B200_WS_GROUPS": "3"},
    {"HIFIR_B200_WS_WINDOW": "1"},
    {"HIFIR_B200_WS_WINDOW": "4"},
    {"HIFIR_B200_WS_FUSE": "0"},
    {"HIFIR_B200_MERGE_SLCAP": "1e3"},
    {"HIFIR_B200_MERGE_SLCAP": "3e4"},
    {"HIFIR_B200_MERGE_SLCAP": "3e5"},
    {"HIFIR_B200_MERGE": "0"},
    {"HIFIR_B200_SWEEP": "stream"},
]


def _config_id(cfg):
    return "-".join(f"{k[len('HIFIR_B200_'):].lower()}{v}" for k, v in cfg.items())


def _check_solves(c, G, nrhs=20):
    """2 single solves and one block of nrhs columns against the oracle; returns the worst error"""
    worst = 0.0
    for j in range(2):
        e = relerr(G.solve(c.rhs(j)), c.solve_ref(j))
        worst = max(worst, e)
        assert e <= c.tol, (j, e)
    X = G.solve_mrhs(_mrhs_block(c, nrhs))
    for k in range(nrhs):
        e = relerr(X[:, k], c.solve_ref(MRHS_SEED + k))
        worst = max(worst, e)
        assert e <= c.tol, (k, e)
    return worst


@gpu
@pytest.mark.parametrize("cfg", SWEEP_CONFIGS, ids=_config_id)
@pytest.mark.parametrize("name", ["P64", "P64f"])
def test_sweep_configuration_at_scale(built, name, cfg, monkeypatch, record_property):
    """Every configuration the attach accepts (read at attach; WS_PIPE at launch).  A plan that is not the
    fused 24 x 2 one sends solve_mrhs to streaming plans of its own (Lm / Um)."""
    c = case(name)
    for k, v in cfg.items():
        monkeypatch.setenv(k, v)
    with c.attach() as G:
        record_property("worst_relerr", _check_solves(c, G))


# switches cached in function-local statics: the first read in a process wins, so each runs in a child
CHILD = textwrap.dedent("""
    import json, sys
    sys.path.insert(0, sys.argv[1])
    import numpy as np
    import hifir_b200 as hb
    from hifir_b200 import problems as P
    from oracle import factor as F
    spec = json.loads(sys.argv[2])
    out = {}
    for name, gen, size, dtype in spec["cases"]:
        A = getattr(P, gen)(size)
        with hb.GpuHif(F.multilevel_levels(A, np.dtype(dtype))) as G:
            G.set_matrix(A)
            if spec["kind"] == "mrhs":
                for nrhs in (20, 70):
                    out[f"{name}/mrhs{nrhs}"] = G.solve_mrhs(P.seeded_rhs(A[0], spec["seed"], nrhs=nrhs))
                out[f"{name}/solve"] = G.solve(P.seeded_rhs(A[0], 0))
            else:
                for which in ("fgmres", "gmres"):
                    for maxit in (7, 23):
                        b = P.seeded_rhs(A[0], 0)
                        r = G.fgmres(b, 10, 1e-6, maxit) if which == "fgmres" else G.gmres(b, 10, 1e-6, maxit)
                        out[f"{name}/{which}{maxit}"] = r[0]
                        out[f"{name}/{which}{maxit}/counts"] = np.array(r[1:])
    np.savez(spec["out"], **out)
""")


def _run_child(env_over, kind, names, tmp_path):
    out = str(tmp_path / "child.npz")
    spec = dict(kind=kind, seed=MRHS_SEED, out=out,
                cases=[(nm, FIXTURES[nm][0].__name__, FIXTURES[nm][1], np.dtype(FIXTURES[nm][2]).name) for nm in names])
    env = dict(os.environ, **env_over)
    r = subprocess.run([sys.executable, "-c", CHILD, ROOT, json.dumps(spec)], env=env, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    with np.load(out) as z:
        return {k: z[k] for k in z.files}


@gpu
@pytest.mark.parametrize("env", [{"HIFIR_B200_MRHS_BATCH": "2"}, {"HIFIR_B200_MRHS_BATCH": "8"},
                                 {"HIFIR_B200_MRHS_WIDE": "0"}, {"HIFIR_B200_MRHS_WIDE": "16"},
                                 {"HIFIR_B200_MRHS_WIDE": "32"}], ids=_config_id)
def test_mrhs_switches_in_a_fresh_process(built, env, tmp_path, record_property):
    got = _run_child(env, "mrhs", ["P64", "P64f"], tmp_path)
    worst = 0.0
    for name in ("P64", "P64f"):
        c = case(name)
        e = relerr(got[f"{name}/solve"], c.solve_ref(0))
        worst = max(worst, e)
        assert e <= c.tol, (name, e)
        for nrhs in (20, 70):
            X = got[f"{name}/mrhs{nrhs}"]
            for k in range(nrhs):
                e = relerr(X[:, k], c.solve_ref(MRHS_SEED + k))
                worst = max(worst, e)
                assert e <= c.tol, (name, nrhs, k, e)
    record_property("worst_relerr", worst)


# ------------------------------------------------------------------ 5. Krylov iterates after a fixed step count
KRYLOV_CASES = ("P64", "C96", "S400")


def _check_fixed_steps(c, which, maxit, x, flag, iters, nmv):
    xr, rflag, riters, rnmv = c.krylov_ref(0, which, 10, maxit)
    assert rflag == 2 and flag == 2 and iters == riters, (c.name, which, maxit, flag, iters, riters)
    if which == "fgmres":
        assert nmv == rnmv, (nmv, rnmv)
    e = relerr(x, xr)
    assert e <= c.kgate, (c.name, which, maxit, e)
    return e


@gpu
@pytest.mark.parametrize("maxit", [7, 23])
@pytest.mark.parametrize("which", ["fgmres", "gmres"])
@pytest.mark.parametrize("name", KRYLOV_CASES)
def test_krylov_after_fixed_steps(built, name, which, maxit, record_property):
    """restart 10: maxit 23 crosses two restarts (FGMRES doubles the refinement count of its inner apply on
    every restart)"""
    c = case(name)
    G = c.handle()
    b = c.rhs(0)
    if which == "fgmres":
        x, flag, iters, nmv = G.fgmres(b, restart=10, maxit=maxit)
    else:
        (x, flag, iters), nmv = G.gmres(b, restart=10, maxit=maxit), None
    record_property("relerr", _check_fixed_steps(c, which, maxit, x, flag, iters, nmv))


@gpu
@pytest.mark.parametrize("env", [{"HIFIR_B200_MGS_PERSIST": "0"}, {"HIFIR_B200_MGS_FUSED": "0"}], ids=_config_id)
def test_krylov_gram_schmidt_variants_in_a_fresh_process(built, env, tmp_path, record_property):
    """the per-step fused Gram-Schmidt kernel and the unfused dot / axpy pair on the same cases"""
    got = _run_child(env, "krylov", KRYLOV_CASES, tmp_path)
    worst = 0.0
    for name in KRYLOV_CASES:
        c = case(name)
        for which in ("fgmres", "gmres"):
            for maxit in (7, 23):
                counts = got[f"{name}/{which}{maxit}/counts"]
                nmv = int(counts[2]) if which == "fgmres" else None
                worst = max(worst, _check_fixed_steps(c, which, maxit, got[f"{name}/{which}{maxit}"], int(counts[0]),
                                                      int(counts[1]), nmv))
    record_property("worst_relerr", worst)


@gpu
def test_krylov_past_the_persistent_gram_schmidt_limit(built, record_property):
    """P156: the slice of the persistent kernel would exceed its 200 KB, the loop runs mgs_step_kernel"""
    c = case("P156")
    assert c.n > PERSIST_LIMIT
    G = c.handle()
    b = c.rhs(0)
    e = _check_fixed_steps(c, "fgmres", 7, *G.fgmres(b, restart=10, maxit=7))
    x, flag, iters = G.gmres(b, restart=10, maxit=7)
    e = max(e, _check_fixed_steps(c, "gmres", 7, x, flag, iters, None))
    record_property("worst_relerr", e)
    c.close()  # 3.8 M rows: give the memory back


@gpu
def test_converged_fgmres_on_the_benchmark_workload(built, record_property):
    """C96, FGMRES(30) to rtol 1e-6: the configuration the benchmark times"""
    c = case("C96")
    b = c.rhs(0)
    x, flag, iters, nmv = c.handle().fgmres(b, restart=30, rtol=1e-6)
    _, rflag, riters, rnmv = c.krylov_ref(0, "fgmres", 30, 500)
    assert flag == rflag == 0 and abs(iters - riters) <= 1, (flag, rflag, iters, riters)
    assert abs(nmv - rnmv) <= _nmv_tol(riters, rnmv), (nmv, rnmv)
    res = np.linalg.norm(b - P.csr_matvec(c.A, x)) / np.linalg.norm(b)
    assert res <= 2e-6, res
    record_property("residual", res)


# ------------------------------------------------------------------ 6. reductions
@gpu
@pytest.mark.parametrize("n", [151_551, 151_552, 151_553, 1_000_003, 3_796_416])
def test_norm2_across_grid_stride_passes(built, n, record_property):
    """kRB * kRT = 151 552 elements per grid-stride pass of reduce_kernel; exactly rounded host reference
    m sqrt(fsum((v / m)^2)); power-of-two scales commute with every rounding of the max-scaled norm"""
    import torch
    G = case("N48").handle()
    v = np.random.default_rng(n).uniform(-1, 1, n)
    m = float(np.abs(v).max())
    ref = m * math.sqrt(math.fsum((v / m) ** 2))
    worst, base = 0.0, None
    for p in (0, 600, -600):
        s = math.ldexp(1.0, p)
        d = torch.from_numpy(v * s).cuda()
        got = G.norm2_dev(d.data_ptr(), n)
        assert got == G.norm2_dev(d.data_ptr(), n), "run-to-run"
        e = abs(got - ref * s) / (ref * s)
        worst = max(worst, e)
        assert e <= 1e-14, (n, p, got, ref * s)
        if base is None:
            base = got
        assert got == math.ldexp(base, p), (n, p)
    record_property("relerr", worst)


# ------------------------------------------------------------------ 7. block Krylov at scale
BLOCK_SEED = 300
BOUNDARY_COLS = (0, 15, 16, 31, 32, 63, 64, 69)


def _single_device(c, G, which, k):
    """the single-rhs device solver on block column k (restart 10, maxit 12), shared between widths"""
    def run():
        b = c.rhs(BLOCK_SEED + k)
        if which == "fgmres":
            return G.fgmres(b, restart=10, maxit=12)
        x, f, it = G.gmres(b, restart=10, maxit=12)
        return x, f, it, it
    return c.ref(("device", which, k), run)


@gpu
@pytest.mark.parametrize("nc", [2, 17, 33, 70])
@pytest.mark.parametrize("which", ["fgmres", "gmres"])
@pytest.mark.parametrize("name", ["P64", "P64f"])
def test_block_krylov_at_scale(built, name, which, nc, record_property):
    c = case(name)
    G = c.handle()
    B = P.seeded_rhs(c.n, BLOCK_SEED, nrhs=nc)
    if which == "fgmres":
        X, flags, iters, nmv = G.fgmres_mrhs(B, restart=10, maxit=12)
    else:
        X, flags, iters = G.gmres_mrhs(B, restart=10, maxit=12)
        nmv = iters
    worst = 0.0
    for k in (k for k in BOUNDARY_COLS if k < nc):
        xr, rflag, riters, rnmv = c.krylov_ref(BLOCK_SEED + k, which, 10, 12)
        assert flags[k] == rflag and iters[k] == riters, (k, flags[k], rflag, iters[k], riters)
        if which == "fgmres":
            assert nmv[k] == rnmv, (k, nmv[k], rnmv)
        e = relerr(X[:, k], xr)
        worst = max(worst, e)
        assert e <= c.kgate, (k, e)
    for k in range(nc):
        x, f, it, nm = _single_device(c, G, which, k)
        assert (flags[k], iters[k], nmv[k]) == (f, it, nm), (k, flags[k], f, iters[k], it, nmv[k], nm)
        assert relerr(X[:, k], x) <= c.kgate, k
    record_property("worst_relerr", worst)


@gpu
@pytest.mark.parametrize("which", ["fgmres", "gmres"])
def test_block_krylov_placement_and_scale_invariance(built, which):
    """One 70-column block: a column's result depends neither on its position inside the first pass of the
    batched apply nor on a power-of-two scale of its right-hand side (bitwise, inside one call); a zero column
    stays exact zeros; the second pass (other ready-bit parity of the multi-rhs epoch) agrees to rounding."""
    c = case("P64")
    G = c.handle()
    b = c.rhs(0)
    B = P.seeded_rhs(c.n, 500, nrhs=70)
    for k in (0, 31, 32, 63, 64):
        B[:, k] = b
    B[:, 5], B[:, 6], B[:, 7] = math.ldexp(1.0, 600) * b, math.ldexp(1.0, -600) * b, 0.0
    if which == "fgmres":
        X, flags, iters, nmv = G.fgmres_mrhs(B, restart=10)
    else:
        X, flags, iters = G.gmres_mrhs(B, restart=10)
        nmv = iters
    counts = lambda k: (flags[k], iters[k], nmv[k])  # noqa: E731
    assert flags[0] == 0, counts(0)
    for k in (31, 32, 63):
        assert np.array_equal(X[:, k], X[:, 0]) and counts(k) == counts(0), k
    for k, p in ((5, 600), (6, -600)):
        assert counts(k) == counts(0), k
        assert np.array_equal(X[:, k], math.ldexp(1.0, p) * X[:, 0]), (k, relerr(X[:, k], math.ldexp(1.0, p) * X[:, 0]))
    assert np.all(X[:, 7] == 0.0) and counts(7) == (0, 0, 0)
    assert counts(64) == counts(0) and relerr(X[:, 64], X[:, 0]) <= 1e-12, relerr(X[:, 64], X[:, 0])


@gpu
@pytest.mark.parametrize("which", ["fgmres", "gmres"])
def test_single_rhs_krylov_scale_invariance(built, which):
    """two fresh handles with identical call histories: scaling b by 2^600 / 2^-600 scales x exactly"""
    c = case("P64")
    b = c.rhs(0)
    scales = (math.ldexp(1.0, 600), math.ldexp(1.0, -600))
    with c.attach() as G1, c.attach() as G2:
        for s in scales:
            if which == "fgmres":
                r1, r2 = G1.fgmres(b, restart=10), G2.fgmres(s * b, restart=10)
            else:
                r1, r2 = G1.gmres(b, restart=10), G2.gmres(s * b, restart=10)
            assert r1[1] == 0 and r1[1:] == r2[1:], (r1[1:], r2[1:])
            assert np.array_equal(r2[0], s * r1[0]), relerr(r2[0], s * r1[0])
