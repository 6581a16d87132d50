"""Attach-time merge policy (merge.cu, MergeParams::plan_cost): the per-factor plan chosen by the
cost model solves exactly what the factor solves, is chosen deterministically, and is never
predicted slower than the plan of the former fixed caps.  CPU only: the host hooks merge and pack
as attach does and run the packed sweep on the host."""
import os

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spl

import hifir_b200 as hb
from hifir_b200 import problems as P

CASES = [("poisson", P.poisson3d, 24), ("convdiff", P.convdiff3d, 24), ("stokes", P.stokes2d_mac, 48)]


@pytest.fixture(scope="module")
def lib():
    from hifir_b200 import build
    build.build()
    return hb.lib()


_levels = {}


def factors(name, gen, size, dtype=np.float64):
    key = (name, size, np.dtype(dtype).name)
    if key not in _levels:
        from oracle import factor as F
        _levels[key] = F.multilevel_levels(gen(size), dtype)
    return _levels[key]


def blocks(levels):
    for lvl, L in enumerate(levels):
        if not L["m"]:
            continue
        for name, upper in (("L", False), ("U", True)):
            if len(L[name][3]):
                yield lvl, L, name, upper


def old_caps_env(block):
    sl = min(1.2e6, max(3.0e5, len(block[3]) / 14.0))
    return {"HIFIR_B200_MERGE_SLCAP": repr(sl), "HIFIR_B200_MERGE_GAIN": repr(3.0 * sl)}


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["double", "single"])
def test_chosen_plan_solves_the_factor(lib, case, dtype):
    levels = factors(*case, dtype=dtype)
    rng = np.random.default_rng(11)
    for lvl, L, name, upper in blocks(levels):
        m = L["m"]
        rhs = rng.uniform(-1, 1, m)
        d = np.asarray(L["d"], dtype=np.float64)
        x, _ = hb.debug_sweep_host(L[name], upper, rhs, d if upper else None)
        nr, nc, cs, ri, va = L[name]
        T = sp.csc_matrix((np.asarray(va, dtype=np.float64), ri, cs), shape=(m, m)) + sp.identity(m, format="csc")
        ref = spl.spsolve_triangular(T.tocsr(), rhs / d if upper else rhs, lower=not upper)
        err = np.linalg.norm(x - ref) / np.linalg.norm(ref)
        # single precision: the merged values (rows of W^{-1}) are stored rounded to float, as attach does
        assert err <= (1e-13 if dtype == np.float64 else 2e-6), (case[0], lvl, name, err)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_plan_choice_is_deterministic(lib, case):
    levels = factors(*case)
    rhs = np.random.default_rng(2)
    for lvl, L, name, upper in blocks(levels):
        b = rhs.uniform(-1, 1, L["m"])
        d = L["d"] if upper else None
        p0, p1 = hb.debug_merge_plan(L[name], upper), hb.debug_merge_plan(L[name], upper)
        assert p0 == p1, (case[0], lvl, name)
        x0, s0 = hb.debug_sweep_host(L[name], upper, b, d)
        x1, s1 = hb.debug_sweep_host(L[name], upper, b, d)
        assert s0 == s1 and np.array_equal(x0, x1), (case[0], lvl, name)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_chosen_plan_is_predicted_no_slower_than_the_fixed_caps(lib, case, monkeypatch):
    levels = factors(*case)
    for lvl, L, name, upper in blocks(levels):
        new = hb.debug_merge_plan(L[name], upper)
        with monkeypatch.context() as mp:
            for k, v in old_caps_env(L[name]).items():
                mp.setenv(k, v)
            old = hb.debug_merge_plan(L[name], upper)
        assert new["entries"] == old["entries"] and new["steps"] <= new["depth"]
        assert new["predicted_us"] <= old["predicted_us"] * (1 + 1e-12), (case[0], lvl, name, new, old)


def test_environment_caps_override_the_model(lib, monkeypatch):
    """HIFIR_B200_MERGE_SLCAP / _GAIN fix the caps (no model); HIFIR_B200_MERGE=0 leaves the factor unmerged."""
    L = factors(*CASES[0])[0]
    chosen = hb.debug_merge_plan(L["L"], False)
    monkeypatch.setenv("HIFIR_B200_MERGE", "0")
    plain = hb.debug_merge_plan(L["L"], False)
    assert plain["steps"] == plain["depth"] and plain["merged_entries"] == plain["entries"]
    monkeypatch.delenv("HIFIR_B200_MERGE")
    monkeypatch.setenv("HIFIR_B200_MERGE_SLCAP", "1e3")
    small = hb.debug_merge_plan(L["L"], False)
    assert small["merged_entries"] <= chosen["merged_entries"] or small["steps"] >= chosen["steps"]
    assert chosen["steps"] < plain["steps"]
