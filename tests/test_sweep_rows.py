"""The triangular sweeps row by row.

Every other device check is normwise: a single row off by 1e-10 ||x||_inf moves ||x - x_ref|| / ||x_ref|| by
about 1e-10 / sqrt(n), which passes a 1e-12 gate at these sizes.  Merged factors carry fill entries that are
products of many factor entries, some of them tiny: dropping one, or gathering a stale value through one,
perturbs only a few rows.  Here:

  * a device sweep must equal, bit for bit, the host emulation of the packed plan the device holds (copied back
    from the device, replayed with the device's per-lane fma order, its shfl_xor butterfly and its readiness
    tags: every published value has its last mantissa bit replaced by the parity before anyone reads it);
  * every row of that result must satisfy the ORIGINAL factor (L_B, or U_B with d) to a componentwise backward
    error gate computed in extended precision -- the plan is the right reformulation, row by row;
  * the full apply (S, SH, M, MH, refinement, multi-rhs, float factors) is gated per row in the inf-norm against
    the C oracle, the operations interleaved on one handle with a different b each time, so that a stale value
    never equals the current one.

The device part shares the factors and handles of test_scale_parity.py; the host-only part runs in the CPU suite
on the same factors (their build is paid for by the regime guard there)."""
import numpy as np
import pytest
import scipy.sparse as sp

import hifir_b200 as hb
from conftest import GOLDEN_CASES, load_golden
from test_scale_parity import MRHS_SEED, built, case  # noqa: F401  (built: module fixture)

gpu = pytest.mark.gpu
ROW_CASES = ("P64", "C96", "S400", "N48", "P64f")

# Componentwise backward error of a sweep against the original factor, max over rows of
#   |r_i - x_i - (T x)_i| / (|r_i| + |x_i| + (|T| |x|)_i)       (extended precision)
# Worst observed: device sweeps on a B200 (1000 W power limit) 2.3e-14 in double (S400, default plan), 4.1e-7 with
# float factors (P64f: the merged values are rounded to float, the original factor's values are not); host
# emulation of the plans below 2.7e-14 (C96, streaming plan).  A fill entry of relative size 1e-10 dropped from
# a double plan shows as about 1e-10.
BERR_GATE = 1e-13
BERR_GATE_SINGLE = 3e-6
# Full apply against the oracle, max_i |x_i - x_ref,i| / ||x_ref||_inf.  Worst observed on a B200 (1000 W power
# limit): 3.2e-15 in double (S400, solve_mrhs of 70 columns), 9.2e-9 with float factors (P64f).
APPLY_INF_GATE = 5e-14
APPLY_INF_GATE_SINGLE = 1e-7


def _tri(block, transpose=False):
    """the CCS block as an extended-precision CSR matrix (transposed: the twin's factor)"""
    nr, nc, cs, ri, va = block
    T = sp.csc_matrix((np.asarray(va, dtype=np.longdouble), np.asarray(ri), np.asarray(cs)), shape=(nr, nc))
    return sp.csr_matrix(T.T if transpose else T)


def backward_error(T, r, x):
    """per-row componentwise backward error of x as the solution of (I + T) x = r; returns (worst, row)"""
    rl, xl = np.asarray(r, dtype=np.longdouble), np.asarray(x, dtype=np.longdouble)
    num = np.abs(rl - xl - T @ xl)
    den = np.abs(rl) + np.abs(xl) + abs(T) @ np.abs(xl)
    w = np.where(den > 0, num / np.where(den > 0, den, 1), num)
    i = int(np.argmax(w))
    return float(w[i]), i


class Factors:
    """L_B, U_B and d of one level in extended precision, for the handle or its transposed twin
    (twin: L' = U_B^T, U' = L_B^T, the same d)"""

    def __init__(self, lev, transposed):
        self.L = _tri(lev["U"] if transposed else lev["L"], transposed)
        self.U = _tri(lev["L"] if transposed else lev["U"], transposed)
        self.d = np.asarray(lev["d"], dtype=np.longdouble)


def _as_double(words):
    return np.asarray(words, dtype=np.uint64).view(np.float64)


def _rows_of(slot_of, slots):
    inv = {int(s): r for r, s in enumerate(slot_of)}
    return [inv.get(int(s), f"aux slot {int(s)}") for s in slots]


# ------------------------------------------------------------------ host only (CPU suite)
HOST_PLANS = [{}, {"HIFIR_B200_MERGE_SLCAP": "1e3"}, {"HIFIR_B200_MERGE_SLCAP": "3e5"}, {"HIFIR_B200_MERGE": "0"},
              {"HIFIR_B200_SWEEP": "stream"}]


def _plan_id(cfg):
    return "-".join(f"{k[len('HIFIR_B200_'):].lower()}{v}" for k, v in cfg.items()) or "default"


@pytest.mark.parametrize("cfg", HOST_PLANS, ids=_plan_id)
@pytest.mark.parametrize("name", ROW_CASES)
def test_emulated_sweep_rows_at_scale(built, name, cfg, monkeypatch, record_property):  # noqa: F811
    """every level's L_B and U_B, merged and packed as attach does, solved with the packed data on the host:
    every row satisfies the original factor"""
    for k, v in cfg.items():
        monkeypatch.setenv(k, v)
    c = case(name)
    gate = BERR_GATE_SINGLE if c.single else BERR_GATE
    rng = np.random.default_rng(7)
    worst = 0.0
    for lv, lev in enumerate(c.levels):
        m = lev["m"]
        if not m:
            continue
        F = Factors(lev, False)
        d = np.asarray(lev["d"], dtype=np.float64)
        b = rng.uniform(-1, 1, m)
        x, _ = hb.debug_sweep_host(lev["L"], False, b, None)
        e, i = backward_error(F.L, b, x)
        worst = max(worst, e)
        assert e <= gate, (name, lv, "L", i, e)
        x, _ = hb.debug_sweep_host(lev["U"], True, b, d)
        e, i = backward_error(F.U, b.astype(np.longdouble) / F.d, x)
        worst = max(worst, e)
        assert e <= gate, (name, lv, "U", i, e)
    record_property("worst_backward_error", worst)


@pytest.mark.parametrize("sweep", ["ws", "stream"])
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_tagged_emulation_stays_within_ulps(name, sweep, monkeypatch):
    """the readiness tag moves every published value by at most one ulp: per row, the tagged emulation
    (parity 0 and 1) stays within a few ulps of the scale of that row's substitution"""
    monkeypatch.setenv("HIFIR_B200_SWEEP", sweep)
    g = load_golden(name)
    rng = np.random.default_rng(3)
    for lev in g.levels:
        m = lev["m"]
        if not m:
            continue
        F = Factors(lev, False)
        d = np.asarray(lev["d"], dtype=np.float64)
        b = rng.uniform(-1, 1, m)
        for blk, upper, T in (("L", False, F.L), ("U", True, F.U)):
            x0, _ = hb.debug_sweep_host(lev[blk], upper, b, d if upper else None)
            r = b.astype(np.longdouble) / F.d if upper else b.astype(np.longdouble)
            scale = np.abs(r) + np.abs(x0.astype(np.longdouble)) + abs(T) @ np.abs(x0.astype(np.longdouble))
            for parity in (0, 1):
                xt, _ = hb.debug_sweep_host(lev[blk], upper, b, d if upper else None, parity=parity)
                assert np.all((xt.view(np.uint64) & np.uint64(1)) == parity), (name, blk, parity)
                ulps = np.abs(xt.astype(np.longdouble) - x0) / (scale * np.finfo(np.float64).eps)
                i = int(np.argmax(ulps))
                assert ulps[i] <= 8, (name, blk, parity, i, float(ulps[i]))


# ------------------------------------------------------------------ device sweeps, bit for bit
DEVICE_PLANS = [{}, {"HIFIR_B200_WS_FUSE": "0"}, {"HIFIR_B200_MERGE": "0"}, {"HIFIR_B200_SWEEP": "stream"},
                {"HIFIR_B200_WS_WARPS": "16", "HIFIR_B200_WS_STAGES": "4"},
                {"HIFIR_B200_WS_WARPS": "32", "HIFIR_B200_WS_STAGES": "2"}]
DEVICE_CASES = [(name, {}) for name in ROW_CASES] + [(name, cfg) for cfg in DEVICE_PLANS[1:] for name in ("P64", "P64f")]


def _check_sweep(G, c, lv, factor, transposed, rhs, F, gate):
    """one device sweep: bitwise against the emulation of its own bytes, then per row against the original
    factor; returns the worst backward error"""
    r = G.debug_sweep_dev(lv, factor, rhs, transposed=transposed)
    words, emul = r["words"], r["emul"]
    where = (c.name, lv, factor, "twin" if transposed else "handle", "parity", r["parity"])
    if not np.array_equal(words, emul):
        bad = np.flatnonzero(words != emul)
        slot_of = r["slot_of"] if r["slot_of_l"] is None else np.concatenate([r["slot_of_l"], r["slot_of"]])
        pytest.fail(f"{where}: {bad.size} of {words.size} words differ from the emulation; first slots "
                    f"{bad[:8].tolist()} = rows {_rows_of(slot_of, bad[:8])}; device {_as_double(words[bad[:4]])} "
                    f"emulation {_as_double(emul[bad[:4]])}")
    rows = r["slot_of"] if r["slot_of_l"] is None else np.concatenate([r["slot_of_l"], r["slot_of"]])
    assert np.all((words[rows] & np.uint64(1)) == r["parity"]), where  # every row carries this call's tag
    worst = 0.0
    x = r["x"]
    if factor == "L":
        checks = [(F.L, rhs, x, "L")]
    elif factor == "U":
        checks = [(F.U, rhs.astype(np.longdouble) / F.d, x, "U")]
    else:  # fused: the L part and the U part, each against its own factor
        z = _as_double(words[r["slot_of_l"]])
        checks = [(F.L, rhs, z, "L"), (F.U, z.astype(np.longdouble) / F.d, x, "U")]
    for T, rr, xx, part in checks:
        e, i = backward_error(T, rr, xx)
        worst = max(worst, e)
        assert e <= gate, (where, part, "row", i, e)
    return worst


@gpu
@pytest.mark.parametrize("name,cfg", DEVICE_CASES, ids=[f"{n}-{_plan_id(c)}" for n, c in DEVICE_CASES])
def test_device_sweeps_bitwise_and_per_row(built, name, cfg, monkeypatch, record_property):  # noqa: F811
    """every level, L and U of the handle and of its transposed twin, three right-hand sides in a row (the third
    the negation of the second: a stale gather differs from the current value)"""
    c = case(name)
    for k, v in cfg.items():
        monkeypatch.setenv(k, v)
    gate = BERR_GATE_SINGLE if c.single else BERR_GATE
    G = c.handle() if not cfg else c.attach()
    fused = not cfg or (cfg.get("HIFIR_B200_WS_FUSE") != "0" and cfg.get("HIFIR_B200_SWEEP") != "stream")
    worst, sweeps = 0.0, 0
    try:
        for lv, lev in enumerate(c.levels):
            m = lev["m"]
            if not m:
                continue
            for transposed in (False, True):
                F = Factors(lev, transposed)
                for factor in (("LU",) if fused else ("L", "U")):
                    rng = np.random.default_rng(1000 * lv + 10 * transposed + len(factor))
                    b1, b2 = rng.uniform(-1, 1, m), rng.uniform(-1, 1, m)
                    for rhs in (b1, b2, -b2):
                        worst = max(worst, _check_sweep(G, c, lv, factor, transposed, rhs, F, gate))
                        sweeps += 1
        if cfg:  # a plan other than the fused 24 x 2 one: solve_mrhs runs the 8-column chunks on plans of its own
            record_property("worst_inf_mrhs", _mrhs_per_row(c, G, 20))
    finally:
        if cfg:
            G.close()
    record_property("worst_backward_error", worst)
    record_property("sweeps", sweeps)


# ------------------------------------------------------------------ full apply, per row
def _inf_err(x, ref):
    ref = np.asarray(ref, dtype=np.float64)
    return float(np.max(np.abs(np.asarray(x) - ref)) / np.max(np.abs(ref)))


MRHS_SHIFTS = {8: 0, 20: 30, 64: 50, 70: 7}  # column k of a width-w block = seed MRHS_SEED + (k + shift) % 70


def _mrhs_per_row(c, G, w):
    """one block of w columns, every column against the oracle per row; returns the worst error"""
    gate = APPLY_INF_GATE_SINGLE if c.single else APPLY_INF_GATE
    seeds = [MRHS_SEED + (k + MRHS_SHIFTS[w]) % 70 for k in range(w)]
    X = G.solve_mrhs(np.stack([c.rhs(s) for s in seeds], axis=1))
    worst = 0.0
    for k, s in enumerate(seeds):
        e = _inf_err(X[:, k], c.solve_ref(s))
        worst = max(worst, e)
        assert e <= gate, (c.name, f"mrhs{w}", k, e)
    return worst


@gpu
@pytest.mark.parametrize("name", ROW_CASES)
def test_apply_per_row_interleaved(built, name, record_property):  # noqa: F811
    """S, SH, M, MH, refinement and multi-rhs of widths 8, 20, 64 and 70 interleaved on one handle, a different b
    every time, every row against the oracle: the apply's real buffers and epochs (epoch, epoch_m, epoch_p) and
    the multi-rhs column kernel"""
    c = case(name)
    G, Oh = c.handle(), c.oracle
    gate = APPLY_INF_GATE_SINGLE if c.single else APPLY_INF_GATE
    worst = {}

    def check(what, x, ref):
        e = _inf_err(x, ref)
        worst[what] = max(worst.get(what, 0.0), e)
        assert e <= gate, (name, what, e)

    def single(op, j):
        b = c.rhs(j)
        if op == "S":
            check("S", G.solve(b), c.solve_ref(j))
        elif op == "hifir":
            check("hifir3", G.apply(b, nirs=3)[0], c.ref(("hifir", j, 3), lambda: Oh.hifir(b, 3)))
        else:
            o = getattr(hb, "LHF_" + op)
            check(op, G.apply(b, op=o)[0], c.ref((op, j), lambda: Oh.apply_op(int(o), b)))

    def mrhs(w):
        e = _mrhs_per_row(c, G, w)
        worst[f"mrhs{w}"] = max(worst.get(f"mrhs{w}", 0.0), e)

    transposed_ops = not c.nsp  # the null-space filter case: as test_apply_parity_at_scale
    seq = [("S", 10), ("M", 11), ("mrhs", 8), ("SH", 12), ("S", 13), ("MH", 14), ("hifir", 15), ("mrhs", 20),
           ("S", 16), ("mrhs", 64), ("SH", 17), ("M", 18), ("mrhs", 70), ("S", 19), ("MH", 20), ("mrhs", 8),
           ("hifir", 21), ("S", 22)]
    for op, arg in seq:
        if op == "mrhs":
            if not c.nsp:
                mrhs(arg)
        elif op in ("SH", "M", "MH") and not transposed_ops:
            single("S", arg)
        else:
            single(op, arg)
    for k, v in worst.items():
        record_property(f"worst_inf_{k}", v)
