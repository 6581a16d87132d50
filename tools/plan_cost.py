"""Developer tool (host only): the attach-time merge plans of every triangular factor and their
predicted sweep times under the library's cost model (MergeParams::plan_cost, csrc/hifgpu.h).

    python tools/plan_cost.py [workload] [size] [--cfg "ENV=value,..."] ...

Without --cfg it prints the cost-model policy (the default), the plan of the former fixed caps
(sl_cap = clamp(nnz/14, 3e5, 1.2e6), gain = 3 sl_cap) and the unmerged factor.  Per factor: merged
depth (dependent steps), stored entries, rows, packed megabytes of the warp streams and the
prediction; per configuration the total over the 2 sweeps of every LDU solve of one apply."""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import bench
import hifir_b200 as hb


def old_caps(block):
    sl = min(1.2e6, max(3.0e5, len(block[3]) / 14.0))
    return f"HIFIR_B200_MERGE_SLCAP={sl:.0f},HIFIR_B200_MERGE_GAIN={3 * sl:.0f}"


def with_env(cfg, fn):
    keys = []
    for kv in filter(None, cfg.split(",")):
        k, v = kv.split("=")
        os.environ[k] = v
        keys.append(k)
    try:
        return fn()
    finally:
        for k in keys:
            os.environ.pop(k, None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workload", nargs="?", default="poisson")
    ap.add_argument("size", nargs="?", type=int, default=128)
    ap.add_argument("--cfg", action="append", default=None)
    ap.add_argument("--no-pack", action="store_true", help="skip the packed size (the warp-stream packing)")
    args = ap.parse_args()
    A, lv = bench.cached_levels(args.workload, args.size)
    cfgs = args.cfg or ["", "old", "HIFIR_B200_MERGE=0"]
    for cfg in cfgs:
        total, steps = 0.0, 0
        name = {"": "cost model (default)", "old": "fixed caps (previous default)"}.get(cfg, cfg)
        print(f"== {name}", flush=True)
        for li, L in enumerate(lv):
            if not L["m"]:
                continue
            rhs = np.random.default_rng(li).uniform(-1, 1, L["m"])
            for nm, upper in (("L", False), ("U", True)):
                blk = L[nm]
                c = old_caps(blk) if cfg == "old" else cfg
                t0 = time.time()
                p = with_env(c, lambda: hb.debug_merge_plan(blk, upper))
                t_plan = time.time() - t0
                mb = float("nan")
                if not args.no_pack:
                    _, st = with_env(c, lambda: hb.debug_sweep_host(blk, upper, rhs, L["d"] if upper else None))
                    mb = st["bytes"] / 1e6
                k = 2 if L["n"] > L["m"] else 1  # a level with a Schur complement solves twice (down and up)
                total += k * p["predicted_us"]
                steps += k * p["steps"]
                print(f"  {nm}{li}: entries {p['entries'] / 1e6:.2f} M ({p['entries'] * 12 / 1e6:.1f} MB), depth "
                      f"{p['depth']} -> {p['steps']}, merged entries {p['merged_entries'] / 1e6:.2f} M, rows "
                      f"{p['merged_rows'] / 1e6:.2f} M, packed {mb:.1f} MB, predicted {p['predicted_us']:.1f} us"
                      f"  (plan {t_plan:.1f} s)", flush=True)
        print(f"  per apply: {steps} dependent steps, predicted sweep time {total / 1e3:.3f} ms", flush=True)


if __name__ == "__main__":
    main()
