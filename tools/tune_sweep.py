"""Developer tool (GPU box): one factorization, several attach-time configurations.

    python tools/tune_sweep.py --size 128 --cfg "HIFIR_B200_MERGE=0" --cfg "HIFIR_B200_MERGE_GAIN=30000" ...

Each --cfg is a comma separated list of ENV=value pairs read by the library at attach time.
Prints ms per apply, the per-kernel profile and the parity against the reference's own apply."""
import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)


def main():
    import torch

    import hifir_b200 as hb
    from bench import factorize, make_problem
    from hifir_b200 import build, problems as P

    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="poisson")
    ap.add_argument("--size", type=int, default=128)
    ap.add_argument("--cfg", action="append", default=[])
    ap.add_argument("--steps", type=int, default=30)
    args = ap.parse_args()
    build.build()
    A = make_problem(args.workload, args.size)
    M = factorize(A)
    levels = M.levels()
    n = A[0]
    bh = P.seeded_rhs(n, 0)
    xr = M.solve(bh)
    b = torch.from_numpy(bh).cuda()
    x = torch.empty_like(b)
    for cfg in args.cfg or [""]:
        keys = []
        for kv in filter(None, cfg.split(",")):
            k, v = kv.split("=")
            os.environ[k] = v
            keys.append(k)
        t0 = time.time()
        try:
            G = hb.GpuHif(levels)
        except Exception as e:  # noqa: BLE001
            print(f"[{cfg}] attach failed: {e}", flush=True)
            for k in keys:
                os.environ.pop(k, None)
            continue
        t_attach = time.time() - t0
        side = torch.cuda.Stream()
        torch.cuda.set_stream(side)
        G.set_stream(side.cuda_stream)
        try:
            for _ in range(3):
                G.solve_dev(b.data_ptr(), x.data_ptr())
            G.synchronize()
            err = float(np.linalg.norm(x.cpu().numpy() - xr) / np.linalg.norm(xr))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                G.solve_dev(b.data_ptr(), x.data_ptr())
            e1.record()
            torch.cuda.synchronize()
            G.synchronize()
            ms = e0.elapsed_time(e1) / args.steps
            prof = {}
            for _ in range(3):
                for name, t in G.profile_solve_dev(b.data_ptr(), x.data_ptr()):
                    prof[name] = t
            st = G.stats()
            print(f"[{cfg}] apply {ms:.3f} ms  parity {err:.1e}  attach {t_attach:.1f}s  device {st['device_bytes'] / 1e9:.2f} GB",
                  flush=True)
            print("    " + " ".join(f"{k}={v * 1e3:.1f}" for k, v in prof.items() if v * 1e3 >= 1), flush=True)
        except Exception as e:  # noqa: BLE001
            print(f"[{cfg}] failed: {e}", flush=True)
        G.close() if hasattr(G, "close") else None
        del G
        for k in keys:
            os.environ.pop(k, None)


if __name__ == "__main__":
    main()
