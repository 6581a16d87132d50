"""Developer tool (GPU box): per-segment trace of the warp-stream sweeps.

    python tools/trace_ws.py --size 128 [--level 0 --which 0] [--cfg ENV=val,...]

Prints where a sweep's time goes: per level set the completion step, and per segment the waits
(admission, first gather round trip, re-poll rounds, publish)."""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)


def analyse(tr, name):
    t0 = tr[:, 0].astype(np.int64)
    t1 = tr[:, 1].astype(np.int64)
    t2 = (tr[:, 2] >> np.uint64(8)).astype(np.int64)
    rounds = (tr[:, 2] & np.uint64(255)).astype(np.int64)
    t3 = (tr[:, 3] >> np.uint64(16)).astype(np.int64)
    lvl = (tr[:, 3] & np.uint64(0x7fff)).astype(np.int64)
    copy = (tr[:, 3] & np.uint64(0x8000)) != 0
    ok = t0 > 0
    base = t0[ok].min()
    t0 = t0 - base
    t1, t2, t3 = t0 + t1, t0 + t2, t0 + t3
    print(f"{name}: segments {ok.sum()} (copy {copy.sum()}) levels {lvl.max() + 1} sweep {t3[ok].max() / 1e3:.1f} us")
    nc = ok & ~copy
    print(f"   per segment (non-copy): admission wait mean {np.mean(t1[nc] - t0[nc]) / 1e3:.2f} us, first gathers "
          f"{np.mean(t2[nc] - t1[nc]) / 1e3:.2f} us, re-poll + publish {np.mean(t3[nc] - t2[nc]) / 1e3:.2f} us, "
          f"rounds mean {rounds[nc].mean():.2f} max {rounds[nc].max()}, life {np.mean(t3[nc] - t0[nc]) / 1e3:.2f} us")
    nl = lvl.max() + 1
    done = np.zeros(nl)
    first = np.zeros(nl)
    cnt = np.zeros(nl, dtype=np.int64)
    for l in range(nl):
        sel = ok & (lvl == l)
        if sel.any():
            done[l] = t3[sel].max()
            first[l] = t0[sel].min()
            cnt[l] = sel.sum()
    step = np.diff(done)
    print(f"   level completion step: mean {step.mean() / 1e3:.2f} us median {np.median(step) / 1e3:.2f} max {step.max() / 1e3:.2f}")
    print("   level: segs  first-decode  done  step | mean(first gathers) mean(repoll) mean(rounds)")
    for l in list(range(0, min(nl, 12))) + list(range(12, nl, max(1, nl // 12))):
        sel = nc & (lvl == l)
        if not sel.any():
            continue
        print(f"   {l:4d}: {cnt[l]:6d} {first[l] / 1e3:8.1f} {done[l] / 1e3:8.1f} {(done[l] - done[l - 1]) / 1e3 if l else 0:6.2f} | "
              f"{np.mean(t2[sel] - t1[sel]) / 1e3:6.2f} {np.mean(t3[sel] - t2[sel]) / 1e3:6.2f} {rounds[sel].mean():5.1f}  "
              f"adm {np.mean(t1[sel] - t0[sel]) / 1e3:5.2f}")


def main():
    import torch

    import hifir_b200 as hb
    from bench import factorize, make_problem
    from hifir_b200 import build, problems as P

    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="poisson")
    ap.add_argument("--size", type=int, default=128)
    ap.add_argument("--cfg", default="")
    ap.add_argument("--sweeps", default="0:0,0:1,1:0,1:1")
    args = ap.parse_args()
    build.build()
    os.environ.setdefault("HIFIR_B200_WS_FUSE", "0")  # the trace numbers the segments of ONE sweep
    for kv in filter(None, args.cfg.split(",")):
        k, v = kv.split("=")
        os.environ[k] = v
    A = make_problem(args.workload, args.size)
    M = factorize(A)
    G = hb.GpuHif(M.levels())
    n = A[0]
    b = torch.from_numpy(P.seeded_rhs(n, 0)).cuda()
    x = torch.empty_like(b)
    side = torch.cuda.Stream()
    torch.cuda.set_stream(side)
    G.set_stream(side.cuda_stream)
    for _ in range(3):
        G.solve_dev(b.data_ptr(), x.data_ptr())
    G.synchronize()
    for sw in args.sweeps.split(","):
        lv, which = (int(v) for v in sw.split(":"))
        tr = G.trace_sweep(b.data_ptr(), x.data_ptr(), lv, which)
        analyse(tr, f"[{args.cfg}] lv{lv} {'down' if which < 2 else 'up'} {'U' if which & 1 else 'L'}")
        np.save(os.path.join(ROOT, "gpurun_out", f"trace_lv{lv}_{which}.npy"), tr)


if __name__ == "__main__":
    main()
