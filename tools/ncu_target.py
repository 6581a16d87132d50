"""Developer tool (GPU box): a short program for ncu -- factorize, attach, a few applies.
    python tools/ncu_target.py [--size 128] [--applies 3]"""
import argparse, os, sys
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
    ap.add_argument("--applies", type=int, default=3)
    ap.add_argument("--nrhs", type=int, default=1)
    args = ap.parse_args()
    build.build()
    A = make_problem(args.workload, args.size)
    M = factorize(A)
    G = hb.GpuHif(M.levels())
    print("sweep_bytes", G.stats()["sweep_bytes"], "sweep_entries", G.stats()["sweep_entries"])
    n = A[0]
    bh = P.seeded_rhs(n, 0)
    b = torch.from_numpy(bh).cuda()
    x = torch.empty_like(b)
    side = torch.cuda.Stream()
    torch.cuda.set_stream(side)
    G.set_stream(side.cuda_stream)
    for _ in range(args.applies):
        G.solve_dev(b.data_ptr(), x.data_ptr())
    G.synchronize()
    if args.nrhs > 1:
        B = torch.from_numpy(P.seeded_rhs(n, 0, nrhs=args.nrhs)).cuda()
        X = torch.empty_like(B)
        for _ in range(args.applies):
            G.solve_mrhs_dev(args.nrhs, B.data_ptr(), X.data_ptr())
        G.synchronize()
        print("mrhs column 0 vs single", float((X[:, 0] - x).norm() / x.norm()))
    xr = M.solve(bh)
    print("parity", float(np.linalg.norm(x.cpu().numpy() - xr) / np.linalg.norm(xr)))


if __name__ == "__main__":
    main()
