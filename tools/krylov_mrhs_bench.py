"""Developer tool (GPU box): block FGMRES(30) over many right-hand sides (lhfdGpuFgmresMrhs) against a loop of
single-rhs solves (lhfdGpuFgmres) over the same columns, on the factors of bench.cached_levels.

Cases: conv-diff 96^3 with 16 and 64 columns, Poisson 128^3 with 16 columns; rtol 1e-6.  Both arms are warmed
up in the same process, then timed alternately with the host clock around the (synchronous) calls, median of 3.
Prints the device and its power limit, column-solves/s of both arms, the per-column iteration counts and the
largest relative difference between the two solutions.  Then one block solve per case runs under torch.profiler
(a run of its own) and its device time is split into apply, SpMV, Gram-Schmidt and solution update; what the
wall time holds beyond the kernels is launch gaps and host round trips.

    python tools/krylov_mrhs_bench.py [workload size nrhs ...]
"""
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

CASES = (("convdiff", 96, 16), ("convdiff", 96, 64), ("poisson", 128, 16))
RESTART, RTOL, MAXIT, REPEATS = 30, 1e-6, 500, 3

# kernel name -> part of the block solve (the block Krylov kernels of csrc/krylov.cu; everything else is the
# batched apply inside the block refinement)
PARTS = (("spmv", ("spmv_cols_kernel",)),
         ("gram-schmidt", ("mgs_step_cols_kernel", "reduce_cols_kernel", "final_cols_kernel", "div_cols_kernel",
                           "zero_cols_kernel")),
         ("update", ("axpy_cols_kernel",)))


def part_of(name):
    for part, keys in PARTS:
        if any(k in name for k in keys):
            return part
    return "apply"


def device_line():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "power limit not readable"
    return f"device: {name}; power limit, max SM clock: {q}"


def profile_block(G, B):
    """device time of one block solve per part (ms), and its wall time"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        t0 = time.perf_counter()
        G.fgmres_mrhs(B, restart=RESTART, rtol=RTOL, maxit=MAXIT)
        wall = time.perf_counter() - t0
    split = {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = getattr(e, "cuda_time_total", 0.0)
        if us:
            p = part_of(e.key)
            split[p] = split.get(p, 0.0) + us / 1e3
    return split, wall * 1e3


def run_case(workload, size, nrhs):
    import hifir_b200 as hb
    from bench import cached_levels
    from hifir_b200 import problems as P
    A, levels = cached_levels(workload, size)
    n = A[0]
    B = P.seeded_rhs(n, 0, nrhs=nrhs)
    with hb.GpuHif(levels) as G:
        G.set_matrix(A)

        def block():
            return G.fgmres_mrhs(B, restart=RESTART, rtol=RTOL, maxit=MAXIT)

        def loop():
            out = [G.fgmres(np.ascontiguousarray(B[:, k]), restart=RESTART, rtol=RTOL, maxit=MAXIT) for k in range(nrhs)]
            return (np.stack([o[0] for o in out], axis=1), np.array([o[1] for o in out]), np.array([o[2] for o in out]),
                    np.array([o[3] for o in out]))

        rb, rl = block(), loop()  # warm-up: allocates the bases, builds the plans and graphs of both arms
        tb, tl = [], []
        for _ in range(REPEATS):
            t0 = time.perf_counter()
            rb = block()
            tb.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            rl = loop()
            tl.append(time.perf_counter() - t0)
        Xb, fb, ib, nb = rb
        Xl, fl, il, nl = rl
        diff = max(float(np.linalg.norm(Xb[:, k] - Xl[:, k]) / np.linalg.norm(Xl[:, k])) for k in range(nrhs))
        relres = max(float(np.linalg.norm(B[:, k] - P.csr_matvec(A, Xb[:, k])) / np.linalg.norm(B[:, k]))
                     for k in range(nrhs))
        mb, ml = statistics.median(tb), statistics.median(tl)
        print(f"== {workload} {size}^3  n={n}  nrhs={nrhs}  FGMRES({RESTART}) rtol {RTOL:g}", flush=True)
        print(f"block: median {mb * 1e3:.1f} ms of {[round(t * 1e3, 1) for t in tb]} -> {nrhs / mb:.1f} column-solves/s")
        print(f"loop:  median {ml * 1e3:.1f} ms of {[round(t * 1e3, 1) for t in tl]} -> {nrhs / ml:.1f} column-solves/s")
        print(f"block / loop speed-up: {ml / mb:.2f}x")
        print(f"iters  block: {ib.tolist()}\n       loop:  {il.tolist()}")
        print(f"num_mv block: {nb.tolist()}\n       loop:  {nl.tolist()}")
        print(f"flags  block: {fb.tolist()}  loop: {fl.tolist()}")
        print(f"max relative difference block vs loop x: {diff:.3e}; max ||b - A x|| / ||b|| (block): {relres:.3e}")
        print(f"device bytes of the handle: {G.stats()['device_bytes'] / 1e9:.2f} GB", flush=True)
        split, wall = profile_block(G, B)
        total = sum(split.values())
        parts = ", ".join(f"{k} {v:.1f} ms" for k, v in sorted(split.items(), key=lambda kv: -kv[1]))
        print(f"profiled block solve: wall {wall:.1f} ms, kernels {total:.1f} ms ({parts}); "
              f"outside kernels {wall - total:.1f} ms", flush=True)


def main():
    from hifir_b200 import build
    build.build()
    print(device_line(), flush=True)
    args = sys.argv[1:]
    cases = [(args[i], int(args[i + 1]), int(args[i + 2])) for i in range(0, len(args), 3)] if args else CASES
    for c in cases:
        run_case(*c)


if __name__ == "__main__":
    main()
