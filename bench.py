#!/usr/bin/env python
"""bench.py -- M^-1 applies/s of the multilevel HIF preconditioner on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Workload (configs[1]): synthetic 3D Poisson 7-point 128^3 (n = 2 097 152), nrhs = 1.  One "step"
= one M^-1 apply (hif::HIF::solve semantics) of a seeded right-hand side.

  value : applies/s with b and x resident in HBM (lhfdGpuSolveDev), whole job over all ranks
  e2e   : applies/s through lhfdGpuSolve with pinned HOST b/x (H2D + apply + D2H per step)
  roofline : algorithmic bytes per apply (SURVEY.md 8d) / measured time vs measured HBM copy peak
  cpu_baseline : the C restatement of the reference's serial apply (oracle/hif_oracle.c), 1 core

Multi-GPU: the apply does not shard (sequential levels); every rank holds a factor replica and
applies to its own right-hand sides -> weak scaling, no collective on the hot path; results are
gathered with one NCCL all_gather after the timed region.

Factors: multilevel HIF factors computed on the host by oracle/factor.py (scaling, permutations, D-ILU
leading blocks, E/F blocks, sparse Schur levels, dense QRCP last level), so that the benchmark needs
nothing outside the repository.  The factorization runs before the timed region and is never part of a
reported number; the parity check before timing compares with the C oracle on the same factors.

--dump-outputs DIR writes what the timed path returned in its last step as DIR/<name>.npy (float64;
a fixed seeded sample of rows when the whole would exceed 64 MB), so that two builds can be compared
output for output: the inputs depend only on the arguments.  Both arms apply step k to right-hand
side k % NB_RHS, so their dumps are solutions of the same system.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CACHE_DIR = os.environ.get("HIFIR_B200_CACHE", "/tmp/hifir_b200_cache")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------- workloads
def make_problem(workload, size):
    from hifir_b200 import problems as P
    gen = {"poisson": P.poisson3d, "neumann": P.neumann3d, "convdiff": P.convdiff3d, "stokes": P.stokes2d_mac}[workload]
    return gen(size)


def workload_name(workload, size, nrhs):
    shape = f"{size}^3" if workload != "stokes" else f"MAC {size}x{size}"
    return f"{workload} {shape} nrhs={nrhs}"


FACTORS = "multilevel D-ILU, independent-set Schur levels, dense QRCP last level (oracle/factor.py)"


class HostFactor:
    """Factors for the device backend plus the C oracle applied to the same factors (parity check and
    CPU baseline): solve / hifir / krylov / set_nsp_const are those of oracle.port.OracleHif."""

    def __init__(self, A, levels):
        from oracle import port as O
        self._levels = levels
        self.oracle = O.OracleHif(levels, A)
        self.nnz = sum(len(L[k][3]) for L in levels for k in "LUEF")

    def levels(self):
        return self._levels

    def __getattr__(self, name):
        return getattr(self.oracle, name)


def factorize(A, nsp=False, dtype=np.float64):
    """Host factorization (oracle/factor.py), wrapped with the C oracle on the same factors.
    dtype=float32: single-precision factors of the double matrix (lhfs* / lhfsd* entry points)."""
    from oracle import factor as F
    t0 = time.time()
    M = HostFactor(A, F.multilevel_levels(A, dtype))
    if nsp:
        M.set_nsp_const()
    log(f"[bench] factorize: {time.time() - t0:.1f} s, levels {len(M.levels())}, nnz {M.nnz}")
    return M


def cached_levels(workload, size):
    """Per-level factors for developer tools: factorize(), cached on local disk (uncompressed npz)
    so that several processes on one box factorize once; the key names the factor producer."""
    from hifir_b200.levels_io import arrays_to_levels, levels_to_arrays
    from oracle import factor as F
    path = os.path.join(CACHE_DIR, f"{workload}{size}_{F.NAME_KEY}.npz")
    A = make_problem(workload, size)
    if os.path.exists(path):
        with np.load(path) as z:
            return A, arrays_to_levels({k: z[k] for k in z.files})
    M = factorize(A)
    levels = M.levels()
    os.makedirs(CACHE_DIR, exist_ok=True)
    np.savez(path, **levels_to_arrays(levels))
    return A, levels


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.device), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ----------------------------------------------------------------------------- reference arm
NB_RHS = 4  # step k of either arm applies to right-hand side k % NB_RHS


def cpu_apply_rate(M, n, applies, warm=1, nirs=1, A=None):
    """The C oracle's apply; nirs > 1: a step is one hifir(A, b, nirs, x) = nirs applies (the
    right-hand sides are then consistent, b = A v, as config 5 asks).  Returns (rate, seconds, x of the
    last step)."""
    bs = [step_rhs(A, n, j, nirs) for j in range(NB_RHS)]
    f = (lambda b: M.solve(b)) if nirs <= 1 else (lambda b: M.hifir(b, nirs))
    for _ in range(warm):
        f(bs[0])
    t0 = time.perf_counter()
    for k in range(applies):
        x = f(bs[k % NB_RHS])
    dt = time.perf_counter() - t0
    return applies / dt, dt, x


def step_rhs(A, n, j, nirs):
    """right-hand side j of a step: U(-1,1) seeded (apply), or the consistent b = A v_j of the
    refinement configs (v_j = sin(0.37 i + j), SURVEY.md 8d config 5)"""
    from hifir_b200 import problems as P
    if nirs <= 1:
        return P.seeded_rhs(n, j)
    return P.csr_matvec(A, np.sin(0.37 * np.arange(n) + j))


def _ref_batched_worker(wid, T, workload, size, nrhs, steps, ready, go, out):
    """One process of the batched CPU arm: factorizes, then applies the C oracle to its columns
    wid, wid + T, ... of the block, `steps` times (the oracle, like hif::HIF, applies one column at a time
    on one thread)."""
    from hifir_b200 import problems as P
    A = make_problem(workload, size)
    M = factorize(A)
    cols = list(range(wid, nrhs, T))  # this worker's columns of the block
    B = P.seeded_rhs(A[0], 0, nrhs=nrhs)
    bs = [np.ascontiguousarray(B[:, k]) for k in cols]
    if bs:
        M.solve(bs[0])
    ready.put(wid)
    go.wait()
    t0 = time.time()
    for _ in range(steps):
        for b in bs:
            M.solve(b)
    out.put((wid, len(bs) * steps, t0, time.time()))


def run_reference_batched(args):
    """--impl reference --nrhs K: a batched CPU apply is a column loop of single solves (the reference's own
    multi-rhs driver is defective, SURVEY.md App. B-1); T processes apply disjoint columns concurrently."""
    import multiprocessing as mp
    nproc = os.cpu_count() or 1
    T = max(1, min(nproc, 8, args.nrhs))
    A = make_problem(args.workload, args.size)
    n = A[0]
    steps = args.steps  # a step = one block of nrhs columns
    ctx = mp.get_context("spawn")
    ready, out, go = ctx.Queue(), ctx.Queue(), ctx.Event()
    ws = [ctx.Process(target=_ref_batched_worker,
                      args=(w, T, args.workload, args.size, args.nrhs, steps, ready, go, out)) for w in range(T)]
    for w in ws:
        w.start()
    for _ in ws:
        ready.get()
    go.set()
    res = [out.get() for _ in ws]
    for w in ws:
        w.join()
    cols = sum(r[1] for r in res)
    wall = max(r[3] for r in res) - min(r[2] for r in res)
    rate = cols / wall
    sample = (f"{steps} blocks of {args.nrhs} columns: {T} processes, each applying its "
              f"{-(-args.nrhs // T)} columns of the block with the C oracle's solve; {cols} applies in {wall:.1f} s")
    line = {
        "impl": "reference", "metric": "M^-1 applies/sec", "value": rate, "unit": "applies/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.workload, args.size, args.nrhs), "n": n,
                   "params": FACTORS, "l2_policy": L2_POLICY},
        "cpu_baseline": {"value": rate, "unit": "applies/s", "cores": T, "kind": "oracle", "sample": sample},
        "e2e": {"value": rate, "unit": "applies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_reference(args, rank, world):
    if rank != 0:
        return
    if args.nrhs > 1:
        return run_reference_batched(args)
    A = make_problem(args.workload, args.size)
    n = A[0]
    single = args.precision == "single"
    nirs = args.nirs
    M = factorize(A, nsp=args.workload == "neumann",
                  dtype=np.float32 if single else np.float64)
    steps = args.steps
    cpu_apply_rate(M, n, max(1, min(args.warmup, 3)), warm=0, nirs=nirs, A=A)
    rate, dt, x = cpu_apply_rate(M, n, steps, warm=0, nirs=nirs, A=A)
    rate *= nirs  # applies/s: a refinement step holds nirs applies
    sample = (f"{steps} serial applies of the C oracle, each a full apply of the workload") if nirs <= 1 else (
              f"{steps} hifir(A, b, nirs={nirs}) solves of the C oracle = {steps * nirs} applies + {steps * (nirs - 1)} A x")
    line = {
        "impl": "reference", "metric": "M^-1 applies/sec", "value": rate, "unit": "applies/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32" if single else "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.workload, args.size, args.nrhs) + (" single-precision factors" if single else "")
                   + (f" hifir nirs={nirs}" if nirs > 1 else ""),
                   "n": n, "params": FACTORS, "l2_policy": L2_POLICY},
        "cpu_baseline": {"value": rate, "unit": "applies/s", "cores": 1, "kind": "oracle", "sample": sample},
        "e2e": {"value": rate, "unit": "applies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, x=x)
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- our arm
def sweep_bytes(levels):
    """Algorithmic bytes of each triangular sweep launch (factor stream + rhs read + x write)."""
    out = {}
    for l, L in enumerate(levels):
        m = L["m"]
        for nm_, key in (("L", "L"), ("U", "U")):
            nnz = len(L[key][3])
            sv = L[key][4].dtype.itemsize  # 8, or 4 for the factors of hif::HIF<float>
            out[f"lv{l}.{nm_}"] = nnz * (4 + sv) + (m + 1) * 4 + (sv * m if nm_ == "U" else 0) + 16 * m
    return out


def run_mrhs(args, rank, world, local_rank):
    """Config 4 style run: one row-interleaved block B[n, nrhs], columns sharded over the ranks
    (every rank holds a factor replica), X gathered with one NCCL all_gather after the timed region."""
    import torch
    import torch.distributed as dist

    import hifir_b200 as hb
    from hifir_b200 import build, problems as P
    from hifir_b200.sharding import gather_columns, local_columns, shard_range

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback exists)"
    torch.cuda.set_device(local_rank)
    build.build()
    A = make_problem(args.workload, args.size)
    n, nrhs = A[0], args.nrhs
    M = factorize(A)
    levels = M.levels()
    G = hb.GpuHif(levels, device=local_rank)
    st = G.stats()
    stream = torch.cuda.current_stream()
    G.set_stream(stream.cuda_stream)
    B = P.seeded_rhs(n, 0, nrhs=nrhs)
    Bl = local_columns(B, world, rank)
    nloc = Bl.shape[1]
    Bh = torch.from_numpy(Bl).pin_memory()
    Bd = Bh.cuda()
    Xd = torch.empty_like(Bd)
    Xh = torch.empty_like(Bh).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if nloc:
        G.solve_mrhs_dev(nloc, Bd.data_ptr(), Xd.data_ptr(), 0)
        G.synchronize()
        b0, _ = shard_range(nrhs, world, rank)
        xr = M.solve(np.ascontiguousarray(B[:, b0]))
        parity = float(np.linalg.norm(Xd[:, 0].cpu().numpy() - xr) / np.linalg.norm(xr))
        assert parity <= 1e-12, f"parity gate failed: {parity}"
    else:
        parity = 0.0
    for _ in range(args.warmup):
        if nloc:
            G.solve_mrhs_dev(nloc, Bd.data_ptr(), Xd.data_ptr(), 0)
    launches0 = G.stats()["launch_count"]
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        if nloc:
            G.solve_mrhs_dev(nloc, Bd.data_ptr(), Xd.data_ptr(), 0)
    e1.record(stream)
    barrier()
    clocks = sampler.stop()
    G.synchronize()
    ms_total = e0.elapsed_time(e1)
    launches = G.stats()["launch_count"] - launches0
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        if nloc:
            hb._chk(hb.lib().lhfdGpuSolveMrhs(G._h, nloc, Bh.data_ptr(), Xh.data_ptr()))
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    barrier()
    t = torch.tensor([ms_total, e2e_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    X = gather_columns(Xd, nrhs, world, rank, dist=dist if world > 1 else None, device="cuda")  # off the timed path
    ms_total, e2e_ms = float(t[0]), float(t[1])
    if rank != 0:
        return
    ms_step = ms_total / args.steps
    peak, peak_src = hbm_peak()
    cpu = None
    if world == 1 and not args.no_cpu:
        # the reference's multi-rhs driver is defective (SURVEY.md App. B-1): its batched apply IS a
        # column loop of hif::HIF::solve on one core; a bounded sample of columns of this block
        ncols = max(1, min(nrhs, args.cpu_applies))
        t0 = time.perf_counter()
        for k in range(ncols):
            M.solve(np.ascontiguousarray(B[:, k]))
        dt = time.perf_counter() - t0
        cpu = {"value": ncols / dt, "unit": "applies/s", "cores": 1, "kind": "oracle",
               "sample": f"{ncols} of the {nrhs} columns, one serial C oracle solve each on the same factors ({dt:.1f} s)"}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, X=X.cpu().numpy())
    nloc0 = max(1, shard_range(nrhs, world, 0)[1])
    width = 64 if nloc0 >= 64 else 32 if nloc0 > 16 else 16 if nloc0 > 8 else 8  # mrhs.cu: apply_mrhs_dev
    chunks = -(-nloc0 // width)
    bytes_step = world * (st["bytes_factors"] + st["bytes_dense"]) + nrhs * st["bytes_vec_per_rhs"]
    line = {
        "metric": "M^-1 applies/sec", "value": nrhs * args.steps / (ms_total * 1e-3), "unit": "applies/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.workload, args.size, nrhs), "n": n, "levels": st["levels"],
                   "nnz_factors": st["nnz"], "params": FACTORS,
                   "l2_policy": "inputs larger than L2",
                   "parallelism": f"replicas, {nrhs} columns sharded over {world} GPU(s), {width} columns per pass"},
        "roofline": {"bound": "hbm", "kernel": "whole batched apply", "achieved": bytes_step / (ms_step * 1e-3) / 1e9,
                     "peak": peak * world, "unit": "GB/s", "frac": bytes_step / (ms_step * 1e-3) / 1e9 / (peak * world),
                     "traffic": None, "algorithmic_bytes_per_step": bytes_step, "peak_source": peak_src,
                     "passes_per_step": chunks},
        "cpu_baseline": cpu,
        "e2e": {"value": nrhs * args.steps / (e2e_ms * 1e-3), "unit": "applies/s",
                "h2d_bytes_per_step": 8 * n * nrhs, "d2h_bytes_per_step": 8 * n * nrhs,
                "api": "lhfdGpuSolveMrhs (pinned host buffers)"},
        "gpu_launches": launches, "clocks": clocks, "parity_vs_oracle": parity,
        "gathered_shape": list(X.shape),
    }
    print(json.dumps(line), flush=True)


DUMP_BYTES = 63 << 20  # array data of --dump-outputs: the .npy headers stay inside 64 MB


def dump_outputs(path, **arrays):
    """Write each array as path/<name>.npy in float64.  When all of them together exceed DUMP_BYTES,
    each is replaced by a fixed, seeded, sorted sample of its rows."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = max(1, len(a) * DUMP_BYTES // total)
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def pin_to_gpu_numa(local_rank):
    """Bind this rank to the host cores of the NUMA node its GPU hangs off (pinned-memory copies of 8
    ranks all served by node 0 were the e2e limiter of round 1).  Best effort: returns a description."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local_rank)],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        bus = out[-12:] if len(out) >= 12 else out  # 0000:xx:yy.z
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            # virtualised boxes do not expose the PCI device's node: ask NVML for the cores next to the GPU
            import pynvml
            pynvml.nvmlInit()
            hdl = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
            words = pynvml.nvmlDeviceGetCpuAffinity(hdl, ((os.cpu_count() or 64) + 63) // 64)
            cpus = [64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1]
            allowed = sorted(set(cpus) & os.sched_getaffinity(0))
            if allowed and len(allowed) < len(os.sched_getaffinity(0)):
                os.sched_setaffinity(0, allowed)
                return f"nvml cpu affinity, {len(allowed)} cores ({allowed[0]}-{allowed[-1]})"
            return f"numa node unknown (nvml affinity = all {len(allowed)} allowed cores)"
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.extend(range(int(lo), int(hi or lo) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return f"numa node {node}, {len(allowed)} cores"
        return f"numa node {node} (no allowed cores there)"
    except Exception as e:  # noqa: BLE001
        return f"not pinned ({type(e).__name__})"


# timing rule of the contract (the same words in both arms' `config`): no L2 flush between steps because one
# step streams far more than the cache holds
L2_POLICY = "inputs larger than L2: the factors one apply streams exceed the 126 MB L2 at 128^3, no flush between steps"
REPEATS = 5  # timed repeats of the --steps steps; the median is reported (SURVEY.md 8d)


def timed_repeats(step, steps, barrier, stream, repeats=REPEATS):
    """`repeats` device-timed runs of `steps` calls of step(k) -> list of milliseconds (this rank)"""
    import torch
    out = []
    for _ in range(repeats):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for k in range(steps):
            step(k)
        e1.record(stream)
        barrier()
        out.append(e0.elapsed_time(e1))
    return out


def max_over_ranks(values, world, dist):
    """element-wise MAX over the ranks of a list of floats"""
    import torch
    t = torch.tensor(values, dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def extra_workload(kind, args, rank, world, local_rank, barrier, stream):
    """Sub-record of the bench line for one of the other BASELINE configs, measured on every rank
    (no collective inside: the caller gathers).  kind: 'mrhs' (config 4: conv-diff 96^3, nrhs = 64
    columns sharded over the ranks), 'hifir' (config 5: Neumann 128^3, hifir(nirs = 4), one system per
    rank), 'stokes' (config 3: Stokes MAC 577^2 apply)."""
    import torch

    import hifir_b200 as hb
    from hifir_b200 import problems as P
    from hifir_b200.sharding import local_columns, shard_range
    wl, size = {"mrhs": ("convdiff", 96), "hifir": ("neumann", 128), "stokes": ("stokes", 577)}[kind]
    if args.extras_small:
        size = {"mrhs": 24, "hifir": 24, "stokes": 48}[kind]
    steps = max(2, min(args.steps, args.extra_steps))
    A = make_problem(wl, size)
    n = A[0]
    nsp = wl == "neumann"
    t0 = time.time()
    M = factorize(A, nsp=nsp)
    t_fact = time.time() - t0
    G = hb.GpuHif(M.levels(), device=local_rank)
    G.set_stream(stream.cuda_stream)
    if nsp:
        G.set_nsp_const()
    st = G.stats()
    rec = {"workload": workload_name(wl, size, 64 if kind == "mrhs" else 1), "n": n, "levels": st["levels"],
           "factorize_s": round(t_fact, 1), "steps": steps, "repeats": 3}
    try:
        if kind == "mrhs":
            nrhs = 64
            B = P.seeded_rhs(n, 0, nrhs=nrhs)
            Bl = local_columns(B, world, rank)
            nloc = Bl.shape[1]
            Bd = torch.from_numpy(Bl).cuda()
            Xd = torch.empty_like(Bd)
            G.solve_mrhs_dev(nloc, Bd.data_ptr(), Xd.data_ptr(), 0)
            G.synchronize()
            b0, _ = shard_range(nrhs, world, rank)
            errs = []
            for c in sorted({0, nloc - 1}):
                xr = M.solve(np.ascontiguousarray(B[:, b0 + c]))
                errs.append(float(np.linalg.norm(Xd[:, c].cpu().numpy() - xr) / np.linalg.norm(xr)))
            ms = timed_repeats(lambda k: G.solve_mrhs_dev(nloc, Bd.data_ptr(), Xd.data_ptr(), 0), steps, barrier, stream, 3)
            rec.update(parity_vs_oracle=max(errs), local_ms=ms, nrhs=nrhs, local_columns=nloc,
                       bytes_per_block=world * (st["bytes_factors"] + st["bytes_dense"]) + nrhs * st["bytes_vec_per_rhs"])
        elif kind == "hifir":
            G.set_matrix(A)
            nirs = 4
            bh = step_rhs(A, n, rank, nirs)  # one system per rank: its own consistent right-hand side
            bd = torch.from_numpy(bh).cuda()
            xd = torch.empty_like(bd)
            G.hifir_dev(bd.data_ptr(), nirs, xd.data_ptr())
            G.synchronize()
            xr = M.hifir(bh, nirs)
            err = float(np.linalg.norm(xd.cpu().numpy() - xr) / np.linalg.norm(xr))
            ms = timed_repeats(lambda k: G.hifir_dev(bd.data_ptr(), nirs, xd.data_ptr()), steps, barrier, stream, 3)
            rec.update(parity_vs_oracle=err, local_ms=ms, nirs=nirs)
        else:
            bh = P.seeded_rhs(n, rank)
            bd = torch.from_numpy(bh).cuda()
            xd = torch.empty_like(bd)
            G.solve_dev(bd.data_ptr(), xd.data_ptr(), 0)
            G.synchronize()
            xr = M.solve(bh)
            err = float(np.linalg.norm(xd.cpu().numpy() - xr) / np.linalg.norm(xr))
            ms = timed_repeats(lambda k: G.solve_dev(bd.data_ptr(), xd.data_ptr(), 0), steps, barrier, stream, 3)
            rec.update(parity_vs_oracle=err, local_ms=ms, depths=G.depths().tolist(),
                       bytes_per_apply=st["bytes_factors"] + st["bytes_dense"] + st["bytes_vec_per_rhs"])
        G.synchronize()
    finally:
        G.close()
    return rec


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    import hifir_b200 as hb
    from hifir_b200 import build, problems as P

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback exists)"
    torch.cuda.set_device(local_rank)
    pinned = pin_to_gpu_numa(local_rank)
    build.build()
    A = make_problem(args.workload, args.size)
    n = A[0]
    nsp = args.workload == "neumann"
    single = args.precision == "single"
    t0 = time.time()
    M = factorize(A, nsp=nsp, dtype=np.float32 if single else np.float64)
    t_fact = time.time() - t0
    levels = M.levels()
    t0 = time.time()
    G = hb.GpuHif(levels, device=local_rank)
    assert G.single == single
    G.set_matrix(A)
    if nsp:
        G.set_nsp_const()
    st = G.stats()
    t_attach = time.time() - t0
    log(f"[bench] rank {rank}: attach {t_attach:.1f} s, device bytes {st['device_bytes'] / 1e9:.2f} GB, "
        f"depths {G.depths().tolist()}, {pinned}")
    stream = torch.cuda.Stream()  # a side stream: the apply schedule is captured into CUDA graphs
    torch.cuda.set_stream(stream)
    G.set_stream(stream.cuda_stream)

    nb = NB_RHS
    nirs = args.nirs  # > 1: a step is one hifir(A, b, nirs, x) = nirs applies + nirs - 1 residuals (config 5)
    b_host = [torch.from_numpy(step_rhs(A, n, rank * nb + j, nirs)).pin_memory() for j in range(nb)]
    b_dev = [b.cuda() for b in b_host]
    x_dev = torch.empty(n, dtype=torch.float64, device="cuda")
    x_host = [torch.empty(n, dtype=torch.float64).pin_memory() for _ in range(2)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_dev(k):
        if nirs <= 1:
            G.solve_dev(b_dev[k % nb].data_ptr(), x_dev.data_ptr(), 0)
        else:  # hif::HIF::hifir: last_dim = size_t(-1), full-rank dense solve (builder.hpp:461)
            G.hifir_dev(b_dev[k % nb].data_ptr(), nirs, x_dev.data_ptr())

    pipelined = nirs <= 1 and not single  # lhfdGpuSolveAsync: H2D(k+1) | apply(k) | D2H(k-1)

    def step_host(k):
        if pipelined:
            G.solve_async(b_host[k % nb].numpy(), x_host[k % 2].numpy())
        elif nirs <= 1:
            G.solve(b_host[k % nb].numpy(), out=x_host[0].numpy())
        else:
            x_host[0].numpy()[:] = G.apply(b_host[k % nb].numpy(), nirs=nirs)[0]

    # ---- parity spot check before timing (against the C oracle's apply of the same factors)
    step_dev(0)
    G.synchronize()
    xr = M.solve(b_host[0].numpy()) if nirs <= 1 else M.hifir(b_host[0].numpy(), nirs)
    parity = float(np.linalg.norm(x_dev.cpu().numpy() - xr) / np.linalg.norm(xr))
    log(f"[bench] rank {rank}: parity vs oracle apply = {parity:.2e}")
    gate = 1e-5 if single else 1e-12  # north_star tolerances (float / double)
    assert parity <= gate, f"parity gate failed: {parity}"

    # ---- device-resident timing: REPEATS x --steps steps, median
    for k in range(max(args.warmup, 2 * nb)):
        step_dev(k)
    G.synchronize()
    launches0 = G.stats()["launch_count"]
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_rep = timed_repeats(step_dev, args.steps, barrier, stream)
    clocks = sampler.stop()
    G.synchronize()  # also surfaces a tripped spin limit
    launches = (G.stats()["launch_count"] - launches0) // REPEATS

    # ---- end to end through the host-buffer C-ABI call (pinned host memory, copies inside the timed region)
    for k in range(min(4, args.warmup)):
        step_host(k)
    G.synchronize()
    e2e_rep = []
    for _ in range(3):
        barrier()
        t0 = time.perf_counter()
        for k in range(args.steps):
            step_host(k)
        G.synchronize()
        e2e_rep.append((time.perf_counter() - t0) * 1e3)
        barrier()
    if pipelined:  # the pipelined entry returns what the synchronous one returns
        G.solve_async(b_host[0].numpy(), x_host[0].numpy())
        G.synchronize()
        assert np.linalg.norm(x_host[0].numpy() - xr) <= gate * np.linalg.norm(xr), "pipelined host solve differs"

    red = max_over_ranks(ms_rep + e2e_rep, world, dist)
    ms_rep, e2e_rep = red[:REPEATS], red[REPEATS:]
    ms_total, e2e_ms = statistics.median(ms_rep), statistics.median(e2e_rep)
    if world > 1:
        # result gather, off the timed path (the only NCCL traffic of this benchmark)
        out = [torch.empty_like(x_dev) for _ in range(world)]
        dist.all_gather(out, x_dev)
    # x_dev still holds the last timed step's result (the host-buffer steps use their own buffers); later
    # calls reuse it.  With several ranks: one row per rank, the gathered result.
    x_last = None
    if args.dump_outputs:
        x_last = x_dev.cpu().numpy() if world == 1 else torch.stack(out).cpu().numpy()
    ms_step = ms_total / args.steps / nirs  # per APPLY (a refinement step holds nirs of them)

    # ---- FGMRES-HIFIR solve time on every rank (second half of BASELINE.json's metric)
    extra = {}
    if not args.no_fgmres and not single:
        bk = P.csr_matvec(A, np.ones(n)) if not nsp else P.csr_matvec(A, np.sin(0.37 * np.arange(n)))
        G.fgmres(bk)  # warm-up (allocates the Krylov basis)
        barrier()
        t0 = time.perf_counter()
        xg, flag, iters, nmv = G.fgmres(bk)
        tg = time.perf_counter() - t0
        tmax = max_over_ranks([tg], world, dist)[0]
        extra["fgmres"] = {"gpu_time_s": tmax, "gpu_time_s_rank0": tg, "iters": iters, "num_mv": nmv, "flag": flag,
                           "restart": 30, "rtol": 1e-6, "systems": world,
                           "relres": float(np.linalg.norm(bk - P.csr_matvec(A, xg)) / np.linalg.norm(bk))}
        if world == 1 and not args.no_cpu:
            t0 = time.perf_counter()
            _, rflag, riters, rnmv = M.krylov(bk, "fgmres")
            extra["fgmres"].update(cpu_time_s=time.perf_counter() - t0, cpu_iters=riters, cpu_num_mv=rnmv,
                                   cpu_threads=1)

    # ---- the other BASELINE configs (3, 4, 5) as sub-records, measured on every rank
    st = G.stats()
    prof = {}
    if rank == 0:  # dominant kernel, timed live with events inside an instrumented (eager) apply
        for rep in range(5):
            for name, ms in G.profile_solve_dev(b_dev[0].data_ptr(), x_dev.data_ptr(), 0):
                prof.setdefault(name, []).append(ms)
        prof = {k: statistics.median(v) for k, v in prof.items()}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        applies = max(1, args.cpu_applies // nirs)
        rate, dt, _ = cpu_apply_rate(M, n, applies, nirs=nirs, A=A)
        cpu = {"value": rate * nirs, "unit": "applies/s", "cores": 1, "kind": "oracle",
               "sample": (f"{applies} C oracle applies" if nirs <= 1 else f"{applies} C oracle hifir(nirs={nirs}) solves") +
                         f" of the same workload on the same factors ({dt:.1f} s, serial)"}
    arena = None
    if args.arena_check and world == 1:
        # factor arena file (csrc/arena.cu): write, attach from the file, compare with the live attach
        path = os.path.join(CACHE_DIR, f"bench_{args.workload}{args.size}_{args.precision}.hifb")
        os.makedirs(CACHE_DIR, exist_ok=True)
        t0 = time.time()
        hb.save_arena(path, levels, True)
        t_save = time.time() - t0
        t0 = time.time()
        F = hb.attach_arena(path, device=local_rank)
        t_file = time.time() - t0
        if nsp:
            F.set_nsp_const()
        # a result carries the ready-bit parity of its apply in the last mantissa bit (common.cuh): compare
        # with the applies of both parities of the file-attached handle
        xb = G.solve(b_host[0].numpy())
        xa = [F.solve(b_host[0].numpy()) for _ in range(2)]
        arena = {"file_bytes": os.path.getsize(path), "save_s": t_save, "attach_file_s": t_file,
                 "attach_live_s": t_attach, "factorize_s_not_needed": t_fact,
                 "bit_identical_to_live_attach": bool(any(np.array_equal(x, xb) for x in xa)),
                 "max_rel_diff": float(max(np.linalg.norm(x - xb) for x in xa) / np.linalg.norm(xb))}
        F.close()
        os.remove(path)
    G.close()
    del M
    extras = {}
    for kind in [k for k in args.extras.split(",") if k in ("mrhs", "hifir", "stokes")]:
        barrier()
        try:
            rec = extra_workload(kind, args, rank, world, local_rank, barrier, stream)
        except Exception as e:  # noqa: BLE001 -- a failing extra must not take the headline down
            rec = {"error": f"{type(e).__name__}: {e}"[:300]}
        if world > 1:
            allrec = [None] * world
            dist.all_gather_object(allrec, rec)
        else:
            allrec = [rec]
        if rank == 0:
            errs = [r["error"] for r in allrec if "error" in r]
            if errs:
                extras[kind] = {"error": errs[0]}
                continue
            r0 = dict(allrec[0])
            ms = statistics.median([max(r["local_ms"][i] for r in allrec) for i in range(len(r0["local_ms"]))])  # max over ranks
            r0.pop("local_ms")
            r0["parity_vs_oracle"] = max(r["parity_vs_oracle"] for r in allrec)
            r0["ms_per_step"] = ms / r0["steps"]
            peak = hbm_peak()[0]
            if kind == "mrhs":
                r0.update(metric="column applies/s, 64 columns sharded over the ranks (strong scaling)",
                          value=r0["nrhs"] * r0["steps"] / (ms * 1e-3), scaling="strong",
                          roofline_frac=r0["bytes_per_block"] / (r0["ms_per_step"] * 1e-3) / 1e9 / (peak * world))
            elif kind == "hifir":
                r0.update(metric="applies/s inside hifir(A, b, 4, x), one system per rank (weak scaling)",
                          value=world * r0["nirs"] * r0["steps"] / (ms * 1e-3), scaling="weak",
                          solves_per_s=world * r0["steps"] / (ms * 1e-3))
            else:
                r0.update(metric="applies/s, one replica per rank (weak scaling)",
                          value=world * r0["steps"] / (ms * 1e-3), scaling="weak",
                          roofline_frac=r0["bytes_per_apply"] / (r0["ms_per_step"] * 1e-3) / 1e9 / peak)
            extras[kind] = r0
    if rank != 0:
        return

    bytes_apply = st["bytes_factors"] + st["bytes_dense"] + st["bytes_vec_per_rhs"]
    if nirs > 1:  # SURVEY.md 8(d): a refinement adds the bytes of A and 3 vectors, nirs - 1 times per solve
        bytes_apply += (nirs - 1) * (len(A[2]) * 12 + (n + 1) * 4 + 3 * 8 * n) // nirs
    peak, peak_src = hbm_peak()
    achieved = bytes_apply / (ms_step * 1e-3) / 1e9
    sb = sweep_bytes(levels)
    # dominant kernel = wsweep_kernel (all triangular sweeps of one apply are launches of it)
    sweep_ms = {k: v for k, v in prof.items() if k.endswith((".L", ".U", ".LU"))}
    sw_bytes = sum(sum(sb[k.split(".")[0] + "." + f] for f in k.split(".")[-1]) for k in sweep_ms)
    sw_ms = sum(sweep_ms.values())
    nl = max(1, len(sweep_ms))  # launches of the dominant kernel per apply
    k_ach = sw_bytes / (sw_ms * 1e-3) / 1e9
    # DRAM traffic of the dominant kernel: from the ncu capture of THIS kernel on THIS workload
    # (tools/ncu_traffic.py writes profiles/ncu_traffic.json); dropped when the packed factor differs
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        try:
            t = json.load(open(tpath)).get(workload_name(args.workload, args.size, 1), {})
            if t.get("kernel") == "wsweep_kernel" and abs(t.get("sweep_bytes", 0) - st["sweep_bytes"]) <= 0.02 * st["sweep_bytes"]:
                traffic, traffic_src = t.get("dram_bytes_per_launch"), t.get("source")
        except Exception:
            traffic = None
    # second ceiling of the sweeps: every factor entry gathers one solution value from L2 and an SM
    # accepts one L2 sector request per clock (measured: 289 G gathers/s on B200, tools/lat_bench.cu)
    gather_peak = 289e9
    roofline = {"bound": "hbm", "kernel": f"wsweep_kernel ({nl} launches per apply: one fused L-then-U sweep per level, "
                                          f"down and up)",
                "achieved": k_ach, "peak": peak, "unit": "GB/s", "frac": k_ach / peak, "traffic": traffic,
                "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": sw_bytes / nl, "ms_per_launch": sw_ms / nl,
                "share_of_step": sw_ms / max(1e-9, sum(prof.values())), "peak_source": peak_src,
                "streamed_bytes_per_launch": st["sweep_bytes"] / nl,
                "streamed_gbs": st["sweep_bytes"] / (sw_ms * 1e-3) / 1e9,
                "l2_gather": {"gathers_per_launch": st["sweep_entries"] / nl,
                              "achieved_g_per_s": st["sweep_entries"] / (sw_ms * 1e-3) / 1e9,
                              "peak_g_per_s": gather_peak / 1e9,
                              "frac": st["sweep_entries"] / (sw_ms * 1e-3) / gather_peak},
                "apply": {"kernels": st["kernels_per_apply"], "algorithmic_bytes": bytes_apply, "achieved": achieved,
                          "frac": achieved / peak},
                "latency_floor": {"dependent_steps_per_apply_reference": st["depth_total"],
                                  "dependent_steps_per_apply_merged": st["depth_merged"],
                                  "us_per_merged_step_achieved": sw_ms * 1e3 / max(1, st["depth_merged"])},
                "kernels_ms": {k: round(v, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1])[:12]},
                "timing": "kernels_ms: CUDA events around every kernel of an eager apply (median of 5); the timed "
                          "region itself launches each apply as one CUDA graph"}

    line = {
        "metric": "M^-1 applies/sec", "value": world * args.steps * nirs / (ms_total * 1e-3), "unit": "applies/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
        "repeats": REPEATS, "ms_per_step_repeats": [round(v / args.steps, 5) for v in ms_rep],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 factors (hif::HIF<float>), f64 vectors and accumulation" if single else "f64",
        "data": "synthetic",
        "config": {"workload": workload_name(args.workload, args.size, 1) + (" single-precision factors" if single else "")
                   + (f" hifir nirs={nirs}" if nirs > 1 else ""),
                   "n": n, "params": FACTORS, "l2_policy": L2_POLICY},
        "run": {"levels": st["levels"], "nnz_factors": st["nnz"],
                "l2_policy": f"inputs larger than L2: {bytes_apply / 1e9:.2f} GB streamed per apply vs 126 MB L2",
                "parallelism": "replicas, independent right-hand sides per GPU" if world > 1 else "1 GPU",
                "host_binding": pinned, "attach_s": round(t_attach, 1), "factorize_s": round(t_fact, 1)},
        "roofline": roofline, "cpu_baseline": cpu,
        "e2e": {"value": world * args.steps * nirs / (e2e_ms * 1e-3), "unit": "applies/s", "h2d_bytes_per_step": 8 * n,
                "d2h_bytes_per_step": 8 * n, "ms_per_step": e2e_ms / args.steps,
                "copy_gb_per_s_per_rank": 16 * n * args.steps / (e2e_ms * 1e-3) / 1e9,
                "api": ("lhfdGpuSolveAsync + lhfdGpuSynchronize (pinned host buffers; H2D, apply and D2H of consecutive "
                        "steps overlap; every step copies its b in and its x out)") if pipelined else
                       ((("lhfsdGpuSolve" if single else "lhfdGpuSolve") if nirs <= 1 else
                         ("lhfsdGpuApply" if single else "lhfdGpuApply") + f"(LHF_S, nirs={nirs})") + " (pinned host buffers)")},
        "gpu_launches": launches, "clocks": clocks, "parity_vs_oracle": parity,
    }
    if arena:
        line["arena"] = arena
    if nirs > 1:
        line["hifir"] = {"nirs": nirs, "solves_per_s": world * args.steps / (ms_total * 1e-3),
                         "ms_per_solve": ms_total / args.steps,
                         "step": f"hif::HIF::hifir(A, b, {nirs}, x): {nirs} applies + {nirs - 1} residuals b - A x, "
                                 "independent systems per GPU"}
    line.update(extra)
    line.update(extras)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, x=x_last)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="poisson", choices=["poisson", "neumann", "convdiff", "stokes"])
    ap.add_argument("--size", type=int, default=128)
    ap.add_argument("--nrhs", type=int, default=1,
                    help="> 1: batched multi-rhs mode (config 4), columns sharded over the ranks (strong scaling)")
    ap.add_argument("--precision", default="double", choices=["double", "single"],
                    help="single: hif::HIF<float,int> factors (mixed precision, lhfsdGpuSolve), parity gate 1e-5")
    ap.add_argument("--nirs", type=int, default=1,
                    help="> 1: a step is one hifir(A, b, nirs, x) iterative-refinement solve (config 5: neumann, nirs=4)")
    ap.add_argument("--arena-check", action="store_true",
                    help="also write a factor arena file, attach from it and compare (csrc/arena.cu)")
    ap.add_argument("--cpu-applies", type=int, default=40)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-fgmres", action="store_true")
    ap.add_argument("--extras", default="mrhs,hifir,stokes",
                    help="other BASELINE configs measured as sub-records of the line: mrhs (config 4), hifir (config 5), "
                         "stokes (config 3); '' = none")
    ap.add_argument("--extra-steps", type=int, default=10)
    ap.add_argument("--extras-small", action="store_true", help="developer: small sizes for the extras")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float64, at most 64 MB in all)")
    args = ap.parse_args()
    args.warmup = max(3, args.warmup)
    if args.dump_outputs and args.impl == "reference" and args.nrhs > 1:
        ap.error("--dump-outputs: the batched reference arm applies in worker processes and returns no outputs")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.nrhs > 1:
            run_mrhs(args, rank, world, local_rank)
        else:
            run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
