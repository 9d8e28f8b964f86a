#!/usr/bin/env python
"""bench.py -- LU GFLOP/s (FP64, (2/3)N^3) of the CONFLUX hot path on 1/2/4/8 B200 (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...     (N > 1: one rank per GPU)

A "step" is one LU factorisation of one synthetic matrix (lu_params::InitMatrix generator, seed 42):
    N=1: 16384 x 16384, v=256, grid 1x1x1   (BASELINE.json configs[1])
    N=2: 32768 x 32768, v=512, grid 1x1x2   (auto grid of 2 ranks, lu_params.hpp:21-47)
    N=4: 32768 x 32768, v=512, grid 2x2x1   (configs[2])
    N=8: 65536 x 65536, v=512, grid 2x2x2   (configs[3])
`value` times K steps with the matrix already resident in HBM (pristine device copy -> working copy -> factor),
`e2e` times K steps through the public LU_rep call with the host->device copy of one matrix per step from pinned
memory and the device->host read of the permutation inside the timed region (streamed: the upload of the next
matrix overlaps the current factorisation; `e2e.single_shot` is the un-overlapped latency of one call).  PyTorch is plumbing only
(torch.distributed bootstrap, pinned host memory).
`--dump-outputs DIR` writes, after the timed steps, what the last one handed its caller (see dump_outputs()), so that
two builds can be compared output for output on the same seeded input.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {1: (16384, 256, (1, 1, 1)), 2: (32768, 512, (1, 1, 2)), 4: (32768, 512, (2, 2, 1)),
             8: (65536, 512, (2, 2, 2))}
FP64_TENSOR_NOMINAL_TFLOPS = 40.0  # NVIDIA B200 datasheet (FP64 / FP64 tensor), context only


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        # median over the samples taken under load (upper half of the sorted clocks)
        load = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": load[len(load) // 2] if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


CPU_THREAD_CAP = 32  # OpenBLAS (pthreads) + the reference's OpenMP loops oversubscribe badly beyond this


def cpu_threads():
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, min(n, CPU_THREAD_CAP))


def host_mem_bytes():
    try:
        return os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_PHYS_PAGES")
    except (ValueError, OSError):
        return 0


_CPU_SNIPPET = r"""
import os, sys, json
cores = %(cores)d
def _busy():                              # per-CPU busy jiffies from /proc/stat
    out = {}
    for ln in open("/proc/stat"):
        f = ln.split()
        if f[0].startswith("cpu") and f[0] != "cpu":
            t = [int(x) for x in f[1:9]]
            out[int(f[0][3:])] = (sum(t) - t[3] - t[4], sum(t))
    return out
try:                                      # pin the whole process (BLAS pthreads + OpenMP inherit it) to the `cores` CPUs
    import time                           # that are idle right now: the box is shared, the first CPUs usually are not
    allowed = sorted(os.sched_getaffinity(0))
    a = _busy(); time.sleep(0.5); b = _busy()
    load = [(b[c][0] - a[c][0]) / max(1, b[c][1] - a[c][1]) if c in a and c in b else 1.0 for c in allowed]
    k = min(cores, len(allowed))          # the least-loaded window of CONSECUTIVE CPUs (one socket / NUMA node as a rule)
    best = min(range(len(allowed) - k + 1), key=lambda i: (round(sum(load[i:i + k]), 1), i))
    os.sched_setaffinity(0, allowed[best:best + k])
except Exception:
    pass
sys.path.insert(0, %(root)r)
from oracle import ref
if not ref.available():
    print(json.dumps({"kind": "unavailable"})); sys.exit(0)
n, v, g, P = %(n)d, %(v)d, %(grid)r, %(P)d
thr = max(1, cores // P)
ref.lu_bench(%(warm_n)d, %(warm_v)d, *g, n_warm=0, n_rep=1, budget_s=1e9, blas_threads=thr)      # thread pools warm
r = ref.lu_bench(n, v, *g, n_warm=%(n_warm)d, n_rep=%(n_rep)d, budget_s=%(budget)f, blas_threads=thr)
print(json.dumps({"kind": "reference", "inner_ms": r["inner_ms"], "outer_ms": r["outer_ms"], "blas_threads": thr}))
"""


def cpu_reference_run(n, v, grid, cores, n_warm, n_rep, budget_s, timeout_s):
    """The reference's own CPU LU_rep (oracle/_ref = the /root/reference sources + OpenBLAS, ranks = threads) in ONE child
    process: one lu_params object, thread pools warmed by a small factorisation, n_warm untimed + up to n_rep timed
    repetitions of the stated configuration, time-boxed.  Returns the child's dict or {"kind": "unavailable: ..."}."""
    P = grid[0] * grid[1] * grid[2]
    thr = max(1, cores // P)
    # (no OMP_PROC_BIND: OpenBLAS' pthreads inherit the one-CPU mask of the bound OpenMP thread that creates them -- measured
    # 13.7 s instead of 0.3 s for N=2048; the process-wide affinity set in the child is what keeps the numbers stable)
    env = dict(os.environ, OMP_NUM_THREADS=str(thr), OPENBLAS_NUM_THREADS=str(thr))
    env.pop("OMP_PROC_BIND", None)
    code = _CPU_SNIPPET % dict(root=ROOT, n=n, v=v, grid=tuple(grid), P=P, cores=cores, warm_n=min(n, 8 * v * grid[0]),
                               warm_v=v, n_warm=n_warm, n_rep=n_rep, budget=budget_s)
    try:
        out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=timeout_s)
        return json.loads(out.stdout.strip().splitlines()[-1])
    except Exception as e:  # noqa: BLE001
        return {"kind": "unavailable: %s" % type(e).__name__}


def reference_plan(gpus):
    """(N, v, grid, note) the CPU arm runs for `--gpus N`: the stated configuration whenever it fits the host's memory
    and a few minutes of CPU time; the 8-GPU configuration (N=65536, 2x2x2: ~40 min and ~400 GiB on the host) is
    measured at N=32768 with the same v and grid and reported as a RATE, labelled as such."""
    N, v, grid = WORKLOADS[gpus]
    P = grid[0] * grid[1] * grid[2]
    note = None
    if gpus == 8:
        N, note = 32768, "rate measured at N=32768 (same v, same grid); the N=65536 run needs ~40 min of host time"
    d = -(-N // (v * grid[0])) * v
    need = 6 * P * d * (-(-N // (v * grid[1])) * v) * 8      # data, A11Buff, A11BuffTemp, A10resultBuff, C + panels
    mem = host_mem_bytes()
    if mem and need > 0.7 * mem and P > 1:
        grid = (1, 1, 1)
        note = (note + "; " if note else "") + "grid 1x1x1 on the host (the rank-thread grid needs %.0f GiB)" % (need / 2 ** 30)
    return N, v, grid, note


def workload_string(N, v, grid, override=False):
    return f"LU N={N} v={v} grid {grid[0]}x{grid[1]}x{grid[2]}" + (" (size override, not the BASELINE config)" if override else "")


GENERATOR = "lu_params::InitMatrix mt19937_64(42+rank), 5+U[0,1)"


def l2_string(N, v, grid):
    Ml = -(-N // (v * grid[0])) * v
    Nl = -(-N // (v * grid[1])) * v
    return "inputs larger than L2 (local matrix %.1f GiB)" % (Ml * Nl * 8 / 2 ** 30)


def run_reference_arm(args, rank):
    if rank != 0:
        return
    cores = cpu_threads()
    N, v, grid = WORKLOADS[args.gpus]
    n_s, v_s, g_s, note = reference_plan(args.gpus)
    if args.N:  # testing only: the line says so
        N, n_s = args.N, args.N
        v = v_s = args.v or v
        note = "size override (testing), not the BASELINE config"
    budget = float(os.environ.get("CFLX_REF_BUDGET_S", "300"))
    t0 = time.time()
    n_warm = 1 if n_s <= 16384 else 0        # big configurations: the small warm-up factorisation only (one rep is minutes)
    d = cpu_reference_run(n_s, v_s, g_s, cores, min(args.warmup, n_warm), args.steps, budget, timeout_s=budget * 4 + 600)
    if not d.get("inner_ms"):
        print(json.dumps({"impl": "reference", "unavailable": "CPU reference run failed or timed out (%s)" % d.get("kind")}))
        return
    done = len(d["inner_ms"])
    ms_step = sum(d["inner_ms"]) / done
    val = (2.0 / 3.0) * n_s ** 3 / (ms_step * 1e-3) / 1e9
    sample = (f"reference LU_rep N={n_s} v={v_s} grid {g_s[0]}x{g_s[1]}x{g_s[2]} (ranks = threads), {done} of {args.steps} "
              f"timed factorisation(s) in one process after a warm-up, time-boxed to {budget:.0f} s; ms = what LU_rep returns "
              f"(main loop, conflux_opt.hpp:1807); OpenBLAS 0.3.15, {cores} pinned cores = {g_s[0] * g_s[1] * g_s[2]} rank(s) x "
              f"{d.get('blas_threads')} threads; MKL/MPI are not in the image" + (f"; {note}" if note else ""))
    print(json.dumps({
        "impl": "reference", "metric": "LU GFLOP/s (FP64, (2/3)N^3)", "value": val, "unit": "GFLOP/s", "n_gpus": args.gpus,
        "steps": args.steps, "steps_done": done, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_string(N, v, grid, bool(args.N)), "generator": GENERATOR, "l2": l2_string(N, v, grid)},
        "measured_on": workload_string(n_s, v_s, g_s), "extrapolated": bool(n_s != N),
        "cpu_baseline": {"value": val, "unit": "GFLOP/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": val, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "outer_ms_per_step": sum(d["outer_ms"]) / done, "wall_s": time.time() - t0}))


def load_golden_perm(N, v, grid):
    """Reference pivot sequence for this exact configuration (tests/golden/lu_perms_bench.npz, produced by running the
    reference itself: tests/golden/make_golden_bench.py), or None."""
    import numpy as np
    path = os.path.join(ROOT, "tests", "golden", "lu_perms_bench.npz")
    if not os.path.exists(path):
        return None
    G = np.load(path)
    for name in ("C2", "C3"):
        if name in G and name + "_case" in G and tuple(int(x) for x in G[name + "_case"]) == (N, v) + tuple(grid):
            return G[name]
    return None


def load_traffic(M, N, K, kernel="dmma"):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the trailing-update kernel, from the committed
    summary of an `ncu --set full` capture (profiles/r02_gemm_traffic.json, written by tools/summarize_ncu.py)."""
    path = os.path.join(ROOT, "profiles", "r02_gemm_traffic.json")
    try:
        d = json.load(open(path))
    except Exception:  # noqa: BLE001
        return None, None
    for e in d.get("launches", []):
        if (e.get("kernel", "dmma"), e.get("M"), e.get("N"), e.get("K")) == (kernel, M, N, K):
            return e.get("dram_bytes"), e.get("source")
    return None, None


DUMP_FACTOR_BYTES = 48 << 20     # --dump-outputs: sampled factor rows over all ranks (the whole dump stays under 64 MB)


def dump_outputs(dirname, rank, n_holders, factor=None, factor_name=None, perm=None):
    """--dump-outputs: writes DIR/<name>.npy in float64.  `perm` (the pivot sequence, identical on every rank) goes to
    lu_perm.npy from rank 0; `factor` (this rank's Ml x Nl block of the factors, None on ranks that hold none) is too
    large to write whole, so a fixed seeded set of its rows goes to <factor_name>_r<rank>.npy and their local indices to
    <factor_name>_rows_r<rank>.npy.  The n_holders ranks that hold factors share DUMP_FACTOR_BYTES."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    if perm is not None and rank == 0:
        np.save(os.path.join(dirname, "lu_perm.npy"), perm.astype(np.float64))
    if factor is not None:
        n = max(1, min(factor.shape[0], DUMP_FACTOR_BYTES // (n_holders * factor.shape[1] * 8)))
        rows = np.sort(np.random.default_rng(rank).choice(factor.shape[0], size=n, replace=False))
        np.save(os.path.join(dirname, f"{factor_name}_r{rank}.npy"), factor[rows])
        np.save(os.path.join(dirname, f"{factor_name}_rows_r{rank}.npy"), rows.astype(np.float64))


CHOL_WORKLOAD = (32768, 512)     # BASELINE.json configs[4]: cholesky_miniapp --dim=32768 --tile=512 (8 x B200)


def run_cholesky(args, rank, world, local_rank):
    """`--algo cholesky`: the CONFCHOX path (BASELINE config C5) at --gpus N, strong scaling (same matrix at every N), the
    reference's automatic grid (Cholesky.cpp:75-111: 8 -> 4x2x1).  Same JSON contract as the LU line."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import conflux_b200 as cb
    from conflux_b200 import _lib
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("gloo", rank=rank, world_size=world)
    N, v = CHOL_WORKLOAD
    if args.N:
        N = args.N
    if args.v:
        v = args.v
    comm = cb.Comm.from_torch_distributed(device=local_rank) if world > 1 else cb.Comm(1, 0, None, local_rank)
    ch = cb.cholesky.initialize(N, v, (0, 0, 0), comm)
    host = cb.pinned_empty((ch.Ml, ch.Nl))
    host[...] = ch.data
    ch.data = host
    flops = float(ch.N) ** 3 / 3.0

    def barrier():
        comm.barrier()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    peak = cb.dbg.fp64_peak_ex(0)[0] if rank == 0 else None
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ch.parallelCholesky(upload=True)
    for _ in range(max(args.warmup, 3) - 1):
        ch.parallelCholesky(upload=False)
    cnt = ctypes.c_int64()
    _lib.lib().cflx_chol_launch_count(ch._h, ctypes.byref(cnt), 1)
    barrier()
    dev_ms = 0.0
    for _ in range(args.steps):
        dev_ms += ch.parallelCholesky(upload=False)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    _lib.lib().cflx_chol_launch_count(ch._h, ctypes.byref(cnt), 1)
    dev_ms = max_over_ranks(dev_ms)
    ms_step = dev_ms / args.steps
    value = flops / (ms_step * 1e-3) / 1e9
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ch.parallelCholesky(upload=True)
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / args.steps
    if args.dump_outputs:       # the factor of the last timed step; only layer 0 holds it
        dump_outputs(args.dump_outputs, rank, ch.PX * ch.PY, ch.local_factor() if ch.pz == 0 else None, "chol_factor")
    resid_abs, resid = ch.validate()
    if rank == 0:
        grid = (ch.PX, ch.PY, ch.PZ)
        line = {"metric": "Cholesky GFLOP/s (FP64, (1/3)N^3)", "value": value, "unit": "GFLOP/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"cholesky N={ch.N} v={ch.v} grid {grid[0]}x{grid[1]}x{grid[2]}",
                           "generator": "CholeskyIO::generateInputMatrixDistributed (tile = lower(R^T R), srand(1), diagonal 2*Kappa*max row sum)",
                           "l2": "inputs larger than L2 (local matrix %.1f GiB)" % (ch.Ml * ch.Nl * 8 / 2 ** 30)},
                "timing": "CUDA events on the launching stream around each factorisation loop, max over ranks",
                "e2e": {"value": flops / (e2e_ms * 1e-3) / 1e9, "unit": "GFLOP/s", "ms_per_step": e2e_ms,
                        "h2d_bytes_per_step": int(ch.Ml * ch.Nl * 8), "d2h_bytes_per_step": 0},
                "gpu_launches": int(cnt.value), "clocks": clocks,
                "roofline": {"bound": "tensor", "kernel": "whole path (gemm_tn_kernel, DMMA.8x8x4, does the rank-v updates)",
                             "achieved": value / 1e3 / args.gpus, "peak": peak, "unit": "TFLOP/s per GPU",
                             "frac": value / 1e3 / args.gpus / peak if peak else None, "traffic": None},
                "parity": {"residual_A_minus_LLt_rel_frobenius": resid, "residual_A_minus_LLt_abs_frobenius": resid_abs,
                           "residual_tolerance": 1e-12, "residual_how": "cflx_chol_validate: update sweep replayed with the stored factor on the grid"}}
        if args.gpus == 1 and not args.no_cpu_baseline:
            import scipy.linalg
            n_s = 8192
            A = np.random.default_rng(0).standard_normal((n_s, 64))
            S = A @ A.T + n_s * np.eye(n_s)
            t1 = time.perf_counter()
            scipy.linalg.cholesky(S, lower=True, overwrite_a=True, check_finite=False)
            dt = time.perf_counter() - t1
            line["cpu_baseline"] = {"value": n_s ** 3 / 3.0 / dt / 1e9, "unit": "GFLOP/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": f"LAPACK dpotrf (scipy/OpenBLAS) N={n_s}, one call -- the reference's own checker "
                                              "(cholesky_helper.cpp:183-217); its MPI driver needs >= 4 ranks and MPI, absent here"}
        print(json.dumps(line))
    ch.finalize()
    comm.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--algo", default="lu", choices=["lu", "cholesky"], help="cholesky = BASELINE config C5 (not the driver's default)")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--N", type=int, default=0, help="override the matrix size (testing only; the line says so)")
    ap.add_argument("--v", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-validate", action="store_true", help="skip the grid-wide residual (debugging only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computes; --impl reference has no outputs to write")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if args.algo == "cholesky":
        if world != args.gpus:
            raise SystemExit(f"--gpus {args.gpus} needs WORLD_SIZE == {args.gpus} (launch N>1 with torchrun)")
        run_cholesky(args, rank, world, local_rank)
        return
    if args.gpus not in WORKLOADS or world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} needs WORLD_SIZE == {args.gpus} in {sorted(WORKLOADS)} (launch N>1 with torchrun)")
    if args.warmup < 3:
        args.warmup = 3

    import numpy as np
    import torch
    import torch.distributed as dist
    import conflux_b200 as cb
    from conflux_b200 import _lib

    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("gloo", rank=rank, world_size=world)
    N, v, (Px, Py, Pz) = WORKLOADS[args.gpus]
    override = bool(args.N)
    if args.N:
        N = args.N
    if args.v:
        v = args.v
    L = _lib.lib()
    comm = cb.Comm.from_torch_distributed(device=local_rank) if world > 1 else cb.Comm(1, 0, None, local_rank)
    gv = cb.lu_params(N, N, v, Px, Py, Pz, comm)
    # pinned host staging for the end-to-end arm
    host = cb.pinned_empty((gv.Ml, gv.Nl))        # cudaHostAlloc through the library (torch never touches CUDA here)
    host[...] = gv.data
    gv.data = host
    perm = np.zeros(gv.M, dtype=np.int32)
    flops = (2.0 / 3.0) * float(gv.N) ** 3

    def barrier():
        comm.barrier()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # FP64 tensor-pipe peak of THIS GPU, measured before the runs (burst) -- MEASURED_PEAKS.json has no FP64 entry
    peak_burst = cb.dbg.fp64_peak_ex(0)[0] if rank == 0 else None
    tcgen05 = bool(L.cflx_lu_uses_tcgen05(gv._h))
    # raw int8 rate of the tensor pipe (back-to-back tcgen05.mma 128x256x32, operands resident): the ceiling of the tcgen05 path
    i8_tmacs = cb.dbg.umma_peak(0, 256) if (rank == 0 and tcgen05) else None
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # ---- device-resident arm -------------------------------------------------------------------------------
    cb.LU_rep(gv, None, perm, upload=True)
    for _ in range(args.warmup - 1):
        cb.LU_rep(gv, None, None, upload=False)
    cnt = ctypes.c_int64()
    L.cflx_lu_launch_count(gv._h, ctypes.byref(cnt), 1)
    L.cflx_lu_set_kernel_timing(gv._h, 1)
    barrier()
    t0 = time.perf_counter()
    dev_ms, gemm_ms, gemm_flops = 0.0, 0.0, 0.0
    for _ in range(args.steps):
        dev_ms += cb.LU_rep(gv, None, None, upload=False)   # device-timed main loop (CUDA events on the rank's stream)
        a, b = ctypes.c_double(), ctypes.c_double()
        L.cflx_lu_trailing_stats(gv._h, ctypes.byref(a), ctypes.byref(b))
        gemm_ms += a.value
        gemm_flops += b.value
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop() if rank == 0 else None
    L.cflx_lu_launch_count(gv._h, ctypes.byref(cnt), 1)
    launches = cnt.value
    L.cflx_lu_set_kernel_timing(gv._h, 0)
    wall_ms = max_over_ranks(wall_ms)
    dev_ms = max_over_ranks(dev_ms)
    # the timed region is the reference's: the main loop between two grid barriers (conflux_opt.hpp:531-532,1805),
    # measured with CUDA events on each rank's launching stream, summed over the K steps, max over ranks
    ms_step = dev_ms / args.steps
    value = flops / (ms_step * 1e-3) / 1e9

    # ---- end-to-end arm: H2D of one matrix + one factorisation + D2H of the permutation, every step -----------------
    # (a) streamed: back-to-back factorisations with double-buffered input -- every step uploads one full matrix from
    # pinned host memory on a copy stream (the input of the NEXT step, cflx_lu_queue_next_local), factors the matrix
    # the previous step uploaded, and reads its permutation back: K uploads, K factorisations, K read-backs per K steps
    cb.LU_rep(gv, None, perm, upload=True, next_data=gv.data)
    cb.LU_rep(gv, None, perm, upload=False, next_data=gv.data)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cb.LU_rep(gv, None, perm, upload=False, next_data=gv.data)
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / args.steps
    e2e_val = flops / (e2e_ms * 1e-3) / 1e9
    # (b) single shot: upload, then factor, then read back, nothing overlapped (the latency of ONE call; step 0 of a
    # factorisation touches the whole matrix, so the transfer cannot hide inside a single run -- DESIGN.md section 5)
    for _ in range(2):
        cb.LU_rep(gv, None, perm, upload=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cb.LU_rep(gv, None, perm, upload=True)
    barrier()
    e2e1_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / args.steps
    e2e1_val = flops / (e2e1_ms * 1e-3) / 1e9
    if args.dump_outputs:       # what LU_rep(gv, C, perm) hands over after the last timed step; only layer 0 holds factors
        C = None
        if gv.pk == 0:
            C = np.empty((gv.Ml, gv.Nl))
            _lib.check(L.cflx_lu_get_factors(gv._h, C.ctypes.data, None), "lu_get_factors")
        dump_outputs(args.dump_outputs, rank, Px * Py, C, "lu_factors", perm)

    # ---- parity of the run that was just timed (every rank takes part: the residual is a grid collective) ------------
    ok_perm = sorted(perm.tolist()) == list(range(gv.M))
    resid_abs = resid = None
    if not args.no_validate:
        resid_abs, resid = cb.validate(gv)            # ||PA-LU||_F and /||A||_F on the GPU grid, full BASELINE size
    golden = load_golden_perm(gv.N, gv.v, (Px, Py, Pz))
    pivots_equal = bool(np.array_equal(perm, golden)) if golden is not None else None

    if rank == 0:
        dmma_peak = peak_burst
        g_tf = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else None
        n1 = gv.Ml - gv.v                             # first-step shape of the trailing update (the ncu-captured launch)
        traffic, traffic_src = load_traffic(n1, gv.Nl - gv.v, gv.nlayr, "ozaki" if tcgen05 else "dmma")
        # FP64-equivalent ceiling of the int8 path: 36 exact int8 plane products per FP64 product
        i8_equiv = (2.0 * i8_tmacs / 36.0) if i8_tmacs else None
        roof_peak = i8_equiv if tcgen05 else dmma_peak
        grid = (Px, Py, Pz)
        line = {
            "metric": "LU GFLOP/s (FP64, (2/3)N^3)", "value": value, "unit": "GFLOP/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_string(gv.N, gv.v, grid, override), "generator": GENERATOR,
                       "l2": l2_string(gv.N, gv.v, grid)},
            "timing": "CUDA events on the launching stream around each factorisation's main loop, max over ranks",
            "wall_ms_per_step_incl_restore_copy": wall_ms / args.steps,
            "e2e": {"value": e2e_val, "unit": "GFLOP/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": int(gv.Ml * gv.Nl * 8),
                    "d2h_bytes_per_step": int(gv.M * 4),
                    "mode": "streamed: every step uploads one matrix (pinned host -> HBM, copy stream) while the matrix uploaded "
                            "by the previous step is factored, then reads the permutation back (public LU_rep(next_data=...))",
                    "single_shot": {"value": e2e1_val, "ms_per_step": e2e1_ms,
                                    "mode": "upload, factor, read back in sequence: the latency of one isolated call"}},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "tensor",
                         "kernel": ("ozaki_gemm_kernel (int8 tcgen05.mma + TMEM + TMA, 36 exact digit-plane products per FP64 product)"
                                    if tcgen05 else "gemm_tn_kernel (FP64 DMMA.8x8x4)") + ", trailing update",
                         "achieved": g_tf, "peak": roof_peak, "unit": "TFLOP/s (FP64-equivalent)" if tcgen05 else "TFLOP/s",
                         "frac": (g_tf / roof_peak) if (g_tf and roof_peak) else None,
                         "frac_of_fp64_dmma_peak": (g_tf / dmma_peak) if g_tf else None, "fp64_dmma_peak": dmma_peak,
                         "int8_pipe_measured_pops": (2.0 * i8_tmacs / 1e3) if i8_tmacs else None,
                         # dram__bytes_read+write of ONE launch of the first-step shape, read from the committed summary of
                         # an `ncu --set full` capture; algorithmic bytes = 16*M*N + 8*K*(M+N) (C read+write, operands once)
                         "traffic": traffic, "traffic_source": traffic_src,
                         "traffic_launch": f"M={n1} N={gv.Nl - gv.v} K={gv.nlayr} (step 0), algorithmic "
                                           f"{16.0 * n1 * (gv.Nl - gv.v) + 8.0 * gv.nlayr * (n1 + gv.Nl - gv.v):.4g} B",
                         "peak_source": ("tcgen05 path: peak = raw int8 rate of the tensor pipe measured live (cflx_dbg_umma_peak: back-to-back "
                                         "tcgen05.mma.kind::i8 128x256x32, one CTA per SM; nominal 4.5 POP/s) x 2 / 36 digit-plane products; "
                                         if tcgen05 else "") +
                                        "fp64_dmma_peak = FP64 tensor (DMMA.8x8x4) burst peak measured live by cflx_dbg_fp64_peak_ex "
                                        "(best ~2 ms launch; = 148 SM x 4 x 32 flop/clk x 1.965 GHz); MEASURED_PEAKS.json has no "
                                        "FP64 / int8 entry; nominal FP64 %.0f TFLOP/s" % FP64_TENSOR_NOMINAL_TFLOPS,
                         "share_of_step": gemm_ms / dev_ms if dev_ms else None,
                         "whole_path_frac": value / 1e3 / (args.gpus * dmma_peak)},
            "parity": {"permutation_is_permutation": bool(ok_perm), "pivots_equal_reference": pivots_equal,
                       "pivots_reference": ("tests/golden/lu_perms_bench.npz (the reference itself, same N, v, grid)"
                                            if golden is not None else "no golden for this configuration (host memory)"),
                       "residual_PA_minus_LU_rel_frobenius": resid, "residual_PA_minus_LU_abs_frobenius": resid_abs,
                       "residual_tolerance": 1e-12,
                       "residual_how": "cflx_lu_validate: masked L/U SUMMA over the grid (conflux_miniapp.cpp:349-500)"},
        }
        if args.gpus == 1 and not args.no_cpu_baseline:
            cores = cpu_threads()
            n_s = 8192
            d = cpu_reference_run(n_s, 256, (1, 1, 1), cores, 1, 2, 40.0, timeout_s=240)
            if not d.get("inner_ms"):      # a crowded host: a sample 8x smaller rather than no number at all
                n_s = 4096
                d = cpu_reference_run(n_s, 256, (1, 1, 1), cores, 1, 2, 20.0, timeout_s=180)
            ms = min(d["inner_ms"]) if d.get("inner_ms") else None
            line["cpu_baseline"] = {"value": ((2.0 / 3.0) * n_s ** 3 / (ms * 1e-3) / 1e9) if ms else None, "unit": "GFLOP/s",
                                    "cores": cores, "kind": d.get("kind"),
                                    "sample": f"reference LU_rep N={n_s} v=256 grid 1x1x1, best of {len(d.get('inner_ms', []))} after a "
                                              f"warm-up, one process, OpenBLAS 0.3.15 ({cores} pinned cores of "
                                              f"{os.cpu_count()}); MKL/MPI are not in the image"}
        print(json.dumps(line))
    gv.free_comms()
    comm.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
