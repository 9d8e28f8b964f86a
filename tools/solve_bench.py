"""tools/solve_bench.py -- measures LU_solve (cflx_lu_solve) at the bench sizes, ranks as threads of one process.

    python tools/solve_bench.py --out DIR [--reps 12] [--nrhs 1,16,18,256,4096]

Workloads: C2 = N 16384, v 256 on 1x1x1; C3 = N 32768, v 512 on 2x2x1 when 4 GPUs are visible.  For each workload and
nrhs it reports the one-time preparation (host clock around the first solve after the factorisation, which returns
after a device synchronise), the solve time (ms_out, median after one warm-up), 2 M^2 nrhs / t, and the floor: the
larger of streaming the factors once (8 Ml Nl bytes per rank at 7.7 TB/s) and the flops at the measured DMMA burst
rate.  nrhs = 16 is the widest right-hand-side block of the bandwidth-bound update kernel, 18 the narrowest on the
DMMA GEMM.  Writes DIR/solve_bench.json."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import conflux_b200 as cb  # noqa: E402
from oracle import layout, solve_ref  # noqa: E402
from tests._harness import n_gpus, run_ranks  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def run(name, N, v, Px, Py, Pz, nrhs_list, reps, dmma_tflops):
    d = layout.dims(N, v, Px, Py, Pz)
    M = d["M"]
    rng = np.random.default_rng(1)
    Bs = {n: rng.standard_normal((M, n)) for n in nrhs_list}
    parts = {n: solve_ref.scatter_rows(Bs[n], N, v, Px, Py, Pz) for n in nrhs_list}

    def body(comm):
        gv = cb.lu_params(N, N, v, Px, Py, Pz, comm)
        fac_ms = cb.LU_rep(gv)
        res = dict(fac_ms=fac_ms, A=gv.data if min(nrhs_list) <= 16 else None, rows={})
        for i, n in enumerate(nrhs_list):
            B = parts[n][gv.rank]
            comm.barrier()
            t0 = time.perf_counter()
            X, _ = cb.LU_solve(gv, B)
            first = (time.perf_counter() - t0) * 1e3
            times = [cb.LU_solve(gv, B)[1] for _ in range(reps)]
            res["rows"][n] = dict(first_ms=first, times=times, X=X if n <= 16 else None, prep=(i == 0))
        gv.free_comms()
        return res

    rs = run_ranks(d["P"], body)
    A = layout.assemble([r["A"] for r in rs], N, v, Px, Py, Pz) if rs[0]["A"] is not None else None
    out = []
    bytes_floor = 8.0 * d["Ml"] * d["Nl"] / HBM_BYTES_PER_S * 1e3
    for n in nrhs_list:
        per_rank = [np.median(r["rows"][n]["times"]) for r in rs]
        ms = float(max(per_rank))
        flops = 2.0 * M * M * n
        flop_floor = flops / (dmma_tflops * 1e12 * d["P"]) * 1e3 if dmma_tflops else 0.0
        row = dict(workload=name, N=N, v=v, grid=[Px, Py, Pz], nrhs=n, factor_ms=rs[0]["fac_ms"], solve_ms=ms,
                   first_solve_ms=max(r["rows"][n]["first_ms"] for r in rs),
                   gflops=flops / (ms * 1e-3) / 1e9, floor_ms=max(bytes_floor, flop_floor),
                   floor_bound="hbm" if bytes_floor >= flop_floor else "dmma", update_path="skinny" if n <= 16 else "dmma")
        if rs[0]["rows"][n]["prep"]:
            row["prep_ms"] = row["first_solve_ms"] - ms     # first solve = one-time preparation + one solve (+ I/O)
        if A is not None and n <= 16:
            X = solve_ref.gather_cols([r["rows"][n]["X"] for r in rs], N, v, Px, Py, Pz)
            row["backward_error"] = float(np.linalg.norm(Bs[n] - A @ X) / (np.linalg.norm(A) * np.linalg.norm(X)))
        print(json.dumps(row), flush=True)
        out.append(row)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=12)
    ap.add_argument("--nrhs", default="1,16,18,256,4096")
    a = ap.parse_args()
    nrhs = [int(x) for x in a.nrhs.split(",")]
    os.makedirs(a.out, exist_ok=True)
    burst, _ = cb.dbg.fp64_peak_ex(0)
    res = dict(card=card(), dmma_burst_tflops=burst, hbm_tb_s=HBM_BYTES_PER_S / 1e12, rows=[])
    res["rows"] += run("C2", 16384, 256, 1, 1, 1, nrhs, a.reps, burst)
    if n_gpus() >= 4:
        res["rows"] += run("C3", 32768, 512, 2, 2, 1, nrhs, a.reps, burst)
    with open(os.path.join(a.out, "solve_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(card=res["card"], dmma_burst_tflops=burst)))


if __name__ == "__main__":
    main()
