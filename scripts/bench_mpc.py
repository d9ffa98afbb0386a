"""Closed-loop MPC throughput: ilqgb_mpc (every step on the device) against the loop a caller writes without it (per step
ilqgb_solve_host on pinned buffers, then the shift and the disturbance in numpy), and ilqgb_shift on its own.

Workload: car parking, T = 500, max_iter 10 per step, S = 20 steps, w = workloads.disturbance(scale 0.01); --batch sizes (default
65 536 and 262 144 problems) on --gpus GPUs through ilqgb_create_multi.  After a warm-up closed loop of the same shape the two
legs alternate --reps times; each leg is timed by the host clock around calls that end in a synchronise.  The logs of the two
legs (x0 and applied u of every step, cost, iterations, result) must be bit-identical, otherwise the script exits non-zero.
ilqgb_shift is timed with CUDA events around each call on one GPU (a start between two calls, outside the events); its bytes are
those of the records it touches, at 32-byte sector granularity, against the HBM bandwidth measured on a B200 and recorded in
profiles/bench_r02f_1gpu.json.  One JSON line per batch size goes to stdout (and, with --out FILE, is appended to FILE).

    python scripts/bench_mpc.py [--gpus N] [--batch 65536,262144] [--reps 2] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "ddp-generator_b200"))

import torch  # noqa: E402  (pinned host memory and CUDA events)

import ilqg_b200  # noqa: E402
from ilqg_b200 import workloads as W  # noqa: E402

LOG_KEYS = ("x", "u", "cost", "iterations", "success")


def gpu_facts(n):
    """Name and power limit of the GPUs in use, read in the same run (read-only query)."""
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, check=True)
    rows = [[f.strip() for f in line.split(",")] for line in q.stdout.strip().splitlines()][:n]
    return [{"index": int(r[0]), "name": r[1], "power_limit_w": float(r[2])} for r in rows]


def hbm_peak():
    rec = json.loads(open(os.path.join(ROOT, "profiles", "bench_r02f_1gpu.json")).readline())["roofline"]
    return float(rec["peak"]), "profiles/bench_r02f_1gpu.json (HBM bandwidth measured on B200)"


def make_solver(B, T, max_iter, gpus, **kw):
    s = ilqg_b200.BatchSolver("car", 0, B, T, devices=gpus, **kw) if gpus > 1 else ilqg_b200.BatchSolver("car", 0, B, T, **kw)
    s.set_options({"max_iter": max_iter})
    s.set_params(W.CAR_PARAMS)
    return s


def leg_fused(s, x0, u0, w, S):
    t = time.perf_counter()
    logs = s.mpc(x0, u0, S, w)
    return time.perf_counter() - t, logs


def leg_host(s, x0, u0, w, S, pin):
    """Today's loop: one end-to-end solve per step from pinned buffers, the next input shifted on the host."""
    xi, ui, xo, uo, co, it, re = pin
    B = x0.shape[0]
    logs = dict(x=np.empty((B, S + 1, x0.shape[1])), u=np.empty((B, S, ui.shape[2])), cost=np.empty((B, S)),
                iterations=np.empty((B, S), np.int32), success=np.empty((B, S), np.int32))
    ptr = lambda a: a.ctypes.data
    t = time.perf_counter()
    xi[:] = x0
    ui[:] = u0
    for st in range(S):
        s.solve_host_ptr(ptr(xi), ptr(ui), ptr(xo), ptr(uo), ptr(co), ptr(it), ptr(re), None)
        logs["x"][:, st] = xi
        logs["u"][:, st] = uo[:, 0]
        logs["cost"][:, st] = co
        logs["iterations"][:, st] = it
        logs["success"][:, st] = re
        np.add(xo[:, 1], w[:, st], out=xi)
        ui[:, :-1] = uo[:, 1:]
        ui[:, -1] = uo[:, -1]
    logs["x"][:, S] = xi
    return time.perf_counter() - t, logs


def time_shift(B, T, max_iter, x0, u0, calls):
    """ilqgb_shift(1) alone on one GPU: CUDA events on the handle's stream around each call."""
    st = torch.cuda.Stream()
    s = make_solver(B, T, max_iter, 1, stream=st.cuda_stream)
    s.upload(x0, u0)
    s.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(calls + 3)]
    for a, b in ev:
        a.record(st)
        s.shift(1)
        b.record(st)
        s.start()          # a shift needs a solution to shift: the initial rollout of the shifted input
    st.synchronize()
    ms = np.array([a.elapsed_time(b) for a, b in ev[3:]])
    nx, nu = s.nx, s.nu
    s.close()
    # per problem: the u sectors of T records read and written (records are whole 32-byte sectors), the x sector of x[1] read,
    # x0 written ([NX][Bp], 8 bytes per state)
    sect = ((nx + nu) * 8 - 1) // 32 - (nx * 8) // 32 + 1
    nbytes = B * (T * 2 * 32 * sect + 32 + 8 * nx)
    peak, src = hbm_peak()
    gbs = nbytes / (np.median(ms) * 1e-3) / 1e9
    return {"calls": calls, "ms_median": float(np.median(ms)), "ms_min": float(ms.min()), "ms_max": float(ms.max()),
            "bytes": int(nbytes), "achieved_gbs": gbs, "hbm_peak_gbs": peak, "peak_source": src, "frac_of_peak": gbs / peak,
            "note": "one GPU, chunks automatic; the source is the buffer the initial rollout wrote (cur = 1), so no aliasing"}


def run(B, args, facts):
    T, S = args.horizon, args.steps
    x0, u0 = W.car_batch(B, T=T, seed=2)
    w = W.disturbance(B, S, 4, 0.01, seed=12)
    s = make_solver(B, T, args.max_iter, args.gpus)
    pinned = [torch.empty(shape, dtype=dt).pin_memory() for shape, dt in
              (((B, 4), torch.float64), ((B, T, 2), torch.float64), ((B, T + 1, 4), torch.float64), ((B, T, 2), torch.float64),
               ((B,), torch.float64), ((B,), torch.int32), ((B,), torch.int32))]
    pin = [t.numpy() for t in pinned]
    leg_fused(s, x0, u0, w, S)                           # warm-up: every kernel, the staging buffers, the log arrays
    t_a, t_b, identical = [], [], True
    for _ in range(args.reps):
        ta, la = leg_fused(s, x0, u0, w, S)
        tb, lb = leg_host(s, x0, u0, w, S, pin)
        t_a.append(ta)
        t_b.append(tb)
        identical = identical and all(np.array_equal(la[k], lb[k]) for k in LOG_KEYS)
    s.close()
    iters = int(la["iterations"].sum())
    a, b = ({"seconds": min(t), "seconds_all": t, "problem_steps_per_s": B * S / min(t), "iterations_per_s": iters / min(t)}
            for t in (t_a, t_b))
    del pin, pinned
    rec = {"metric": "closed-loop MPC problem-steps/s (car parking T=500)", "batch": B, "n_gpus": args.gpus, "steps": S,
           "horizon": T, "max_iter": args.max_iter, "disturbance_scale": 0.01, "reps": args.reps, "logs_bit_identical": identical,
           "iterations_total": iters, "fused_ilqgb_mpc": a, "host_loop_solve_host": b, "speedup": b["seconds"] / a["seconds"],
           "gpus": facts, "timing": "host clock around calls that end in a synchronise; best of --reps, legs alternated"}
    rec["shift"] = time_shift(B // args.gpus, T, args.max_iter, x0[: B // args.gpus], u0[: B // args.gpus], args.shift_calls)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--batch", default="65536,262144", help="comma-separated batch sizes")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--horizon", type=int, default=500)
    ap.add_argument("--max-iter", type=int, default=10)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--shift-calls", type=int, default=50)
    ap.add_argument("--out", help="append the JSON lines to this file")
    args = ap.parse_args()
    facts = gpu_facts(args.gpus)
    ok = True
    for B in (int(b) for b in args.batch.split(",")):
        rec = run(B, args, facts)
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")
        ok = ok and rec["logs_bit_identical"]
    if not ok:
        print("bench_mpc: the logs of ilqgb_mpc and of the host loop differ", file=sys.stderr)
        sys.exit(1)


if __name__ == "__main__":
    main()
