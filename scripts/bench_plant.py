"""Closed loops against sampled plants: what a plant costs ilqgb_mpc, and what it saves against the host loop a MATLAB user
writes for a Monte-Carlo robustness study (solve, then the plant stepped with iLQG<Name>MMex modes 16 and 0).

Workload: car parking, T = 500, max_iter 10 per step, S = 20 steps, w = workloads.disturbance(scale 0.01), --batch sizes (default
65 536 and 262 144 problems) on one GPU.  ilqgb_mpc runs in four forms, alternated --reps times after one warm-up loop each, timed
by the host clock around calls that end in a synchronise (best of --reps):
  none      no plant (k_mpc_advance);
  identity  a plant equal to the model, n_sub 1: its logs must be bit-identical to `none`;
  sampled   per-problem plants workloads.car_plant(spread 0.1), n_sub 1;
  sampled10 the same plants with n_sub 10 and h = 0.003 (the model's h / 10).
The host loop is ilqgb_solve_host on pinned buffers, then ilqgb_eval mode 16 and mode 0 on a second handle that holds the sampled
plants; its logs must be bit-identical to `sampled`.  k_mpc_plant alone is timed against k_mpc_advance with CUDA events around
each of --shift-calls ilqgb_shift(1) calls (a start between two calls, outside the events).  The script exits non-zero when a
pair of logs that must agree does not.  One JSON line per batch size goes to stdout (and, with --out FILE, is appended to FILE).

    python scripts/bench_plant.py [--batch 65536,262144] [--reps 2] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "ddp-generator_b200"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402  (pinned host memory and CUDA events)

import bench_mpc as BM  # noqa: E402  (GPU facts, solver set-up, the fused leg)
from ilqg_b200 import workloads as W  # noqa: E402

LOG_KEYS = BM.LOG_KEYS
FORMS = ("none", "identity", "sampled", "sampled10")


def attach(s, form, plants):
    s.clear_plant()
    if form == "identity":
        s.set_plant_substeps(1)
    elif form == "sampled":
        s.set_plant_substeps(1)
        s.set_plant_params_batch(plants)
    elif form == "sampled10":
        s.set_plant_substeps(10)
        s.set_plant_params({"h": [0.003]})
        s.set_plant_params_batch(plants)


def eval_into(s, mode, x, u, out):
    s._chk(s.lib.ilqgb_eval(s.h, mode, 0, x.ctypes.data, u.ctypes.data, out.ctypes.data))


def leg_host(s, plant, x0, u0, w, S, pin):
    """The MATLAB loop: one end-to-end solve per step from pinned buffers; the plant's clamp (mode 16) and dynamics (mode 0) on the
    plant handle; the next input shifted on the host."""
    xi, ui, xo, uo, co, it, re, ua = pin
    B = x0.shape[0]
    logs = dict(x=np.empty((B, S + 1, x0.shape[1])), u=np.empty((B, S, ui.shape[2])), cost=np.empty((B, S)),
                iterations=np.empty((B, S), np.int32), success=np.empty((B, S), np.int32))
    ptr = lambda a: a.ctypes.data
    u_app, xn = np.empty((B, ui.shape[2])), np.empty((B, x0.shape[1]))
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
        u_app[:] = uo[:, 0]
        eval_into(plant, 16, xi, u_app, ua)
        eval_into(plant, 0, xi, ua, xn)
        np.add(xn, w[:, st], out=xi)
        ui[:, :-1] = uo[:, 1:]
        ui[:, -1] = uo[:, -1]
    logs["x"][:, S] = xi
    return time.perf_counter() - t, logs


def time_advance(B, T, max_iter, x0, u0, plants, calls):
    """ilqgb_shift(1) alone, as k_mpc_advance (no plant) and as k_mpc_plant (sampled plants, n_sub 1 and 10), CUDA events around
    each call on the handle's stream"""
    st = torch.cuda.Stream()
    s = BM.make_solver(B, T, max_iter, 1, stream=st.cuda_stream)
    s.upload(x0, u0)
    s.start()
    out = {}
    for form in ("none", "sampled", "sampled10"):
        attach(s, form, plants)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(calls + 3)]
        for a, b in ev:
            a.record(st)
            s.shift(1)
            b.record(st)
            s.start()
        st.synchronize()
        ms = np.array([a.elapsed_time(b) for a, b in ev[3:]])
        out[{"none": "k_mpc_advance", "sampled": "k_mpc_plant_nsub1", "sampled10": "k_mpc_plant_nsub10"}[form]] = {
            "ms_median": float(np.median(ms)), "ms_min": float(ms.min()), "ms_max": float(ms.max())}
    npf = s.get("plant").shape[1]
    s.close()
    # bytes k_mpc_plant moves per problem beyond k_mpc_advance's: the plant's parameter column (npf doubles) and x0 (nx doubles)
    # read; it reads u[0] where k_mpc_advance reads x[1], one sector each
    out["extra_bytes_per_problem"] = 8 * (npf + 4)
    out["calls"] = calls
    out["note"] = "one GPU, chunks automatic; the source is the buffer the initial rollout wrote (cur = 1), so no aliasing"
    return out


def run(B, args, facts):
    T, S = args.horizon, args.steps
    x0, u0 = W.car_batch(B, T=T, seed=2)
    w = W.disturbance(B, S, 4, 0.01, seed=12)
    plants = W.car_plant(B, 0.1, seed=13)
    s = BM.make_solver(B, T, args.max_iter, 1)
    plant = BM.make_solver(B, T, args.max_iter, 1)
    plant.set_params_batch(plants)
    plant.lib.ilqgb_eval.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    pinned = [torch.empty(shape, dtype=dt).pin_memory() for shape, dt in
              (((B, 4), torch.float64), ((B, T, 2), torch.float64), ((B, T + 1, 4), torch.float64), ((B, T, 2), torch.float64),
               ((B,), torch.float64), ((B,), torch.int32), ((B,), torch.int32), ((B, 2), torch.float64))]
    pin = [t.numpy() for t in pinned]
    for form in FORMS:                                    # warm-up: every kernel, the staging buffers, the plant tables
        attach(s, form, plants)
        BM.leg_fused(s, x0, u0, w, S)
    times = {f: [] for f in FORMS + ("host",)}
    logs = {}
    for _ in range(args.reps):
        for form in FORMS:
            attach(s, form, plants)
            t, logs[form] = BM.leg_fused(s, x0, u0, w, S)
            times[form].append(t)
        t, logs["host"] = leg_host(s, plant, x0, u0, w, S, pin)
        times["host"].append(t)
    s.close()
    plant.close()
    same = lambda a, b, keep=slice(None): all(np.array_equal(logs[a][k][keep], logs[b][k][keep], equal_nan=True) for k in LOG_KEYS)
    # a problem whose initial rollout failed goes on from its nominal x[1] without a plant, from the plant step with one
    ok = np.all(logs["none"]["success"] != -1, axis=1)
    legs = {f: {"seconds": min(t), "seconds_all": t, "problem_steps_per_s": B * S / min(t),
                "iterations_per_s": int(logs[f]["iterations"].sum()) / min(t)} for f, t in times.items()}
    base = legs["none"]["seconds"]
    for f in FORMS[1:]:
        legs[f]["overhead_vs_none"] = legs[f]["seconds"] / base - 1.0
    del pin, pinned
    rec = {"metric": "closed-loop MPC against sampled plants, problem-steps/s (car parking T=500)", "batch": B, "n_gpus": 1, "steps": S,
           "horizon": T, "max_iter": args.max_iter, "disturbance_scale": 0.01, "plant_spread": 0.1, "reps": args.reps,
           "identity_logs_bit_identical": same("none", "identity", ok), "identity_problems_excluded": int((~ok).sum()),
           "host_logs_bit_identical": same("sampled", "host"),
           "sampled_differs_from_none": not same("none", "sampled"), "fused": {f: legs[f] for f in FORMS},
           "host_loop_solve_host_eval": legs["host"], "speedup_vs_host": legs["host"]["seconds"] / legs["sampled"]["seconds"],
           "gpus": facts, "timing": "host clock around calls that end in a synchronise; best of --reps, forms alternated"}
    rec["advance"] = time_advance(B, T, args.max_iter, x0, u0, plants, args.shift_calls)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", default="65536,262144", help="comma-separated batch sizes")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--horizon", type=int, default=500)
    ap.add_argument("--max-iter", type=int, default=10)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--shift-calls", type=int, default=50)
    ap.add_argument("--out", help="append the JSON lines to this file")
    args = ap.parse_args()
    facts = BM.gpu_facts(1)
    ok = True
    for B in (int(b) for b in args.batch.split(",")):
        rec = run(B, args, facts)
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")
        ok = ok and rec["identity_logs_bit_identical"] and rec["host_logs_bit_identical"] and rec["sampled_differs_from_none"]
    if not ok:
        print("bench_plant: logs that must agree differ (or the sampled plants changed nothing)", file=sys.stderr)
        sys.exit(1)


if __name__ == "__main__":
    main()
