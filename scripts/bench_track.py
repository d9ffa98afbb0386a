"""Per-problem parameter tracks on the car-tracking problem (cartrack, T = 500, FULL_DDP = 0).

1. Cost of reading tracks: the same batch solved with the reference path as shared [k]-indexed parameters and as per-problem
   tracks that hold the same values in every row.  The results must be bit-identical; ilqgb_timing gives the derivative and
   line-search time per pass (CUDA events around every launch of a class, TIMING handle).
2. Closed loop: S = 20 steps of max_iter 10 with a moving window, ilqgb_mpc with tracks against the loop a caller writes without
   them (per step ilqgb_set_param_track with the window [b, s : s + T + 1] re-uploaded, then ilqgb_solve_host on pinned buffers,
   the shift and the disturbance in numpy).  The logs must be bit-identical.  Host clock around calls that end in a synchronise;
   after a warm-up loop the legs alternate --reps times and the best of each is kept.
One JSON line per batch size (default 65 536 and 262 144 problems, one GPU) goes to stdout and, with --out FILE, is appended to FILE.
The script exits non-zero if any comparison differs.

    python scripts/bench_track.py [--batch 65536,262144] [--reps 2] [--out FILE]
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

import torch  # noqa: E402  (pinned host memory)

import ilqg_b200  # noqa: E402
from ilqg_b200 import workloads as W  # noqa: E402

LOG_KEYS = ("x", "u", "cost", "iterations", "success")
OUT_KEYS = ("x", "u", "cost", "iterations", "success", "n_linesearch")


def gpu_facts():
    """Name and power limit of GPU 0, read in the same run (read-only query)."""
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, check=True)
    r = [f.strip() for f in q.stdout.strip().splitlines()[0].split(",")]
    return {"index": int(r[0]), "name": r[1], "power_limit_w": float(r[2])}


def make_solver(B, T, max_iter, params, flags=0):
    s = ilqg_b200.BatchSolver("cartrack", 0, B, T, flags=flags)
    s.set_options({"max_iter": max_iter})
    s.set_params(params)
    return s


def read_cost(B, T, steps, x0, u0, params):
    """shared [k]-indexed parameters against tracks with the same values; per-pass kernel time of each class"""
    same = {k: np.ascontiguousarray(np.broadcast_to(np.asarray(params[k])[None], (B, T + 1))) for k in ("xr", "yr")}
    legs = {}
    outs = {}
    for name in ("shared", "tracks", "shared", "tracks"):     # second round timed: modules loaded, buffers sized
        s = make_solver(B, T, steps, params, flags=ilqg_b200.TIMING)
        if name == "tracks":
            for k, v in same.items():
                s.set_param_track(k, v)
        s.upload(x0, u0)
        s.sync()
        s.timing(reset=True)
        t = time.perf_counter()
        s.run()
        s.sync()
        wall = time.perf_counter() - t
        tm = s.timing(reset=True)
        outs[name] = s.download()
        s.close()
        passes = max(tm["derivs"][1], 1)
        legs[name] = {"solve_s": wall, "passes": tm["derivs"][1],
                      "derivs_ms_per_pass": tm["derivs"][0] / passes, "linesearch_ms_per_pass": tm["linesearch"][0] / passes,
                      "backpass_ms_per_pass": tm["backpass"][0] / passes}
    identical = all(np.array_equal(outs["shared"][k], outs["tracks"][k]) for k in OUT_KEYS)
    return {"max_iter": steps, "shared": legs["shared"], "tracks": legs["tracks"], "results_bit_identical": identical,
            "extra_bytes_note": "per evaluated step a track read adds 2 x 8 B per problem (xr, yr) against the 208 B the car's "
                                "derivative kernel reads; not measured separately"}


def leg_fused(B, T, S, max_iter, params, tracks, x0, u0, w):
    s = make_solver(B, T, max_iter, params)
    for k, v in tracks.items():
        s.set_param_track(k, v)
    s.sync()
    t = time.perf_counter()
    logs = s.mpc(x0, u0, S, w)
    dt = time.perf_counter() - t
    assert s.track_offset() == S - 1
    s.close()
    return dt, logs


def leg_host(B, T, S, max_iter, params, tracks, x0, u0, w, pin):
    """Without device-side windows: re-upload the window of every track and solve end to end, every step."""
    xi, ui, xo, uo, co, it, re = pin
    s = make_solver(B, T, max_iter, params)
    logs = dict(x=np.empty((B, S + 1, 4)), u=np.empty((B, S, 2)), cost=np.empty((B, S)),
                iterations=np.empty((B, S), np.int32), success=np.empty((B, S), np.int32))
    ptr = lambda a: a.ctypes.data
    s.sync()
    t = time.perf_counter()
    xi[:] = x0
    ui[:] = u0
    for st in range(S):
        for k, v in tracks.items():
            s.set_param_track(k, v[:, st:st + T + 1])
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
    dt = time.perf_counter() - t
    s.close()
    return dt, logs


def run(B, args, facts):
    T, S = args.horizon, args.steps
    x0, u0, tracks = W.cartrack_batch(B, T=T, extra=S - 1, seed=4)
    params = dict(W.CARTRACK_PARAMS, xr=tracks["xr"][0, :T + 1], yr=tracks["yr"][0, :T + 1])
    rec = {"metric": "parameter tracks, cartrack T=500 FULL_DDP=0", "batch": B, "horizon": T, "gpu": facts}
    rec["read_cost"] = read_cost(B, T, args.passes, x0, u0, params)
    w = W.disturbance(B, S, 4, 0.01, seed=12)
    pinned = [torch.empty(shape, dtype=dt).pin_memory() for shape, dt in
              (((B, 4), torch.float64), ((B, T, 2), torch.float64), ((B, T + 1, 4), torch.float64), ((B, T, 2), torch.float64),
               ((B,), torch.float64), ((B,), torch.int32), ((B,), torch.int32))]
    pin = [t.numpy() for t in pinned]
    leg_fused(B, T, S, args.max_iter, params, tracks, x0, u0, w)          # warm-up
    ta, tb, identical = [], [], True
    for _ in range(args.reps):
        a, la = leg_fused(B, T, S, args.max_iter, params, tracks, x0, u0, w)
        b, lb = leg_host(B, T, S, args.max_iter, params, tracks, x0, u0, w, pin)
        ta.append(a)
        tb.append(b)
        identical = identical and all(np.array_equal(la[k], lb[k]) for k in LOG_KEYS)
    del pin, pinned
    fa, fb = ({"seconds": min(t), "seconds_all": t, "problem_steps_per_s": B * S / min(t)} for t in (ta, tb))
    rec["closed_loop"] = {"steps": S, "max_iter": args.max_iter, "disturbance_scale": 0.01, "reps": args.reps,
                          "fused_ilqgb_mpc_tracks": fa, "host_loop_set_param_track_solve_host": fb, "speedup": fb["seconds"] / fa["seconds"],
                          "logs_bit_identical": identical, "iterations_total": int(la["iterations"].sum()),
                          "timing": "host clock around calls that end in a synchronise; best of --reps, legs alternated"}
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", default="65536,262144", help="comma-separated batch sizes")
    ap.add_argument("--horizon", type=int, default=500)
    ap.add_argument("--passes", type=int, default=20, help="max_iter of the read-cost solves")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--max-iter", type=int, default=10)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", help="append the JSON lines to this file")
    args = ap.parse_args()
    facts = gpu_facts()
    ok = True
    for B in (int(b) for b in args.batch.split(",")):
        rec = run(B, args, facts)
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")
        ok = ok and rec["read_cost"]["results_bit_identical"] and rec["closed_loop"]["logs_bit_identical"]
    if not ok:
        print("bench_track: results with tracks differ from the comparison leg", file=sys.stderr)
        sys.exit(1)


if __name__ == "__main__":
    main()
