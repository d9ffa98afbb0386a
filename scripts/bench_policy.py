"""Feedback policy of a solved batch: what ilqgb_policy costs, and how fast ilqgb_policy_rollout rolls the policy out from M
perturbed initial states per problem.

Workload: car parking, T = 500, solved with max_iter 10 from workloads.car_batch; --batch sizes (default 65 536 and 262 144
problems) on one GPU, one chunk, so that a call is one launch and its kernel time is that launch's.  Samples:
workloads.perturbed_states(x*_0, M, 0.05) for M in --m (default 1, 4, 16, 64), no trajectories stored.  Recorded per batch size, with the card's name and power limit read in the same run:
  policy        host clock around ilqgb_policy + a synchronise (best of --reps), and the fraction of problems with policy_ok == 0;
  rollout[M]    ilqgb_policy_rollout of all M samples in one call: end-to-end seconds (host clock, pageable numpy arrays, copies
                included; best of --reps) and k_policy_rollout's kernel time (torch.profiler, in a profiled call of its own, after
                a profiled warm-up call whose record is dropped);
  separate[M]   the same samples as M calls with M = 1 (what sharing the nominal between a problem's samples buys), timed the same way;
                their results must be bit-identical to the single call's, else the script exits non-zero.
Throughput is problem * sample * steps per second of kernel time.  The HBM share puts the algorithmic bytes of the kernel -- the
nominal x|u, l and L records once per (problem, step), the samples' x0 in and cost / final state / ok out, the per-problem scalars --
over kernel time against the HBM bandwidth measured earlier on a B200 (profiles/bench_r02f_1gpu.json, 6550 GB/s).  One JSON line
per batch size goes to stdout (and, with --out FILE, is appended to FILE).

    python scripts/bench_policy.py [--batch 65536,262144] [--m 1,4,16,64] [--reps 2] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "ddp-generator_b200"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402  (torch.profiler: kernel time)

import bench_mpc as BM  # noqa: E402  (GPU facts, HBM peak, solver set-up)
from ilqg_b200 import workloads as W  # noqa: E402

KERNEL = "k_policy_rollout"


def best(f, reps):
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        f()
        ts.append(time.perf_counter() - t)
    return min(ts), ts


def kernel_seconds(f):
    """device time of every k_policy_rollout launch inside f(), summed"""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        f()
        torch.cuda.synchronize()
    tot, n = 0.0, 0
    for e in prof.key_averages():
        if KERNEL in e.key:
            us = getattr(e, "device_time_total", None)
            tot += float(us if us is not None else e.cuda_time_total)
            n += e.count
    return tot * 1e-6, n


def algorithmic_bytes(s, B, M, T):
    """bytes k_policy_rollout must move for B problems x M samples: each nominal record once per (problem, step), each sample's
    x0 in and cost, final state and ok out, per problem cur, policy_ok, w_pen_l, w_pen_f (car: no multipliers, shared parameters)"""
    nx, nu = s.nx, s.nu
    rxu, rlm, rls = (nx + nu + 3) // 4 * 4, (nu * nx + 3) // 4 * 4, (nu + 1) // 2 * 2
    return 8 * B * T * (rxu + rlm + rls) + B * M * (8 * nx + 8 + 8 * nx + 4) + B * (4 + 4 + 16)


def run(B, args, facts, peak):
    T = args.horizon
    x0, u0 = W.car_batch(B, T=T, seed=2)
    s = BM.make_solver(B, T, args.max_iter, 1, chunks=1)
    s.upload(x0, u0)
    s.run()
    s.sync()
    s.policy()
    s.sync()                                                     # warm-up
    t_pol, t_pol_all = best(lambda: (s.policy(), s.sync()), args.reps)
    pok = s.get_int("policy_ok")
    xs0 = s.get("x")[:, 0]
    rec = {"metric": "feedback-policy rollouts, problem*sample*steps/s of kernel time (car parking T=500)", "batch": B, "n_gpus": 1,
           "horizon": T, "max_iter": args.max_iter, "chunks": s.chunks(), "gpus": facts, "hbm_peak_bytes_per_s": peak[0] * 1e9,
           "hbm_peak_source": peak[1], "policy": {"seconds": t_pol, "seconds_all": t_pol_all,
                                                   "policy_ok_zero_fraction": float((pok == 0).mean()),
                                                   "result_counts": {str(k): int(v) for k, v in zip(*np.unique(s.download(False)["success"], return_counts=True))}},
           "rollout": {}, "consistent": True}
    for M in args.m:
        x0s = W.perturbed_states(xs0, M, 0.05, seed=5)
        one = s.policy_rollout(x0s)                                 # warm-up, and the results the separate calls must reproduce
        kernel_seconds(lambda: s.policy_rollout(x0s))               # the profiler's own warm-up
        t_one, t_one_all = best(lambda: s.policy_rollout(x0s), args.reps)
        k_one, n_one = kernel_seconds(lambda: s.policy_rollout(x0s))
        cols = [np.ascontiguousarray(x0s[:, i:i + 1]) for i in range(M)]
        sep = [s.policy_rollout(c) for c in cols]
        same = all(np.array_equal(np.concatenate([r[k] for r in sep], axis=1), one[k], equal_nan=True) for k in ("cost", "x_final", "ok"))
        t_sep, t_sep_all = best(lambda: [s.policy_rollout(c) for c in cols], args.reps)
        k_sep, n_sep = kernel_seconds(lambda: [s.policy_rollout(c) for c in cols])
        work = B * M * T
        byt = algorithmic_bytes(s, B, M, T)
        rec["rollout"][str(M)] = {
            "one_call": {"seconds_end_to_end": t_one, "seconds_all": t_one_all, "kernel_seconds": k_one, "kernel_launches": n_one,
                         "problem_sample_steps_per_s": work / k_one if k_one else None,
                         "algorithmic_bytes": byt, "hbm_share": byt / k_one / (peak[0] * 1e9) if k_one else None},
            "m_calls_of_one": {"seconds_end_to_end": t_sep, "seconds_all": t_sep_all, "kernel_seconds": k_sep, "kernel_launches": n_sep,
                               "problem_sample_steps_per_s": work / k_sep if k_sep else None,
                               "algorithmic_bytes": M * algorithmic_bytes(s, B, 1, T)},
            "kernel_speedup_of_sharing": k_sep / k_one if k_one else None,
            "ok_fraction": float(one["ok"].mean()), "bit_identical_to_m_calls": bool(same)}
        rec["consistent"] = rec["consistent"] and same
    s.close()
    rec["timing"] = ("host clock around calls that end in a synchronise (best of --reps); kernel time from torch.profiler in a "
                     "separate profiled call")
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", default="65536,262144", help="comma-separated batch sizes")
    ap.add_argument("--m", default="1,4,16,64", help="comma-separated samples per problem")
    ap.add_argument("--horizon", type=int, default=500)
    ap.add_argument("--max-iter", type=int, default=10)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", help="append the JSON lines to this file")
    args = ap.parse_args()
    args.m = [int(m) for m in args.m.split(",")]
    facts = BM.gpu_facts(1)
    peak = BM.hbm_peak()
    ok = True
    for B in (int(b) for b in args.batch.split(",")):
        rec = run(B, args, facts, peak)
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")
        ok = ok and rec["consistent"]
    if not ok:
        print("bench_policy: M calls of one sample differ from one call of M samples", file=sys.stderr)
        sys.exit(1)


if __name__ == "__main__":
    main()
