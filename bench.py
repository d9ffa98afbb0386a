#!/usr/bin/env python
"""bench.py -- batched iLQG iterations/sec on the car-parking problem (T=500), BASELINE.json's metric.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE config 4 -- B = 262144 car-parking problems (n=4, m=2, T=500, FULL_DDP=0) with
random initial states and controls (SURVEY.md 8d), strong-scaled: the B problems are split evenly over the N ranks,
one process per GPU, no collective on the solve path (torch.distributed is used for the timing barrier and the
final reduction of counters only).
A "step" is one pass of the iLQG loop (derivative kernel, backward-pass kernel, line-search kernel) over the rank's
whole shard; K steps = a solve with max_iter = K, which makes K passes unless every problem of the shard has stopped before
(`passes` in the JSON line is the number made; fewer than K is also reported on stderr).  W warm-up steps run first on the
same inputs (a throw-away solve with max_iter = W).  `value` = (line searches performed by all problems on all ranks) / (max over ranks of
the device time of the K timed steps incl. the initial rollout), inputs resident in HBM.  `e2e` = the same count
over the time of ONE call of the public C ABI's end-to-end entry (ilqgb_solve_host): upload (pinned host -> HBM) + solve +
download of x, u, cost, iterations (HBM -> pinned host), pipelined per chunk stream.  The iteration count follows SURVEY.md 8d: loop passes that reached line_search.

Both timed legs directly follow a warm-up solve of W passes through the same entry point (stated in config.timing), so both
start with the clocks up and the staging buffers of the end-to-end path allocated.  (An idle gap in front of a leg was tried
and dropped: the clocks of an idle B200 take long enough to come back up that a 0.12 s leg -- the 8-GPU share -- lost 10 %.)

`extra` (N = 1 only) holds the other BASELINE configs with the same fields in short form: config 3 (car, B = 4096), config 5
(synthetic quadrotor n = 12, m = 4, T = 1000, FULL_DDP = 1, B = 16384; fp64-issue roofline of k_backpass_warp) and config 4 at
the surveyed max_iter = 50.  Each carries a bit-exactness flag against the CPU reference on a sample; any false flag makes
the process exit non-zero after the JSON line is printed.

`--gpus N` without torchrun (WORLD_SIZE unset) drives N GPUs from this one process through ilqgb_create_multi.

`--dump-outputs DIR` writes what the end-to-end leg's call returned after its last timed step (the same results as the
resident leg: the run checks the costs of both bit for bit), as float64 .npy files in DIR:
cost.npy, iterations.npy, result.npy, n_linesearch.npy of every problem (a seeded sample of 2^19 problems above that batch) with
their problem numbers in problem_index.npy, and the trajectories x.npy [n][T+1][4] and u.npy [n][T][2] of a seeded sample of 1024
problems (traj_index.npy); under 64 MB at any batch.  The inputs are a fixed function of the problem number, so two builds run with
the same arguments can be compared output for output.

`--impl reference` times the reference's own C solver (oracle/_ref, the unmodified sources compiled -O3
-ffp-contract=off; falls back to the oracle port if that library is not present) on all host cores, one solver
instance per thread, on a bounded sample of the same batch.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "ddp-generator_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "batched iLQG iterations/sec (car-parking T=500)"
UNIT = "iterations/s"
T_HOR = 500
PROBLEM, FULL_DDP = "car", 0


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        if os.environ.get("BENCH_NO_SAMPLER"):      # development aid: measure the poller's own influence
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """index of the next sample: brackets a timed region while the poller keeps running (starting nvidia-smi right in front
        of a 0.1 s region perturbs it: measured 0.131 s against 0.116 s at 32768 problems)"""
        return len(self.lines)

    def summary(self, i0=0, i1=None):
        """samples taken inside [i0, i1), widened by one sample on each side when the region was shorter than the polling interval"""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        i1 = len(self.lines) if i1 is None else i1
        lines = self.lines[max(i0 - 1, 0):i1 + 1]
        return self._digest(lines)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        return self._digest(self.lines)

    def _digest(self, lines):
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                pw.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "sm_mhz_min": float(min(sm)) if sm else None, "power_w_max": float(max(pw)) if pw else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
def make_inputs(first, count, pinned):
    """Counter-based synthetic inputs for problems first..first+count-1, written into (pinned) host arrays."""
    from ilqg_b200 import workloads as W

    x0, u0 = pinned
    CH = 16384
    for s in range(0, count, CH):
        n = min(CH, count - s)
        a, b = W.car_batch(n, T=T_HOR, first=first + s)
        x0[s:s + n] = a
        u0[s:s + n] = b


DUMP_PROBLEMS, DUMP_TRAJECTORIES = 1 << 19, 1024


def dump_outputs(path, x, u, cost, iterations, result, n_linesearch):
    """The arrays a caller of the timed solve receives, as float64 .npy files; samples are seeded and depend on the batch only."""
    os.makedirs(path, exist_ok=True)
    B = cost.shape[0]

    def sample(n):
        return np.arange(B) if B <= n else np.sort(np.random.default_rng(0).choice(B, size=n, replace=False))

    pi, ti = sample(DUMP_PROBLEMS), sample(DUMP_TRAJECTORIES)
    arrays = {"problem_index": pi, "cost": cost[pi], "iterations": iterations[pi], "result": result[pi], "n_linesearch": n_linesearch[pi],
              "traj_index": ti, "x": x[ti], "u": u[ti]}
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), np.asarray(a, dtype=np.float64))


def cpu_reference_run(n_problems, max_iter, threads, first=0, problem=PROBLEM, ddp=FULL_DDP, inputs=None, params=None):
    """Solve problems first..first+n-1 with the reference's C solver (or the port) on `threads` host threads."""
    import oracle_lib
    from ilqg_b200 import workloads as W

    kind = "reference" if oracle_lib.available("reference", problem, ddp, fast=True) else "port"
    if not oracle_lib.available(kind, problem, ddp, fast=True):
        return None
    O = oracle_lib.OracleLib(kind, problem, ddp, fast=True)
    x0, u0 = inputs if inputs is not None else W.car_batch(n_problems, T=T_HOR, first=first)
    params = params if params is not None else W.CAR_PARAMS
    t0 = time.perf_counter()
    out = O.solve_batch(x0, u0, params, {"max_iter": float(max_iter)}, threads)
    dt = time.perf_counter() - t0
    its = int(out["n_linesearch"].sum())
    return dict(kind=kind, seconds=dt, iterations=its, value=its / dt, cores=threads, n_problems=n_problems, out=out)


def cpu_single_instance():
    """BASELINE config 1 on the host: one car instance (T=500, max_iter=200) with the reference's single-threaded build
    and with its experimental -DMULTI_THREADED=1 pipeline (north star: both are reported, neither is the target)."""
    import oracle_lib
    from ilqg_b200 import workloads as W

    out = {}
    x0, u0 = W.car_single()
    for key, kind, fast in (("single_thread", "reference", True), ("multi_threaded_2", "reference-mt", False)):
        if not oracle_lib.available(kind, PROBLEM, FULL_DDP, fast):
            continue
        s = oracle_lib.OracleLib(kind, PROBLEM, FULL_DDP, fast).solver(T_HOR)
        s.set_opts({"max_iter": 200})
        s.set_params(W.CAR_PARAMS)
        best = None
        for _ in range(3):
            s.init(x0, u0)
            t0 = time.perf_counter()
            s.solve()
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        n = s.scalar("n_linesearch")
        out[key] = {"iterations_per_s": n / best, "ms_per_iteration": 1e3 * best / n, "iterations": int(n), "final_cost": s.scalar("cost")}
        s.close()
    return out


def run_reference_arm(args, rank):
    if rank != 0:
        return
    cores = host_cores()
    per_core = max(2, int(1250 * 25 / max(args.steps, 1)))       # ~25 s at ~1250 it/s/core
    n = min(args.batch, per_core * cores)
    cpu_reference_run(min(n, 2 * cores), max(args.warmup, 1), cores)          # warm-up
    r = cpu_reference_run(n, args.steps, cores)
    if r is None:
        print(json.dumps({"impl": "reference", "unavailable": "neither oracle/_ref nor the oracle port is built"}))
        return
    sample = f"first {n} problems of the batch, max_iter={args.steps}, one solver instance per thread"
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * r["seconds"] / max(args.steps, 1), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": cores, "kind": r["kind"], "sample": sample},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(args):
    return {"workload": f"car-parking n=4 m=2 T={T_HOR} FULL_DDP=0, batch {args.batch} random initial states "
                        f"(BASELINE config 4), max_iter={args.steps}, default options",
            "batch": args.batch, "horizon": T_HOR, "max_iter": args.steps, "sharding": "contiguous blocks of batch/N problems per GPU",
            "l2": "working set (>=160 KB per problem, tens of GB per GPU) is far larger than the 126 MB L2",
            "timing": "each timed leg (resident, end to end) directly follows a warm-up solve of W passes through the same entry point; "
                      f"the kernels-alone leg starts after {IDLE_S} s of idle like the burst measurement of the HBM peak it is compared with"}


IDLE_S = 1.5


def algorithmic_bytes(nx, nu, nv, T):
    """Bytes per problem and unit of work, two conventions.  `alg` = SURVEY.md 8(d): only the doubles the algorithm needs (car:
    derivative sweep 192 B/step, back pass 240 B/step, stored rollout 176 B/step, parallel-alpha tail 128 B/step).  `rec` = what
    the kernels address: x|u and L records rounded up to 32-byte sectors, l to 16 bytes (car: 208 / 240 / 208 / 144 B per step)."""
    nq = nx * (nx + 1) // 2
    rxu, rll = 8 * ((nx + nu + 3) // 4) * 4, 8 * ((nu * nx + 3) // 4) * 4 + 8 * ((nu + 1) // 2) * 2     # x|u record; L record + l record
    xu, ll = 8 * (nx + nu), 8 * (nu + nu * nx)
    fin = 8 * (nx + nq)
    return {
        "alg": {"derivs": T * (xu + 8 * nv) + (8 * nx + fin), "backpass": T * (8 * nv + 8 * nu + ll) + fin,
                "rollout": T * (xu + ll + xu) + 8 * nx, "tail": T * (xu + ll)},
        "rec": {"derivs": T * (rxu + 8 * nv) + (rxu + fin), "backpass": T * (8 * nv + 8 * nu + rll) + fin,
                "rollout": T * (rxu + rll + rxu) + rxu, "tail": T * (rxu + rll)},
    }


def fp64_peak():
    for name in ("fp64_peak_r02.json", "fp64_peak_r01.json"):
        fp = os.path.join(ROOT, "profiles", name)
        if os.path.exists(fp):
            return json.load(open(fp))["dmul_dadd_instr_per_s"], f"profiles/{name} (csrc/fp64_peak.cu on B200: DMUL+DADD, no FMA)"
    return 1.847e13, "csrc/fp64_peak.cu on B200 (DMUL+DADD, no FMA)"


def kernels_alone(problem, ddp, n_k, T, params, x0_ptr, u0_ptr, steps, device, stream, nx, nu):
    """Roofline leg: the kernels of a solve timed ALONE (one stream, CUDA events around every launch, recorded by the library on
    the launching stream) on n_k problems, after an idle; work units are counted by the kernels themselves."""
    import ilqg_b200

    K = ilqg_b200.BatchSolver(problem, ddp, n_k, T, device=device, flags=ilqg_b200.TIMING, stream=stream, chunks=1)
    K.set_params(params)
    K.set_options({"max_iter": steps})
    K.upload_ptr(x0_ptr, u0_ptr)
    K.sync()
    ksampler = ClockSampler(device)
    ksampler.start()
    time.sleep(IDLE_S)
    i0 = ksampler.mark()
    K.run()
    K.sync()
    kclocks = ksampler.summary(i0, ksampler.mark())
    ksampler.stop()
    ktime = K.timing(reset=True)
    cnt = {k: int(K.get_int(f).sum()) for k, f in (("derivs", "n_derivs"), ("backpass", "n_backpass"), ("rollout", "n_rollouts"), ("tail", "n_tails"))}
    nv = K.L.deriv_doubles_per_step
    K.close()
    per = algorithmic_bytes(nx, nu, nv, T)
    tot = {c: {"derivs": cnt["derivs"] * per[c]["derivs"], "backpass": cnt["backpass"] * per[c]["backpass"],
               "linesearch": cnt["rollout"] * per[c]["rollout"] + cnt["tail"] * per[c]["tail"]} for c in ("alg", "rec")}
    kernels = {}
    all_ms = max(sum(v[0] for v in ktime.values()), 1e-9)
    for k in ("derivs", "backpass", "linesearch"):
        ms, n = ktime[k]
        if n and ms > 0:
            kernels[k] = {"ms_total": ms, "launches": n, "ms_per_launch": ms / n, "algorithmic_bytes": tot["alg"][k],
                          "record_bytes": tot["rec"][k], "achieved_gbs": tot["alg"][k] / (ms * 1e-3) / 1e9,
                          "achieved_gbs_record_bytes": tot["rec"][k] / (ms * 1e-3) / 1e9, "share_of_step": ms / all_ms}
    if "backpass" in kernels:
        # fp64-issue bound: algorithmic multiply+add count per (problem, step) from SURVEY.md 8d (dense formula, regType 1, no
        # clamp; + the FULL_DDP tensor terms) against the DMUL+DADD instruction rate measured on a B200 (FMA is off-limits)
        n_, m_ = nx, nu
        pairs = 2 * n_**3 + 5 * n_**2 * m_ + 3 * n_ * m_**2 + n_**2 + 4 * n_ * m_ + 2 * m_**2 + m_
        if ddp:
            pairs += n_**2 * m_ + n_ * (m_ * (m_ + 1) // 2) + n_ * (n_ * (n_ + 1) // 2)
        peak64, src = fp64_peak()
        dp = 2.0 * pairs * cnt["backpass"] * T / (kernels["backpass"]["ms_total"] * 1e-3)
        kernels["backpass"]["fp64"] = {"algorithmic_dp_instr_per_step": 2 * pairs, "achieved_dp_instr_per_s": dp,
                                       "peak_dp_instr_per_s": peak64, "frac": dp / peak64, "peak_source": src}
    return kernels, kclocks, cnt


def roofline_of(kernels, dom, n_k, kclocks, names):
    peak, peak_src = measured_peak_hbm()
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get(dom, {}).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    k = kernels[dom]
    return {"kernel": names[dom], "bound": "hbm", "achieved": k["achieved_gbs"], "peak": peak, "peak_source": peak_src, "unit": "GB/s",
            "frac": k["achieved_gbs"] / peak, "frac_record_bytes": k["achieved_gbs_record_bytes"] / peak, "traffic": traffic,
            "algorithmic_bytes_per_launch": k["algorithmic_bytes"] / k["launches"], "record_bytes_per_launch": k["record_bytes"] / k["launches"],
            "timed_on": f"{n_k} problems (one chunk of the timed run), kernels alone on one stream, after {IDLE_S} s idle",
            "clocks": kclocks,
            "note": "achieved/frac: SURVEY.md 8(d) algorithmic bytes (car: 176 B per stored rollout step, 128 B per tail step, 240 B per "
                    "back-pass step, 192 B per derivative step) x units counted by the kernels; *_record_bytes: the sector-padded records the "
                    "kernels address; traffic: ncu dram bytes per launch of this kernel class at the same launch size (profiles/traffic.json)"}


def short_config(tag, problem, ddp, B, T, params, inputs, max_iter, sample_n, device, nx, nu, workload):
    """One of the other BASELINE configs: resident value, end-to-end value, roofline of its dominant kernel class and a
    bit-exactness check of a sample against the CPU reference (checker only).  One GPU."""
    import torch

    import ilqg_b200

    x0, u0 = inputs
    x0_t = torch.from_numpy(np.ascontiguousarray(x0)).pin_memory()
    u0_t = torch.from_numpy(np.ascontiguousarray(u0)).pin_memory()
    xo = torch.empty((B, T + 1, nx), dtype=torch.float64).pin_memory()
    uo = torch.empty((B, T, nu), dtype=torch.float64).pin_memory()
    co = torch.empty(B, dtype=torch.float64).pin_memory()
    io, ro, no = (torch.empty(B, dtype=torch.int32).pin_memory() for _ in range(3))
    stream = torch.cuda.current_stream().cuda_stream
    S = ilqg_b200.BatchSolver(problem, ddp, B, T, device=device, stream=stream)
    S.set_params(params)
    S.set_options({"max_iter": 3})
    S.solve_host_ptr(x0_t.data_ptr(), u0_t.data_ptr(), xo.data_ptr(), uo.data_ptr(), co.data_ptr(), io.data_ptr(), ro.data_ptr(), no.data_ptr())
    S.set_options({"max_iter": max_iter})
    S.upload_ptr(x0_t.data_ptr(), u0_t.data_ptr())
    S.set_options({"max_iter": 3})
    S.run()
    S.set_options({"max_iter": max_iter})
    S.upload_ptr(x0_t.data_ptr(), u0_t.data_ptr())
    l0 = S.launch_count()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall = time.perf_counter()
    e0.record()
    S.run()
    e1.record()
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall
    ms = e0.elapsed_time(e1)
    assert stream != 0 and 0.8 * t_wall * 1e3 <= ms <= 1.02 * t_wall * 1e3, (ms, t_wall)
    launches = S.launch_count() - l0
    S.download_ptr(None, None, co.data_ptr(), io.data_ptr(), ro.data_ptr(), no.data_ptr())
    n_ls = int(no.numpy().sum())
    cost_res = co.numpy().copy()
    S.set_options({"max_iter": 3})
    S.solve_host_ptr(x0_t.data_ptr(), u0_t.data_ptr(), xo.data_ptr(), uo.data_ptr(), co.data_ptr(), io.data_ptr(), ro.data_ptr(), no.data_ptr())
    S.set_options({"max_iter": max_iter})
    t0 = time.perf_counter()
    S.solve_host_ptr(x0_t.data_ptr(), u0_t.data_ptr(), xo.data_ptr(), uo.data_ptr(), co.data_ptr(), io.data_ptr(), ro.data_ptr(), no.data_ptr())
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    n_ls_e2e = int(no.numpy().sum())
    same_e2e = bool(np.array_equal(cost_res, co.numpy()))
    chunks = S.chunks()
    split = int(S.get_int("bp_split")[0])   # lanes per problem the backward pass ran with (4: k_backpass_split, small batches)
    S.close()
    n_k = max(1, B // chunks)
    kernels, kclocks, _ = kernels_alone(problem, ddp, n_k, T, params, x0_t.data_ptr(), u0_t.data_ptr(), max_iter, device, stream, nx, nu)
    dom = max(kernels, key=lambda k: kernels[k]["ms_total"])
    names = {"derivs": "k_derivs", "backpass": "k_backpass_warp" if nx > 6 else ("k_backpass_split" if split else "k_backpass"), "linesearch": "k_ls_round"}
    roof = roofline_of(kernels, dom, n_k, kclocks, names)
    if dom == "backpass":       # fp64-issue bound kernel: report it against the fp64 instruction peak, keep the HBM figure beside it
        f = kernels["backpass"]["fp64"]
        roof = {"kernel": names[dom], "bound": "fp64-issue", "achieved": f["achieved_dp_instr_per_s"] / 1e12, "peak": f["peak_dp_instr_per_s"] / 1e12,
                "unit": "T dp-instr/s (DMUL+DADD)", "frac": f["frac"], "peak_source": f["peak_source"], "hbm": roof}
    cores = host_cores()
    r = cpu_reference_run(sample_n, max_iter, cores, problem=problem, ddp=ddp, inputs=(x0[:sample_n], u0[:sample_n]), params=params)
    parity = bool(np.array_equal(r["out"]["cost"], cost_res[:sample_n])) if r else None
    return {"config": tag, "workload": workload, "value": n_ls / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / max(max_iter, 1), "steps": max_iter,
            "e2e": {"value": n_ls_e2e / t_e2e, "unit": UNIT, "seconds": t_e2e, "h2d_bytes": (x0_t.numel() + u0_t.numel()) * 8,
                    "d2h_bytes": (xo.numel() + uo.numel() + co.numel()) * 8 + 12 * B, "equals_resident": same_e2e},
            "gpu_launches": launches, "streams_per_gpu": chunks, "roofline": roof,
            "kernels": {k: {kk: vv for kk, vv in v.items() if kk in ("ms_per_launch", "launches", "share_of_step", "achieved_gbs", "fp64")} for k, v in kernels.items()},
            "cpu_reference": {"value": r["value"], "cores": cores, "kind": r["kind"], "sample": f"first {sample_n} problems, max_iter={max_iter}"} if r else None,
            "gpu_costs_bit_identical_on_sample": parity}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=262144)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the other BASELINE configs (config 3, config 5, config 4 at max_iter=50)")
    ap.add_argument("--chunks", type=int, default=0, help="concurrent streams per GPU (0 = automatic)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed solve returned as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist

    import ilqg_b200

    if args.dump_outputs and world > 1:
        raise SystemExit("bench.py: --dump-outputs needs the whole batch in one process (--gpus N without torchrun drives N GPUs)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a CUDA device: the solver has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    # one process driving several GPUs (not under torchrun): the C ABI's multi-device handle shards the batch itself
    multi = args.gpus if (world == 1 and args.gpus > 1) else 0
    n_gpus = multi or world

    def barrier():
        if world > 1:
            dist.barrier()
        if multi:
            for d in range(multi):
                torch.cuda.synchronize(d)
        else:
            torch.cuda.synchronize()

    def reduce(v, op):
        if world == 1:
            return v
        t = torch.tensor([float(v)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    # ---- shard and inputs (pinned host memory) ---------------------------------------------------------------------
    from ilqg_b200.sharding import shard_range

    first, count = shard_range(args.batch, rank, world)
    nx, nu = 4, 2
    x0_t = torch.empty((count, nx), dtype=torch.float64).pin_memory()
    u0_t = torch.empty((count, T_HOR, nu), dtype=torch.float64).pin_memory()
    make_inputs(first, count, (x0_t.numpy(), u0_t.numpy()))
    x_out = torch.empty((count, T_HOR + 1, nx), dtype=torch.float64).pin_memory()
    u_out = torch.empty((count, T_HOR, nu), dtype=torch.float64).pin_memory()
    cost_out = torch.empty(count, dtype=torch.float64).pin_memory()
    it_out = torch.empty(count, dtype=torch.int32).pin_memory()
    res_out = torch.empty(count, dtype=torch.int32).pin_memory()
    nls_out = torch.empty(count, dtype=torch.int32).pin_memory()
    host_ptrs = (x0_t.data_ptr(), u0_t.data_ptr(), x_out.data_ptr(), u_out.data_ptr(), cost_out.data_ptr(), it_out.data_ptr(),
                 res_out.data_ptr(), nls_out.data_ptr())

    from ilqg_b200 import workloads as W

    # The library's streams are non-blocking: they do NOT order with the legacy default stream, so events recorded there would
    # not bracket the solve (round 1 did that and under-measured the timed region: its event fired when the last passes were
    # ISSUED).  Everything here runs on one explicit stream that the handle adopts as its main stream (fork / join point).
    torch.cuda.set_stream(torch.cuda.Stream(device=dev))
    stream = torch.cuda.current_stream().cuda_stream
    assert stream != 0
    S = ilqg_b200.BatchSolver(PROBLEM, FULL_DDP, count, T_HOR, device=local_rank, flags=0, stream=stream, chunks=args.chunks,
                              devices=multi or None)
    S.set_params(W.CAR_PARAMS)

    # ---- warm-up: W passes on the same inputs, through both entry points ------------------------------------------------------
    sampler = ClockSampler(local_rank)      # polls from here on; the timed regions are bracketed by sample indices
    sampler.start()
    S.set_options({"max_iter": args.warmup})
    S.solve_host_ptr(*host_ptrs)          # also allocates the staging buffers of the end-to-end path
    S.upload_ptr(x0_t.data_ptr(), u0_t.data_ptr())
    S.run()
    S.sync()

    # ---- timed region 1: inputs resident, K passes ---------------------------------------------------------------------------
    S.set_options({"max_iter": args.steps})
    S.upload_ptr(x0_t.data_ptr(), u0_t.data_ptr())
    S.sync()
    launches0 = S.launch_count()
    barrier()
    i0 = sampler.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall = time.perf_counter()
    e0.record()
    S.run()
    e1.record()
    S.sync()                                  # this rank's own work (all its devices) ...
    t_wall = time.perf_counter() - t_wall
    barrier()                                 # ... then everybody's
    clocks = sampler.summary(i0, sampler.mark())
    ms_dev = e0.elapsed_time(e1)
    if not (0.8 * t_wall * 1e3 <= ms_dev <= 1.02 * t_wall * 1e3):   # the events must bracket the work the host waited for
        raise SystemExit(f"bench.py: device time {ms_dev:.1f} ms does not match the wall clock {t_wall * 1e3:.1f} ms around the same region")
    launches = S.launch_count() - launches0
    S.download_ptr(None, None, cost_out.data_ptr(), it_out.data_ptr(), res_out.data_ptr(), nls_out.data_ptr())
    n_ls = int(nls_out.numpy().sum())
    cost_resident = cost_out.numpy().copy()
    # passes of the iLQG loop the timed solve made: --steps unless every problem of the shard stopped earlier
    passes = int(reduce(int(it_out.numpy().max()), dist.ReduceOp.MAX if world > 1 else None))

    ms_max = reduce(ms_dev, dist.ReduceOp.MAX if world > 1 else None)
    its_total = reduce(n_ls, dist.ReduceOp.SUM if world > 1 else None)
    value = its_total / (ms_max * 1e-3)

    # ---- timed region 2: end to end through the C ABI with host buffers (preceded, like region 1, by W warm-up passes) --------
    S.set_options({"max_iter": args.warmup})
    S.solve_host_ptr(*host_ptrs)
    S.set_options({"max_iter": args.steps})
    barrier()
    i0 = sampler.mark()
    t0 = time.perf_counter()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    S.solve_host_ptr(*host_ptrs)
    e3.record()
    torch.cuda.synchronize()
    wall_e2e = time.perf_counter() - t0
    ms_e2e = max(e2.elapsed_time(e3), wall_e2e * 1e3)
    barrier()
    eclocks = sampler.summary(i0, sampler.mark())
    sampler.stop()
    n_ls_e2e = int(nls_out.numpy().sum())
    deterministic = bool(np.array_equal(cost_resident, cost_out.numpy()))
    if args.dump_outputs:   # the host buffers hold what this leg's call returned; no copy beyond the timed one
        dump_outputs(args.dump_outputs, x_out.numpy(), u_out.numpy(), cost_out.numpy(), it_out.numpy(), res_out.numpy(), nls_out.numpy())
    ms_e2e_max = reduce(ms_e2e, dist.ReduceOp.MAX if world > 1 else None)
    its_e2e = reduce(n_ls_e2e, dist.ReduceOp.SUM if world > 1 else None)
    h2d = x0_t.numel() * 8 + u0_t.numel() * 8
    d2h = (x_out.numel() + u_out.numel() + cost_out.numel()) * 8 + (it_out.numel() + res_out.numel() + nls_out.numel()) * 4
    h2d_tot = reduce(h2d, dist.ReduceOp.SUM if world > 1 else None)
    d2h_tot = reduce(d2h, dist.ReduceOp.SUM if world > 1 else None)
    chunks_per_gpu = S.chunks() // max(multi, 1)

    # ---- roofline of the dominant kernel: kernels timed ALONE on the problems of one chunk of this rank's shard, i.e. at
    #      exactly the launch size the timed run uses --------------------------------------------------------------------------
    n_k = max(1, count // S.chunks())
    kernels, kclocks, _ = kernels_alone(PROBLEM, FULL_DDP, n_k, T_HOR, W.CAR_PARAMS, x0_t.data_ptr(), u0_t.data_ptr(), args.steps,
                                        local_rank, stream, nx, nu)
    dom = max(kernels, key=lambda k: kernels[k]["ms_total"]) if kernels else None
    names = {"derivs": "k_derivs", "backpass": "k_backpass", "linesearch": "k_ls_round"}
    roofline = roofline_of(kernels, dom, n_k, kclocks, names) if dom else None
    if dom == "backpass":       # fp64-issue bound kernel: its roofline is the fp64 instruction peak; the HBM view stays beside it
        f = kernels["backpass"]["fp64"]
        roofline = {"kernel": names[dom], "bound": "fp64-issue", "achieved": f["achieved_dp_instr_per_s"] / 1e12, "peak": f["peak_dp_instr_per_s"] / 1e12,
                    "unit": "T dp-instr/s (DMUL+DADD)", "frac": f["frac"], "peak_source": f["peak_source"], "traffic": roofline["traffic"], "hbm": roofline}
    # the line search and the backward pass take about the same share of a pass; both views are always in the record
    rooflines = {k: roofline_of(kernels, k, n_k, kclocks, names) for k in kernels}

    # ---- CPU baseline on the host cores (rank 0, N = 1 only) -----------------------------------------------------------------
    cpu = None
    parity_flags = []
    if rank == 0 and n_gpus == 1 and not args.no_cpu_baseline:
        cores = host_cores()
        n = min(args.batch, max(cores * 2, int(cores * 1250 * 15 / max(args.steps, 1))))
        r = cpu_reference_run(n, args.steps, cores)
        if r:
            # the sample doubles as a parity check of the timed GPU results (checker only, never the product path)
            same = bool(np.array_equal(r["out"]["cost"], cost_resident[:n])) if first == 0 else None
            parity_flags.append(same)
            cpu = {"value": r["value"], "unit": UNIT, "cores": cores, "kind": r["kind"],
                   "sample": f"first {n} problems of the batch, max_iter={args.steps}, one solver instance per thread, {r['seconds']:.1f} s",
                   "note": "a sample of the batch, rate extrapolated; the reference core is compiled -O3 -ffp-contract=off against the same "
                           "generated problem code as the GPU, i.e. with csrc/dm_math.h for sin/cos/asin (3.5 % slower than glibc libm, DESIGN.md 6)",
                   "gpu_costs_bit_identical_on_sample": same, "config1_single_instance": cpu_single_instance()}

    # ---- the other BASELINE configs (N = 1 only) ---------------------------------------------------------------------------------
    extra = None
    if rank == 0 and n_gpus == 1 and not args.no_extra and not args.no_cpu_baseline:
        S.close()
        S = None
        del x_out, u_out
        extra = []
        extra.append(short_config("config3", "car", 0, 4096, T_HOR, W.CAR_PARAMS, W.car_batch(4096, T=T_HOR), 50, 256, local_rank, 4, 2,
                                  "car-parking n=4 m=2 T=500 FULL_DDP=0, batch 4096 (BASELINE config 3), max_iter=50"))
        qB = 16384
        extra.append(short_config("config5", "quad", 1, qB, W.QUAD_T, W.QUAD_PARAMS, W.quad_batch(qB, T=W.QUAD_T), 20, 32, local_rank, 12, 4,
                                  "synthetic quadrotor n=12 m=4 T=1000 FULL_DDP=1 box-constrained, batch 16384 (BASELINE config 5), max_iter=20"))
        if args.steps != 50 and args.batch == 262144:
            x0n, u0n = x0_t.numpy(), u0_t.numpy()
            extra.append(short_config("config4_max_iter50", "car", 0, args.batch, T_HOR, W.CAR_PARAMS, (x0n, u0n), 50, 2048, local_rank, 4, 2,
                                      "car-parking n=4 m=2 T=500 FULL_DDP=0, batch 262144 (BASELINE config 4 as surveyed), max_iter=50"))
        parity_flags += [e["gpu_costs_bit_identical_on_sample"] for e in extra]

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps, "passes": passes, "warmup": args.warmup,
            "ms_per_step": ms_max / max(args.steps, 1), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(args), "clocks": clocks,
            "e2e": {"value": its_e2e / (ms_e2e_max * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d_tot / max(args.steps, 1),
                    "d2h_bytes_per_step": d2h_tot / max(args.steps, 1), "h2d_bytes": h2d_tot, "d2h_bytes": d2h_tot,
                    "seconds": ms_e2e_max * 1e-3, "clocks": eclocks},
            "gpu_launches": launches, "roofline": roofline, "roofline_hbm_by_kernel": {k: {kk: v[kk] for kk in ("achieved", "frac", "frac_record_bytes", "traffic", "algorithmic_bytes_per_launch")} for k, v in rooflines.items()},
            "kernels": kernels, "cpu_baseline": cpu,
            "iterations_total": its_total, "seconds": ms_max * 1e-3, "seconds_wall_rank0": t_wall, "deterministic_rerun": deterministic,
            "streams_per_gpu": chunks_per_gpu, "process_model": "one process, ilqgb_create_multi" if multi else "one process per GPU",
            "extra": extra,
        }
        print(json.dumps(line))
        sys.stdout.flush()
        if passes < args.steps:
            sys.stderr.write(f"bench.py: every problem stopped after {passes} of the {args.steps} passes --steps allows\n")
    if S is not None:
        S.close()
    if world > 1:
        dist.destroy_process_group()
    if any(f is False for f in parity_flags) or not deterministic:
        sys.stderr.write("bench.py: GPU results differ from the CPU reference on the checked sample (or between reruns)\n")
        sys.exit(3)


if __name__ == "__main__":
    main()
