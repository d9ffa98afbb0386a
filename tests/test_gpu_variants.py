"""Every kernel variant the solver can dispatch to, forced in turn on the same inputs.  Each cell checks that
- everything the solve writes is bit-identical to the oracle called once per problem with that problem's parameters (and,
  for tracks, its window), gains l, L and the expected reduction dV included;
- everything, the per-step box-QP clamp records included, is bit-identical to the other variants of the same axis;
- the variant ran (the ilqgb_get_int test hooks "cw_lpp", "bp_split", "bp_latency", "ls_tail_from", "ls_commit_par"), and the
  inputs exercised it: problems of one warp take different numbers of iterations, back passes fail and are retried, QPs clamp,
  the line search backtracks deep.

Axes: the warp-cooperative backward pass at 32, 16 and 8 lanes per problem (the quadrotor, and the lane-per-problem problems
through the test build in ddp-generator_b200/lib_coop/ that forces it on); the backward-pass kernels (k_backpass_split, both
register builds of k_backpass); the line search (sequential rounds before the parallel-alpha tail, checkpointed or sequential
commit); each with shared and per-problem parameter sets, and per-problem tracks with per-problem parameters."""
import os

import numpy as np
import pytest

import ilqg_b200
import parity_util as PU
from ilqg_b200 import workloads as W

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COOP_LIB = os.path.join(ROOT, "ddp-generator_b200", "lib_coop")
ORACLE_KEYS = PU.assert_same.__defaults__[0] + ("l", "L", "dV0", "dV1")
KEYS = ("result", "iterations", "n_ls", "n_bp", "cost", "lambda", "g_norm", "w_pen_l", "w_pen_f", "dV0", "dV1", "tr_alpha",
        "tr_lambda", "tr_newcost", "tr_clamp", "x", "u", "l", "L")          # as tests/test_gpu_split.py
HOOKS = ("bp_split", "cw_lpp", "bp_latency", "ls_tail_from", "ls_commit_par")
N_ALPHA = 8
CW_WARPS = 4      # warps per block of k_backpass_warp


class Case:
    """One set of inputs: shared parameters, optional per-problem parameter sets pp {name: [B, size]} and tracks
    {name: [B, len]} read from window offset `off`."""

    def __init__(self, problem, ddp, T, params, x0, u0, opts, pp=None, tracks=None, off=0):
        self.problem, self.ddp, self.T, self.params, self.x0, self.u0, self.opts = problem, ddp, T, params, x0, u0, opts
        self.pp, self.tracks, self.off = pp or {}, tracks or {}, off
        self.B = x0.shape[0]

    def params_of(self, b):
        p = dict(self.params, **{k: v[b] for k, v in self.pp.items()})
        return dict(p, **{k: v[b, self.off:self.off + self.T + 1] for k, v in self.tracks.items()})


def run(c, tuning=None, lib_dir=None):
    """Solve the batch on the GPU: per-problem records shaped like parity_util.oracle_record, and the hooks."""
    s = ilqg_b200.BatchSolver(c.problem, c.ddp, c.B, c.T, flags=ilqg_b200.TRACE, lib_dir=lib_dir)
    s.set_options(c.opts)
    s.set_params(c.params)
    if c.pp:
        s.set_params_batch(c.pp)
    for k, v in c.tracks.items():
        s.set_param_track(k, v)
    if c.tracks:
        s.set_track_offset(c.off)
    for k, v in (tuning or {}).items():
        s.set_tuning(k, v)
    out = s.solve(c.x0, c.u0)
    sc = {k: s.get(k) for k in ("lambda", "g_norm", "w_pen_l", "w_pen_f", "dV0", "dV1")}
    l, L = s.get("l"), s.get("L")
    tr_l, tr_c = s.get("tr_lambda"), s.get("tr_newcost")
    tr_a, tr_cl = s.get_int("tr_alpha"), s.get_int("tr_clamp")
    nbp = s.get_int("n_backpass")
    hooks = {k: s.get_int(k) for k in HOOKS}
    s.close()
    recs = []
    for b in range(c.B):
        n = int(out["n_linesearch"][b])
        recs.append(dict(result=int(out["success"][b]), iterations=int(out["iterations"][b]), cost=out["cost"][b],
                         x=out["x"][b], u=out["u"][b], l=l[b], L=L[b], n_ls=n, n_bp=int(nbp[b]),
                         tr_lambda=tr_l[b][:n], tr_alpha=tr_a[b][:n], tr_newcost=tr_c[b][:n], tr_clamp=tr_cl[b],
                         **{k: v[b] for k, v in sc.items()}))
    for k, v in hooks.items():
        assert np.all(v == v[0]), f"hook {k} differs between problems of one chunk"
    return recs, {k: int(v[0]) for k, v in hooks.items()}


_ORACLE, _BASE = {}, {}


def oracle(name, c):
    if name not in _ORACLE:
        kind = PU.oracle_kinds(c.problem, c.ddp)[0]
        opts = {k: float(v) if np.isscalar(v) else v for k, v in c.opts.items()}
        _ORACLE[name] = [PU.oracle_record(kind, c.problem, c.ddp, c.T, c.params_of(b), c.x0[b], c.u0[b], opts) for b in range(c.B)]
    return _ORACLE[name]


def check(name, c, recs, base):
    """recs against the oracle (every problem) and against the axis' baseline variant `base` (records of the same inputs)."""
    for b, (g, o) in enumerate(zip(recs, oracle(name, c))):
        if not o["init_ok"]:
            assert g["result"] == -1 and g["n_ls"] == 0, f"{name} b{b}: failed initial rollout not reported"
            continue
        PU.assert_same(g, o, f"{name} b{b} vs oracle", keys=ORACLE_KEYS)
    for b, (g, r) in enumerate(zip(recs, base)):
        for k in KEYS:
            assert np.array_equal(np.asarray(g[k]), np.asarray(r[k]), equal_nan=True), f"{name} b{b}: {k} differs from the baseline variant"


def clamped(recs, inputs=None):
    """number of (problem, step) box-QP solutions with a clamped input (of `inputs`, default any)"""
    mask = sum(3 << (2 * i) for i in inputs) if inputs is not None else 0xffff
    return sum(int(np.count_nonzero(np.asarray(r["tr_clamp"]) & mask)) for r in recs)


def deep(recs):
    """accepted or rejected line-search results at alpha index >= 4"""
    return sum(int((np.asarray(r["tr_alpha"]) >= 4).sum()) for r in recs)


def retried(recs):
    return sum(r["n_bp"] > r["iterations"] for r in recs)


def mixed_groups(recs, size):
    """groups of `size` consecutive problems (the problems of one warp or block) whose iteration counts differ"""
    it = [r["iterations"] for r in recs]
    return sum(len(set(it[g:g + size])) > 1 for g in range(0, len(it), size))


# ---- 1. the warp-cooperative backward pass on the quadrotor, 32 / 16 / 8 lanes per problem ----------------------------------
QUAD_OPTS = {"default": {"max_iter": 30}, "reg2": {"max_iter": 25, "regType": 2},
             "lmax": {"max_iter": 30, "lambdaInit": 1e-3, "lambdaMin": 1e-6, "lambdaMax": 1e-2}}
QUAD_FAIL = 5      # a problem whose initial rollout fails, sharing its warp at 16 and 8 lanes per problem


def quad_case(ddp, opts):
    B, T = 37, 130
    x0, u0 = W.quad_batch(B, T=T, seed=23)
    x0[QUAD_FAIL, 10] = x0[QUAD_FAIL, 11] = 1e200      # wq * wr overflows: the NaN guard fails the first step
    rng = np.random.default_rng(29)
    uh = W.QUAD_PARAMS["uh"][0]
    tight = rng.random(B) < 0.5                       # half of the problems get a narrow thrust box: their QPs clamp
    ulim = np.where(tight[:, None], [[0.85 * uh, 1.15 * uh]], [W.QUAD_PARAMS["ulim"]])
    cf = np.asarray(W.QUAD_PARAMS["cf"])[None, :] * (0.3 + 1.4 * rng.random((B, 12)))
    return Case("quad", ddp, T, W.QUAD_PARAMS, x0, u0, QUAD_OPTS[opts], pp={"ulim": ulim, "cf": cf})


@pytest.mark.parametrize("lpp", [32, 16, 8])
@pytest.mark.parametrize("opts", list(QUAD_OPTS))
@pytest.mark.parametrize("ddp", [0, 1])
def test_quad_cooperative_lanes_per_problem(ddp, opts, lpp):
    name = f"quad ddp{ddp} {opts}"
    c = quad_case(ddp, opts)
    if name not in _BASE:
        _BASE[name] = run(c, {"cw_lpp": 32})[0]
    recs, hooks = run(c, {"cw_lpp": lpp})
    assert hooks["cw_lpp"] == lpp
    check(name, c, recs, _BASE[name])
    ppw = 32 // lpp
    assert mixed_groups(recs, ppw if ppw > 1 else CW_WARPS) > 0, "every warp's problems took the same number of iterations"
    fail_grp = range(QUAD_FAIL // ppw * ppw, QUAD_FAIL // ppw * ppw + ppw)
    assert recs[QUAD_FAIL]["result"] == -1 and all(recs[b]["result"] != -1 for b in fail_grp if b != QUAD_FAIL)
    assert clamped(recs) > 100
    if ddp == 1 or opts == "lmax":
        assert retried(recs) > 0, "no back pass failed"


# ---- 2. the cooperative backward pass forced on for the lane-per-problem problems (ddp-generator_b200/lib_coop/) -----------
def coop_case(which, ddp):
    if which in ("car", "car_reg2"):
        B, T = 13, 90
        x0, u0 = W.car_batch(B, T=T, seed=33)
        opts = {"max_iter": 30} if which == "car" else {"max_iter": 25, "regType": 2}
        return Case("car", ddp, T, W.CAR_PARAMS, x0, u0, opts)
    if which == "carhx":
        B, T = 11, 90
        x0, u0 = W.car_batch(B, T=T, seed=37)
        x0[:, 3] = 1.5                              # moving: the steering limit limW / (1 + kv v^2) depends on the state
        u0 = u0 * 4.0
        return Case("carhx", ddp, T, W.CARHX_PARAMS, x0, u0, {"max_iter": 30})
    if which == "pend":
        x0, u0 = W.pend_batch(9)
        return Case("pend", ddp, W.PEND_T, W.PEND_PARAMS, x0, u0, W.PEND_OPTS)
    params, x0, u0, opts = W.brachi_hli(120)
    B = 3
    return Case("brachi_hli", ddp, 120, params, np.tile(x0, (B, 1)), u0[None] * np.array([1.0, 0.8, 1.2])[:, None, None], opts)


@pytest.mark.parametrize("lpp", [32, 16, 8])
@pytest.mark.parametrize("ddp", [0, 1])
@pytest.mark.parametrize("which", ["car", "car_reg2", "carhx", "pend", "brachi_hli"])
def test_forced_cooperative_backward_pass(which, ddp, lpp):
    name = f"coop {which} ddp{ddp}"
    c = coop_case(which, ddp)
    if name not in _BASE:
        base, hooks = run(c)                         # the default library: k_backpass_split or k_backpass
        assert hooks["cw_lpp"] == 0
        _BASE[name] = base
    recs, hooks = run(c, {"cw_lpp": lpp}, lib_dir=COOP_LIB)
    assert hooks["cw_lpp"] == lpp, "the lib_coop build did not run the cooperative backward pass"
    check(name, c, recs, _BASE[name])
    if c.B > 32 // lpp:
        assert mixed_groups(recs, 32 // lpp if lpp < 32 else CW_WARPS) > 0
    if which == "carhx":
        assert clamped(recs, inputs=[0]) > 20, "the speed-dependent steering limit never clamps"
    elif which in ("car", "car_reg2"):
        assert clamped(recs) > 0
    if ddp == 1 and which in ("car", "car_reg2"):
        assert retried(recs) > 0


# ---- 3. backward-pass kernels x parameter sets ----------------------------------------------------------------------------
BP = {"split": {"bp_split": 4}, "lane_latency": {"bp_split": 0, "bp_latency": 1}, "lane_128reg": {"bp_split": 0, "bp_latency": 0}}


def bp_case(which, ddp, pp):
    rng = np.random.default_rng(43)
    if which in ("car", "carhx"):
        B, T = 37, 100
        x0, u0 = W.car_batch(B, T=T, seed=47)
        params = W.CAR_PARAMS if which == "car" else W.CARHX_PARAMS
        if which == "carhx":
            x0[:, 3] = 1.5
            u0 = u0 * 4.0
        per = {}
        if pp:
            per = {"limW": np.stack([-0.2 - 0.3 * rng.random(B), 0.2 + 0.3 * rng.random(B)], axis=1),
                   "cf": np.asarray(params["cf"])[None, :] * (0.5 + rng.random((B, 4))), "d": 1.5 + rng.random((B, 1))}
        return Case(which, ddp, T, params, x0, u0, {"max_iter": 30}, pp=per)
    if which == "pend":
        B = 11
        x0, u0 = W.pend_batch(B)
        per = {"lim": np.stack([-1.0 - 2.0 * rng.random(B), 1.0 + 2.0 * rng.random(B)], axis=1), "thmin": 0.3 + 0.4 * rng.random((B, 1))} if pp else {}
        return Case("pend", ddp, W.PEND_T, W.PEND_PARAMS, x0, u0, W.PEND_OPTS, pp=per)
    params, x0, u0, opts = W.brachi_hli(120)
    B = 5
    per = {"g": 9.81 * (0.7 + 0.6 * rng.random((B, 1)))} if pp else {}
    return Case("brachi_hli", ddp, 120, params, np.tile(x0, (B, 1)), np.tile(u0[None], (B, 1, 1)), opts, pp=per)


@pytest.mark.parametrize("pp", [False, True], ids=["shared", "per_problem"])
@pytest.mark.parametrize("which,ddp,variant", [(p, d, v) for p, d in (("car", 0), ("car", 1), ("carhx", 0), ("carhx", 1), ("pend", 1), ("brachi_hli", 0))
                                               for v in BP if not (p == "carhx" and v == "split")])   # carhx: state-dependent limits, k_backpass only
def test_backward_pass_kernels(which, ddp, variant, pp):
    name = f"bp {which} ddp{ddp} pp{int(pp)}"
    c = bp_case(which, ddp, pp)
    if name not in _BASE:
        _BASE[name] = run(c, BP["lane_latency"])[0]
    recs, hooks = run(c, BP[variant])
    assert hooks["cw_lpp"] == 0 and hooks["bp_split"] == BP[variant]["bp_split"]
    if variant != "split":
        assert hooks["bp_latency"] == BP[variant]["bp_latency"]
    check(name, c, recs, _BASE[name])
    if which in ("car", "carhx"):
        assert clamped(recs, inputs=[0] if which == "carhx" else None) > 20
    if ddp == 1 and which == "car":
        assert retried(recs) > 0


# ---- 4. line search: sequential rounds before the parallel-alpha tail, checkpointed or sequential commit -------------------
def ls_case(T, pp):
    """large steps leave the domain of the dynamics (NaN guard) while small ones are fine: the search backtracks deep"""
    B = 12
    x0, u0 = W.car_batch(B, T=T, seed=91)
    x0[:, 3] = 1.5
    u0 = u0 * 5
    params = dict(W.CAR_PARAMS, d=[0.05], limA=[-20.0, 20.0])
    per = {}
    if pp:
        rng = np.random.default_rng(53)
        per = {"d": 0.04 + 0.02 * rng.random((B, 1)), "cf": np.asarray(params["cf"])[None, :] * (0.5 + rng.random((B, 4)))}
    return Case("car", 0, T, params, x0, u0, {"max_iter": 15}, pp=per)


@pytest.mark.parametrize("commit", ["parallel", "sequential"])
@pytest.mark.parametrize("tail_from", [0, 1, 2, 3, 4, N_ALPHA])
@pytest.mark.parametrize("pp", [False, True], ids=["shared", "per_problem"])
@pytest.mark.parametrize("T", [80, 20])
def test_line_search_schedules(T, pp, tail_from, commit, monkeypatch):
    """T = 80 is not a multiple of the 32 commit segments; T = 20 has fewer steps than segments."""
    name = f"ls T{T} pp{int(pp)}"
    c = ls_case(T, pp)
    if name not in _BASE:
        _BASE[name] = run(c, {"ls_tail_from": N_ALPHA})[0]
    if commit == "sequential":
        monkeypatch.setenv("ILQG_LS_COMMIT_PAR", "0")     # read when the handle allocates its workspace
    recs, hooks = run(c, {"ls_tail_from": tail_from})
    assert hooks["ls_tail_from"] == tail_from and hooks["ls_commit_par"] == (commit == "parallel")
    check(name, c, recs, _BASE[name])
    assert deep(recs) > (20 if T == 80 else 5), "the line search never backtracked deep"


# ---- 5. per-problem tracks together with per-problem parameter sets ----------------------------------------------------------
TRACK_VARIANTS = {"default": {}, "lane_latency": BP["lane_latency"], "lane_128reg": BP["lane_128reg"], "tail0": {"ls_tail_from": 0},
                  "tail2": {"ls_tail_from": 2}, "sequential": {"ls_tail_from": N_ALPHA}}


@pytest.mark.parametrize("variant", list(TRACK_VARIANTS))
@pytest.mark.parametrize("ddp", [0, 1])
def test_tracks_with_per_problem_parameters(ddp, variant):
    B, T, off = 9, 60, 4
    x0, u0, tracks = W.cartrack_batch(B, T=T, extra=10, seed=59)
    params = dict(W.CARTRACK_PARAMS, **{k: v[0, :T + 1] for k, v in tracks.items()})
    rng = np.random.default_rng(61)
    pp = {"limW": np.stack([-0.1 - 0.4 * rng.random(B), 0.1 + 0.4 * rng.random(B)], axis=1),
          "cu": np.asarray(params["cu"])[None, :] * (0.5 + rng.random((B, 2)))}
    c = Case("cartrack", ddp, T, params, x0, u0, {"max_iter": 15}, pp=pp, tracks=tracks, off=off)
    name = f"tracks ddp{ddp}"
    if name not in _BASE:
        _BASE[name] = run(c, BP["lane_latency"])[0]
    recs, hooks = run(c, TRACK_VARIANTS[variant])
    for k, v in TRACK_VARIANTS[variant].items():
        assert hooks[k] == v
    check(name, c, recs, _BASE[name])
    assert clamped(recs) > 0
