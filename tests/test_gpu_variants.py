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

import parity_util as PU
from ilqg_b200 import workloads as W

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COOP_LIB = os.path.join(ROOT, "ddp-generator_b200", "lib_coop")
N_ALPHA = 8
_BASE = {}      # records of each axis' baseline variant, by case name


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
    return PU.Case("quad", ddp, T, W.QUAD_PARAMS, x0, u0, QUAD_OPTS[opts], pp={"ulim": ulim, "cf": cf})


@pytest.mark.parametrize("lpp", [32, 16, 8])
@pytest.mark.parametrize("opts", list(QUAD_OPTS))
@pytest.mark.parametrize("ddp", [0, 1])
def test_quad_cooperative_lanes_per_problem(ddp, opts, lpp):
    name = f"quad ddp{ddp} {opts}"
    c = quad_case(ddp, opts)
    if name not in _BASE:
        _BASE[name] = PU.run(c, {"cw_lpp": 32})[0]
    recs, hooks = PU.run(c, {"cw_lpp": lpp})
    assert hooks["cw_lpp"] == lpp
    PU.check(name, c, recs, _BASE[name])
    ppw = 32 // lpp
    assert PU.mixed_groups(recs, ppw if ppw > 1 else PU.CW_WARPS) > 0, "every warp's problems took the same number of iterations"
    fail_grp = range(QUAD_FAIL // ppw * ppw, QUAD_FAIL // ppw * ppw + ppw)
    assert recs[QUAD_FAIL]["result"] == -1 and all(recs[b]["result"] != -1 for b in fail_grp if b != QUAD_FAIL)
    assert PU.clamped(recs) > 100
    if ddp == 1 or opts == "lmax":
        assert PU.retried(recs) > 0, "no back pass failed"


# ---- 2. the cooperative backward pass forced on for the lane-per-problem problems (ddp-generator_b200/lib_coop/) -----------
def coop_case(which, ddp):
    if which in ("car", "car_reg2"):
        B, T = 13, 90
        x0, u0 = W.car_batch(B, T=T, seed=33)
        opts = {"max_iter": 30} if which == "car" else {"max_iter": 25, "regType": 2}
        return PU.Case("car", ddp, T, W.CAR_PARAMS, x0, u0, opts)
    if which == "carhx":
        B, T = 11, 90
        x0, u0 = W.car_batch(B, T=T, seed=37)
        x0[:, 3] = 1.5                              # moving: the steering limit limW / (1 + kv v^2) depends on the state
        u0 = u0 * 4.0
        return PU.Case("carhx", ddp, T, W.CARHX_PARAMS, x0, u0, {"max_iter": 30})
    if which == "pend":
        x0, u0 = W.pend_batch(9)
        return PU.Case("pend", ddp, W.PEND_T, W.PEND_PARAMS, x0, u0, W.PEND_OPTS)
    params, x0, u0, opts = W.brachi_hli(120)
    B = 3
    return PU.Case("brachi_hli", ddp, 120, params, np.tile(x0, (B, 1)), u0[None] * np.array([1.0, 0.8, 1.2])[:, None, None], opts)


@pytest.mark.parametrize("lpp", [32, 16, 8])
@pytest.mark.parametrize("ddp", [0, 1])
@pytest.mark.parametrize("which", ["car", "car_reg2", "carhx", "pend", "brachi_hli"])
def test_forced_cooperative_backward_pass(which, ddp, lpp):
    name = f"coop {which} ddp{ddp}"
    c = coop_case(which, ddp)
    if name not in _BASE:
        base, hooks = PU.run(c)                         # the default library: k_backpass_split or k_backpass
        assert hooks["cw_lpp"] == 0
        _BASE[name] = base
    recs, hooks = PU.run(c, {"cw_lpp": lpp}, lib_dir=COOP_LIB)
    assert hooks["cw_lpp"] == lpp, "the lib_coop build did not run the cooperative backward pass"
    PU.check(name, c, recs, _BASE[name])
    if c.B > 32 // lpp:
        assert PU.mixed_groups(recs, 32 // lpp if lpp < 32 else PU.CW_WARPS) > 0
    if which == "carhx":
        assert PU.clamped(recs, inputs=[0]) > 20, "the speed-dependent steering limit never clamps"
    elif which in ("car", "car_reg2"):
        assert PU.clamped(recs) > 0
    if ddp == 1 and which in ("car", "car_reg2"):
        assert PU.retried(recs) > 0


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
        return PU.Case(which, ddp, T, params, x0, u0, {"max_iter": 30}, pp=per)
    if which == "pend":
        B = 11
        x0, u0 = W.pend_batch(B)
        per = {"lim": np.stack([-1.0 - 2.0 * rng.random(B), 1.0 + 2.0 * rng.random(B)], axis=1), "thmin": 0.3 + 0.4 * rng.random((B, 1))} if pp else {}
        return PU.Case("pend", ddp, W.PEND_T, W.PEND_PARAMS, x0, u0, W.PEND_OPTS, pp=per)
    params, x0, u0, opts = W.brachi_hli(120)
    B = 5
    per = {"g": 9.81 * (0.7 + 0.6 * rng.random((B, 1)))} if pp else {}
    return PU.Case("brachi_hli", ddp, 120, params, np.tile(x0, (B, 1)), np.tile(u0[None], (B, 1, 1)), opts, pp=per)


@pytest.mark.parametrize("pp", [False, True], ids=["shared", "per_problem"])
@pytest.mark.parametrize("which,ddp,variant", [(p, d, v) for p, d in (("car", 0), ("car", 1), ("carhx", 0), ("carhx", 1), ("pend", 1), ("brachi_hli", 0))
                                               for v in BP if not (p == "carhx" and v == "split")])   # carhx: state-dependent limits, k_backpass only
def test_backward_pass_kernels(which, ddp, variant, pp):
    name = f"bp {which} ddp{ddp} pp{int(pp)}"
    c = bp_case(which, ddp, pp)
    if name not in _BASE:
        _BASE[name] = PU.run(c, BP["lane_latency"])[0]
    recs, hooks = PU.run(c, BP[variant])
    assert hooks["cw_lpp"] == 0 and hooks["bp_split"] == BP[variant]["bp_split"]
    if variant != "split":
        assert hooks["bp_latency"] == BP[variant]["bp_latency"]
    PU.check(name, c, recs, _BASE[name])
    if which in ("car", "carhx"):
        assert PU.clamped(recs, inputs=[0] if which == "carhx" else None) > 20
    if ddp == 1 and which == "car":
        assert PU.retried(recs) > 0


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
    return PU.Case("car", 0, T, params, x0, u0, {"max_iter": 15}, pp=per)


@pytest.mark.parametrize("commit", ["parallel", "sequential"])
@pytest.mark.parametrize("tail_from", [0, 1, 2, 3, 4, N_ALPHA])
@pytest.mark.parametrize("pp", [False, True], ids=["shared", "per_problem"])
@pytest.mark.parametrize("T", [80, 20])
def test_line_search_schedules(T, pp, tail_from, commit, monkeypatch):
    """T = 80 is not a multiple of the 32 commit segments; T = 20 has fewer steps than segments."""
    name = f"ls T{T} pp{int(pp)}"
    c = ls_case(T, pp)
    if name not in _BASE:
        _BASE[name] = PU.run(c, {"ls_tail_from": N_ALPHA})[0]
    if commit == "sequential":
        monkeypatch.setenv("ILQG_LS_COMMIT_PAR", "0")     # read when the handle allocates its workspace
    recs, hooks = PU.run(c, {"ls_tail_from": tail_from})
    assert hooks["ls_tail_from"] == tail_from and hooks["ls_commit_par"] == (commit == "parallel")
    PU.check(name, c, recs, _BASE[name])
    assert PU.deep(recs) > (20 if T == 80 else 5), "the line search never backtracked deep"


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
    c = PU.Case("cartrack", ddp, T, params, x0, u0, {"max_iter": 15}, pp=pp, tracks=tracks, off=off)
    name = f"tracks ddp{ddp}"
    if name not in _BASE:
        _BASE[name] = PU.run(c, BP["lane_latency"])[0]
    recs, hooks = PU.run(c, TRACK_VARIANTS[variant])
    for k, v in TRACK_VARIANTS[variant].items():
        assert hooks[k] == v
    PU.check(name, c, recs, _BASE[name])
    assert PU.clamped(recs) > 0
