"""Every kernel at problem dimensions no shipped problem has: the test-only problems tests/data/shape_<nx>x<nu>.mac, built by
__graft_entry__.build_shape_problems() into ddp-generator_b200/build_shapes/.

    (4, 1)   one input and several states; NX+NU odd; a 1 x 1 box QP
    (3, 4)   more inputs than states; odd nx
    (6, 3)   the largest lane-per-problem state; k_backpass_split's columns and off-diagonals split unevenly over 4 lanes; NX+NU = 9
    (7, 5)   the smallest cooperative state; NU*NX = 35; the lane-parallel QP inverse with idle lanes at every lane count
    (10, 9)  a 9 x 9 box QP: more inputs than 8 lanes (sequential inverse at 8 lanes per problem)
    (16, 9)  the workspace of 8 lanes per problem does not fit in a block's shared memory: cw_lpp 8 is refused

Each solve cell forces one backward-pass variant, checks everything the solve writes against the oracle called once per problem
and against the shape's baseline variant (parity_util.check), that the variant ran, and that its inputs exercised it: iterations
differ inside a warp, back passes fail and are retried, every input clamps (the middle one of three between two free ones too),
the line search backtracks to alpha index 4 or deeper.  On the shapes with odd record lengths, the closed loop, shift, the feedback
policy and chunking are checked against the oracle as well."""
import os

import numpy as np
import pytest

import ilqg_b200
import oracle_lib
import parity_util as PU
import policy_util
import test_gpu_mpc as MPC
from shapes_util import COOP, LANE, name_of, params_of
from ilqg_b200 import workloads as W

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPE_ROOT = os.path.join(ROOT, "ddp-generator_b200", "build_shapes")
SHAPE_LIB = os.path.join(SHAPE_ROOT, "lib")
ODD = [(4, 1), (6, 3), (7, 5)]
BP = {"split": {"bp_split": 4}, "lane_latency": {"bp_split": 0, "bp_latency": 1}, "lane_128reg": {"bp_split": 0, "bp_latency": 0}}
# lanes per problem whose workspace fits in the 227 KB of shared memory a B200 gives one block (coop_smem_bytes: 8 lanes per problem of
# (16, 9) need about 363 KB, test_workspace_that_does_not_fit_is_refused)
FITS = {(7, 5): (32, 16, 8), (10, 9): (32, 16, 8), (16, 9): (32, 16)}
_BASE = {}


def inputs(shape, B, T, seed):
    """initial states beyond pi / 2, where the final cost 1 - cos is concave: the back passes of FULL_DDP = 0 fail too"""
    rng = np.random.default_rng(seed)
    return rng.uniform(-2.5, 2.5, (B, shape[0])), 0.1 * rng.standard_normal((B, T, shape[1]))


def shape_case(shape, ddp, pp=False):
    B = 37 if shape in LANE else 13
    T = 40
    x0, u0 = inputs(shape, B, T, seed=71 + shape[0] * 16 + shape[1])
    per = {}
    if pp:
        rng = np.random.default_rng(73)
        lim = np.asarray(params_of(shape)["uhi"])[None, :] * (0.6 + 0.8 * rng.random((B, shape[1])))
        per = {"ulo": -lim, "uhi": lim, "cf": 5.0 * (0.5 + rng.random((B, shape[0])))}
    return PU.Case(name_of(shape), ddp, T, params_of(shape), x0, u0, {"max_iter": 100}, pp=per)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def mixed_clamps(recs, nu):
    """box-QP solutions in which an input is clamped while both its neighbours are free"""
    n = 0
    for r in recs:
        c = np.asarray(r["tr_clamp"]) & 0xffff
        code = [(c >> (2 * i)) & 3 for i in range(nu)]
        n += sum(int(((code[i] != 0) & (code[i - 1] == 0) & (code[i + 1] == 0)).sum()) for i in range(1, nu - 1))
    return n


def exercised(recs, shape, per_warp):
    assert PU.mixed_groups(recs, per_warp) > 0, "every warp's problems took the same number of iterations"
    assert PU.retried(recs) > 0, "no back pass failed"
    for i in range(shape[1]):
        assert PU.clamped(recs, inputs=[i]) > 0, f"input {i} never clamps"
    if shape[1] >= 3:
        assert mixed_clamps(recs, shape[1]) > 0, "no clamped input between two free ones"
    assert PU.deep(recs) > 0, "the line search never backtracked to alpha index 4"


# ---- 1. the lane-per-problem backward passes: k_backpass_split and both register builds of k_backpass -----------------------------
@pytest.mark.parametrize("variant", list(BP))
@pytest.mark.parametrize("ddp", [0, 1])
@pytest.mark.parametrize("shape,pp", [(s, False) for s in LANE] + [((6, 3), True)], ids=lambda v: f"{v[0]}x{v[1]}" if isinstance(v, tuple) else ("per_problem" if v else "shared"))
def test_lane_per_problem_shapes(shape, pp, ddp, variant):
    name = f"{name_of(shape)} ddp{ddp} pp{int(pp)}"
    c = shape_case(shape, ddp, pp)
    if name not in _BASE:
        _BASE[name] = PU.run(c, BP["lane_latency"], lib_dir=SHAPE_LIB)[0]
    recs, hooks = PU.run(c, BP[variant], lib_dir=SHAPE_LIB)
    assert hooks["cw_lpp"] == 0 and hooks["bp_split"] == BP[variant]["bp_split"]
    if variant != "split":
        assert hooks["bp_latency"] == BP[variant]["bp_latency"]
    PU.check(name, c, recs, _BASE[name])
    exercised(recs, shape, 4 if variant == "split" else 32)      # problems per warp: 4 with four lanes each, else 32


# ---- 2. the warp-cooperative backward pass at 32, 16 and 8 lanes per problem, wherever the workspace fits ------------------------
@pytest.mark.parametrize("shape,ddp,lpp", [(s, d, lpp) for s in COOP for d in (0, 1) for lpp in FITS[s]],
                         ids=lambda v: f"{v[0]}x{v[1]}" if isinstance(v, tuple) else str(v))
def test_cooperative_shapes(shape, ddp, lpp):
    name = f"{name_of(shape)} ddp{ddp}"
    c = shape_case(shape, ddp)
    if name not in _BASE:
        base, hooks = PU.run(c, lib_dir=SHAPE_LIB)         # the default: 32 lanes per problem
        assert hooks["cw_lpp"] == 32
        _BASE[name] = base
    recs, hooks = PU.run(c, {"cw_lpp": lpp}, lib_dir=SHAPE_LIB)
    assert hooks["cw_lpp"] == lpp
    PU.check(name, c, recs, _BASE[name])
    exercised(recs, shape, 32 // lpp if lpp < 32 else PU.CW_WARPS)


# ---- 3. lanes per problem whose workspace a block cannot hold ------------------------------------------------------------------
def test_workspace_that_does_not_fit_is_refused(monkeypatch):
    """(16, 9) at 8 lanes per problem needs more shared memory per block than the device gives: set_tuning refuses it, names the
    bytes, and the handle keeps solving at its previous setting; ILQG_CW_LPP=8 fails at create.  (10, 9) takes 8 lanes."""
    c = shape_case((16, 9), 1)
    s = ilqg_b200.BatchSolver(c.problem, 1, c.B, c.T, lib_dir=SHAPE_LIB)
    s.set_options(c.opts)
    s.set_params(c.params)
    s.set_tuning("cw_lpp", 16)
    with pytest.raises(RuntimeError, match=r"cw_lpp 8: .* needs \d+ bytes of shared memory per block, the device allows \d+"):
        s.set_tuning("cw_lpp", 8)
    out = s.solve(c.x0, c.u0)
    assert (s.get_int("cw_lpp") == 16).all()
    ora = PU.oracle(f"{name_of((16, 9))} ddp1", c)
    for b in range(c.B):
        assert out["cost"][b] == ora[b]["cost"] and np.array_equal(out["u"][b], ora[b]["u"]), b
    s.close()
    monkeypatch.setenv("ILQG_CW_LPP", "8")
    with pytest.raises(RuntimeError, match=r"ilqgb_create failed: cw_lpp 8: .* needs \d+ bytes"):
        ilqg_b200.BatchSolver(c.problem, 1, c.B, c.T, lib_dir=SHAPE_LIB)
    monkeypatch.delenv("ILQG_CW_LPP")
    s = ilqg_b200.BatchSolver(name_of((10, 9)), 0, 4, 10, lib_dir=SHAPE_LIB)
    s.set_tuning("cw_lpp", 8)
    s.close()


# ---- 4. around the solve, on the shapes with odd record lengths ------------------------------------------------------------------
def around_case(shape, ddp, B=6, T=30):
    x0, u0 = inputs(shape, B, T, seed=91 + shape[0])
    return x0, u0, params_of(shape, dt=0.1), {"max_iter": 15}


@pytest.mark.parametrize("ddp", [0, 1])
@pytest.mark.parametrize("shape", ODD, ids=lambda s: f"{s[0]}x{s[1]}")
def test_closed_loop_and_shift(shape, ddp):
    """mpc() is the oracle called once per step; shift(n) then run() is the oracle on x[n] and the solution shifted by n."""
    problem = name_of(shape)
    x0, u0, params, opts = around_case(shape, ddp)
    w = W.disturbance(x0.shape[0], 3, shape[0], 0.01, seed=95)
    log, final = MPC.gpu_mpc(problem, ddp, x0, u0, params, opts, 3, w, lib_dir=SHAPE_LIB)
    ora, ora_final = MPC.oracle_loop(problem, ddp, x0, u0, params, opts, 3, w)
    MPC.assert_logs(log, ora, f"{problem} mpc")
    MPC.assert_logs(final, ora_final, f"{problem} mpc final plan", keys=("x", "u"))
    O = oracle_lib.OracleLib(PU.oracle_kinds(problem, ddp)[0], problem, ddp)
    s = MPC.solver(problem, ddp, x0.shape[0], u0.shape[1], params, opts, lib_dir=SHAPE_LIB)
    for n in (0, 1, 3):
        d = s.solve(x0, u0)
        s.shift(n)
        assert np.array_equal(s.get("x0"), d["x"][:, n])
        s.run()
        got = s.download()
        want = O.solve_batch(d["x"][:, n], MPC.shifted(d["u"], n), params, {k: float(v) for k, v in opts.items()}, 1, want_traj=True)
        MPC.assert_logs(dict(got, result=got["success"]), want, f"{problem} shift {n}",
                        keys=("x", "u", "cost", "iterations", "result", "n_linesearch"))
    s.close()


@pytest.mark.parametrize("ddp", [0, 1])
@pytest.mark.parametrize("shape", ODD, ids=lambda s: f"{s[0]}x{s[1]}")
def test_policy(shape, ddp):
    """policy() gains are the oracle's calc_derivs + back_pass; policy_rollout is its forward pass at alpha 0 from each sample;
    policy_eval is the rollout's control"""
    problem = name_of(shape)
    x0, u0, params, opts = around_case(shape, ddp)
    B, T = u0.shape[:2]
    s = MPC.solver(problem, ddp, B, T, params, opts, lib_dir=SHAPE_LIB)
    s.upload(x0, u0)
    s.run()
    s.policy()
    got = dict(l=s.get("l"), L=s.get("L"), dV0=s.get("dV0"), dV1=s.get("dV1"), g_norm=s.get("g_norm"), policy_ok=s.get_int("policy_ok"))
    x0s = W.perturbed_states(x0, 4, 0.05, seed=97)
    x0s[:, 0] = s.get("x")[:, 0]
    r = s.policy_rollout(x0s, want_traj=True)
    O = policy_util.oracle(problem, ddp, os.path.join(SHAPE_ROOT, "problems"))
    checked = 0
    for b in range(B):
        o = policy_util.Solved(O, T, params, {k: float(v) for k, v in opts.items()}, x0[b], u0[b])
        ref = o.policy()
        assert got["policy_ok"][b] == ref["policy_ok"], b
        if ref["policy_ok"]:
            for k in ("l", "L", "dV0", "dV1", "g_norm"):
                assert np.array_equal(bits(got[k][b]), bits(ref[k])), (b, k)
            for i in range(x0s.shape[1]):
                rr = o.rollout(x0s[b, i])
                assert r["ok"][b, i] == rr["ok"], (b, i)
                if rr["ok"]:
                    checked += 1
                    for k in ("cost", "x_final", "x", "u"):
                        assert np.array_equal(r[k][b, i], rr[k]), (b, i, k)
        o.close()
    assert checked >= 2 * B
    ok = r["ok"].all(axis=1)
    for k in (0, T // 2, T - 1):
        u = s.policy_eval(k, r["x"][:, 1, k])
        assert np.array_equal(u[ok], r["u"][ok, 1, k]), k
    s.close()


@pytest.mark.parametrize("shape", ODD, ids=lambda s: f"{s[0]}x{s[1]}")
def test_three_chunks_match_one(shape):
    """chunks scatter and gather records of every length; a closed loop and policy rollouts over 3 chunks are those of 1"""
    problem = name_of(shape)
    x0, u0, params, opts = around_case(shape, 1, B=70)
    w = W.disturbance(x0.shape[0], 3, shape[0], 0.01, seed=99)
    x0s = W.perturbed_states(x0, 3, 0.05, seed=101)
    res = []
    for chunks in (1, 3):
        s = MPC.solver(problem, 1, x0.shape[0], u0.shape[1], params, opts, chunks=chunks, lib_dir=SHAPE_LIB)
        assert s.chunks() == chunks
        log = s.mpc(x0, u0, 3, w)
        final = s.download()
        s.policy()
        res.append((log, final, s.policy_rollout(x0s, want_traj=True)))
        s.close()
    (l1, f1, r1), (l3, f3, r3) = res
    MPC.assert_logs(l3, l1, f"{problem} chunks=3")
    MPC.assert_logs(f3, f1, f"{problem} chunks=3 final plan", keys=("x", "u", "cost"))
    for k in ("cost", "x_final", "ok", "x", "u"):
        assert np.array_equal(r3[k], r1[k], equal_nan=True), k
    assert len(np.unique(l1["iterations"])) > 1
