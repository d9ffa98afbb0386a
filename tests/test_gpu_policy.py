"""Feedback policy of a solved batch (ilqgb_policy, ilqgb_policy_rollout, ilqgb_policy_eval), bit for bit against the oracle.
The gains are the reference's calc_derivs + back_pass on the tOptSet iLQG() left behind; a rollout is forward_pass's feedback
branch at alpha = 0 from another initial state (tests/policy_util.py), with the plant's parameters where the handle has one."""
import numpy as np
import pytest

import ilqg_b200
import policy_util
from ilqg_b200 import workloads as W

pytestmark = pytest.mark.gpu

UNTOUCHED_F = ("x", "u", "cost", "lambda", "dlambda", "w_pen_l", "w_pen_f", "mu_r", "mu_f")
UNTOUCHED_I = ("iterations", "result", "status", "cur")


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def same_bits(a, b):
    return np.array_equal(bits(a), bits(b))


class Case:
    def __init__(self, problem, ddp, x0, u0, params, opts, model_batch=None, tracks=None, off=0, plant=None, plant_batch=None):
        self.problem, self.ddp, self.x0, self.u0, self.params, self.opts = problem, ddp, x0, u0, params, opts
        self.model_batch, self.tracks, self.off = model_batch or {}, tracks or {}, off
        self.plant, self.plant_batch = plant or {}, plant_batch or {}
        self.B, self.T = u0.shape[0], u0.shape[1]

    def model(self, b):
        p = dict(self.params, **{k: np.asarray(v)[b] for k, v in self.model_batch.items()})
        return dict(p, **{k: v[b, self.off:self.off + self.T + 1] for k, v in self.tracks.items()})

    def plant_params(self, b):
        p = dict(self.model(b), **self.plant)
        return dict(p, **{k: np.asarray(v)[b] for k, v in self.plant_batch.items()})

    def solver(self, **kw):
        s = ilqg_b200.BatchSolver(self.problem, self.ddp, self.B, self.T, **kw)
        s.set_options(self.opts)
        s.set_params(self.params)
        if self.model_batch:
            s.set_params_batch(self.model_batch)
        for k, v in self.tracks.items():
            s.set_param_track(k, v)
        if self.off:
            s.set_track_offset(self.off)
        if self.plant or self.plant_batch:
            s.set_plant_params(self.plant)
            s.set_plant_params_batch(self.plant_batch)
        return s

    def solved(self, **kw):
        s = self.solver(**kw)
        s.upload(self.x0, self.u0)
        s.run()
        return s

    def oracle(self, b):
        return policy_util.Solved(policy_util.oracle(self.problem, self.ddp), self.T, self.model(b), {k: float(v) for k, v in self.opts.items()},
                                  self.x0[b], self.u0[b])


def make_case(name, B=6, T=60):
    if name in ("car0", "car1"):
        x0, u0 = W.car_batch(B, T=T, seed=301)
        return Case("car", int(name[-1]), x0, u0, W.CAR_PARAMS, {"max_iter": 10})
    if name == "car0_plant":
        x0, u0 = W.car_batch(B, T=T, seed=302)
        return Case("car", 0, x0, u0, W.CAR_PARAMS, {"max_iter": 10}, plant={"d": [2.2], "limA": [-1.0, 1.0]})
    if name == "car1_plant_batch":
        x0, u0 = W.car_batch(B, T=T, seed=303)
        return Case("car", 1, x0, u0, W.CAR_PARAMS, {"max_iter": 10}, plant_batch=W.car_plant(B, 0.2, seed=304))
    if name == "car0_follow":
        x0, u0 = W.car_batch(B, T=T, seed=305)
        lim = np.stack([-1.0 - np.linspace(0, 1, B), 1.0 + np.linspace(0, 1, B)], axis=1)
        return Case("car", 0, x0, u0, W.CAR_PARAMS, {"max_iter": 10}, model_batch={"limA": lim}, plant={"d": [1.8]})
    if name == "carhx0":
        x0, u0 = W.car_batch(B, T=T, seed=306)
        x0[:, 3] = np.linspace(-3.0, 3.0, B)      # moving: the speed-dependent steering limit binds
        return Case("carhx", 0, x0, u0, W.CARHX_PARAMS, {"max_iter": 10})
    if name == "pend0":
        x0, u0 = W.pend_batch(B, T=T, seed=307)
        return Case("pend", 0, x0, u0, W.PEND_PARAMS, dict(W.PEND_OPTS, max_iter=30))
    if name == "brachi_hli0":
        params, bx0, bu0, opts = W.brachi_hli(T)
        x0 = np.repeat(bx0[None], B, 0) * (1 + np.arange(B))[:, None]
        u0 = np.repeat(bu0[None], B, 0) * (1 + 0.1 * np.arange(B))[:, None, None]
        return Case("brachi_hli", 0, x0, u0, params, opts)
    if name == "quad1":
        x0, u0 = W.quad_batch(3, T=T, seed=308)
        return Case("quad", 1, x0, u0, W.QUAD_PARAMS, {"max_iter": 8})
    if name.startswith("cartrack"):
        off = int(name[-1])
        x0, u0, tr = W.cartrack_batch(B, T=T, extra=off, seed=309)
        params = dict(W.CARTRACK_PARAMS, **{k: v[0, :T + 1] for k, v in tr.items()})
        return Case("cartrack", 0, x0, u0, params, {"max_iter": 15}, tracks=tr, off=off)
    raise KeyError(name)


def snapshot(s):
    return {**{k: s.get(k) for k in UNTOUCHED_F}, **{k: s.get_int(k) for k in UNTOUCHED_I}, "download": s.download()}


def assert_snapshot(a, b, what):
    for k in UNTOUCHED_F + UNTOUCHED_I:
        assert same_bits(a[k], b[k]) if k in UNTOUCHED_F else np.array_equal(a[k], b[k]), f"{what}: {k} changed"
    for k, v in a["download"].items():
        assert np.array_equal(v, b["download"][k], equal_nan=True), f"{what}: download {k} changed"


# ---- 1. gains ---------------------------------------------------------------------------------------------------------------
GAIN_CASES = [("car0", 0), ("car0", 4), ("car1", 0), ("car1", 4), ("carhx0", 0), ("pend0", 0), ("pend0", 4), ("brachi_hli0", 0),
              ("brachi_hli0", 4), ("quad1", 0), ("cartrack0", 0), ("cartrack0", 4), ("cartrack5", 0), ("cartrack5", 4)]


@pytest.mark.parametrize("name,split", GAIN_CASES)
def test_policy_gains_are_calc_derivs_and_back_pass(name, split):
    case = make_case(name)
    s = case.solved()
    before = snapshot(s)
    s.set_tuning("bp_split", split)
    s.policy()
    if case.problem in ("car", "pend", "brachi_hli", "cartrack"):
        assert (s.get_int("bp_split") == split).all()
    assert_snapshot(snapshot(s), before, name)
    got = dict(l=s.get("l"), L=s.get("L"), dV0=s.get("dV0"), dV1=s.get("dV1"), g_norm=s.get("g_norm"), bp_done=s.get_int("bp_done"),
               policy_ok=s.get_int("policy_ok"))
    ran = 0
    for b in range(case.B):
        o = case.oracle(b)
        assert o.init_ok, (name, b)
        ref = o.policy()
        o.close()
        assert got["policy_ok"][b] == ref["policy_ok"] and got["bp_done"][b] == ref["bp_done"], (name, b)
        if not ref["policy_ok"]:
            continue
        ran += 1
        for k in ("l", "L"):
            assert same_bits(got[k][b], ref[k]), (name, b, k)
        for k in ("dV0", "dV1", "g_norm"):
            assert same_bits(got[k][b], ref[k]), (name, b, k)
    assert ran >= case.B // 2
    s.close()


# ---- 2. rollouts against the oracle ---------------------------------------------------------------------------------------------
ROLLOUT_CASES = ["car0", "car1", "car0_plant", "car1_plant_batch", "car0_follow", "carhx0", "pend0", "quad1", "cartrack5"]


def perturbed(case, s, M, seed):
    x0s = W.perturbed_states(case.x0, M, 0.05, seed=seed)
    x0s[:, 0] = s.get("x")[:, 0]
    return x0s


@pytest.mark.parametrize("name", ROLLOUT_CASES)
def test_policy_rollouts_are_the_oracle(name):
    case = make_case(name)
    s = case.solved()
    s.policy()
    before = snapshot(s)
    x0s = perturbed(case, s, 5, seed=401)
    r = s.policy_rollout(x0s, want_traj=True)
    assert_snapshot(snapshot(s), before, name)         # the handle is untouched
    nom = before["download"]
    ok_b = s.get_int("policy_ok")
    plant = bool(case.plant or case.plant_batch)
    checked = 0
    for b in range(case.B):
        if not ok_b[b]:
            assert (r["ok"][b] == 0).all() and np.isnan(r["cost"][b]).all()
            continue
        if not plant:      # sample 0 starts at x*_0: the plan itself
            assert np.array_equal(r["x"][b, 0], nom["x"][b]) and np.array_equal(r["u"][b, 0], nom["u"][b]), (name, b)
        o = case.oracle(b)
        o.policy()
        if plant:
            o.set_params(case.plant_params(b))
        for i in range(x0s.shape[1]):
            ref = o.rollout(x0s[b, i])
            assert r["ok"][b, i] == ref["ok"], (name, b, i)
            if not ref["ok"]:
                continue
            checked += 1
            for k in ("cost", "x_final", "x", "u"):
                assert same_bits(r[k][b, i], ref[k]), (name, b, i, k)
        o.close()
    assert checked >= 2 * case.B
    assert not np.array_equal(r["u"][:, 1], nom["u"])       # the perturbed samples move off the plan
    s.close()


# ---- 3. the control law on its own -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["car0", "carhx0", "cartrack5"])
def test_policy_eval_is_the_rollouts_control(name):
    case = make_case(name)
    s = case.solved()
    s.policy()
    r = s.policy_rollout(perturbed(case, s, 2, seed=402), want_traj=True)
    ok = r["ok"].all(axis=1)
    assert ok.sum() >= case.B // 2
    for i in range(2):
        for k in range(case.T):
            u = s.policy_eval(k, r["x"][:, i, k])
            assert same_bits(u[ok], r["u"][ok, i, k]), (name, i, k)
    s.close()


# ---- 4. groups, chunks and devices ----------------------------------------------------------------------------------------------
def test_policy_rollout_groups_chunks_and_devices(monkeypatch):
    B, T, M = 96, 40, 7
    case = make_case("car0_plant", B=B, T=T)
    s = case.solved()
    s.policy()
    x0s = W.perturbed_states(case.x0, M, 0.05, seed=403)
    full = s.policy_rollout(x0s, want_traj=True)
    keys = ("cost", "x_final", "ok")
    bare = s.policy_rollout(x0s)
    for k in keys:
        assert np.array_equal(bare[k], full[k], equal_nan=True), k
    monkeypatch.setenv("ILQG_POLICY_STAGE", str(B * 3 * (10 + (T + 1) * 4 + T * 2)))   # groups of 3 samples, the last one of 1
    grouped = s.policy_rollout(x0s, want_traj=True)
    monkeypatch.delenv("ILQG_POLICY_STAGE")
    for k in keys + ("x", "u"):
        assert np.array_equal(grouped[k], full[k], equal_nan=True), k
    assert full["ok"].sum() >= B * M // 2
    s.close()
    s3 = case.solved(chunks=3)
    assert s3.chunks() == 3
    s3.policy()
    three = s3.policy_rollout(x0s, want_traj=True)
    s3.close()
    for k in keys + ("x", "u"):
        assert np.array_equal(three[k], full[k], equal_nan=True), k
    if ilqg_b200.Library("car", 0).device_count() < 2:
        pytest.skip("one GPU: the two-device comparison needs two")
    s2 = case.solved(devices=2)
    s2.policy()
    two = s2.policy_rollout(x0s, want_traj=True)
    s2.close()
    for k in keys + ("x", "u"):
        assert np.array_equal(two[k], full[k], equal_nan=True), k


# ---- 5. failures ---------------------------------------------------------------------------------------------------------------
def test_failed_problem_has_no_policy_and_leaves_the_others():
    case = make_case("car0")
    bad = make_case("car0")
    bad.x0 = bad.x0.copy()
    bad.x0[2] = np.nan                     # the initial rollout fails: result -1
    x0s = W.perturbed_states(case.x0, 4, 0.05, seed=404)
    outs = []
    for c in (case, bad):
        s = c.solved()
        s.policy()
        outs.append((s.download(), s.get_int("policy_ok"), s.policy_rollout(x0s, want_traj=True)))
        s.close()
    (d0, ok0, r0), (d1, ok1, r1) = outs
    assert d1["success"][2] == -1 and ok1[2] == 0 and ok0[2] == 1
    assert (r1["ok"][2] == 0).all() and np.isnan(r1["cost"][2]).all() and np.isnan(r1["x_final"][2]).all()
    assert np.isnan(r1["x"][2]).all() and np.isnan(r1["u"][2]).all()
    keep = np.arange(case.B) != 2
    for k in ("cost", "x_final", "ok", "x", "u"):
        assert same_bits(r1[k][keep], r0[k][keep]), k


# ---- 6. rejected arguments ----------------------------------------------------------------------------------------------------
def test_rejected_arguments_change_nothing():
    case = make_case("car0")
    s = case.solved()
    with pytest.raises(RuntimeError, match="ilqgb_policy"):          # no policy yet
        s.policy_rollout(W.perturbed_states(case.x0, 2, 0.05, seed=405))
    s.policy()
    x0s = W.perturbed_states(case.x0, 3, 0.05, seed=405)
    ref = s.policy_rollout(x0s, want_traj=True)
    before = snapshot(s)
    with pytest.raises(RuntimeError, match="M must be"):
        s.policy_rollout(np.zeros((case.B, 0, 4)))
    for bad in (np.zeros((case.B, 3)), np.zeros((case.B + 1, 3, 4)), np.zeros((case.B, 3, 5))):
        with pytest.raises(ValueError):
            s.policy_rollout(bad)
    with pytest.raises(ValueError):
        s.policy_eval(0, np.zeros((case.B, 5)))
    for k in (-1, case.T):
        with pytest.raises(RuntimeError, match="k must be"):
            s.policy_eval(k, np.zeros((case.B, 4)))
    s.set_plant_substeps(2)
    with pytest.raises(RuntimeError, match="n_sub"):
        s.policy_rollout(x0s)
    s.clear_plant()
    assert_snapshot(snapshot(s), before, "after rejected calls")
    again = s.policy_rollout(x0s, want_traj=True)
    for k in ref:
        assert same_bits(again[k], ref[k]), k
    # stale: after an upload, a shift or a closed loop
    for stale in (lambda: s.upload(case.x0, case.u0), lambda: (s.run(), s.shift(1)), lambda: s.mpc(case.x0, case.u0, 2)):
        s.upload(case.x0, case.u0)
        s.run()
        s.policy()
        s.policy_rollout(x0s)
        stale()
        with pytest.raises(RuntimeError, match="ilqgb_policy"):
            s.policy_rollout(x0s)
        with pytest.raises(RuntimeError, match="ilqgb_policy"):
            s.policy_eval(0, case.x0)
    s.close()
