"""Closed loops against a plant that differs from the model (ilqgb_set_plant_param*, ilqgb_set_plant_substeps).  The controller
solves with the model's parameters; the next x0 is the plant stepped from the solve's x0 through the applied controls, each
held for n_sub sub-steps of clampU then f with the plant's parameters.  The oracle's plant step is the oracle with horizon n_sub
initialised at xp with u[j] repeated (tests/test_plant.py checks it against MMex modes 16 then 0).  That rollout evaluates
sub-step i at k = i where the device uses k = j; no problem's dynamics or input limits read a [k]-indexed parameter (only costs
and constraints of brachi_hli and cartrack do), so the two agree.  Every comparison is bit for bit."""
import ctypes as C

import numpy as np
import pytest

import ilqg_b200
import oracle_lib
import parity_util as PU
from ilqg_b200 import workloads as W

pytestmark = pytest.mark.gpu

LOG_KEYS = ("x", "u", "cost", "iterations", "success")
OUT_KEYS = ("x", "u", "cost", "iterations", "success", "n_linesearch")
CAR_OPTS = {"max_iter": 10}


def shifted(u, n=1):
    T = u.shape[1]
    return u[:, np.minimum(np.arange(T) + n, T - 1)]


def assert_same(a, b, what, keys=LOG_KEYS):
    for k in keys:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.shape == y.shape, f"{what}: {k} shape {x.shape} vs {y.shape}"
        assert np.array_equal(x, y, equal_nan=x.dtype.kind == "f"), f"{what}: {k} differs"


def per_problem(params, batch, b):
    """the parameter struct of problem b: shared values overridden by row b of the per-problem ones"""
    return dict(params, **{k: np.asarray(v)[b] for k, v in (batch or {}).items()})


def flat(lib, p):
    """the effective parameter vector of one problem in ilqgb_get "plant" order (non-[k] parameters in declaration order)"""
    return np.concatenate([np.asarray(p[n], dtype=float).ravel() for n, z in zip(lib.param_names, lib.param_sizes) if z != -1])


class Case:
    """model (shared + per-problem parameters, tracks), plant (shared + per-problem overrides, n_sub), inputs of one loop"""

    def __init__(self, problem, ddp, x0, u0, params, opts, S, w=None, model_batch=None, tracks=None, off=0,
                 plant=None, plant_batch=None, n_sub=1):
        self.problem, self.ddp, self.x0, self.u0, self.params, self.opts, self.S, self.w = problem, ddp, x0, u0, params, opts, S, w
        self.model_batch, self.tracks, self.off = model_batch or {}, tracks or {}, off
        self.plant, self.plant_batch, self.n_sub = plant or {}, plant_batch or {}, n_sub
        self.B, self.T = u0.shape[0], u0.shape[1]

    def model(self, b, step):
        p = per_problem(self.params, self.model_batch, b)
        return dict(p, **{k: v[b, self.off + step:self.off + step + self.T + 1] for k, v in self.tracks.items()})

    def plant_params(self, b, n_sub):
        p = dict(per_problem(self.params, self.model_batch, b), **self.plant)
        p = per_problem(p, self.plant_batch, b)
        return dict(p, **{k: np.zeros(n_sub + 1) for k in self.tracks})   # [k]-indexed: read by no dynamics or limit

    def solver(self, plant=True, flags=0, **kw):
        s = ilqg_b200.BatchSolver(self.problem, self.ddp, self.B, self.T, flags=flags, **kw)
        s.set_options(self.opts)
        s.set_params(self.params)
        if self.model_batch:
            s.set_params_batch(self.model_batch)
        for k, v in self.tracks.items():
            s.set_param_track(k, v)
        if self.off:
            s.set_track_offset(self.off)
        if plant:
            self.attach(s)
        return s

    def attach(self, s):
        s.set_plant_substeps(self.n_sub)
        s.set_plant_params(self.plant)
        s.set_plant_params_batch(self.plant_batch)

    def gpu(self, plant=True, **kw):
        s = self.solver(plant, **kw)
        log = s.mpc(self.x0, self.u0, self.S, self.w)
        final = s.download()
        s.close()
        return log, final


def oracle_plant(case, xp, u, n):
    """xp [B, nx] stepped through u[:, 0..n-1], n_sub oracle sub-steps per control"""
    O = oracle_lib.OracleLib(PU.oracle_kinds(case.problem, 0)[0], case.problem, 0)
    s = O.solver(case.n_sub)
    out = xp.copy()
    for b in range(case.B):
        s.set_params(case.plant_params(b, case.n_sub))
        for j in range(n):
            s.init(out[b], np.tile(u[b, j], (case.n_sub, 1)))
            out[b] = s.get("x")[case.n_sub]
    s.close()
    return out


def oracle_loop(case):
    """the reference once per step and problem with the model's parameters; x0 <- plant(x0, u[0]) + w[:, s]"""
    O = oracle_lib.OracleLib(PU.oracle_kinds(case.problem, case.ddp)[0], case.problem, case.ddp)
    opts = {k: float(v) for k, v in case.opts.items()}
    log = {k: [] for k in LOG_KEYS}
    x, u = case.x0.copy(), case.u0.copy()
    for st in range(case.S):
        rs = [O.solve_batch(x[b:b + 1], u[b:b + 1], case.model(b, st), opts, 1, want_traj=True) for b in range(case.B)]
        r = {k: np.concatenate([q[k] for q in rs]) for k in ("x", "u", "cost", "iterations", "result")}
        for k, v in zip(LOG_KEYS, (x, r["u"][:, 0], r["cost"], r["iterations"], r["result"])):
            log[k].append(v)
        x = oracle_plant(case, x, r["u"], 1)
        if case.w is not None:
            x = x + case.w[:, st]
        u = shifted(r["u"])
    log["x"].append(x)
    return {k: np.stack(v, axis=1) for k, v in log.items()}, dict(x=r["x"], u=r["u"])


def car_case(ddp, B=8, T=60, S=5, seed=201, w=False, **kw):
    x0, u0 = W.car_batch(B, T=T, seed=seed)
    return Case("car", ddp, x0, u0, W.CAR_PARAMS, CAR_OPTS, S, W.disturbance(B, S, 4, 0.01, seed=seed + 1) if w else None, **kw)


def make_case(name):
    if name == "car0_shared":
        return car_case(0, plant={"d": [2.2]})
    if name == "car1_batch_w":
        return car_case(1, seed=211, w=True, plant_batch=W.car_plant(8, 0.1, seed=212))
    if name == "car0_nsub4":
        return car_case(0, seed=221, plant={"h": [0.03 / 4]}, plant_batch=W.car_plant(8, 0.1, seed=222), n_sub=4)
    if name == "carhx0":
        x0, u0 = W.car_batch(8, T=60, seed=231)
        x0[:, 3] = np.linspace(-3.0, 3.0, 8)      # moving: the speed-dependent steering limit binds
        return Case("carhx", 0, x0, u0, W.CARHX_PARAMS, CAR_OPTS, 4, plant_batch={"kv": np.linspace(0.2, 1.5, 8)[:, None]})
    if name == "pend0":
        x0, u0 = W.pend_batch(8, T=100, seed=241)
        return Case("pend", 0, x0, u0, W.PEND_PARAMS, dict(W.PEND_OPTS, max_iter=30), 4, plant={"gl": [9.81 * 1.1], "dt": [0.01]},
                    n_sub=2)
    if name == "quad1":
        x0, u0 = W.quad_batch(3, T=100, seed=251)
        return Case("quad", 1, x0, u0, W.QUAD_PARAMS, {"max_iter": 10}, 3, plant_batch=W.quad_plant(3, 0.2, seed=252))
    if name.startswith("cartrack"):
        off, S, B, T = int(name[-1]), 4, 6, 60
        x0, u0, tr = W.cartrack_batch(B, T=T, extra=S + off, seed=261)
        params = dict(W.CARTRACK_PARAMS, **{k: v[0, :T + 1] for k, v in tr.items()})
        return Case("cartrack", 0, x0, u0, params, {"max_iter": 15}, S, tracks=tr, off=off,
                    plant_batch={"d": W.car_plant(B, 0.1, seed=262)["d"]})
    if name == "car0_follow":
        lim = np.stack([-1.0 - np.linspace(0, 1, 8), 1.0 + np.linspace(0, 1, 8)], axis=1)
        return car_case(0, seed=271, model_batch={"limA": lim}, plant={"d": [1.8]})
    raise KeyError(name)


# ---- 1. the reference once per step against the plant --------------------------------------------------------------------
@pytest.mark.parametrize("name", ["car0_shared", "car1_batch_w", "car0_nsub4", "carhx0", "pend0", "quad1", "cartrack0", "cartrack5",
                                  "car0_follow"])
def test_closed_loop_against_the_plant_is_the_reference(name):
    case = make_case(name)
    log, final = case.gpu()
    ora, ora_final = oracle_loop(case)
    assert_same(log, ora, name)
    assert_same(final, ora_final, name + " final plan", keys=("x", "u"))
    model, _ = case.gpu(plant=False)
    assert not np.array_equal(log["x"], model["x"])        # the plant is not the model (the car at rest: not in the first step)
    assert np.array_equal(log["x"][:, 0], model["x"][:, 0])


# ---- 2. a plant equal to the model ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["car0_shared", "car1_batch_w", "carhx0", "quad1"])
def test_identity_plant_is_no_plant(name):
    case = make_case(name)
    case.plant, case.plant_batch, case.n_sub = {}, {}, 1
    s = case.solver(plant=False)
    ref = s.mpc(case.x0, case.u0, case.S, case.w)
    ref_final = s.download()
    ok = np.all(ref["success"] != -1, axis=1)          # problems whose initial rollout failed go on from their nominal x[1]
    assert ok.sum() >= case.B // 2
    keep = lambda d: {k: v[ok] for k, v in d.items() if v is not None}
    full = {n: case.params[n] for n, z in zip(s.L.param_names, s.L.param_sizes) if z != -1}
    for what, setup in (("every entry set", lambda: (s.set_plant_substeps(1), s.set_plant_params(full))), ("nothing set", lambda: s.set_plant_substeps(1))):
        s.clear_plant()
        setup()
        got = s.mpc(case.x0, case.u0, case.S, case.w)
        assert_same(keep(got), keep(ref), f"{name} {what}")
        assert_same(keep(s.download()), keep(ref_final), f"{name} {what} final plan", keys=OUT_KEYS)
    s.set_plant_params({"d": [3.0]} if case.problem != "quad" else {"mass": [2.0]})
    s.clear_plant()          # x[1] + w again, bit for bit, also for problems whose initial rollout failed
    again = s.mpc(case.x0, case.u0, case.S, case.w)
    assert_same(again, ref, f"{name} after clear_plant")
    assert_same(s.download(), ref_final, f"{name} after clear_plant final plan", keys=OUT_KEYS)
    s.close()


# ---- 3. fused, stepwise and host loops -----------------------------------------------------------------------------------
def eval_batch(s, mode, x, u):
    L = s.lib
    L.ilqgb_eval.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    out = np.zeros((s.B, L.ilqgb_eval_size(mode)))
    x, u = np.ascontiguousarray(x), np.ascontiguousarray(u)
    s._chk(L.ilqgb_eval(s.h, mode, 0, x.ctypes.data, u.ctypes.data, out.ctypes.data))
    return out


@pytest.mark.parametrize("flags", [0, ilqg_b200.TRACE])
def test_fused_equals_stepwise_and_host_loop(flags):
    """mpc() = a loop of shift(1, w) + run() = the MATLAB loop: solve, then the plant stepped with single evaluations (mode 16
    clamp, mode 0 f) on a second handle that holds the plant's parameters"""
    case = car_case(0, B=40, S=5, seed=281, w=True, plant={"h": [0.015]}, plant_batch=W.car_plant(40, 0.1, seed=282), n_sub=2)
    fused, final = case.gpu(flags=flags)
    s = case.solver(flags=flags)
    s.upload(case.x0, case.u0)
    step = {k: [] for k in LOG_KEYS}
    for st in range(case.S):
        x = s.get("x0")
        s.run()
        d = s.download()
        for k, v in zip(LOG_KEYS, (x, d["u"][:, 0], d["cost"], d["iterations"], d["success"])):
            step[k].append(v)
        s.shift(1, w=case.w[:, st])
    step["x"].append(s.get("x0"))
    s.close()
    assert_same(fused, {k: np.stack(v, axis=1) for k, v in step.items()}, f"stepwise flags={flags}")
    ctl = case.solver(plant=False, flags=flags)
    plant = ilqg_b200.BatchSolver("car", 0, case.B, case.T)
    plant.set_params(dict(case.params, **case.plant))
    plant.set_params_batch(case.plant_batch)
    host = {k: [] for k in LOG_KEYS}
    x, u = case.x0.copy(), case.u0.copy()
    for st in range(case.S):
        d = ctl.solve(x, u)
        for k, v in zip(LOG_KEYS, (x, d["u"][:, 0], d["cost"], d["iterations"], d["success"])):
            host[k].append(v)
        for _ in range(case.n_sub):
            ua = eval_batch(plant, 16, x, d["u"][:, 0])
            x = eval_batch(plant, 0, x, ua)
        x = x + case.w[:, st]
        u = shifted(d["u"])
    host["x"].append(x)
    ctl.close()
    plant.close()
    assert_same(fused, {k: np.stack(v, axis=1) for k, v in host.items()}, f"host loop flags={flags}")
    assert_same(final, d, f"final plan flags={flags}", keys=OUT_KEYS)


# ---- 4. shift ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [0, 1, 7])
def test_shift_steps_the_plant_through_the_applied_controls(n):
    case = car_case(0, B=24, seed=291, plant_batch=W.car_plant(24, 0.1, seed=292), n_sub=3, plant={"h": [0.01]})
    w = W.disturbance(24, 1, 4, 0.01, seed=293)[:, 0]
    x_meas = W.car_batch(24, T=60, seed=294)[0]
    ref = case.solver(plant=False)
    s = case.solver()
    d = s.solve(case.x0, case.u0)
    xp = oracle_plant(case, case.x0, d["u"], n)
    for kw, x_new in (({}, xp), ({"w": w}, xp + w), ({"x0": x_meas}, x_meas)):
        s.solve(case.x0, case.u0)
        s.shift(n, **kw)
        assert np.array_equal(s.get("x0"), x_new), (n, list(kw))
        s.run()
        assert_same(s.download(), ref.solve(x_new, shifted(d["u"], n)), f"n={n} {list(kw)}", keys=OUT_KEYS)
    if n:
        assert not np.array_equal(xp, d["x"][:, n])
    s.close()
    ref.close()


# ---- 5. chunks and devices -----------------------------------------------------------------------------------------------
def chunk_case():
    lim = np.stack([-1.0 - np.linspace(0, 1, 77), 1.0 + np.linspace(0, 1, 77)], axis=1)
    return car_case(0, B=77, S=4, seed=301, w=True, model_batch={"limA": lim}, plant={"h": [0.015]},
                    plant_batch=W.car_plant(77, 0.1, seed=302), n_sub=2)


def expected_plant(case, lib):
    return np.stack([flat(lib, case.plant_params(b, 1)) for b in range(case.B)])


def test_chunks_match_one_stream():
    case = chunk_case()
    one, one_final = case.gpu(chunks=1)
    s = case.solver(chunks=3)
    assert s.chunks() == 3
    assert np.array_equal(s.get("plant"), expected_plant(case, s.L))
    three = s.mpc(case.x0, case.u0, case.S, case.w)
    three_final = s.download()
    s.close()
    assert_same(one, three, "chunks=3")
    assert_same(one_final, three_final, "chunks=3 final plan", keys=OUT_KEYS)
    assert len(np.unique(one["iterations"])) > 1


def test_devices_match_one_device():
    if ilqg_b200.Library("car", 0).device_count() < 2:
        pytest.skip("needs 2 GPUs")
    case = chunk_case()
    one, one_final = case.gpu()
    s = case.solver(devices=2)
    assert np.array_equal(s.get("plant"), expected_plant(case, s.L))
    two = s.mpc(case.x0, case.u0, case.S, case.w)
    two_final = s.download()
    s.close()
    assert_same(one, two, "devices=2")
    assert_same(one_final, two_final, "devices=2 final plan", keys=OUT_KEYS)


# ---- 6. entries never set follow the model -------------------------------------------------------------------------------
def test_unset_plant_entries_follow_the_model():
    case = car_case(0, B=40, S=3, seed=311, plant={"d": [2.2]})
    s = case.solver(chunks=2)
    lib = s.L
    assert np.array_equal(s.get("plant"), expected_plant(case, lib))
    case.params = dict(case.params, h=[0.025])
    s.set_params(case.params)
    case.model_batch = {"limW": np.stack([-0.3 - 0.01 * np.arange(40), 0.3 + 0.01 * np.arange(40)], axis=1)}
    s.set_params_batch(case.model_batch)
    want = expected_plant(case, lib)
    got = s.get("plant")
    assert np.array_equal(got, want)
    cols = np.cumsum([0] + [z for z in lib.param_sizes if z != -1])
    col = {n: slice(cols[i], cols[i + 1]) for i, n in enumerate(n for n, z in zip(lib.param_names, lib.param_sizes) if z != -1)}
    assert np.all(got[:, col["d"]] == 2.2) and np.all(got[:, col["h"]] == 0.025)
    assert np.array_equal(got[:, col["limW"]], case.model_batch["limW"])
    log = s.mpc(case.x0, case.u0, case.S)
    s.close()
    # the same plant with every entry set explicitly
    e = case.solver(plant=False)
    names = [n for n, z in zip(lib.param_names, lib.param_sizes) if z != -1]
    e.set_plant_substeps(1)
    e.set_plant_params_batch({n: want[:, col[n]] for n in names})
    assert np.array_equal(e.get("plant"), want)
    explicit = e.mpc(case.x0, case.u0, case.S)
    e.close()
    assert_same(log, explicit, "follow the model")
    ora, _ = oracle_loop(case)
    assert_same(log, ora, "follow the model vs reference")


# ---- 7. a plant that blows up ----------------------------------------------------------------------------------------------
def test_non_finite_plant_state_fails_that_problem_only():
    case = car_case(0, B=8, S=4, seed=321, w=True, plant_batch={"d": np.full((8, 1), 2.1)})
    good, _ = case.gpu()
    case.plant_batch = {"d": np.where(np.arange(8) == 2, 0.0, 2.1)[:, None]}     # d = 0: 0/0 in the heading update
    bad, _ = case.gpu()
    assert np.all(np.isnan(bad["x"][2, 1:]).any(axis=1))
    assert np.all(bad["success"][2, 1:] == -1) and good["success"][2, 1] != -1
    keep = np.arange(8) != 2
    assert_same({k: v[keep] for k, v in bad.items()}, {k: v[keep] for k, v in good.items()}, "other problems")


# ---- 8. rejected arguments -----------------------------------------------------------------------------------------------
def test_rejected_arguments_change_nothing():
    B, T = 4, 20
    x0, u0, tr = W.cartrack_batch(B, T=T, extra=4, seed=331)
    params = dict(W.CARTRACK_PARAMS, **{k: v[0, :T + 1] for k, v in tr.items()})
    s = ilqg_b200.BatchSolver("cartrack", 0, B, T)
    s.set_options({"max_iter": 5})
    s.set_params(params)
    s.set_plant_params({"d": [2.1]})
    ref = s.mpc(x0, u0, 3)
    plant = s.get("plant")
    L, h = s.lib, s.h
    names, sizes = s.L.param_names, s.L.param_sizes
    v = np.ones(B * 4)
    p = v.ctypes.data_as(C.c_void_p)
    bad = [(-1, 1), (len(names), 1), (names.index("xr"), T + 1), (names.index("yr"), 1), (names.index("d"), 2), (names.index("limA"), 1),
           (names.index("limA"), 0)]
    for setter in (L.ilqgb_set_plant_param, L.ilqgb_set_plant_param_batch):
        for i, n in bad:
            assert setter(h, i, p, n) == -1 and L.ilqgb_last_error(h).decode(), (setter, i, n)
        assert setter(h, names.index("d"), None, 1) == -1
    for n_sub in (0, -1, 65):
        assert L.ilqgb_set_plant_substeps(h, n_sub) == -1 and L.ilqgb_last_error(h).decode()
    assert np.array_equal(s.get("plant"), plant)
    assert_same(s.mpc(x0, u0, 3), ref, "after rejected calls")
    for call in (lambda: s.set_plant_params_batch({"d": np.ones((B + 1, 1))}), lambda: s.set_plant_params_batch({"limA": np.ones((B, 1))}),
                 lambda: s.set_plant_params_batch({"d": np.ones((B, 1, 1))})):
        with pytest.raises(ValueError):
            call()
    with pytest.raises(KeyError):
        s.set_plant_params({"nope": [1.0]})
    with pytest.raises(RuntimeError):
        s.set_plant_params({"xr": np.zeros(T + 1)})
    with pytest.raises(RuntimeError):
        s.set_plant_substeps(65)
    assert sizes[names.index("xr")] == -1
    s.close()
