"""Receding horizon on the device (ilqgb_shift, ilqgb_mpc).  One closed-loop step is one call of the reference with the
measured state as x0 and the previous solution, shifted by one step, as u0; the fused loop, the stepwise loop and a host loop
over solve() must all give the reference's results bit for bit."""
import ctypes as C

import numpy as np
import pytest

import ilqg_b200
import oracle_lib
import parity_util as PU
from ilqg_b200 import workloads as W

pytestmark = pytest.mark.gpu

LOG_KEYS = ("x", "u", "cost", "iterations", "success")


def shifted(u, n=1):
    """u[k + n] for k < T - n, then the last control: the MATLAB loop's u0 = [u(:,2:end) u(:,end)] for n = 1."""
    T = u.shape[1]
    return u[:, np.minimum(np.arange(T) + n, T - 1)]


def stack_logs(log):
    return {k: np.stack(v, axis=1) for k, v in log.items()}


def assert_logs(a, b, what, keys=LOG_KEYS):
    for k in keys:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.shape == y.shape, f"{what}: {k} shape {x.shape} vs {y.shape}"
        assert np.array_equal(x, y, equal_nan=x.dtype.kind == "f"), f"{what}: {k} differs"


def oracle_loop(problem, ddp, x0, u0, params, opts, S, w=None):
    """The reference called once per step (init + iLQG(), everything re-initialised): x0 <- x[1] + w[:, s], u0 <- shifted u."""
    O = oracle_lib.OracleLib(PU.oracle_kinds(problem, ddp)[0], problem, ddp)
    opts = {k: float(v) for k, v in opts.items()}
    log = {k: [] for k in LOG_KEYS}
    x0, u = x0.copy(), u0.copy()
    for s in range(S):
        r = O.solve_batch(x0, u, params, opts, 4, want_traj=True)
        for k, v in zip(LOG_KEYS, (x0, r["u"][:, 0], r["cost"], r["iterations"], r["result"])):
            log[k].append(v)
        x0 = r["x"][:, 1] + w[:, s] if w is not None else r["x"][:, 1]
        u = shifted(r["u"])
    log["x"].append(x0)
    return stack_logs(log), dict(x=r["x"], u=r["u"])


def solver(problem, ddp, B, T, params, opts, flags=0, tuning=None, **kw):
    s = ilqg_b200.BatchSolver(problem, ddp, B, T, flags=flags, **kw)
    s.set_options(opts)
    s.set_params(params)
    for k, v in (tuning or {}).items():
        s.set_tuning(k, v)
    return s


def gpu_mpc(problem, ddp, x0, u0, params, opts, S, w=None, **kw):
    s = solver(problem, ddp, x0.shape[0], u0.shape[1], params, opts, **kw)
    log = s.mpc(x0, u0, S, w)
    final = s.download()
    s.close()
    return log, final


def host_loop(problem, ddp, x0, u0, params, opts, S, w=None, **kw):
    """What a caller does without ilqgb_shift / ilqgb_mpc: solve, download, shift on the host, upload."""
    s = solver(problem, ddp, x0.shape[0], u0.shape[1], params, opts, **kw)
    log = {k: [] for k in LOG_KEYS}
    x, u = x0.copy(), u0.copy()
    for st in range(S):
        d = s.solve(x, u)
        for k, v in zip(LOG_KEYS, (x, d["u"][:, 0], d["cost"], d["iterations"], d["success"])):
            log[k].append(v)
        x = d["x"][:, 1] + w[:, st] if w is not None else d["x"][:, 1]
        u = shifted(d["u"])
    log["x"].append(x)
    s.close()
    return stack_logs(log), d


CAR_OPTS = {"max_iter": 10}


def _brachi_hli_case():
    params, x0, u0, opts = W.brachi_hli(100)
    B = 3
    return params, np.tile(x0, (B, 1)), u0[None] * (1.0 + 0.1 * np.arange(B))[:, None, None], opts


@pytest.mark.parametrize("case", ["car0", "car0_w", "car1", "car1_w", "car0_split4", "car0_split0", "pend0", "pend1", "brachi_hli", "quad1"])
def test_closed_loop_is_the_reference_called_once_per_step(case):
    tuning = None
    w = None
    if case.startswith("car"):
        problem, ddp, B, T, S = "car", int(case[3]), 8, 60, 6
        x0, u0 = W.car_batch(B, T=T, seed=101)
        params, opts = W.CAR_PARAMS, CAR_OPTS
        if case.endswith("_w"):
            w = W.disturbance(B, S, 4, 0.01, seed=102)
        if "split" in case:
            tuning = {"bp_split": int(case[-1])}
    elif case.startswith("pend"):
        problem, ddp, B, T, S = "pend", int(case[4]), 8, 100, 5
        x0, u0 = W.pend_batch(B, T=T, seed=103)
        params, opts = W.PEND_PARAMS, dict(W.PEND_OPTS, max_iter=30)
    elif case == "brachi_hli":
        problem, ddp, T, S = "brachi_hli", 0, 100, 3
        params, x0, u0, opts = _brachi_hli_case()
    else:
        problem, ddp, B, T, S = "quad", 1, 2, 100, 3
        x0, u0 = W.quad_batch(B, T=T, seed=104)
        params, opts = W.QUAD_PARAMS, {"max_iter": 10}
    log, final = gpu_mpc(problem, ddp, x0, u0, params, opts, S, w, tuning=tuning)
    ora, ora_final = oracle_loop(problem, ddp, x0, u0, params, opts, S, w)
    assert_logs(log, ora, case)
    assert_logs(final, ora_final, case + " final plan", keys=("x", "u"))
    assert not np.array_equal(log["x"][:, 0], log["x"][:, -1])    # the loop really moved the state


@pytest.mark.parametrize("flags", [0, ilqg_b200.TRACE])
def test_fused_equals_stepwise_and_host_loop(flags):
    """mpc() = a loop of shift(1, w) + run() (a start after a shift behaves like a fresh upload) = a host loop over solve()."""
    B, T, S = 40, 60, 5
    x0, u0 = W.car_batch(B, T=T, seed=111)
    w = W.disturbance(B, S, 4, 0.01, seed=112)
    fused, final = gpu_mpc("car", 0, x0, u0, W.CAR_PARAMS, CAR_OPTS, S, w, flags=flags)
    s = solver("car", 0, B, T, W.CAR_PARAMS, CAR_OPTS, flags=flags)
    s.upload(x0, u0)
    log = {k: [] for k in LOG_KEYS}
    for st in range(S):
        x = s.get("x0")
        s.run()
        d = s.download()
        for k, v in zip(LOG_KEYS, (x, d["u"][:, 0], d["cost"], d["iterations"], d["success"])):
            log[k].append(v)
        s.shift(1, w=w[:, st])
    log["x"].append(s.get("x0"))
    s.close()
    assert_logs(fused, stack_logs(log), f"stepwise flags={flags}")
    assert np.array_equal(log["x"][-1], d["x"][:, 1] + w[:, -1])
    host, host_final = host_loop("car", 0, x0, u0, W.CAR_PARAMS, CAR_OPTS, S, w, flags=flags)
    assert_logs(fused, host, f"host loop flags={flags}")
    assert_logs(final, host_final, f"final plan flags={flags}", keys=("x", "u", "cost", "iterations", "success"))


@pytest.mark.parametrize("n", [0, 1, 7, 60])
def test_shift_equals_uploading_the_host_shifted_solution(n):
    B, T = 24, 60
    x0, u0 = W.car_batch(B, T=T, seed=121)
    w = W.disturbance(B, 1, 4, 0.01, seed=122)[:, 0]
    x_meas = W.car_batch(B, T=T, seed=123)[0]
    ref = solver("car", 0, B, T, W.CAR_PARAMS, CAR_OPTS)
    s = solver("car", 0, B, T, W.CAR_PARAMS, CAR_OPTS)
    d = s.solve(x0, u0)
    for kw, x_new in (({}, d["x"][:, n]), ({"w": w}, d["x"][:, n] + w), ({"x0": x_meas}, x_meas)):
        s.solve(x0, u0)
        s.shift(n, **kw)
        assert np.array_equal(s.get("x0"), x_new), kw
        s.run()
        got = s.download()
        want = ref.solve(x_new, shifted(d["u"], n))
        assert_logs(got, want, f"n={n} {list(kw)}", keys=("x", "u", "cost", "iterations", "success", "n_linesearch"))
    s.close()
    ref.close()


def _chunk_case():
    B, T, S = 77, 60, 4
    x0, u0 = W.car_batch(B, T=T, seed=131)
    return x0, u0, W.disturbance(B, S, 4, 0.01, seed=132), S


def test_chunks_match_one_stream():
    """Chunks (whole warps, so ragged sizes) run their closed loops independently; the logs are those of one stream."""
    x0, u0, w, S = _chunk_case()
    one, one_final = gpu_mpc("car", 0, x0, u0, W.CAR_PARAMS, CAR_OPTS, S, w, chunks=1)
    s = solver("car", 0, x0.shape[0], u0.shape[1], W.CAR_PARAMS, CAR_OPTS, chunks=3)
    assert s.chunks() == 3
    three = s.mpc(x0, u0, S, w)
    three_final = s.download()
    s.close()
    assert_logs(one, three, "chunks=3")
    assert_logs(one_final, three_final, "chunks=3 final plan", keys=("x", "u", "cost"))
    assert len(np.unique(one["iterations"])) > 1     # ragged convergence: the chunks really run different numbers of passes


def test_devices_match_one_device():
    if ilqg_b200.Library("car", 0).device_count() < 2:
        pytest.skip("needs 2 GPUs")
    x0, u0, w, S = _chunk_case()
    one, one_final = gpu_mpc("car", 0, x0, u0, W.CAR_PARAMS, CAR_OPTS, S, w)
    two, two_final = gpu_mpc("car", 0, x0, u0, W.CAR_PARAMS, CAR_OPTS, S, w, devices=2)
    assert_logs(one, two, "devices=2")
    assert_logs(one_final, two_final, "devices=2 final plan", keys=("x", "u", "cost"))


def test_failing_problem_applies_what_its_nominal_holds():
    """A problem whose initial rollout turns non-finite (result -1) goes on from whatever its nominal trajectory holds, as a
    host loop over solve() would; the other problems of the batch are not affected."""
    B, T, S = 8, 30, 4
    x0, u0 = W.car_batch(B, T=T, seed=141)
    w = W.disturbance(B, S, 4, 0.01, seed=142)
    bad = x0.copy()
    bad[2, 3] = 1e4    # speed so large that sqrt(d^2 - (h v sin w)^2) is NaN (test_gpu_edge.py)
    log, final = gpu_mpc("car", 0, bad, u0, W.CAR_PARAMS, CAR_OPTS, S, w)
    host, host_final = host_loop("car", 0, bad, u0, W.CAR_PARAMS, CAR_OPTS, S, w)
    assert log["success"][2, 0] == -1
    assert_logs(log, host, "failing problem vs host loop")
    assert_logs(final, host_final, "failing problem final plan", keys=("x", "u", "cost", "iterations", "success"))
    clean, _ = gpu_mpc("car", 0, x0, u0, W.CAR_PARAMS, CAR_OPTS, S, w)
    keep = np.arange(B) != 2
    assert_logs({k: v[keep] for k, v in log.items()}, {k: v[keep] for k, v in clean.items()}, "other problems")


def test_rejected_arguments():
    B, T = 4, 20
    x0, u0 = W.car_batch(B, T=T, seed=151)
    s = solver("car", 0, B, T, W.CAR_PARAMS, CAR_OPTS)
    L, h = s.lib, s.h
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    w1, ws = np.zeros((B, 4)), np.zeros((B, 2, 4))

    def rejected(rc):
        assert rc == -1 and L.ilqgb_last_error(h).decode()

    s.upload(x0, u0)
    rejected(L.ilqgb_shift(h, 1, None, None))                       # no start since the upload
    s.run()
    rejected(L.ilqgb_shift(h, -1, None, None))
    rejected(L.ilqgb_shift(h, T + 1, None, None))
    rejected(L.ilqgb_shift(h, 1, p(x0), p(w1)))                     # w is added to the solution's state, not to a given x0
    rejected(L.ilqgb_mpc(h, 2, None, None, None, None, None, None, None, None))   # nothing to continue from after a solve
    assert L.ilqgb_shift(h, 1, None, None) == 0
    rejected(L.ilqgb_shift(h, 1, None, None))                       # a shift needs a start since the last shift
    rejected(L.ilqgb_mpc(h, 0, p(x0), p(u0), None, None, None, None, None, None))
    rejected(L.ilqgb_mpc(h, 2, p(x0), None, None, None, None, None, None, None))
    rejected(L.ilqgb_mpc(h, 2, None, p(u0), None, None, None, None, None, None))
    assert L.ilqgb_mpc(h, 2, None, None, p(ws), None, None, None, None, None) == 0   # continues from the shift
    for call in (lambda: s.mpc(x0[:, :3], u0, 2), lambda: s.mpc(x0, u0[:, :-1], 2), lambda: s.mpc(x0, u0, 2, w=ws[:, :1]),
                 lambda: s.mpc(x0, None, 2), lambda: s.shift(1, x0=x0[:-1]), lambda: s.shift(1, w=ws)):
        with pytest.raises(ValueError):
            call()
    s.close()
