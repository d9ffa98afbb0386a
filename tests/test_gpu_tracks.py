"""Per-problem time-indexed parameter tracks (ilqgb_set_param_track).  A solve with tracks at offset `off` is, for every
problem b, the reference called with name[k] = track[b, off + k]; in a closed loop the window moves one step per shift.
Every comparison is bit for bit."""
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


def shifted(u, n=1):
    T = u.shape[1]
    return u[:, np.minimum(np.arange(T) + n, T - 1)]


def assert_same(a, b, what, keys):
    for k in keys:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.shape == y.shape, f"{what}: {k} shape {x.shape} vs {y.shape}"
        assert np.array_equal(x, y, equal_nan=x.dtype.kind == "f"), f"{what}: {k} differs"


def brachi_hli_case(B, T, extra):
    """brachi_hli with a different ymin track per problem (the demo's ramp, moved up or down and extended at -4)."""
    params, x0, u0, opts = W.brachi_hli(T)
    ramp = np.concatenate([params["ymin"][:T], np.full(extra + 1, -4.0)])
    tracks = {"ymin": ramp[None, :] + 0.05 * np.arange(B)[:, None]}
    params = dict(params, ymin=tracks["ymin"][0, :T + 1])
    return params, np.tile(x0, (B, 1)), np.tile(u0[None], (B, 1, 1)), dict(opts, max_iter=20.0), tracks


def case(problem, B, T, extra, seed=11):
    """(params with shared [k] values, x0, u0, opts, tracks) of a tracking batch"""
    if problem == "cartrack":
        x0, u0, tr = W.cartrack_batch(B, T=T, extra=extra, seed=seed)
        params = dict(W.CARTRACK_PARAMS, **{k: v[0, :T + 1] for k, v in tr.items()})
        return params, x0, u0, {"max_iter": 15.0}, tr
    return brachi_hli_case(B, T, extra)


def window(params, tracks, b, off, T):
    return dict(params, **{k: v[b, off:off + T + 1] for k, v in tracks.items()})


def solver(problem, ddp, B, T, params, opts, tracks, flags=0, tuning=None, **kw):
    s = ilqg_b200.BatchSolver(problem, ddp, B, T, flags=flags, **kw)
    s.set_options(opts)
    s.set_params(params)
    for k, v in tracks.items():
        s.set_param_track(k, v)
    for k, v in (tuning or {}).items():
        s.set_tuning(k, v)
    return s


def gpu_records(s, x0, u0):
    """per-problem records shaped like parity_util.oracle_record (TRACE handle)"""
    out = s.solve(x0, u0)
    sc = {k: s.get(k) for k in ("lambda", "g_norm", "w_pen_l", "w_pen_f")}
    tr_l, tr_c, tr_a, nbp = s.get("tr_lambda"), s.get("tr_newcost"), s.get_int("tr_alpha"), s.get_int("n_backpass")
    recs = []
    for b in range(s.B):
        n = int(out["n_linesearch"][b])
        recs.append(dict(result=int(out["success"][b]), iterations=int(out["iterations"][b]), cost=out["cost"][b], x=out["x"][b],
                         u=out["u"][b], n_ls=n, n_bp=int(nbp[b]), tr_lambda=tr_l[b][:n], tr_alpha=tr_a[b][:n], tr_newcost=tr_c[b][:n],
                         **{k: v[b] for k, v in sc.items()}))
    return recs


# ---- 1. single solves ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tail_from", [0, 2, 8])
@pytest.mark.parametrize("off", [0, 7])
@pytest.mark.parametrize("problem,ddp", [("cartrack", 0), ("cartrack", 1), ("brachi_hli", 0)])
def test_single_solve_reads_the_window_of_each_problem(problem, ddp, off, tail_from):
    B, T = 6, 60
    params, x0, u0, opts, tracks = case(problem, B, T, extra=10)
    s = solver(problem, ddp, B, T, params, opts, tracks, flags=ilqg_b200.TRACE, tuning={"ls_tail_from": tail_from})
    s.set_track_offset(off)
    recs = gpu_records(s, x0, u0)
    s.close()
    kind = PU.oracle_kinds(problem, ddp)[0]
    for b in range(B):
        ora = PU.oracle_record(kind, problem, ddp, T, window(params, tracks, b, off, T), x0[b], u0[b], opts)
        PU.assert_same(recs[b], ora, f"{problem} ddp{ddp} off {off} tail {tail_from} problem {b}")


# ---- 2. identical tracks are the shared parameter -----------------------------------------------------------------------
@pytest.mark.parametrize("problem,ddp", [("cartrack", 0), ("brachi_hli", 0)])
def test_identical_tracks_match_the_shared_parameter(problem, ddp):
    B, T = 40, 50
    params, x0, u0, opts, tracks = case(problem, B, T, extra=0)
    same = {k: np.tile(np.asarray(params[k], dtype=float)[None], (B, 1)) for k in tracks}
    s = solver(problem, ddp, B, T, params, opts, {})
    ref = s.solve(x0, u0)
    s.close()
    s = solver(problem, ddp, B, T, params, opts, same)
    out = s.solve(x0, u0)
    s.close()
    assert_same(out, ref, problem, OUT_KEYS)


# ---- 3. closed loops ----------------------------------------------------------------------------------------------------
def oracle_loop(problem, ddp, x0, u0, params, opts, tracks, S, w=None, off=0):
    """The reference once per step and problem, step s reading the window track[b, off + s : off + s + T + 1]."""
    O = oracle_lib.OracleLib(PU.oracle_kinds(problem, ddp)[0], problem, ddp)
    opts = {k: float(v) for k, v in opts.items()}
    B, T = u0.shape[0], u0.shape[1]
    log = {k: [] for k in LOG_KEYS}
    x, u = x0.copy(), u0.copy()
    for st in range(S):
        rs = [O.solve_batch(x[b:b + 1], u[b:b + 1], window(params, tracks, b, off + st, T), opts, 1, want_traj=True) for b in range(B)]
        r = {k: np.concatenate([q[k] for q in rs]) for k in ("x", "u", "cost", "iterations", "result")}
        for k, v in zip(LOG_KEYS, (x, r["u"][:, 0], r["cost"], r["iterations"], r["result"])):
            log[k].append(v)
        x = r["x"][:, 1] + w[:, st] if w is not None else r["x"][:, 1]
        u = shifted(r["u"])
    log["x"].append(x)
    return {k: np.stack(v, axis=1) for k, v in log.items()}, dict(x=r["x"], u=r["u"])


@pytest.mark.parametrize("name", ["cartrack0", "cartrack0_w", "cartrack1", "cartrack1_w", "cartrack0_split0", "cartrack0_split4", "brachi_hli"])
def test_closed_loop_is_the_reference_on_a_moving_window(name):
    problem = "brachi_hli" if name == "brachi_hli" else "cartrack"
    ddp = 0 if problem == "brachi_hli" else int(name[8])
    B, T, S = 8, 50, 5
    params, x0, u0, opts, tracks = case(problem, B, T, extra=S - 1)
    w = W.disturbance(B, S, x0.shape[1], 0.01, seed=12) if name.endswith("_w") else None
    tuning = {"bp_split": int(name[-1])} if "split" in name else None
    s = solver(problem, ddp, B, T, params, opts, tracks, tuning=tuning)
    log = s.mpc(x0, u0, S, w)
    final = s.download()
    assert s.track_offset() == S - 1
    s.close()
    ora, ora_final = oracle_loop(problem, ddp, x0, u0, params, opts, tracks, S, w)
    assert_same(log, ora, name, LOG_KEYS)
    assert_same(final, ora_final, name + " final plan", ("x", "u"))


# ---- 4. three ways to run a loop ----------------------------------------------------------------------------------------
def test_fused_stepwise_and_host_loops_agree():
    B, T, S = 32, 50, 5
    params, x0, u0, opts, tracks = case("cartrack", B, T, extra=S - 1)
    w = W.disturbance(B, S, 4, 0.01, seed=13)
    s = solver("cartrack", 0, B, T, params, opts, tracks)
    fused = s.mpc(x0, u0, S, w)
    s.close()

    s = solver("cartrack", 0, B, T, params, opts, tracks)
    s.upload(x0, u0)
    step = {k: [] for k in LOG_KEYS}
    x = x0.copy()
    for st in range(S):
        s.run()
        d = s.download()
        for k, v in zip(LOG_KEYS, (x, d["u"][:, 0], d["cost"], d["iterations"], d["success"])):
            step[k].append(v)
        x = d["x"][:, 1] + w[:, st]
        if st < S - 1:
            s.shift(1, w=w[:, st])
    step["x"].append(x)
    assert s.track_offset() == S - 1
    s.close()

    s = solver("cartrack", 0, B, T, params, opts, tracks)
    host = {k: [] for k in LOG_KEYS}
    x, u = x0.copy(), u0.copy()
    for st in range(S):
        s.set_track_offset(st)
        d = s.solve(x, u)
        for k, v in zip(LOG_KEYS, (x, d["u"][:, 0], d["cost"], d["iterations"], d["success"])):
            host[k].append(v)
        x = d["x"][:, 1] + w[:, st]
        u = shifted(d["u"])
    host["x"].append(x)
    s.close()
    step = {k: np.stack(v, axis=1) for k, v in step.items()}
    host = {k: np.stack(v, axis=1) for k, v in host.items()}
    assert_same(step, fused, "shift + run", LOG_KEYS)
    assert_same(host, fused, "host loop", LOG_KEYS)


# ---- 5. chunks advance their windows on their own -----------------------------------------------------------------------
def test_three_chunks_equal_one_stream():
    B, T, S = 96, 50, 5
    params, x0, u0, opts, tracks = case("cartrack", B, T, extra=S - 1)
    logs = []
    for chunks in (1, 3):
        s = solver("cartrack", 0, B, T, params, opts, tracks, chunks=chunks)
        assert s.chunks() == chunks
        logs.append((s.mpc(x0, u0, S), s.download()))
        assert s.track_offset() == S - 1
        s.close()
    assert_same(logs[1][0], logs[0][0], "3 chunks", LOG_KEYS)
    assert_same(logs[1][1], logs[0][1], "3 chunks final plan", ("x", "u"))
    it = logs[0][0]["iterations"]
    assert len(np.unique(it)) > 1, "every problem took the same number of iterations: the chunks would finish together"


# ---- 6. a tracked and a shared [k]-indexed parameter -------------------------------------------------------------------
def test_mixed_tracked_and_shared_parameters():
    B, T, S = 8, 50, 4
    params, x0, u0, opts, tracks = case("cartrack", B, T, extra=S - 1)
    only_x = {"xr": tracks["xr"]}
    s = solver("cartrack", 0, B, T, params, opts, only_x)
    log = s.mpc(x0, u0, S)
    s.close()
    # yr stays params["yr"] at every step: it does not move with the window
    ora, _ = oracle_loop("cartrack", 0, x0, u0, params, opts, only_x, S)
    assert_same(log, ora, "xr tracked, yr shared", LOG_KEYS)

    # set_param on the tracked index makes it shared again: today's results
    s = solver("cartrack", 0, B, T, params, opts, tracks)
    s.set_track_offset(3)
    s.set_params(params)
    out = s.solve(x0, u0)
    s.close()
    s = solver("cartrack", 0, B, T, params, opts, {})
    ref = s.solve(x0, u0)
    s.close()
    assert_same(out, ref, "track dropped", OUT_KEYS)


# ---- 7. single evaluations ----------------------------------------------------------------------------------------------
def evaluate(s, mode, k, x, u):
    L = s.lib
    L.ilqgb_eval_size.argtypes = [C.c_int]
    L.ilqgb_eval.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    out = np.zeros((s.B, L.ilqgb_eval_size(mode)))
    x, u = np.ascontiguousarray(x), np.ascontiguousarray(u)
    s._chk(L.ilqgb_eval(s.h, mode, k, x.ctypes.data, u.ctypes.data, out.ctypes.data))
    return out


def test_single_evaluations_read_the_window():
    B, T, off = 8, 30, 5
    params, x0, u0, opts, tracks = case("cartrack", B, T, extra=off)
    points = [(mode, k) for mode in (0, 1, 5) for k in (0, 1, 17, T - 1)]
    s = solver("cartrack", 0, B, T, params, opts, tracks)
    s.set_track_offset(off)
    got = {p: evaluate(s, p[0], p[1], x0, u0[:, p[1]]) for p in points}
    s.close()
    for b in range(B):
        r = solver("cartrack", 0, B, T, window(params, tracks, b, off, T), opts, {})
        for mode, k in points:
            assert np.array_equal(got[mode, k][b], evaluate(r, mode, k, x0, u0[:, k])[b]), (mode, k, b)
        r.close()


# ---- 8. rejected arguments ----------------------------------------------------------------------------------------------
def test_rejected_arguments_leave_the_offset_unchanged():
    B, T = 8, 30
    params, x0, u0, opts, tracks = case("cartrack", B, T, extra=6)        # len = T + 7
    s = solver("cartrack", 0, B, T, params, opts, tracks)
    L = s.lib
    s.set_track_offset(2)
    v = np.ascontiguousarray(tracks["xr"])

    def rejected(fn, *a):
        with pytest.raises((RuntimeError, ValueError)):
            fn(*a)
        assert s.track_offset() == 2

    rejected(lambda: s._chk(L.ilqgb_set_param_track(s.h, 99, v.ctypes.data, v.shape[1])))     # index out of range
    rejected(lambda: s._chk(L.ilqgb_set_param_track(s.h, -1, v.ctypes.data, v.shape[1])))
    rejected(s.set_param_track, "d", np.ones((B, T + 7)))                                     # not [k]-indexed
    rejected(s.set_param_track, "xr", np.ones((B, T + 2)))                                    # len < offset + n_hor + 1
    rejected(s.set_track_offset, -1)
    rejected(s.set_track_offset, 7)                                                           # window overruns the tracks
    rejected(s.set_param_track, "xr", np.ones(T + 7))                                         # Python shape checks
    rejected(s.set_param_track, "xr", np.ones((B + 1, T + 7)))
    s.set_param_track("yr", np.ones((B, T + 3)))                                              # exactly offset + n_hor + 1
    rejected(s.set_track_offset, 3)                                                           # ... now the shortest track
    s.set_param_track("yr", tracks["yr"])
    s.upload(x0, u0)
    s.run()
    rejected(s.shift, 5)                                                                      # 2 + 5 + T + 1 > T + 7
    rejected(s.mpc, x0, u0, 6)                                                                # 2 + 5 + T + 1 > T + 7
    s.shift(4)
    assert s.track_offset() == 6
    s.close()


# ---- 9. two devices -----------------------------------------------------------------------------------------------------
def test_two_devices_equal_one():
    if ilqg_b200.Library("cartrack", 0).device_count() < 2:
        pytest.skip("needs two GPUs")
    B, T, S = 64, 50, 4
    params, x0, u0, opts, tracks = case("cartrack", B, T, extra=S - 1)
    logs = []
    for devices in (None, 2):
        s = solver("cartrack", 0, B, T, params, opts, tracks, devices=devices)
        logs.append((s.mpc(x0, u0, S), s.download()))
        s.close()
    assert_same(logs[1][0], logs[0][0], "2 devices", LOG_KEYS)
    assert_same(logs[1][1], logs[0][1], "2 devices final plan", ("x", "u"))
