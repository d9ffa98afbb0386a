"""Deterministic synthetic workloads for the BASELINE.json configs (SURVEY.md 8d).

Counter-based streams (SplitMix64 finaliser over (seed, problem, element)) so that every consumer -- the CUDA
path, the CPU oracle, each rank of a sharded run -- can materialise exactly the same inputs for any subset of
problems without sharing RNG state.  Parameters and the single-instance initial state are the ones in the
reference's demos (examples/CarParking/testCar.m:2-16, examples/Brachistochrone/testBrachi.m:7-22).
"""
from __future__ import annotations

import numpy as np

_GOLD = np.uint64(0x9E3779B97F4A7C15)


def _mix(z):
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def uniform01(seed, stream, idx):
    """U(0,1) for counters idx (array) of stream `stream` (array or scalar) under `seed`; 53-bit resolution."""
    with np.errstate(over="ignore"):
        s = _mix(np.uint64(seed) * _GOLD + np.asarray(stream, dtype=np.uint64))
        z = _mix(s + (np.asarray(idx, dtype=np.uint64) + np.uint64(1)) * _GOLD)
    return ((z >> np.uint64(11)).astype(np.float64) + 0.5) * (1.0 / 9007199254740992.0)


def normal(seed, stream, idx):
    """N(0,1) via Box-Muller on two counters per sample."""
    idx = np.asarray(idx, dtype=np.uint64)
    u1 = uniform01(seed, stream, idx * np.uint64(2))
    u2 = uniform01(seed, stream, idx * np.uint64(2) + np.uint64(1))
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)


# ---- closed loops ------------------------------------------------------------------------------------------------------
def disturbance(B, S, nx, scale, seed, first=0):
    """Process noise of a closed loop, w [B, S, nx] = scale * N(0,1), for problems first..first+B-1 and steps 0..S-1."""
    b = np.arange(first, first + B, dtype=np.uint64)
    idx = np.arange(S * nx, dtype=np.uint64)[None, :]
    return scale * normal(seed, b[:, None], idx).reshape(B, S, nx)


def perturbed_states(x0, M, scale, seed, first=0):
    """M initial states per problem around x0 [B, nx] for Monte-Carlo rollouts of a feedback policy (BatchSolver.policy_rollout):
    x0s [B, M, nx] = x0[b] + scale * N(0,1), scale a scalar or one value per state; rows are problems first..first+B-1, so a
    shard regenerates its own."""
    x0 = np.asarray(x0, dtype=np.float64)
    B, nx = x0.shape
    b = np.arange(first, first + B, dtype=np.uint64)
    idx = np.arange(M * nx, dtype=np.uint64)[None, :]
    return x0[:, None, :] + np.asarray(scale, dtype=np.float64) * normal(seed, b[:, None], idx).reshape(B, M, nx)


def _scaled(seed, b, idx, nominal, spread):
    """nominal values scaled by U(1 - spread, 1 + spread), one factor per problem b and element idx"""
    return np.asarray(nominal)[None, :] * (1.0 + spread * (2.0 * uniform01(seed, b[:, None], idx[None, :]) - 1.0))


def car_plant(B, spread, seed, first=0):
    """Sampled car plants for a robustness study: {"d": [B, 1]}, the wheelbase scaled by U(1 - spread, 1 + spread); problems
    first..first+B-1 (BatchSolver.set_plant_params_batch)."""
    b = np.arange(first, first + B, dtype=np.uint64)
    return {"d": _scaled(seed, b, np.arange(1, dtype=np.uint64), CAR_PARAMS["d"], spread)}


def quad_plant(B, spread, seed, first=0):
    """Sampled quadrotor plants: mass [B, 1], inertia J [B, 3] and rotor torque coefficient kq [B, 1], each entry scaled by its
    own U(1 - spread, 1 + spread); problems first..first+B-1."""
    b = np.arange(first, first + B, dtype=np.uint64)
    e = np.arange(5, dtype=np.uint64)
    return {"mass": _scaled(seed, b, e[:1], QUAD_PARAMS["mass"], spread), "J": _scaled(seed, b, e[1:4], QUAD_PARAMS["J"], spread),
            "kq": _scaled(seed, b, e[4:], QUAD_PARAMS["kq"], spread)}


# ---- car parking ---------------------------------------------------------------------------------------------
CAR_PARAMS = {
    "d": [2.0], "h": [0.03],
    "pf": [0.01, 0.01, 0.01, 1.0], "cf": [0.1, 0.1, 1.0, 0.3],
    "cu": [1e-2 * 1.0, 1e-2 * 0.01], "cx": [1e-3 * 1.0, 1e-3 * 1.0], "px": [0.1, 0.1],
    "limW": [-0.5, 0.5], "limA": [-2.0, 2.0],
}
CAR_X0 = np.array([1.0, 1.0, np.pi * 3 / 2, 0.0])
CAR_T = 500


def car_single(T=CAR_T, seed=1):
    """Config 1: x0 of testCar.m:15, u0 = 0.1*N(0,1) (testCar.m:17, made reproducible). u0 is [T][2]."""
    idx = np.arange(T * 2, dtype=np.uint64)
    u0 = 0.1 * normal(seed, 0, idx).reshape(T, 2)
    return CAR_X0.copy(), u0


def car_batch(B, T=CAR_T, seed=2, first=0):
    """Configs 3/4: x0_b = [U(-2,2), U(-2,2), U(0,2pi), 0], u0_b = 0.1*N(0,1); problems first..first+B-1."""
    b = np.arange(first, first + B, dtype=np.uint64)
    x0 = np.zeros((B, 4))
    x0[:, 0] = -2.0 + 4.0 * uniform01(seed, b, 0)
    x0[:, 1] = -2.0 + 4.0 * uniform01(seed, b, 1)
    x0[:, 2] = 2.0 * np.pi * uniform01(seed, b, 2)
    idx = np.arange(T * 2, dtype=np.uint64)[None, :] + np.uint64(16)
    u0 = 0.1 * normal(seed, b[:, None], idx).reshape(B, T, 2)
    return x0, u0


# ---- car tracking a reference path (problem cartrack, authored here) -----------------------------------------------------
CARTRACK_PARAMS = {
    "d": [2.0], "h": [0.03],
    "cu": [1e-2 * 1.0, 1e-2 * 0.01], "cx": [1.0, 1.0], "px": [0.1, 0.1], "cf": [1.0, 1.0],
    "limW": [-0.5, 0.5], "limA": [-2.0, 2.0],
}


def cartrack_batch(B, T=CAR_T, extra=20, seed=4, first=0):
    """Problems first..first+B-1, each following its own constant-speed arc: speed U(0.5, 2), curvature U(-0.2, 0.2), heading
    U(0, 2pi), start U(-2, 2)^2, sampled every h = 0.03 s (the car's step).  Returns x0 [B, 4] (near the start of the path,
    at the path's speed), u0 [B, T, 2] = 0.1*N(0,1) and the tracks {"xr", "yr"}: [B, T + 1 + extra], enough for a closed
    loop of extra + 1 steps."""
    b = np.arange(first, first + B, dtype=np.uint64)
    speed = 0.5 + 1.5 * uniform01(seed, b, 0)
    kappa = -0.2 + 0.4 * uniform01(seed, b, 1)
    head = 2.0 * np.pi * uniform01(seed, b, 2)
    px0 = -2.0 + 4.0 * uniform01(seed, b, 3)
    py0 = -2.0 + 4.0 * uniform01(seed, b, 4)
    s = speed[:, None] * (CARTRACK_PARAMS["h"][0] * np.arange(T + 1 + extra))[None, :]     # arc length at each step
    kap = kappa[:, None]
    straight = np.abs(kap) < 1e-9
    ks = np.where(straight, 1.0, kap)
    th = head[:, None] + kap * s
    xr = px0[:, None] + np.where(straight, s * np.cos(head)[:, None], (np.sin(th) - np.sin(head)[:, None]) / ks)
    yr = py0[:, None] + np.where(straight, s * np.sin(head)[:, None], (np.cos(head)[:, None] - np.cos(th)) / ks)
    x0 = np.zeros((B, 4))
    x0[:, 0] = px0 + 0.2 * (uniform01(seed, b, 5) - 0.5)
    x0[:, 1] = py0 + 0.2 * (uniform01(seed, b, 6) - 0.5)
    x0[:, 2] = head + 0.2 * (uniform01(seed, b, 7) - 0.5)
    x0[:, 3] = speed
    idx = np.arange(T * 2, dtype=np.uint64)[None, :] + np.uint64(16)
    u0 = 0.1 * normal(seed, b[:, None], idx).reshape(B, T, 2)
    return x0, u0, {"xr": xr, "yr": yr}


# ---- brachistochrone ----------------------------------------------------------------------------------------------
def brachi(n):
    """Config 2 (testBrachi.m:7-22): g=9.81, yf=-4, x0=-eps, u0=-1, dx=2*pi/n; options max_iter=20, w_pen_fact2=2.
    (testBrachi.m:13 also sets `w_pen_init`, which setOptParam rejects -- iLQG.c:211-213 -- so it is dropped.)"""
    params = {"dx": [2.0 * np.pi / n], "g": [9.81], "yf": [-4.0]}
    x0 = np.array([-np.finfo(float).eps])
    u0 = -np.ones((n, 1))
    opts = {"max_iter": 20.0, "w_pen_fact2": 2.0}
    return params, x0, u0, opts


# ---- synthetic quadrotor (config 5) ---------------------------------------------------------------------------------
QUAD_T = 1000
_QUAD_UH = 1.0 * 9.81 / 4.0
QUAD_PARAMS = {
    "dt": [0.01], "mass": [1.0], "grav": [9.81], "J": [0.01, 0.01, 0.02], "arm": [0.2], "kq": [0.05],
    "cx": [1e-3] * 3 + [1e-4] * 3 + [1e-3] * 3 + [1e-4] * 3,
    "cf": [10.0] * 3 + [1.0] * 3 + [10.0] * 3 + [1.0] * 3,
    "cu": [1e-3] * 4, "xg": [0.0] * 12, "uh": [_QUAD_UH], "ulim": [0.0, 2.0 * _QUAD_UH],
}


def quad_batch(B, T=QUAD_T, seed=3, first=0):
    """x0 = hover at the origin + U(-0.5, 0.5) on every state, u0 = hover thrust on all rotors (SURVEY 8d config 5)."""
    b = np.arange(first, first + B, dtype=np.uint64)
    x0 = np.stack([-0.5 + uniform01(seed, b, i) for i in range(12)], axis=1)
    u0 = np.full((B, T, 4), _QUAD_UH)
    return x0, u0


# ---- car with a state-dependent steering limit (reference extension: state dependent input constraints) -------------
CARHX_PARAMS = dict(CAR_PARAMS, kv=[0.5])


# ---- Brachistochrone with a running inequality and a [k]-indexed parameter (testBrachi_hli.m:7-32) -----------------
def brachi_hli(n=500):
    params = {"dx": [2.0 * np.pi / n], "g": [9.81], "ymin": np.concatenate([np.linspace(-1.0, -5.0, n), [-4.0]])}
    x0 = np.array([-np.finfo(float).eps])
    u0 = -np.ones((n, 1))
    opts = {"max_iter": 20.0, "w_pen_init_l": 40.0, "w_pen_init_f": 1e-5, "w_pen_max_f": 1.0, "w_pen_fact2": 1.0}
    return params, x0, u0, opts


# ---- twin-motor pendulum: running equality (hle) + terminal inequality (hfi) + torque limits (authored here) ------------
PEND_PARAMS = {"dt": [0.02], "gl": [9.81], "cu": [0.01, 0.03], "cx": [0.1, 0.01], "cf": [5.0, 1.0], "lim": [-3.0, 3.0], "thmin": [0.5]}
PEND_T = 200


def pend_batch(B, T=PEND_T, seed=7, first=0):
    """x0 = [U(1.5, 3), U(-1, 1)], u0 = 0.1*N(0,1) on both motors (unequal: the equality constraint starts violated)."""
    b = np.arange(first, first + B, dtype=np.uint64)
    x0 = np.zeros((B, 2))
    x0[:, 0] = 1.5 + 1.5 * uniform01(seed, b, 0)
    x0[:, 1] = -1.0 + 2.0 * uniform01(seed, b, 1)
    idx = np.arange(T * 2, dtype=np.uint64)[None, :] + np.uint64(16)
    u0 = 0.1 * normal(seed, b[:, None], idx).reshape(B, T, 2)
    return x0, u0


PEND_OPTS = {"max_iter": 60.0, "w_pen_fact2": 2.0}
