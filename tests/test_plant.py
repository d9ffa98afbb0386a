"""Plants of closed loops without a GPU: the samplers of sampled plants, and the oracle's plant step that tests/test_gpu_plant.py
compares with.  That step is the oracle with horizon n_sub, initialised at xp with u[j] repeated n_sub times: its initial
forward_pass clamps u[j] at each sub-step's own state and applies f, which must be what a MATLAB user's loop does with the
generated single-evaluation function, iLQG<Name>MMex mode 16 (clamp) then mode 0 (f), once per sub-step."""
import os

import numpy as np
import pytest

import fake_mex as FM
import oracle_lib
import parity_util as PU
from ilqg_b200 import workloads as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("sampler,names", [(W.car_plant, {"d": 1}), (W.quad_plant, {"mass": 1, "J": 3, "kq": 1})])
def test_plant_samplers_are_deterministic_and_shard(sampler, names):
    a = sampler(40, 0.1, seed=5)
    assert {k: v.shape for k, v in a.items()} == {k: (40, n) for k, n in names.items()}
    b = sampler(40, 0.1, seed=5)
    parts = [sampler(n, 0.1, seed=5, first=f) for f, n in ((0, 13), (13, 20), (33, 7))]
    other = sampler(40, 0.1, seed=6)
    nominal = W.CAR_PARAMS if sampler is W.car_plant else W.QUAD_PARAMS
    for k, v in a.items():
        assert np.array_equal(v, b[k])
        assert np.array_equal(v, np.concatenate([p[k] for p in parts]))
        assert not np.array_equal(v, other[k])
        ratio = v / np.asarray(nominal[k])[None, :]
        assert np.all(ratio >= 0.9) and np.all(ratio <= 1.1) and ratio.min() < 0.95 and ratio.max() > 1.05
        assert len(np.unique(v)) == v.size        # every entry of every problem has its own factor


def oracle_plant_step(problem, xp, u, params, n_sub):
    """xp stepped n_sub times with u held: the oracle's initial rollout over a horizon of n_sub"""
    O = oracle_lib.OracleLib(PU.oracle_kinds(problem, 0)[0], problem, 0)
    s = O.solver(n_sub)
    s.set_params(params)
    s.init(xp, np.tile(u, (n_sub, 1)))
    x = s.get("x")[n_sub]
    s.close()
    return x


@pytest.mark.parametrize("problem", ["car", "quad"])
def test_oracle_plant_step_is_mmex_clamp_then_dynamics(problem):
    path = os.path.join(ROOT, "oracle", "_build", f"libmmexcpu_{problem}.so")
    if not os.path.exists(FM.FAKEMEX) or not os.path.exists(path):
        pytest.fail(f"{path} missing: make -C oracle port")
    g = FM.Gateway(path)
    if problem == "car":
        params = dict(W.CAR_PARAMS, d=[2.2], h=[0.03 / 4])
        x0, u0 = W.car_batch(6, T=4, seed=31)
        u0 = u0 * 8.0           # beyond the steering and acceleration limits: the clamp matters
    else:
        params = dict(W.QUAD_PARAMS, dt=[0.01 / 4], **{k: v[3] for k, v in W.quad_plant(4, 0.2, seed=32).items()})
        x0, u0 = W.quad_batch(6, T=4, seed=33)
        u0 = u0 * (1.0 + np.linspace(-1.5, 1.5, 24).reshape(6, 1, 4))   # some rotors below zero or above the thrust limit
    clamped = 0
    for b in range(x0.shape[0]):
        for n_sub in (1, 4):
            x = x0[b].copy()
            for _ in range(n_sub):
                ua = g(x, u0[b, 0], params, 16.0, 0.0, float(n_sub), nlhs=1)[0].ravel()
                clamped += not np.array_equal(ua, u0[b, 0])
                x = g(x, ua, params, 0.0, 0.0, float(n_sub), nlhs=1)[0].ravel()
            assert np.array_equal(oracle_plant_step(problem, x0[b], u0[b, 0], params, n_sub), x), (problem, b, n_sub)
    assert clamped > 0
