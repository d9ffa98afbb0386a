"""Feedback policy without a GPU: the oracle's definition of a policy rollout, and the sampler of initial states."""
import numpy as np
import pytest

import parity_util as PU
import policy_util
from ilqg_b200 import workloads as W


@pytest.mark.parametrize("problem,T", [("car", 60), ("quad", 40)])
def test_oracle_policy_rollout_from_the_plan_start_is_the_plan(problem, T):
    """calc_derivs + back_pass + forward_pass's feedback branch at alpha = 0 from x*_0 reproduces the nominal x and u: the
    definition the device's rollouts are checked against"""
    if not PU.oracle_kinds(problem, 0):
        pytest.skip("oracle not built")
    O = policy_util.oracle(problem, 0)
    if problem == "car":
        x0, u0 = W.car_batch(3, T=T, seed=31)
        params, opts = W.CAR_PARAMS, {"max_iter": 10.0}
    else:
        x0, u0 = W.quad_batch(2, T=T, seed=32)
        params, opts = W.QUAD_PARAMS, {"max_iter": 8.0}
    for b in range(x0.shape[0]):
        p = policy_util.Solved(O, T, params, opts, x0[b], u0[b])
        assert p.init_ok
        g = p.policy()
        assert g["policy_ok"] == 1
        assert np.any(g["L"] != 0.0)
        r = p.rollout(p.x[0])
        assert r["ok"] == 1
        assert np.array_equal(r["x"], p.x) and np.array_equal(r["u"], p.u)
        assert np.array_equal(p.s.get("x"), p.x)       # the nominal is back in place
        moved = p.rollout(p.x[0] + 0.05)
        assert moved["ok"] == 1 and not np.array_equal(moved["u"], p.u)
        p.close()


def test_perturbed_states_are_deterministic_and_shard():
    x0, _ = W.car_batch(10, T=5, seed=3)
    a = W.perturbed_states(x0, 6, 0.1, seed=9)
    assert a.shape == (10, 6, 4)
    assert np.array_equal(a, W.perturbed_states(x0, 6, 0.1, seed=9))
    assert not np.array_equal(a, W.perturbed_states(x0, 6, 0.1, seed=10))
    assert np.array_equal(a[4:], W.perturbed_states(x0[4:], 6, 0.1, seed=9, first=4))
    dev = a - x0[:, None, :]
    assert 0.05 < dev.std() < 0.2
    per_state = W.perturbed_states(x0, 6, [0.1, 0.1, 0.0, 0.0], seed=9)
    assert np.array_equal(per_state[..., 2:], np.broadcast_to(x0[:, None, 2:], (10, 6, 2)))
