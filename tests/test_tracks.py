"""Tracking workloads without a GPU: the cartrack batch generator and the oracle on a window of the tracks."""
import numpy as np
import pytest

import oracle_lib
import parity_util as PU
from ilqg_b200 import workloads as W


def test_cartrack_batch_is_deterministic_and_shards_are_slices():
    a = W.cartrack_batch(40, T=30, extra=5, seed=9)
    b = W.cartrack_batch(40, T=30, extra=5, seed=9)
    part = W.cartrack_batch(15, T=30, extra=5, seed=9, first=20)
    x0, u0, tr = a
    assert x0.shape == (40, 4) and u0.shape == (40, 30, 2)
    assert set(tr) == {"xr", "yr"} and all(v.shape == (40, 36) for v in tr.values())
    for p, q in ((a[0], b[0]), (a[1], b[1]), (a[2]["xr"], b[2]["xr"]), (a[2]["yr"], b[2]["yr"])):
        assert np.array_equal(p, q)
    assert np.array_equal(part[0], x0[20:35]) and np.array_equal(part[1], u0[20:35])
    for k in ("xr", "yr"):
        assert np.array_equal(part[2][k], tr[k][20:35])
    # one arc per problem: constant spacing along the path (speed * h), starting next to x0
    step = np.hypot(np.diff(tr["xr"], axis=1), np.diff(tr["yr"], axis=1))
    assert np.allclose(step, step[:, :1], rtol=1e-6)
    assert np.all(np.hypot(x0[:, 0] - tr["xr"][:, 0], x0[:, 1] - tr["yr"][:, 0]) < 0.2)


@pytest.mark.parametrize("ddp", [0, 1])
def test_oracle_solves_cartrack_on_a_window_of_the_tracks(ddp):
    kinds = PU.oracle_kinds("cartrack", ddp)
    if not kinds:
        pytest.skip("no cartrack oracle built")
    T, off = 40, 7
    x0, u0, tr = W.cartrack_batch(3, T=T, extra=10, seed=5)
    for b in range(3):
        params = dict(W.CARTRACK_PARAMS, **{k: v[b, off:off + T + 1] for k, v in tr.items()})
        rec = PU.oracle_record(kinds[0], "cartrack", ddp, T, params, x0[b], u0[b], {"max_iter": 20.0})
        assert rec["init_ok"]
        assert rec["cost"] < rec["cost0"], (b, rec["cost"], rec["cost0"])
