"""The single-evaluation gateway (SURVEY.md 8f N3; iLQG_MMex.tem:81-226): `out = iLQG<Name>MMex(x, u, params, mode, k, n_hor)`.

CPU part: the generated reference-ABI file problems/<name>/iLQG_MMex.c (what a reference build gets from iLQG_MMex.tem), driven
through the fake mex API, is checked against finite differences of its own modes 0 / 1 / 2 -- values, shapes and the layout of
the full Hessians and of the three-index second-order dynamics -- and against the solver-side generated code (calc_derivs of
the reference harness).  GPU part: ddp-generator_b200/mex/iLQG_MMex_b200.c over the CUDA library returns the same arrays bit for bit in all
17 modes and raises the same argument errors."""
import os

import numpy as np
import pytest

import fake_mex as FM
import oracle_lib
import shapes_util as SU
from ilqg_b200 import workloads as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
needs_rig = pytest.mark.skipif(not os.path.exists(FM.FAKEMEX), reason="build the fake mex runtime: make -C oracle port")
PARAMS = {"car": W.CAR_PARAMS, "carhx": W.CARHX_PARAMS, "quad": W.QUAD_PARAMS, **{SU.name_of(s): SU.params_of(s) for s in SU.SHAPES}}
DIMS = {"car": (4, 2), "carhx": (4, 2), "quad": (12, 4), **{SU.name_of(s): s for s in SU.SHAPES}}


def gw(kind, problem):
    path = os.path.join(ROOT, "oracle", "_build", f"libmmex{kind}_{problem}.so")
    if not os.path.exists(path):
        pytest.fail(f"{path} missing: make -C oracle port b200")
    return FM.Gateway(path)


def point(problem, seed):
    rng = np.random.default_rng(seed)
    nx, nu = DIMS[problem]
    if problem == "quad":
        x = rng.uniform(-0.4, 0.4, nx)
        u = W.QUAD_PARAMS["uh"][0] * (1.0 + rng.uniform(-0.3, 0.3, nu))
    elif problem.startswith("shape_"):
        x = rng.uniform(-2.0, 2.0, nx)
        u = rng.uniform(-0.2, 0.2, nu)         # inside every box: the clamp mode leaves it alone
    else:
        x = np.array([rng.uniform(-2, 2), rng.uniform(-2, 2), rng.uniform(0, 6), rng.uniform(-1, 1)])
        u = np.array([rng.uniform(-0.4, 0.4), rng.uniform(-1.5, 1.5)])
    return x, u


def call(g, x, u, params, mode, k=3, N=10):
    return g(x, u, params, float(mode), float(k), float(N), nlhs=1)[0]


def fd(fun, z, h=1e-6):
    cols = []
    for i in range(z.size):
        e = np.zeros_like(z); e[i] = h
        cols.append((np.atleast_1d(fun(z + e)) - np.atleast_1d(fun(z - e))) / (2 * h))
    return np.stack(cols, axis=-1)


@needs_rig
@pytest.mark.parametrize("problem", ["car", "quad"] + [SU.name_of(s) for s in SU.SHAPES])
def test_generated_mmex_matches_finite_differences(problem):
    g = gw("cpu", problem)
    p = PARAMS[problem]
    nx, nu = DIMS[problem]
    x, u = point(problem, 5)
    f = lambda xx, uu: call(g, xx, uu, p, 0).ravel()
    L = lambda xx, uu: call(g, xx, uu, p, 1).ravel()
    F = lambda xx: call(g, xx, u, p, 2).ravel()
    shapes = {0: (nx, 1), 1: (1, 1), 2: (1, 1), 3: (1, nx), 4: (nx, nx), 5: (1, nx), 6: (1, nu), 7: (nx, nx), 8: (nu, nu), 9: (nx, nu),
              10: (nx, nx), 11: (nx, nu), 12: (nx, nx, nx), 13: (nu, nu, nx), 14: (nx, nu, nx), 15: (0, 1), 16: (nu, 1)}
    out = {m: call(g, x, u, p, m) for m in range(17)}
    for m, s in shapes.items():
        assert out[m].shape == s, (m, out[m].shape)
    tol = dict(rtol=2e-5, atol=2e-6)
    assert np.allclose(out[3], fd(F, x)[0], **tol)                                               # Fx
    assert np.allclose(out[4], fd(lambda xx: call(g, xx, u, p, 3).ravel(), x), **tol)             # Fxx
    assert np.allclose(out[5], fd(lambda xx: L(xx, u), x)[0], **tol) and np.allclose(out[6], fd(lambda uu: L(x, uu), u)[0], **tol)
    assert np.allclose(out[7], fd(lambda xx: call(g, xx, u, p, 5).ravel(), x), **tol)             # Lxx
    assert np.allclose(out[8], fd(lambda uu: call(g, x, uu, p, 6).ravel(), u), **tol)             # Luu
    assert np.allclose(out[9], fd(lambda uu: call(g, x, uu, p, 5).ravel(), u), **tol)             # Lxu[r, c] = d2L / dx_r du_c
    assert np.allclose(out[10], fd(lambda xx: f(xx, u), x), **tol) and np.allclose(out[11], fd(lambda uu: f(x, uu), u), **tol)
    # second-order dynamics A(c, j, r) = d2 f_r / d c d j
    fx_of_x = fd(lambda xx: call(g, xx, u, p, 10).ravel(order="F"), x).reshape(nx, nx, nx, order="F")      # [r, c, j] = d fx[r,c] / dx_j
    assert np.allclose(out[12], np.transpose(fx_of_x, (1, 2, 0)), **tol)
    fu_of_u = fd(lambda uu: call(g, x, uu, p, 11).ravel(order="F"), u).reshape(nx, nu, nu, order="F")
    assert np.allclose(out[13], np.transpose(fu_of_u, (1, 2, 0)), **tol)
    fx_of_u = fd(lambda uu: call(g, x, uu, p, 10).ravel(order="F"), u).reshape(nx, nx, nu, order="F")      # d fx[r,c] / du_j
    assert np.allclose(out[14], np.transpose(fx_of_u, (1, 2, 0)), **tol)
    # the clamp: inside the box nothing moves, outside it lands on the limits
    assert np.array_equal(out[16].ravel(), u)
    big = call(g, x, u * 0 + 100.0, p, 16).ravel()
    assert (big < 100.0).all()


@needs_rig
def test_generated_mmex_agrees_with_the_solver_side_code():
    """fx, fu, Lx ... from the MMex file equal what calc_derivs of the reference harness leaves in the trajectory (same lowering,
    two emitters): bit for bit."""
    T = 12
    x0, u0 = W.car_batch(1, T=T, seed=9)
    kind = "reference" if oracle_lib.available("reference", "car", 1) else "port"
    s = oracle_lib.OracleLib(kind, "car", 1).solver(T)
    s.set_opts({"max_iter": 3}); s.set_params(W.CAR_PARAMS)
    assert s.init(x0[0], u0[0]) and s.calc_derivs()
    g = gw("cpu", "car")
    xs, us = s.get("x"), s.get("u")
    for k in (0, 5, 11):
        for mode, field, pack in ((10, "fx", None), (11, "fu", None), (5, "cx", None), (6, "cu", None), (9, "cxu", None), (7, "cxx", 4), (8, "cuu", 2)):
            got = call(g, xs[k], us[k], W.CAR_PARAMS, mode, k=k + 1, N=T)
            want = s.get(field)[k]
            if pack:
                full = np.array([[want[(max(r, c) * (max(r, c) + 1)) // 2 + min(r, c)] for c in range(pack)] for r in range(pack)])
                assert np.array_equal(got, full), (k, field)
            else:
                assert np.array_equal(got.ravel(order="F"), want), (k, field)
    s.close()


def test_problems_with_folded_constraints_have_no_mmex():
    assert not os.path.exists(os.path.join(ROOT, "ddp-generator_b200", "problems", "brachi", "iLQG_MMex.c"))
    assert os.path.exists(os.path.join(ROOT, "ddp-generator_b200", "problems", "car", "iLQG_MMex.c"))


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@needs_rig
@pytest.mark.parametrize("problem", ["car", "carhx", "quad"] + [SU.name_of(s) for s in SU.SHAPES])
def test_gpu_gateway_matches_generated_mmex_in_all_modes(problem):
    cpu, gpu = gw("cpu", problem), gw("b200", problem)
    p = PARAMS[problem]
    for seed in range(4):
        x, u = point(problem, 20 + seed)
        if seed == 3:
            u = u * 50.0          # far outside the limits: the clamp mode has something to do
        for mode in range(17):
            a, b = call(cpu, x, u, p, mode, k=seed + 1, N=8), call(gpu, x, u, p, mode, k=seed + 1, N=8)
            assert a.shape == b.shape and np.array_equal(a, b, equal_nan=True), (problem, seed, mode)
    assert gpu.live_allocs == 0


@pytest.mark.gpu
@needs_rig
def test_gpu_gateway_argument_errors_match():
    cpu, gpu = gw("cpu", "car"), gw("b200", "car")
    x, u = point("car", 1)
    good = [x, u, dict(W.CAR_PARAMS), 0.0, 1.0, 10.0]

    def both(args, nlhs=1):
        res = []
        for g in (cpu, gpu):
            try:
                g(*args, nlhs=nlhs)
                res.append(None)
            except FM.MexError as e:
                res.append((e.ident, e.msg))
        return res

    cases = [good[:5], good + [1.0]]
    for i, bad in ((0, np.zeros(5)), (1, np.zeros(3)), (3, np.zeros(2)), (4, np.zeros(2)), (5, np.zeros(2)), (2, np.zeros(3))):
        a = list(good); a[i] = bad; cases.append(a)
    missing = dict(W.CAR_PARAMS); del missing["cf"]; a = list(good); a[2] = missing; cases.append(a)
    wrong = dict(W.CAR_PARAMS); wrong["cf"] = [1.0, 2.0]; a = list(good); a[2] = wrong; cases.append(a)
    sparse = dict(W.CAR_PARAMS); sparse["d"] = FM.Sparse(np.array([2.0])); a = list(good); a[2] = sparse; cases.append(a)
    for c in cases:
        r = both(c)
        assert r[0] is not None and r[0] == r[1], (r, [np.shape(v) if not isinstance(v, dict) else "struct" for v in c])
    r = both(good, nlhs=2)
    assert r[0] is not None and r[0] == r[1]
