"""The reference's example problems (CarParking, Brachistochrone, Brachistochrone with hli), restated as problem files in
tests/data/, through the one-step build `python -m ilqg_gen.make file.mac`: the resulting product libraries solve on the GPU
bit-exactly like the solver core linked against the C generated from the same file -- the unmodified reference core where it
was built against that C, else the oracle port, which reproduces the reference's golden fixtures bit for bit
(test_oracle_golden.py).  __graft_entry__.build() builds the libraries and their checkers (build_mac_examples)."""
import os

import numpy as np
import pytest

import ilqg_b200
import oracle_lib
from ilqg_b200 import workloads as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAC_LIB = os.path.join(ROOT, "ddp-generator_b200", "build_mac", "lib")
MAC_PROBLEMS = os.path.join(ROOT, "ddp-generator_b200", "build_mac", "problems")
GOLD = os.path.join(ROOT, "tests", "golden")


def _case(name):
    if name == "mac_car":
        x0, u0 = W.car_batch(6, T=150, seed=17)
        return 150, W.CAR_PARAMS, x0, u0, {"max_iter": 25.0}
    if name == "mac_brachi":
        params, x0, u0, opts = W.brachi(60)
        return 60, params, x0[None], u0[None], opts
    params, x0, u0, opts = W.brachi_hli(120)
    return 120, params, x0[None], u0[None], opts


def _checker(name, ddp):
    """The reference core where its library is at least as new as the C generated from tests/data/<name>.mac (an older one was
    linked against the C of another problem file and is not rebuilt without the reference's sources), else the oracle port."""
    ref, gen = oracle_lib.lib_path("reference", name, ddp), os.path.join(MAC_PROBLEMS, name, "iLQG_func.c")
    fresh = os.path.exists(ref) and os.path.exists(gen) and os.path.getmtime(ref) >= os.path.getmtime(gen)
    return "reference" if fresh else "port"


def _have(name, ddp):
    return os.path.exists(ilqg_b200.lib_path(name, ddp, MAC_LIB)) and oracle_lib.available(_checker(name, ddp), name, ddp)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mac_car", "mac_brachi", "mac_brachi_hli"])
@pytest.mark.parametrize("ddp", [0, 1])
def test_mac_built_library_matches_reference_core(name, ddp):
    assert _have(name, ddp), "build the .mac examples first: python -c 'import __graft_entry__ as g; g.build()'"
    T, params, x0, u0, opts = _case(name)
    s = ilqg_b200.BatchSolver(name, ddp, x0.shape[0], T, flags=ilqg_b200.TRACE, lib_dir=MAC_LIB)
    s.set_options(opts); s.set_params(params)
    out = s.solve(x0, u0)
    tr_a, tr_l = s.get_int("tr_alpha"), s.get("tr_lambda")
    mu_f = s.get("mu_f") if name != "mac_car" else None
    s.close()
    O = oracle_lib.OracleLib(_checker(name, ddp), name, ddp)
    for b in range(x0.shape[0]):
        h = O.solver(T); h.set_opts(opts); h.set_params(params)
        assert h.init(x0[b], u0[b])
        res = h.solve()
        n = int(h.scalar("n_linesearch"))
        assert out["success"][b] == res and out["iterations"][b] == h.scalar("iterations") and out["n_linesearch"][b] == n
        assert out["cost"][b] == h.scalar("cost")
        assert np.array_equal(out["x"][b], h.get("x")) and np.array_equal(out["u"][b], h.get("u"))
        assert np.array_equal(tr_a[b][:n], h.trace("alpha_idx").astype(int)) and np.array_equal(tr_l[b][:n], h.trace("lambda"))
        if mu_f is not None:
            assert mu_f[b].ravel()[0] == h.get("mult_f")[0]
        h.close()


@pytest.mark.parametrize("name,fixture,T", [("mac_brachi", "brachi_n500_ddp0.npz", 500), ("mac_brachi_hli", "brachi_hli_ddp0.npz", 500),
                                            ("mac_car", "car_T100_b0.npz", 100)])
def test_mac_model_agrees_with_the_handwritten_module(name, fixture, T):
    """CPU: the solver core (the reference's where it is built, else the oracle port) on the C generated from the .mac file
    reaches the solution the fixtures hold (which were recorded with the hand-written problem modules).  The two front ends may
    order floating-point operations differently, so the first pass is compared to 1e-12 relative and -- for the Brachistochrone,
    which is not chaotic -- the final cost to 1e-9."""
    assert oracle_lib.available(_checker(name, 0), name, 0), "build the .mac examples first: python -c 'import __graft_entry__ as g; g.build()'"
    g = np.load(os.path.join(GOLD, fixture))
    params, opts = {"mac_car": (W.CAR_PARAMS, {"max_iter": 30.0}), "mac_brachi": W.brachi(T)[0::3], "mac_brachi_hli": W.brachi_hli(T)[0::3]}[name]
    h = oracle_lib.OracleLib(_checker(name, 0), name, 0).solver(T)
    h.set_opts(opts); h.set_params(params)
    assert h.init(g["x0"], g["u0"])
    assert abs(h.scalar("cost") - float(g["cost0"])) <= 1e-12 * abs(float(g["cost0"]))
    h.solve()
    if name != "mac_car":
        assert abs(h.scalar("cost") - float(g["cost"])) <= 1e-9 * abs(float(g["cost"]))
        assert int(h.scalar("iterations")) == int(g["iterations"])
    h.close()
