"""`.mac` front end (gen/ilqg_gen/macfile.py): the reference's own example files parse into the same models as the
hand-written problem modules, and a problem file written for this repo goes through the whole generator."""
import os
import subprocess
import tempfile

import pytest
import sympy as sp

from ilqg_gen.emit_c import emit_func_c, emit_problem_h
from ilqg_gen.emit_cuda import emit_device
from ilqg_gen.lower import lower
from ilqg_gen.macfile import load_mac
from ilqg_gen.problems import REGISTRY

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference/examples"


def _same(a, b):
    """equal up to symbol identity (assumptions differ between the two front ends)"""
    ra = a.xreplace({s: sp.Symbol(s.name) for s in a.free_symbols})
    rb = b.xreplace({s: sp.Symbol(s.name) for s in b.free_symbols})
    return sp.simplify(ra - rb) == 0


def _same_model(path, mod):
    a, b = lower(load_mac(path)), lower(REGISTRY[mod]())
    assert [d.name for d in a.params] == [d.name for d in b.params] and [d.size for d in a.params] == [d.size for d in b.params]
    assert [s.name for s in a.x] == [s.name for s in b.x] and [s.name for s in a.u] == [s.name for s in b.u]
    assert [x.name for x in a.aux] == [x.name for x in b.aux] and a.n_mu == b.n_mu
    assert all(_same(p, q) for p, q in zip(a.f, b.f))
    for p, q in zip(a.aux, b.aux):
        assert _same(p.expr, q.expr), p.name
    assert _same(a.L, b.L) and _same(a.F, b.F)
    assert [(h["input"], h["sign"]) for h in a.h] == [(h["input"], h["sign"]) for h in b.h]
    assert all(_same(h1["limit"], h2["limit"]) for h1, h2 in zip(a.h, b.h))


@pytest.mark.skipif(not os.path.exists(REF), reason="reference tree not present on this machine")
@pytest.mark.parametrize("mac,mod", [("CarParking/optDefCar.mac", "car"), ("Brachistochrone/optDefBrachi.mac", "brachi"),
                                     ("Brachistochrone/optDefBrachi_hli.mac", "brachi_hli")])
def test_reference_examples_parse_to_the_same_model(mac, mod):
    """The reference's own example files, which this repository does not carry (the reference is GPL-2.0 and never copied
    here): runs only next to a reference checkout and skips elsewhere by design.  test_restated_examples_parse_to_the_same_model
    checks the restatements in tests/data/ the same way on every machine."""
    _same_model(os.path.join(REF, mac), mod)


@pytest.mark.parametrize("mod", ["car", "brachi", "brachi_hli"])
def test_restated_examples_parse_to_the_same_model(mod):
    """tests/data/<mod>.mac, the input of the .mac-built libraries of test_gpu_macfile.py, describes the hand-written model."""
    _same_model(os.path.join(ROOT, "tests", "data", f"{mod}.mac"), mod)


def test_own_mac_file_generates_and_compiles():
    P = load_mac(os.path.join(ROOT, "tests", "data", "pendulum.mac"), "Pendulum")
    m = lower(P)
    assert (m.nx, m.nu) == (2, 1) and [a.name for a in m.aux][:1] == ["acc"]
    assert [d.name for d in m.params] == ["b", "cu", "dt", "g", "l", "m", "q", "qf", "thg", "tmax"]
    assert [(h["input"], h["sign"]) for h in m.h] == [(0, -1), (0, 1)]        # ascending h index: lower bound first
    assert m.n_mu == {"fe": 1, "fi": 0, "le": 0, "li": 0}
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "iLQG_problem.h"), "w").write(emit_problem_h(m))
        open(os.path.join(d, "iLQG_func.c"), "w").write(emit_func_c(m))
        open(os.path.join(d, "pendulum_device.cuh"), "w").write(emit_device(m, "ProbPendulum"))
        inc = ["-I" + d, "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "ddp-generator_b200", "csrc")]
        subprocess.run(["gcc", "-std=gnu11", "-O1", "-ffp-contract=off", "-w", "-DFULL_DDP=1", "-DPRNT=printf", *inc, "-c",
                        os.path.join(d, "iLQG_func.c"), "-o", os.path.join(d, "f.o")], check=True)
        cu = os.path.join(d, "t.cu")
        open(cu, "w").write('#include "ilqg_kernels.cuh"\n#include "pendulum_device.cuh"\n'
                            'template __global__ void ilqg::k_derivs<ProbPendulum, true, false>(ilqg_work, ilqg::ParamBlock<ProbPendulum>);\n'
                            'template __global__ void ilqg::k_backpass<ProbPendulum, true, 8, true>(ilqg_work, ilqg_opts, ilqg::ParamBlock<ProbPendulum>, int);\n'
                            'template __global__ void ilqg::k_ls_round<ProbPendulum, false>(ilqg_work, ilqg_opts, ilqg::ParamBlock<ProbPendulum>, int, int);\n')
        subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-fmad=false", "-diag-suppress", "550,177,20281",
                        *inc, "-c", cu, "-o", os.path.join(d, "t.o")], check=True)


def test_one_step_build_from_mac_file():
    """python -m ilqg_gen.make: .mac file -> generated code -> loadable libraries (the role of the reference's make_iLQG.m)."""
    import ctypes as C

    from ilqg_gen import make

    with tempfile.TemporaryDirectory() as d:
        r = make.build(os.path.join(ROOT, "tests", "data", "pendulum.mac"), out=d)
        assert r["name"] == "pendulum" and r["struct"] == "ProbPendulum" and all(os.path.exists(p) for p in r["libs"])
        for ddp in (0, 1):
            L = C.CDLL(os.path.join(d, "lib", f"libilqg_b200_pendulum_ddp{ddp}.so"))
            L.ilqgb_problem_name.restype = C.c_char_p
            L.ilqgb_param_name.restype = C.c_char_p
            assert (L.ilqgb_nx(), L.ilqgb_nu(), L.ilqgb_full_ddp()) == (2, 1, ddp)
            assert [L.ilqgb_param_name(i).decode() for i in range(L.ilqgb_n_params())] == ["b", "cu", "dt", "g", "l", "m", "q", "qf", "thg", "tmax"]
        D = C.CDLL(os.path.join(d, "lib", "libilqg_dropin_pendulum_ddp0.so"))
        assert all(hasattr(D, s) for s in ("iLQG", "setOptParam", "standard_parameters", "init_opt", "forward_pass", "makeCandidateNominal"))


_BAD = """x: [p, v];
u: [a, w];
f[p]: p + dt*v;
f[v]: v + dt*a;
L: a^2 + w^2;
F: p^2;
%s
"""


@pytest.mark.parametrize("h,msg", [
    ("h[1]: a + w - 1;", "may depend on only one input"),              # genenerator_main.mac:389-390
    ("h[1]: 2*a - 1;", "must be 1 or -1"),                             # genenerator_main.mac:392-393
    ("h[1]: a + a^2 - 1;", "must be 1 or -1"),
    ("s: a*v;\nh[1]: w + 's - 1;", "may depend on only one input|may only depend directly on one input"),   # a second input through an aux value (:386-391)
])
def test_invalid_input_constraints_are_rejected_like_the_reference_generator(h, msg):
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "optDefBad.mac")
        open(path, "w").write(_BAD % h)
        with pytest.raises(ValueError, match=msg):
            lower(load_mac(path))


def test_f_must_be_indexed_by_states_and_k_index_cannot_be_mixed():
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "optDefBad.mac")
        open(path, "w").write(_BAD.replace("f[v]:", "f[q]:") % "")
        with pytest.raises(ValueError, match="indexed by elements of x"):
            load_mac(path)
        open(path, "w").write(_BAD.replace("L: a^2 + w^2;", "L: r[k]*a^2 + r[1]*w^2;") % "")
        with pytest.raises(ValueError, match="index k and other integer index mixed"):      # genenerator_main.mac:146-152
            load_mac(path)


def test_mac_expressions_are_exact_and_sandboxed(tmp_path):
    """Integer arithmetic follows Maxima (2/3 is a rational, p^(1/2) a square root -> sqrt in the generated code), and an
    expression can only use arithmetic, plain calls and subscripts: no attribute access, comprehensions, lambdas, strings."""
    base = "x: [y];\nu: [dy];\nf[y]: y + dy*dx;\nL: %s;\nF: 0;\n"
    f = tmp_path / "t.mac"
    f.write_text(base % "(2/3)*dy^2 + p^(1/2)*y^2")
    P = load_mac(str(f), "T")
    assert sp.simplify(P.L - (sp.Rational(2, 3) * P.u[0] ** 2 + sp.sqrt(sp.Symbol("p", real=True)) * P.x[0] ** 2)) == 0
    assert "dm_sqrt(p[1][0])" in emit_func_c(lower(P))
    for bad in ("y.__class__", "[c for c in y]", "(lambda: 1)()", "__import__(1)", "'a'"):
        f.write_text(base % bad)
        with pytest.raises(ValueError):
            load_mac(str(f), "T")


def test_generator_cli_has_help(tmp_path):
    r = subprocess.run(["python", "-m", "ilqg_gen", "--help"], capture_output=True, text=True, cwd=str(tmp_path),
                       env=dict(os.environ, PYTHONPATH=os.path.join(ROOT, "ddp-generator_b200", "gen")))
    assert r.returncode == 0 and "outroot" in r.stdout and not os.listdir(str(tmp_path))
