"""Oracle side of the feedback-policy tests.  The gains are the reference's calc_derivs + back_pass on the tOptSet that iLQG() left
behind.  A policy rollout from another initial state is forward_pass's feedback branch at alpha = 0: the nominal l is scaled by 0
(ps_scale_l) and forward_pass(alpha = 1) runs from o.x0 = the sample (ps_set_x0), which computes u* + (0 * l) * 1 + L dx, the same
operations in the same order.  (forward_pass(alpha = 0) itself skips the gains.)  The two setters live in
tests/policy_oracle_shim.c, built here once per problem into a temporary directory."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import oracle_lib
import parity_util as PU

ROOT = oracle_lib.ROOT
_SHIMS = {}


def shim(problem, ddp, probdir=None):
    """tests/policy_oracle_shim.c compiled against the problem's structure layout, as the oracle's own C is (oracle/Makefile);
    `probdir`: the root of the generated problem code where it is not the package's problems/"""
    key = (problem, int(ddp))
    if key not in _SHIMS:
        out = os.path.join(tempfile.mkdtemp(prefix="policy_shim_"), f"shim_{problem}_{int(ddp)}.so")
        subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-std=gnu11", "-w", "-DHAVE_OCTAVE", "-DPRNT=h_prnt",
                        f"-DFULL_DDP={int(ddp)}", "-include", os.path.join(ROOT, "oracle", "prnt_decl.h"),
                        "-I" + os.path.join(ROOT, "oracle", "mex_stub"), "-I" + os.path.join(ROOT, "ddp-generator_b200", "csrc"),
                        "-I" + os.path.join(probdir or os.path.join(ROOT, "ddp-generator_b200", "problems"), problem), "-I" + os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "tests", "policy_oracle_shim.c"), "-o", out], check=True)
        L = C.CDLL(out)
        L.ps_set_x0.argtypes = [C.c_void_p, oracle_lib._dp]
        L.ps_scale_l.argtypes = [C.c_void_p, C.c_double]
        _SHIMS[key] = L
    return _SHIMS[key]


def oracle(problem, ddp, probdir=None):
    O = oracle_lib.OracleLib(PU.oracle_kinds(problem, ddp)[0], problem, ddp)
    O.shim = shim(problem, ddp, probdir)
    return O


class Solved:
    """one problem solved by the oracle with the model's parameters; policy() computes its gains, rollout() rolls them out"""

    def __init__(self, O, T, params, opts, x0, u0):
        s = self.s = O.solver(T)
        self.shim = O.shim
        assert self.shim.ps_sizeof_trajEl() == int(s.scalar("sizeof_trajEl")), "shim and oracle disagree on the layout"
        s.set_opts(opts)
        s.set_params(params)
        self.init_ok = bool(s.init(x0, u0))
        self.result = s.solve() if self.init_ok else -1
        self.x, self.u = s.get("x"), s.get("u")

    def policy(self):
        s = self.s
        self.derivs_ok = bool(s.calc_derivs())
        self.bp_ok = s.back_pass() == 0
        self.policy_ok = int(self.derivs_ok and self.bp_ok)
        g = dict(l=s.get("l"), L=s.get("L"), policy_ok=self.policy_ok, bp_done=int(self.bp_ok))
        g.update({k: s.scalar(k) for k in ("dV0", "dV1", "g_norm")})
        self.shim.ps_scale_l(s.h, 0.0)
        assert np.array_equal(s.get("l"), g["l"] * 0.0)
        return g

    def set_params(self, params):
        """the rollouts' parameters (a plant): the trajectory, gains and multipliers stay"""
        self.s.set_params(params)

    def rollout(self, x0):
        s = self.s
        self.shim.ps_set_x0(s.h, np.ascontiguousarray(x0, dtype=np.float64))
        ok, c = s.forward_pass(1.0)
        s.make_candidate_nominal()          # read the candidate, then swap the nominal back
        x, u = s.get("x"), s.get("u")
        s.make_candidate_nominal()
        return dict(ok=int(ok), cost=c, x=x, u=u, x_final=x[-1])

    def close(self):
        self.s.close()
