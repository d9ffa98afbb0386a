"""Shared helpers for parity tests: run the oracle (reference or port) and the CUDA library on the same inputs and
collect comparable records."""
from __future__ import annotations

import numpy as np

import oracle_lib


def oracle_kinds(problem, ddp):
    """Checkers available on this machine: the compiled reference (oracle/_ref) and/or the C port."""
    return [k for k in ("reference", "port") if oracle_lib.available(k, problem, ddp)]


def oracle_record(kind, problem, ddp, T, params, x0, u0, opts, qp_cap=0):
    O = oracle_lib.OracleLib(kind, problem, ddp)
    s = O.solver(T)
    s.set_opts(opts)
    s.set_params(params)
    if qp_cap:
        s.qp_trace_enable(qp_cap)
    ok = s.init(x0, u0)
    rec = dict(init_ok=ok)
    if not ok:
        return rec
    rec["cost0"] = s.scalar("cost")
    rec["result"] = s.solve()
    rec["iterations"] = int(s.scalar("iterations"))
    for k in ("cost", "lambda", "g_norm", "w_pen_l", "w_pen_f", "dV0", "dV1"):
        rec[k] = s.scalar(k)
    for k in ("x", "u", "l", "L"):
        rec[k] = s.get(k)
    rec["mult_f"] = s.get("mult_f")
    rec["tr_lambda"] = s.trace("lambda")
    rec["tr_alpha"] = s.trace("alpha_idx").astype(int)
    rec["tr_newcost"] = s.trace("new_cost")
    rec["tr_iter"] = s.trace("iter").astype(int)
    rec["n_ls"] = rec["tr_lambda"].size
    rec["n_bp"] = s.bp_trace("lambda").size
    if qp_cap:
        rec["qp"] = s.qp_trace()
    s.close()
    return rec


def gpu_records(problem, ddp, T, params, x0, u0, opts, flags=1, tuning=None):
    """Solve a batch on the GPU; returns a list of per-problem records shaped like oracle_record()."""
    import ilqg_b200

    x0 = np.atleast_2d(x0)
    u0 = np.asarray(u0)
    if u0.ndim == 2:
        u0 = u0[None]
    B = x0.shape[0]
    s = ilqg_b200.BatchSolver(problem, ddp, B, T, flags=flags)
    s.set_options(opts)
    s.set_params(params)
    for name, value in (tuning or {}).items():
        s.set_tuning(name, value)
    out = s.solve(x0, u0)
    sc = {k: s.get(k) for k in ("lambda", "g_norm", "w_pen_l", "w_pen_f", "dV0", "dV1")}
    l, L = s.get("l"), s.get("L")
    tr_l, tr_c = s.get("tr_lambda"), s.get("tr_newcost")
    tr_a, tr_cl = s.get_int("tr_alpha"), s.get_int("tr_clamp")
    nbp = s.get_int("n_backpass")
    muf = s.get("mu_f") if s.L.lib.ilqgb_nx() and tr_l is not None else None
    recs = []
    for b in range(B):
        n = int(out["n_linesearch"][b])
        recs.append(dict(result=int(out["success"][b]), iterations=int(out["iterations"][b]), cost=out["cost"][b],
                         x=out["x"][b], u=out["u"][b], l=l[b], L=L[b], n_ls=n, n_bp=int(nbp[b]),
                         tr_lambda=tr_l[b][:n], tr_alpha=tr_a[b][:n], tr_newcost=tr_c[b][:n], tr_clamp=tr_cl[b],
                         **{k: v[b] for k, v in sc.items()}))
    s.close()
    return recs


def assert_same(gpu, ora, what, keys=("result", "iterations", "n_ls", "n_bp", "cost", "lambda", "g_norm", "w_pen_l",
                                       "w_pen_f", "tr_alpha", "tr_lambda", "tr_newcost", "x", "u")):
    for k in keys:
        a, b = np.asarray(gpu[k]), np.asarray(ora[k])
        assert a.shape == b.shape, f"{what}: {k} shape {a.shape} vs {b.shape}"
        assert np.array_equal(a, b), f"{what}: {k} differs (max abs diff {np.max(np.abs(a.astype(float) - b.astype(float)))})"


# ---- one batch solved on the GPU against the oracle called once per problem (test_gpu_variants.py, test_gpu_shapes.py) ----------
ORACLE_KEYS = assert_same.__defaults__[0] + ("l", "L", "dV0", "dV1")
KEYS = ("result", "iterations", "n_ls", "n_bp", "cost", "lambda", "g_norm", "w_pen_l", "w_pen_f", "dV0", "dV1", "tr_alpha",
        "tr_lambda", "tr_newcost", "tr_clamp", "x", "u", "l", "L")          # as tests/test_gpu_split.py
HOOKS = ("bp_split", "cw_lpp", "bp_latency", "ls_tail_from", "ls_commit_par")
CW_WARPS = 4      # warps per block of k_backpass_warp


class Case:
    """One set of inputs: shared parameters, optional per-problem parameter sets pp {name: [B, size]} and tracks
    {name: [B, len]} read from window offset `off`."""

    def __init__(self, problem, ddp, T, params, x0, u0, opts, pp=None, tracks=None, off=0):
        self.problem, self.ddp, self.T, self.params, self.x0, self.u0, self.opts = problem, ddp, T, params, x0, u0, opts
        self.pp, self.tracks, self.off = pp or {}, tracks or {}, off
        self.B = x0.shape[0]

    def params_of(self, b):
        p = dict(self.params, **{k: v[b] for k, v in self.pp.items()})
        return dict(p, **{k: v[b, self.off:self.off + self.T + 1] for k, v in self.tracks.items()})


def run(c, tuning=None, lib_dir=None):
    """Solve the batch on the GPU: per-problem records shaped like parity_util.oracle_record, and the hooks."""
    import ilqg_b200

    s = ilqg_b200.BatchSolver(c.problem, c.ddp, c.B, c.T, flags=ilqg_b200.TRACE, lib_dir=lib_dir)
    s.set_options(c.opts)
    s.set_params(c.params)
    if c.pp:
        s.set_params_batch(c.pp)
    for k, v in c.tracks.items():
        s.set_param_track(k, v)
    if c.tracks:
        s.set_track_offset(c.off)
    for k, v in (tuning or {}).items():
        s.set_tuning(k, v)
    out = s.solve(c.x0, c.u0)
    sc = {k: s.get(k) for k in ("lambda", "g_norm", "w_pen_l", "w_pen_f", "dV0", "dV1")}
    l, L = s.get("l"), s.get("L")
    tr_l, tr_c = s.get("tr_lambda"), s.get("tr_newcost")
    tr_a, tr_cl = s.get_int("tr_alpha"), s.get_int("tr_clamp")
    nbp = s.get_int("n_backpass")
    hooks = {k: s.get_int(k) for k in HOOKS}
    s.close()
    recs = []
    for b in range(c.B):
        n = int(out["n_linesearch"][b])
        recs.append(dict(result=int(out["success"][b]), iterations=int(out["iterations"][b]), cost=out["cost"][b],
                         x=out["x"][b], u=out["u"][b], l=l[b], L=L[b], n_ls=n, n_bp=int(nbp[b]),
                         tr_lambda=tr_l[b][:n], tr_alpha=tr_a[b][:n], tr_newcost=tr_c[b][:n], tr_clamp=tr_cl[b],
                         **{k: v[b] for k, v in sc.items()}))
    for k, v in hooks.items():
        assert np.all(v == v[0]), f"hook {k} differs between problems of one chunk"
    return recs, {k: int(v[0]) for k, v in hooks.items()}


_ORACLE = {}


def oracle(name, c):
    if name not in _ORACLE:
        kind = oracle_kinds(c.problem, c.ddp)[0]
        opts = {k: float(v) if np.isscalar(v) else v for k, v in c.opts.items()}
        _ORACLE[name] = [oracle_record(kind, c.problem, c.ddp, c.T, c.params_of(b), c.x0[b], c.u0[b], opts) for b in range(c.B)]
    return _ORACLE[name]


def check(name, c, recs, base):
    """recs against the oracle (every problem) and against the axis' baseline variant `base` (records of the same inputs)."""
    for b, (g, o) in enumerate(zip(recs, oracle(name, c))):
        if not o["init_ok"]:
            assert g["result"] == -1 and g["n_ls"] == 0, f"{name} b{b}: failed initial rollout not reported"
            continue
        assert_same(g, o, f"{name} b{b} vs oracle", keys=ORACLE_KEYS)
    for b, (g, r) in enumerate(zip(recs, base)):
        for k in KEYS:
            assert np.array_equal(np.asarray(g[k]), np.asarray(r[k]), equal_nan=True), f"{name} b{b}: {k} differs from the baseline variant"


def clamped(recs, inputs=None):
    """number of (problem, step) box-QP solutions with a clamped input (of `inputs`, default any)"""
    mask = sum(3 << (2 * i) for i in inputs) if inputs is not None else 0xffff
    return sum(int(np.count_nonzero(np.asarray(r["tr_clamp"]) & mask)) for r in recs)


def deep(recs):
    """accepted or rejected line-search results at alpha index >= 4"""
    return sum(int((np.asarray(r["tr_alpha"]) >= 4).sum()) for r in recs)


def retried(recs):
    return sum(r["n_bp"] > r["iterations"] for r in recs)


def mixed_groups(recs, size):
    """groups of `size` consecutive problems (the problems of one warp or block) whose iteration counts differ"""
    it = [r["iterations"] for r in recs]
    return sum(len(set(it[g:g + size])) > 1 for g in range(0, len(it), size))
