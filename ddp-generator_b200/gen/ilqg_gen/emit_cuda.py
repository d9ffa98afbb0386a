"""Emit the problem functions as sm_100a __device__ code (one header per problem).

Same statement lists as emit_c.py (lin.Scope), different leaf names: params are a flat array, auxiliary values
are locals recomputed from (x,u) instead of trajectory fields, outputs go to per-thread arrays.  The generic
kernels in csrc/ilqg_kernels.cuh are templated on the struct emitted here.

Reference semantics restated (file:line in /root/reference):
  step()/step_cost()  = one k of forward_pass: calcXVariableAux, clampU, calcXUVariableAux, ddpf, ddpL
                        (iLQG_func.tem:121-185, 40-73, 223-250)
  final_cost()        = calcFVariableAux + ddpF (iLQG_func.tem:179-182)
  derivs()            = calcLAuxDeriv + bp_derivsL + limitsU of one k (iLQG_func.tem:187-221, 75-119, 252-289)
  derivs_final()      = calcFAuxDeriv + bp_derivsF (iLQG_func.tem:291-310)
  consts()/unpack()   = init_running's time-invariant entries (iLQG_func.tem:312-345) / the time-varying ones
  add2()              = the FULL_DDP tensor contractions Vx.fxx, Vx.fuu, Vx.fxu (back_pass.c:95-131), sparse
  mult_*()            = update_multipliers_running/final (iLQG_func.tem:417-509)
"""
from __future__ import annotations

from .lin import Scope, render_operand, render_rhs


class CuNames:
    def __init__(self, m, final=False):
        self.map = {}
        for i, s in enumerate(m.x):
            self.map[s] = f"x[{i}]"
        for i, s in enumerate(m.u):
            self.map[s] = f"u[{i}]"
        kidx = 0
        for d in m.params:
            if d.size == -1:
                self.map[d.symbols[0]] = f"pk({kidx}, k)"
                kidx += 1
            else:
                for ei, s in enumerate(d.symbols):
                    self.map[s] = f"p[{d.flat_index + ei}]"
        for a in m.aux:
            self.map[a.sym] = f"aux_{a.name}"
        for a in m.daux:
            self.map[a.sym] = f"daux_{a.name}"
        self.map[m.w_pen] = "w_pen"
        off = 0
        for kind in (("fe", "fi") if final else ("le", "li")):
            for r in m.mult[kind]:
                self.map[r["mu"]] = f"mu[{off}]"
                off += 1
        # multipliers of the other context are never referenced in this context
        for kind in (("le", "li") if final else ("fe", "fi")):
            for r in m.mult[kind]:
                self.map[r["mu"]] = "mu_wrong_context"

    def __call__(self, s):
        return self.map[s]


def render(sc: Scope, names, tname, indent="        ", guards=True):
    out = []
    for it in sc.items:
        if it[0] == "tmp":
            out.append(f"{indent}const double {it[1]} = {render_rhs(it[2], names)};")
        elif it[0] == "out":
            lhs, decl = tname(it[1])
            out.append(f"{indent}{decl}{lhs} = {render_operand(it[2], names)};")
            if it[3] and guards:
                out.append(f"{indent}ok &= dm_isfinite({lhs});")
        elif it[0] == "sincos":
            out.append(f"{indent}double {it[1]}, {it[2]}; dm_sincos({render_operand(it[3], names)}, &{it[1]}, &{it[2]});")
        elif it[0] == "raw":
            out.append(it[1](names, indent))
    return "\n".join(out)


def emit_device(m, struct_name) -> str:
    nx, nu = m.nx, m.nu
    # flat param indexing (time-invariant params only)
    flat = 0
    nkp = 0
    for d in m.params:
        if d.size == -1:
            d.flat_index = -1
            nkp += 1
        else:
            d.flat_index = flat
            flat += d.size
    NR = CuNames(m, final=False)
    NF = CuNames(m, final=True)

    # canonical order of time-varying entries stored per step
    blocks1 = [("fx", m.fx), ("fu", m.fu), ("cx", m.cx), ("cxx", m.cxx), ("cu", m.cu), ("cuu", m.cuu), ("cxu", m.cxu)]
    blocks2 = [("fxx", m.fxx), ("fuu", m.fuu), ("fxu", m.fxu)]
    v1 = [(k, e) for k, es in blocks1 for e in es if e.time_var]
    v2 = [(k, e) for k, es in blocks2 for e in es if e.time_var]
    v1_pos = {(k, e.idx): i for i, (k, e) in enumerate(v1)}
    v2_pos = {(k, e.idx): i for i, (k, e) in enumerate(v2)}
    n_v1e = len(v1)
    off_lower = n_v1e
    off_upper = n_v1e + nu
    nv1 = n_v1e + 2 * nu
    if m.has_hx:
        off_lsign = nv1
        off_usign = nv1 + nu
        off_lhx = nv1 + 2 * nu
        off_uhx = off_lhx + nx * nu
        nv1 = off_uhx + nx * nu
    nv2 = len(v2)
    n_mu_r = m.n_mu["le"] + m.n_mu["li"]
    n_mu_f = m.n_mu["fe"] + m.n_mu["fi"]

    daux_names = {a.name for a in m.daux}

    def aux_t(t):
        k = t[0]
        if k == "field":      # aux / daux value -> local
            return (f"{'daux_' if t[1] in daux_names else 'aux_'}{t[1]}", "const double ")
        if k == "var":
            return (t[1], "")
        if k == "xnext":
            return (f"x_next[{t[1]}]", "")
        if k == "c":
            return ("c", "")
        if k == "v1":
            return (f"v1[{t[1]}]", "")
        if k == "v2":
            return (f"v2[{t[1]}]", "")
        if k == "arr":
            return (f"{t[1]}[{t[2]}]", "")
        raise ValueError(t)

    def aux_outs(sc, infos, pred):
        for a in infos:
            if pred(a):
                sc.out(("field", a.name), a.expr, not a.atomic)

    o = []
    o.append(f"/* Generated by ilqg_gen (ddp-generator_b200/gen) for problem '{m.name}'. Do not edit. */")
    o.append("#pragma once\n#include \"dm_math.h\"\n")
    o.append(f"struct {struct_name} {{")
    o.append(f"    static constexpr int NX = {nx}, NU = {nu}, NQXX = {m.nqxx}, NQUU = {m.nquu}, NQXU = {m.nqxu};")
    o.append(f"    static constexpr int NPF = {max(flat, 1)}, NPF_USED = {flat}, NKP = {nkp};")
    o.append(f"    static constexpr int N_MU_LE = {m.n_mu['le']}, N_MU_LI = {m.n_mu['li']}, N_MU_FE = {m.n_mu['fe']}, N_MU_FI = {m.n_mu['fi']};")
    o.append(f"    static constexpr int N_MU_R = {n_mu_r}, N_MU_F = {n_mu_f};")
    o.append(f"    static constexpr bool HAS_HX = {'true' if m.has_hx else 'false'};")
    o.append(f"    static constexpr int NV1 = {nv1}, NV2 = {max(nv2, 1)}, NV2_USED = {nv2};")
    o.append(f"    static constexpr int OFF_LOWER = {off_lower}, OFF_UPPER = {off_upper};")
    o.append(f"    static constexpr int NH = {len(m.h)};")
    o.append(f"    static constexpr bool COOP = {'true' if nx > 6 else 'false'};   /* warp-cooperative backward pass (state too large for one lane) */")
    o.append(f"    static const char *name() {{ return \"{m.name}\"; }}")
    o.append("    static int param_count() { return %d; }" % len(m.params))
    o.append("    static const char *param_name(int i) { const char *n[] = {%s}; return n[i]; }"
             % ", ".join([f'"{d.name}"' for d in m.params] + ['""']))
    o.append("    static int param_size(int i) { const int n[] = {%s}; return n[i]; }"
             % ", ".join([str(d.size) for d in m.params] + ["0"]))
    o.append("")
    # pk: accessor of the [k]-indexed parameters, pk(j, k) (PkShared / PkTrack in csrc/ilqg_kernels.cuh)
    ARGS = "const double *p, const PK &pk, int k, int N, double w_pen, const double *mu"
    TPK = "template <class PK> "
    UNUSED = "        (void)p; (void)pk; (void)k; (void)N; (void)w_pen; (void)mu;"

    # ---- rollout step ----------------------------------------------------------------------------------------
    def step_body(cost_only, clamp=True):
        scA = Scope("a")
        aux_outs(scA, m.aux, lambda a: a.used_running and not a.dep_u)
        if not cost_only and clamp:
            for rec in m.h:
                scA.out(("var", "limit"), rec["limit"], False)
                j, cmp_ = rec["input"], (">" if rec["sign"] > 0 else "<")
                scA.raw(lambda names, ind, j=j, cmp_=cmp_: f"{ind}if (u[{j}] {cmp_} limit) u[{j}] = limit;")
        scB = Scope("b")
        aux_outs(scB, m.aux, lambda a: a.used_running and a.dep_u)
        if not cost_only:
            for i, e in enumerate(m.f):
                scB.out(("xnext", i), e, True)
        scB.out(("c",), m.L, True)
        return render(scA, NR, aux_t) + "\n" + render(scB, NR, aux_t)

    o.append("    /* one timestep of the rollout: control already formed in u (pre-clamp); clamps u in place */")
    o.append(f"    {TPK}__device__ __forceinline__ static bool step(const double *x, double *u, {ARGS}, double *x_next, double &c) {{")
    o.append("        bool ok = true; double limit; (void)limit;\n" + UNUSED)
    o.append(step_body(False))
    o.append("        return ok;\n    }\n")
    o.append("    /* dynamics and cost of one timestep at the given u, NOT clamped (single evaluations: iLQG_MMex.tem mode 0) */")
    o.append(f"    {TPK}__device__ __forceinline__ static bool step_free(const double *x, const double *u, {ARGS}, double *x_next, double &c) {{")
    o.append("        bool ok = true;\n" + UNUSED)
    o.append(step_body(False, clamp=False))
    o.append("        return ok;\n    }\n")
    o.append(f"    {TPK}__device__ __forceinline__ static bool step_cost(const double *x, const double *u, {ARGS}, double &c) {{")
    o.append("        bool ok = true;\n" + UNUSED)
    o.append(step_body(True))
    o.append("        return ok;\n    }\n")

    # ---- user outputs g (calcG, iLQG_func.tem:511-521) ----------------------------------------------------------------
    scg = Scope("g")
    aux_outs(scg, m.aux, lambda a: a.used_running)
    for i, e in enumerate(m.g):
        scg.out(("arr", "g", i), e, False)
    o.append(f"    static constexpr int NG = {len(m.g)};")
    o.append(f"    {TPK}__device__ __forceinline__ static void calc_g(const double *x, const double *u, {ARGS}, double *g) {{")
    o.append("        (void)x; (void)u; (void)g;\n" + UNUSED)
    o.append(render(scg, NR, aux_t, guards=False) if m.g else "")
    o.append("    }\n")

    # ---- final cost ------------------------------------------------------------------------------------------
    sc = Scope("f")
    aux_outs(sc, m.aux, lambda a: a.used_final)
    sc.out(("c",), m.F, True)
    o.append(f"    {TPK}__device__ __forceinline__ static bool final_cost(const double *x, {ARGS}, double &c) {{")
    o.append("        bool ok = true;\n" + UNUSED)
    o.append(render(sc, NF, aux_t))
    o.append("        return ok;\n    }\n")

    # ---- derivatives of one step ---------------------------------------------------------------------------------
    def derivs_body(full):
        sc = Scope("d")
        aux_outs(sc, m.aux, lambda a: a.used_running)
        # calcLAuxDeriv evaluates -- and guards -- EVERY auxiliary derivative whatever FULL_DDP is (iLQG_func.tem:252-260: only
        # the fxx/fuu/fxu blocks sit under #if FULL_DDP), so a non-finite second-order auxiliary derivative fails calc_derivs
        # of a FULL_DDP=0 build too.  The first-order-only variant therefore still evaluates them, for their guards alone.
        aux_outs(sc, m.daux, lambda a: a.used_running and (full or _needed_first(a) or not a.atomic))
        for key, e in v1:
            sc.out(("v1", v1_pos[(key, e.idx)]), e.expr, not e.atomic)
        if full:
            for key, e in v2:
                sc.out(("v2", v2_pos[(key, e.idx)]), e.expr, not e.atomic)
        # limitsU
        lines = []
        lines.append("        double lower[NU], upper[NU]; int lower_idx[NU], upper_idx[NU];")
        lines.append("        #pragma unroll\n        for (int i = 0; i < NU; i++) { lower[i] = -dm_inf(); upper[i] = dm_inf(); lower_idx[i] = -1; upper_idx[i] = -1; }")
        sc.raw(lambda names, ind: "\n".join(lines))
        for rec in m.h:
            sc.out(("var", "limit"), rec["limit"], False)
            j, hi = rec["input"], rec["index"]
            if rec["sign"] > 0:
                sc.raw(lambda names, ind, j=j, hi=hi: f"{ind}if (upper[{j}] > limit) {{ upper[{j}] = limit; upper_idx[{j}] = {hi}; }}")
            else:
                sc.raw(lambda names, ind, j=j, hi=hi: f"{ind}if (lower[{j}] < limit) {{ lower[{j}] = limit; lower_idx[{j}] = {hi}; }}")
        sc.raw(lambda names, ind: f"{ind}#pragma unroll\n{ind}for (int i = 0; i < NU; i++) {{ v1[OFF_LOWER + i] = lower[i] - u[i]; v1[OFF_UPPER + i] = upper[i] - u[i]; }}")
        if m.has_hx:
            # active-constraint gradient and sign per input and side (iLQG_func.tem:101-118)
            for rec in m.h:
                for l_, e in enumerate(rec["hx"]):
                    sc.out(("var", f"const double hx_{rec['index']}_{l_}"), e, False)
            for side, idxn, offs, offh in (("lower", "lower_idx", off_lsign, off_lhx), ("upper", "upper_idx", off_usign, off_uhx)):
                for j in range(nu):
                    def emit(names, ind, side=side, idxn=idxn, offs=offs, offh=offh, j=j):
                        ls = [f"{ind}v1[{offs + j}] = 0.0;"]
                        for l_ in range(nx):
                            ls.append(f"{ind}v1[{offh + j * nx + l_}] = 0.0;")
                        for rec in m.h:
                            if rec["input"] != j or (rec["sign"] > 0) != (side == "upper"):
                                continue
                            hi = rec["index"]
                            ls.append(f"{ind}if ({idxn}[{j}] == {hi}) {{ v1[{offs + j}] = {float(rec['sign'])!r};"
                                      + "".join(f" v1[{offh + j * nx + l_}] = hx_{hi}_{l_};" for l_ in range(nx)) + " }")
                        return "\n".join(ls)
                    sc.raw(emit)
        return render(sc, NR, aux_t)

    def _needed_first(a):
        # aux derivatives needed when second-order dynamics blocks are not generated: those reachable from
        # the first-order / cost entries.  Computed lazily below.
        return a.name in needed_no2

    import sympy as sp
    by_sym = {a.sym: a for a in m.aux + m.daux}
    needed_no2 = set()
    stack = []
    for key, e in v1:
        stack.extend(s for s in e.expr.free_symbols if s in by_sym)
    for rec in m.h:
        for e in [rec["limit"]] + rec["hx"]:
            stack.extend(s for s in sp.sympify(e).free_symbols if s in by_sym)
    while stack:
        s = stack.pop()
        a = by_sym[s]
        if a.name in needed_no2:
            continue
        needed_no2.add(a.name)
        stack.extend(t for t in a.expr.free_symbols if t in by_sym)

    o.append("    __device__ __forceinline__ static double dm_inf() { return dm_from_bits(0x7ff0000000000000ull); }\n")
    for full, fname in ((False, "derivs"), (True, "derivs_full")):
        o.append(f"    /* time-varying derivative entries of step k (+ shifted input limits){' incl. second-order dynamics' if full else ''} */")
        o.append(f"    {TPK}__device__ __forceinline__ static bool {fname}(const double *x, const double *u, {ARGS}, double *v1, double *v2) {{")
        o.append("        bool ok = true; double limit; (void)limit; (void)v2;\n" + UNUSED)
        o.append(derivs_body(full))
        o.append("        return ok;\n    }\n")

    # ---- final derivatives (dense: constants and varying alike) ------------------------------------------------------
    sc = Scope("g")
    aux_outs(sc, m.aux, lambda a: a.used_final)
    aux_outs(sc, m.daux, lambda a: a.used_final)
    for e in m.Fcx:
        sc.out(("arr", "cx", e.idx), e.expr, not e.atomic and e.time_var)
    for e in m.Fcxx:
        sc.out(("arr", "cxx", e.idx), e.expr, not e.atomic and e.time_var)
    o.append(f"    {TPK}__device__ __forceinline__ static bool derivs_final(const double *x, {ARGS}, double *cx, double *cxx) {{")
    o.append("        bool ok = true;\n" + UNUSED)
    o.append(render(sc, NF, aux_t))
    o.append("        return ok;\n    }\n")

    # ---- constants + unpack into a dense per-step record ---------------------------------------------------------------
    sc = Scope("k")
    aux_outs(sc, m.aux, lambda a: a.used_running and not a.time_var)
    aux_outs(sc, m.daux, lambda a: a.used_running and not a.time_var)
    for key, es in blocks1:
        for e in es:
            if not e.time_var:
                sc.out(("arr", f"D.{key}", e.idx), e.expr, False)
    o.append("    template <class DT> __device__ __forceinline__ static void consts(const double *p, DT &D) {\n        (void)p;")
    o.append(render(sc, NR, aux_t, guards=False))
    if m.has_hx is False:
        pass
    o.append("    }\n")
    lines = []
    for key, e in v1:
        lines.append(f"        D.{key}[{e.idx}] = v1[{v1_pos[(key, e.idx)]}];")
    lines.append("        #pragma unroll\n        for (int i = 0; i < NU; i++) { D.lower[i] = v1[OFF_LOWER + i]; D.upper[i] = v1[OFF_UPPER + i]; }")
    if m.has_hx:
        lines.append(f"        #pragma unroll\n        for (int i = 0; i < NU; i++) {{ D.lower_sign[i] = v1[{off_lsign} + i]; D.upper_sign[i] = v1[{off_usign} + i]; }}")
        lines.append(f"        #pragma unroll\n        for (int i = 0; i < NX * NU; i++) {{ D.lower_hx[i] = v1[{off_lhx} + i]; D.upper_hx[i] = v1[{off_uhx} + i]; }}")
    o.append("    template <class DT> __device__ __forceinline__ static void unpack(const double *v1, DT &D) {")
    o.append("\n".join(lines))
    o.append("    }\n")

    # ---- FULL_DDP contractions, skipping structurally zero entries (back_pass.c:95-131) ----------------------------------
    def contraction(entries, pos, nout, outname):
        # reference: for j: d1 = 0; for i ascending: d1 += Vx[i]*T[j + i*nout]; out[j] += d1
        ls = []
        ent = {e.idx: e for e in entries}
        sck = Scope("z" + outname[-2:])
        for j in range(nout):
            terms = []
            for i in range(nx):
                e = ent[j + i * nout]
                if e.expr == 0:
                    continue
                if e.time_var:
                    terms.append((i, f"v2[{pos[(outname_key[outname], e.idx)]}]"))
                else:
                    r = sck.ref(e.expr)
                    terms.append((i, render_operand(r, NR)))
            if not terms:
                continue
            ls.append((j, terms))
        pre = render(sck, NR, aux_t, guards=False)
        body = []
        for j, terms in ls:
            body.append("        { double d1 = 0.0;" + "".join(f" d1 += Vx[{i}] * {t};" for i, t in terms) + f" {outname}[{j}] += d1; }}")
        return pre, "\n".join(body)

    outname_key = {"Qxx": "fxx", "Quu": "fuu", "Qxu": "fxu"}
    o.append("    __device__ __forceinline__ static void add2_Qxu(const double *Vx, const double *v2, const double *p, double *Qxu) {\n        (void)Vx; (void)v2; (void)p; (void)Qxu;")
    pre, body = contraction(m.fxu, v2_pos, m.nqxu, "Qxu"); o.append(pre); o.append(body); o.append("    }")
    o.append("    __device__ __forceinline__ static void add2_Quu(const double *Vx, const double *v2, const double *p, double *Quu) {\n        (void)Vx; (void)v2; (void)p; (void)Quu;")
    pre, body = contraction(m.fuu, v2_pos, m.nquu, "Quu"); o.append(pre); o.append(body); o.append("    }")
    o.append("    __device__ __forceinline__ static void add2_Qxx(const double *Vx, const double *v2, const double *p, double *Qxx) {\n        (void)Vx; (void)v2; (void)p; (void)Qxx;")
    pre, body = contraction(m.fxx, v2_pos, m.nqxx, "Qxx"); o.append(pre); o.append(body); o.append("    }\n")

    # ---- structural-zero masks of the first-order blocks (compile-time): the lane-per-problem backward pass skips
    #      multiplications by entries that are identically zero for this problem -------------------------------------------
    for key, entries in blocks1:
        ent = sorted(entries, key=lambda e: e.idx)
        bits = ", ".join("false" if (not e.time_var and e.expr == 0) else "true" for e in ent)
        o.append("    struct Mask_%s { __host__ __device__ static constexpr bool nz(int i) { constexpr bool t[] = {%s}; return t[i]; } };" % (key, bits))
    o.append("")

    # ---- data-driven forms for the warp-cooperative backward pass ------------------------------------------------------
    # (a) destination of every stored time-varying entry inside the dense per-step record (struct Dense in
    #     ilqg_kernels.cuh: fx fu cx cxx cu cuu cxu lower upper lower_sign upper_sign lower_hx upper_hx, contiguous doubles)
    offs, acc_ = {}, 0
    for key, size in (("fx", nx * nx), ("fu", nx * nu), ("cx", nx), ("cxx", m.nqxx), ("cu", nu), ("cuu", m.nquu), ("cxu", m.nqxu),
                      ("lower", nu), ("upper", nu), ("lower_sign", nu), ("upper_sign", nu), ("lower_hx", nx * nu), ("upper_hx", nx * nu)):
        offs[key] = acc_
        acc_ += size
    dst = [offs[k] + e.idx for k, e in v1] + [offs["lower"] + i for i in range(nu)] + [offs["upper"] + i for i in range(nu)]
    if m.has_hx:
        dst += [offs["lower_sign"] + i for i in range(nu)] + [offs["upper_sign"] + i for i in range(nu)]
        dst += [offs["lower_hx"] + i for i in range(nx * nu)] + [offs["upper_hx"] + i for i in range(nx * nu)]
    assert len(dst) == nv1
    o.append("    static constexpr int DENSE_SIZE = %d;" % acc_)
    o.append("    __device__ __forceinline__ static int v1_dst(int j) { static constexpr unsigned short t[] = {%s}; return t[j]; }"
             % ", ".join(str(d) for d in dst))
    # (b) FULL_DDP contractions as sparse term lists per output entry (reference loop: back_pass.c:95-131); constant
    #     (parameter-only) tensor entries get slots in c2[], filled once by consts2()
    sck2 = Scope("q")
    c2_slots = []

    def csr(entries, pos, nout, key):
        ent = {e.idx: e for e in entries}
        start, vi, src = [0], [], []
        for j in range(nout):
            for i in range(nx):
                e = ent[j + i * nout]
                if e.expr == 0:
                    continue
                vi.append(i)
                if e.time_var:
                    src.append(pos[(key, e.idx)])
                else:
                    c2_slots.append(e.expr)
                    src.append(-len(c2_slots))
            start.append(len(vi))
        return start, vi, src

    for nm, entries, nout, key in (("xu", m.fxu, m.nqxu, "fxu"), ("uu", m.fuu, m.nquu, "fuu"), ("xx", m.fxx, m.nqxx, "fxx")):
        start, vi, src = csr(entries, v2_pos, nout, key)
        o.append("    __device__ __forceinline__ static int s2%s_start(int j) { static constexpr unsigned short t[] = {%s}; return t[j]; }" % (nm, ", ".join(map(str, start))))
        o.append("    __device__ __forceinline__ static int s2%s_vx(int t_) { static constexpr unsigned char t[] = {%s}; return t[t_]; }" % (nm, ", ".join(map(str, vi + [0]))))
        o.append("    __device__ __forceinline__ static int s2%s_src(int t_) { static constexpr short t[] = {%s}; return t[t_]; }" % (nm, ", ".join(map(str, src + [0]))))
        # number of terms / of output entries that have terms (the warp-cooperative kernel forms all products lane-parallel and
        # sizes its per-lane term and entry slots from these)
        o.append("    static constexpr int NT2%s = %d, NE2%s = %d;" % (nm.upper(), len(vi), nm.upper(), sum(1 for j in range(nout) if start[j + 1] > start[j])))
    o.append("    static constexpr int NC2 = %d;" % max(len(c2_slots), 1))
    for i, e in enumerate(c2_slots):
        sck2.out(("arr", "c2", i), e, False)
    o.append("    __device__ __forceinline__ static void consts2(const double *p, double *c2) {\n        (void)p; (void)c2;")
    o.append(render(sck2, NR, aux_t, guards=False))
    o.append("    }\n")

    # ---- multiplier updates ----------------------------------------------------------------------------------------------
    # h values of the constraints of one context, evaluated from the state (the reference reads the aux value the
    # last rollout stored in the nominal trajectory, which is the same function of the same x,u)
    def mult_fn(final):
        kinds = ("fe", "fi") if final else ("le", "li")
        NN = NF if final else NR
        sc = Scope("m")
        aux_outs(sc, m.aux, (lambda a: a.used_final) if final else (lambda a: a.used_running))
        off = 0
        for kind in kinds:
            for r in m.mult[kind]:
                sc.out(("arr", "hval", off), r["h"], False)
                if kind in ("fe", "le"):
                    sc.out(("arr", "mu_next", off), r["next"], False)
                else:
                    sc.out(("var", f"const double nA{off}"), r["next_A"], False)
                    sc.out(("var", f"const double nI{off}"), r["next_I"], False)
                    sc.raw(lambda names, ind, off=off: f"{ind}mu_next[{off}] = (hval[{off}] >= 0) ? nA{off} : nI{off};")
                off += 1
        return render(sc, NN, aux_t, guards=False)

    o.append("    /* constraint values and updated multipliers; is_ineq[i] tells which test update_multipliers applies */")
    o.append(f"    {TPK}__device__ __forceinline__ static void mult_running(const double *x, const double *u, {ARGS}, double *hval, double *mu_next) {{")
    o.append(UNUSED + "\n        (void)x; (void)u; (void)hval; (void)mu_next;")
    o.append(mult_fn(False))
    o.append("    }")
    o.append(f"    {TPK}__device__ __forceinline__ static void mult_final(const double *x, {ARGS}, double *hval, double *mu_next) {{")
    o.append(UNUSED + "\n        (void)x; (void)hval; (void)mu_next;")
    o.append(mult_fn(True))
    o.append("    }")
    o.append("};\n")
    return "\n".join(o)
