/* ilqg_kernels.cuh -- batched iLQG / control-limited DDP kernels for sm_100a (B200), templated on a generated
 * problem struct P (problems/<name>/<name>_device.cuh).
 *
 * Execution model ("lane per problem"): the batch of independent problems is the parallel axis.  Lane b of a warp
 * owns problem b for the phases that are sequential in time (backward pass, rollouts) and keeps its value
 * function, Q-function and box-QP state in registers; the derivative pass is parallel over (problem, timestep).
 * Every array in HBM is structure-of-arrays with the problem index fastest ([k][field][b]), so each warp-level load
 * or store touches one fully used 256-byte segment.
 *
 * Bit-exact parity with the reference C solver is a design constraint: every floating-point operation is issued
 * in the reference's order (single accumulators, ascending indices, explicit symmetrisation; see the citations on
 * each function), the translation unit is compiled with -fmad=false, and transcendental functions come from
 * dm_math.h on both sides.
 *
 * Reference functions restated here (file:line in /root/reference):
 *   add_mul_vec / add_square_tri / add_mul2_tri   matMult.c:3-12 / 14-46 / 48-72
 *   box_qp (+ masked Cholesky / inverse)          boxQP.c:39-238, cholesky.c:6-27, 51-74
 *   k_backpass                                    back_pass.c:38-257 + iLQG.c:261-303 (lambda loop, gradient exit)
 *   k_ls_round, k_init                            iLQG_func.tem:121-185 (forward_pass), line_search.c:33-78,
 *                                                 iLQG.c:311-361 (accept / reject), iLQG_mex.c:108-120 (initial)
 *   k_derivs                                      iLQG_func.tem:187-221 (calc_derivs)
 *   k_post                                        iLQG_func.tem:417-509 (update_multipliers) + cost-only pass
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "dm_math.h"
#include "ilqg_work.h"

namespace ilqg {

constexpr int MAX_ALPHA = ILQG_MAX_ALPHA;
constexpr int BP_BLOCK = 64;   /* threads per block for the sequential-in-time kernels */
constexpr int DV_BLOCK = 128;  /* threads per block for the derivative kernel */
#ifndef ILQG_BP_MINBLOCKS
#define ILQG_BP_MINBLOCKS 8   /* 128 registers/thread: 16 warps per SM; measured faster than 212 registers at 8 warps */
#endif
#ifndef ILQG_LS_MINBLOCKS
#define ILQG_LS_MINBLOCKS 1
#endif

enum { ST_RUNNING = 0, ST_DONE = 1 };
enum { POST_NONE = 0, POST_MULT = 1, POST_COST = 2 };

using Opts = ilqg_opts;
using Work = ilqg_work;

template <class P> struct ParamBlock { double v[P::NPF]; };

/* Problem parameters: shared by the batch (kernel-argument block, constant bank) or, when PP, one set per problem read
   from w.pp ([NPF][Bp], problem index fastest) into the thread's registers -- a batch of independent reference calls,
   each with its own parameter struct (iLQG_mex.c:70-84). */
#define ILQG_PARAMS(PP_, b_)                                                                   \
    double pl_[(PP_) ? P::NPF : 1];                                                            \
    const double *pv = pb.v;                                                                   \
    if (PP_) {                                                                                 \
        _Pragma("unroll") for (int i_ = 0; i_ < P::NPF_USED; i_++) pl_[i_] = w.pp[(size_t)i_ * w.Bp + (b_)]; \
        pv = pl_;                                                                              \
    }

/* [k]-indexed parameters (name[k] in a problem file), read by the generated problem functions as pk(j, k).  PkShared: one
   array of n_hor + 1 values per parameter, shared by the batch (w.pk[j][k]).  PkTrack (ilqgb_set_param_track): the parameters
   whose bit is set in w.tr_mask have a track per problem, stored [len][Bp] with the problem index fastest so that the lanes of
   a warp read one coalesced row, and a solve reads step w.tr_off + k of it; the others stay shared.  The bit test is uniform
   over a launch.  Only the kernels that evaluate the problem functions have a track variant (template flag TR); the
   backward passes read derivative entries and consts(p) alone. */
struct PkShared {
    const double *const *p;
    __device__ __forceinline__ double operator()(int j, int k) const { return p[j][k]; }
};
struct PkTrack {
    const double *const *p;
    unsigned mask;
    int off, b;
    size_t Bp;
    __device__ __forceinline__ double operator()(int j, int k) const
    {
        return ((mask >> j) & 1u) ? p[j][(size_t)(off + k) * Bp + b] : p[j][k];
    }
};
template <bool TR> struct PkSel { using type = PkShared; };
template <> struct PkSel<true> { using type = PkTrack; };
template <bool TR> __device__ __forceinline__ typename PkSel<TR>::type make_pk(const ilqg_work &w, int b)
{
    if constexpr (TR) return PkTrack{w.pk, w.tr_mask, w.tr_off, b, (size_t)w.Bp};
    else return PkShared{w.pk};
}
#define ILQG_PK(TR_, b_) const auto pk = make_pk<TR_>(w, (b_));

#ifndef ILQG_FORCE_COOP
#define ILQG_FORCE_COOP 0
#endif
/* problems whose backward-pass state does not fit one lane's registers use the warp-cooperative kernel */
template <class P> __host__ __device__ constexpr bool use_coop() { return P::COOP || ILQG_FORCE_COOP; }

__device__ __forceinline__ double dmax(double a, double b) { return (a > b) ? a : b; }
__device__ __forceinline__ double dmin(double a, double b) { return (a < b) ? a : b; }
__host__ __device__ constexpr int utri(int r, int c) { return (c * (c + 1)) / 2 + r; }
__host__ __device__ constexpr int symtri(int r, int c) { return r > c ? utri(c, r) : utri(r, c); }

/* ---- small dense algebra, operation order of matMult.c ----------------------------------------------------------
 * MA / MC are compile-time masks of the structurally non-zero entries of the operands a / c (generated per problem;
 * AllNZ for run-time dense operands).  A term whose factor is structurally zero is skipped: it could only add +-0 to
 * a finite sum, so every non-zero result is unchanged (DESIGN.md section 2).  -DILQG_EXPLOIT_ZEROS=0 keeps all terms. */
#ifndef ILQG_EXPLOIT_ZEROS
#define ILQG_EXPLOIT_ZEROS 1
#endif
struct AllNZ { __host__ __device__ static constexpr bool nz(int) { return true; } };
template <class M> __host__ __device__ constexpr bool mnz(int i) { return !ILQG_EXPLOIT_ZEROS || M::nz(i); }

template <int NR, int NC, class MB = AllNZ>
__device__ __forceinline__ void add_mul_vec(double *base, const double *a, const double *b)
{
#pragma unroll
    for (int c = 0; c < NC; c++)
#pragma unroll
        for (int r = 0; r < NR; r++)
            if (mnz<MB>(r + c * NR)) base[c] += a[r] * b[r + c * NR];
}

template <int NR, int NC, class MA = AllNZ>
__device__ __forceinline__ void add_square_tri(double *base, const double *B, const double *a)
{
    double ba[NR * NC];
#pragma unroll
    for (int c = 0; c < NC; c++)
#pragma unroll
        for (int r = 0; r < NR; r++) {
            double acc = 0.0;
#pragma unroll
            for (int s = 0; s < NR; s++)
                if (mnz<MA>(s + c * NR)) acc += B[symtri(r, s)] * a[s + c * NR];
            ba[r + c * NR] = acc;
        }
#pragma unroll
    for (int c = 0; c < NC; c++)
#pragma unroll
        for (int r = 0; r <= c; r++) {
            double acc = 0.0;
#pragma unroll
            for (int s = 0; s < NR; s++)
                if (mnz<MA>(s + r * NR)) acc += a[s + r * NR] * ba[s + c * NR];
            if (r != c) {
#pragma unroll
                for (int s = 0; s < NR; s++)
                    if (mnz<MA>(s + c * NR)) acc += a[s + c * NR] * ba[s + r * NR];
                acc *= 0.5;
            }
            base[utri(r, c)] += acc;
        }
}

template <int NRA, int NCA, int NCC, class MA = AllNZ, class MC = AllNZ>
__device__ __forceinline__ void add_mul2_tri(double *base, const double *B, const double *a, const double *c)
{
    double bc[NRA * NCC];
#pragma unroll
    for (int j = 0; j < NCC; j++)
#pragma unroll
        for (int r = 0; r < NRA; r++) {
            double acc = 0.0;
#pragma unroll
            for (int s = 0; s < NRA; s++)
                if (mnz<MC>(s + j * NRA)) acc += B[symtri(r, s)] * c[s + j * NRA];
            bc[r + j * NRA] = acc;
        }
#pragma unroll
    for (int i = 0; i < NCA; i++)
#pragma unroll
        for (int j = 0; j < NCC; j++) {
            double acc = 0.0;
#pragma unroll
            for (int s = 0; s < NRA; s++)
                if (mnz<MA>(s + i * NRA)) acc += a[s + i * NRA] * bc[s + j * NRA];
            base[i + j * NCA] += acc;
        }
}

/* ---- projected-Newton box QP ------------------------------------------------------------------------------------------
 * The reference compacts the free rows/columns before factorising (boxQP.c:129-146).  Here the factor U and the
 * inverse live in FULL index space and clamped indices are skipped by predicate: the same multiplications and
 * additions happen in the same order, but every array index is a compile-time constant, so all QP state stays in
 * registers. */
template <int M>
__device__ __forceinline__ double qp_value(const double *H, const double *g, const double *x)
{
    double val = 0.0;
#pragma unroll
    for (int i = 0; i < M; i++) {
        double hx = 0.0;
#pragma unroll
        for (int j = 0; j < M; j++)
            hx += H[symtri(i, j)] * x[j];
        val += x[i] * (g[i] + 0.5 * hx);
    }
    return val;
}

/* CL > 0 (warp-cooperative callers, CL lanes hold identical QP state): the columns of the explicit inverse are computed by
   different lanes -- lane c of the group solves the two triangular systems of column c, skipping by predicate the terms the
   reference's loops start behind (i < col), then the columns are exchanged by shuffle.  Same operations in the same order
   for every entry of the free block (checked on the host against the sequential form: bit-identical), 2M instead of
   M(M+1) divisions per lane. */
template <int M, int CL = 0>
__device__ __forceinline__ int box_qp(const double *H, const double *g, const double *lower, const double *upper,
                                      double *x, int *clamped, double *invH, int &n_free_out, int co_lane = 0, unsigned co_mask = 0u,
                                      int co_base = 0)
{
    constexpr int MP = (M * (M + 1)) / 2;
    const double min_grad = 1e-8, min_rel_improve = 1e-8, step_dec = 0.6, min_step = 1e-22, armijo = 0.1;
    double U[MP], grad[M], gc[M], search[M], w[M];
    double value, oldvalue = 0.0;
#pragma unroll
    for (int i = 0; i < MP; i++) U[i] = 1.0;   /* entries of clamped rows/columns are don't-care but must be defined */

#pragma unroll
    for (int i = 0; i < M; i++) {
        if (x[i] > upper[i]) x[i] = upper[i];
        if (x[i] < lower[i]) x[i] = lower[i];
        clamped[i] = 0;
    }
    value = qp_value<M>(H, g, x);

    for (int iter = 0; iter < 100; iter++) {
        if (iter > 0 && (oldvalue - value) < min_rel_improve * fabs(oldvalue))
            return 4;
        oldvalue = value;

        int n_free = 0;
        bool changed = false, all_clamped = true;
        double gsq = 0.0;
#pragma unroll
        for (int i = 0; i < M; i++) {
            double hx = 0.0;
#pragma unroll
            for (int j = 0; j < M; j++)
                hx += H[symtri(i, j)] * x[j];
            grad[i] = g[i] + hx;
            const int was = clamped[i];
            if (x[i] <= lower[i] && grad[i] > 0)
                clamped[i] = 1;
            else if (x[i] >= upper[i] && grad[i] < 0)
                clamped[i] = 2;
            else {
                clamped[i] = 0;
                all_clamped = false;
                gsq += grad[i] * grad[i];
                n_free++;
            }
            if ((!was) != (!clamped[i]))
                changed = true;
        }
        n_free_out = n_free;
        if (all_clamped)
            return 6;

        if (iter == 0 || changed) {
            /* U'U = H(free,free)  (cholesky.c:6-27), straight-line: every entry is evaluated and the clamp pattern
               only SELECTS which terms enter a sum; entries that involve a clamped index hold don't-care values that
               no later read uses.  Same operations in the same order on the free block, no divergent branches. */
            bool pd = true;
#pragma unroll
            for (int col = 0; col < M; col++) {
#pragma unroll
                for (int row = 0; row <= col; row++) {
                    const bool act = !clamped[col] && !clamped[row];
                    double dot = 0;
#pragma unroll
                    for (int k = 0; k < row; k++) {
                        const double t = dot + U[utri(k, col)] * U[utri(k, row)];
                        dot = clamped[k] ? dot : t;
                    }
                    const double rem = H[utri(row, col)] - dot;
                    if (row == col) {
                        if (act && rem <= 0.0) pd = false;
                        U[utri(row, col)] = sqrt(rem);
                    } else {
                        U[utri(row, col)] = 1.0 / U[utri(row, row)] * rem;
                    }
                }
            }
            if (!pd)
                return -1;
            /* explicit inverse, one unit right-hand side per free column (cholesky.c:51-74), same scheme */
            if (CL >= M && M > 2) {
                const int col = co_lane < M ? co_lane : 0;
                double wv[M];
#pragma unroll
                for (int k = 0; k < M; k++) {
                    double wk = (k == col) ? 1.0 : 0.0;
#pragma unroll
                    for (int i = 0; i < k; i++) {
                        const double t = wk - wv[i] * U[utri(i, k)];
                        wk = (clamped[i] || i < col) ? wk : t;
                    }
                    wv[k] = wk / U[utri(k, k)];
                }
#pragma unroll
                for (int k = M - 1; k >= 0; k--) {
                    double wk = wv[k];
#pragma unroll
                    for (int i = k + 1; i < M; i++) {
                        const double t = wk - wv[i] * U[utri(k, i)];
                        wk = clamped[i] ? wk : t;
                    }
                    wv[k] = wk / U[utri(k, k)];
                }
#pragma unroll
                for (int c = 0; c < M; c++)
#pragma unroll
                    for (int k = c; k < M; k++) invH[utri(c, k)] = __shfl_sync(co_mask, wv[k], co_base + c);
            } else
#pragma unroll
            for (int col = 0; col < M; col++) {
                w[col] = 1.0;
#pragma unroll
                for (int k = col + 1; k < M; k++)
                    w[k] = 0.0;
#pragma unroll
                for (int k = col; k < M; k++) {
                    double wk = w[k];
#pragma unroll
                    for (int i = col; i < k; i++) {
                        const double t = wk - w[i] * U[utri(i, k)];
                        wk = clamped[i] ? wk : t;
                    }
                    w[k] = wk / U[utri(k, k)];
                }
#pragma unroll
                for (int k = M - 1; k >= col; k--) {
                    double wk = w[k];
#pragma unroll
                    for (int i = k + 1; i < M; i++) {
                        const double t = wk - w[i] * U[utri(k, i)];
                        wk = clamped[i] ? wk : t;
                    }
                    wk = wk / U[utri(k, k)];
                    w[k] = wk;
                    invH[utri(col, k)] = wk;
                }
            }
        }
        if (gsq < min_grad * min_grad)
            return 5;

        /* search = -Hfree^-1 (g + H x_clamped) - x on the free set (boxQP.c:153-177) */
#pragma unroll
        for (int i = 0; i < M; i++) {
            double hc = 0.0;
#pragma unroll
            for (int j = 0; j < M; j++) {
                const double t = hc + H[symtri(i, j)] * x[j];
                hc = clamped[j] ? t : hc;
            }
            gc[i] = g[i] + hc;
        }
#pragma unroll
        for (int i = 0; i < M; i++) {
            double sd = -x[i];
#pragma unroll
            for (int j = 0; j < M; j++) {
                const double t = sd - invH[symtri(i, j)] * gc[j];
                sd = clamped[j] ? sd : t;
            }
            search[i] = clamped[i] ? 0.0 : sd;
        }
        double sdotg = 0.0;
#pragma unroll
        for (int i = 0; i < M; i++)
            sdotg += search[i] * grad[i];
        if (sdotg >= 0.0)
            return -2;

        /* Armijo backtracking along the projected step (boxQP.c:198-227) */
        double step = 1.0, vc;
        double xc[M];
        for (;;) {
#pragma unroll
            for (int i = 0; i < M; i++) {
                xc[i] = x[i] + step * search[i];
                if (xc[i] > upper[i]) xc[i] = upper[i];
                if (xc[i] < lower[i]) xc[i] = lower[i];
            }
            vc = qp_value<M>(H, g, xc);
            if (((vc - oldvalue) / (step * sdotg)) >= armijo)
                break;
            step = step * step_dec;
            if (step < min_step)
                return 2;
        }
#pragma unroll
        for (int i = 0; i < M; i++)
            x[i] = xc[i];
        value = vc;
    }
    return 1;
}

/* ---- per-(step, problem) records in HBM ---------------------------------------------------------------------------
 * The data a rollout reads and writes is stored as one small contiguous record per (timestep, problem):
 *   XU[buf][k][b][RXU] = x (NX) | u (NU) | pad        LL[buf][k][b][RLM] = L (NU*NX) | pad        Ll[buf][k][b][RLS] = l (NU) | pad
 * with the x|u and L records rounded up to 32-byte sectors and the small l record to 16 bytes (two problems per sector).  The
 * gains and the feed-forward term are separate arrays since round 2: DRAM is fetched in 64-byte granules, a 96-byte l|L record
 * of a problem whose neighbours are not in the (compacted) list cost 2-3 granules for 80 useful bytes (round 1 measured 239 B
 * read per step in round 1 of the line search against 160 B in round 0); a 64-byte L record is exactly one granule.  Any lane -> problem mapping (the line search works on compacted
 * problem lists) then moves only fully used sectors, and a warp with lane == problem still reads one contiguous run. */
template <class P> struct Rec {
    static constexpr int RXU = ((P::NX + P::NU + 3) / 4) * 4;
    static constexpr int RLM = ((P::NU * P::NX + 3) / 4) * 4;   /* gains L */
    static constexpr int RLS = ((P::NU + 1) / 2) * 2;            /* feed-forward l */
};

template <int N> __device__ __forceinline__ void ld_rec(const double *p, double *out)
{
    const double2 *p2 = reinterpret_cast<const double2 *>(p);
#pragma unroll
    for (int i = 0; i < (N + 1) / 2; i++) {
        const double2 v = p2[i];
        out[2 * i] = v.x;
        if (2 * i + 1 < N) out[2 * i + 1] = v.y;
    }
}

/* stores whole 16-byte pairs: `in` must hold N rounded up to even (pad with anything finite) */
template <int N> __device__ __forceinline__ void st_rec(double *p, const double *in)
{
    double2 *p2 = reinterpret_cast<double2 *>(p);
#pragma unroll
    for (int i = 0; i < N / 2; i++) p2[i] = make_double2(in[2 * i], in[2 * i + 1]);
}

/* ---- asynchronous global->shared copies (LDGSTS) for software pipelining --------------------------------------------- */
__device__ __forceinline__ void cp_async8(double *smem_dst, const double *gmem_src)
{
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

/* ---- per-step dense record the backward pass works on ------------------------------------------------------------- */
template <class P> struct Dense {
    double fx[P::NX * P::NX], fu[P::NX * P::NU], cx[P::NX], cxx[P::NQXX], cu[P::NU], cuu[P::NQUU], cxu[P::NQXU];
    double lower[P::NU], upper[P::NU];
    double lower_sign[P::NU], upper_sign[P::NU], lower_hx[P::NX * P::NU], upper_hx[P::NX * P::NU];
};

__device__ __forceinline__ void finish(const Work &w, int b, int iter, int result)
{
    w.status[b] = ST_DONE;
    w.iterations[b] = iter;
    w.result[b] = result;
}

__device__ __forceinline__ void raise_lambda(const Opts &o, double &lambda, double &dlambda)
{
    dlambda = dmax(dlambda * o.lambdaFactor, o.lambdaFactor);   /* iLQG.c:272-273, 342-343 */
    lambda = dmax(lambda * dlambda, o.lambdaMin);
}

__device__ __forceinline__ void lower_lambda(const Opts &o, double &lambda, double &dlambda)
{
    dlambda = dmin(dlambda / o.lambdaFactor, 1.0 / o.lambdaFactor);   /* iLQG.c:298-299, 317-318 */
    lambda = lambda * dlambda * (double)(lambda > o.lambdaMin);
}

/* =====================================================================================================================
 * K1: derivative pass, one thread per (problem, timestep); k == T evaluates the final-cost derivatives.
 * ===================================================================================================================== */
/* rewrite one double in place: a store of exactly what is there, which the compiler must not drop */
__device__ __forceinline__ void rewrite8(double *p)
{
    double v;
    asm volatile("ld.global.cg.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    *p = v;
}

template <class P, bool FULL, bool PP, bool TR = false>
__global__ void __launch_bounds__(DV_BLOCK) k_derivs(Work w, ParamBlock<P> pb)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    const int k = blockIdx.y;
    /* fresh: this problem needs new derivatives (iLQG.c:240-253).  The entry-major stores below put four neighbouring problems
       into one 32-byte sector, and a partially written sector costs a DRAM read-modify-write (measured with ncu once ~10 % of a
       batch had finished: +2 GB DRAM reads per sweep and twice the kernel time).  So a sector is either skipped or written
       whole: a lane that is not fresh but shares a sector with a fresh one re-evaluates its entries -- same nominal and
       parameters, hence the same bits for a running problem; a finished problem's entries are never read again -- or, when the
       derivatives depend on multipliers / penalty weights that may have moved since they were last evaluated (the reference
       does not refresh them after a rejected step, iLQG.c:345-349), stores back what is there. */
    constexpr bool KEEP = (P::N_MU_R + P::N_MU_F) > 0;
    const bool inb = b < w.B;
    const bool fresh = inb && w.status[b] == ST_RUNNING && w.new_deriv[b];
    bool fill = false;
    if (!use_coop<P>()) {
        const unsigned m = __ballot_sync(0xffffffffu, fresh);
        fill = inb && !fresh && ((m >> (threadIdx.x & 28)) & 0xfu) != 0u;
    }
    if (!fresh && !fill) return;
    const size_t Bp = w.Bp;
    if (KEEP && fill) {
        if (k < w.T) {
            double *o1 = w.V1 + (size_t)k * P::NV1 * Bp + b;
#pragma unroll
            for (int i = 0; i < P::NV1; i++) rewrite8(o1 + i * Bp);
            if (FULL) {
                double *o2 = w.V2 + (size_t)k * P::NV2 * Bp + b;
#pragma unroll
                for (int i = 0; i < P::NV2_USED; i++) rewrite8(o2 + i * Bp);
            }
        } else {
            double *fd = w.FD + b;
#pragma unroll
            for (int i = 0; i < P::NX + P::NQXX; i++) rewrite8(fd + i * Bp);
        }
        return;
    }
    ILQG_PARAMS(PP, b)
    ILQG_PK(TR, b)
    const int cur = w.cur[b];
    constexpr int RXU = Rec<P>::RXU;
    double xu[RXU], mu[P::N_MU_R + P::N_MU_F + 1];
    ld_rec<P::NX + P::NU>(w.XU[cur] + ((size_t)k * Bp + b) * RXU, xu);
    const double *x = xu, *u = xu + P::NX;
    bool ok;
    if (k < w.T) {
#pragma unroll
        for (int i = 0; i < P::N_MU_R; i++) mu[i] = w.muR[((size_t)k * P::N_MU_R + i) * Bp + b];
        double v1[P::NV1], v2[P::NV2];
        const double w_pen = w.w_pen_l[b];
        if (FULL)
            ok = P::derivs_full(x, u, pv, pk, k, w.T, w_pen, mu, v1, v2);
        else
            ok = P::derivs(x, u, pv, pk, k, w.T, w_pen, mu, v1, v2);
        if (use_coop<P>()) { /* one contiguous record per (step, problem): the consumer is a whole warp per problem */
            double *o1 = w.V1 + ((size_t)k * Bp + b) * P::NV1;
#pragma unroll
            for (int i = 0; i < P::NV1; i++) o1[i] = v1[i];
            if (FULL) {
                double *o2 = w.V2 + ((size_t)k * Bp + b) * P::NV2;
#pragma unroll
                for (int i = 0; i < P::NV2_USED; i++) o2[i] = v2[i];
            }
        } else {
            double *o1 = w.V1 + (size_t)k * P::NV1 * Bp + b;
#pragma unroll
            for (int i = 0; i < P::NV1; i++) o1[i * Bp] = v1[i];
            if (FULL) {
                double *o2 = w.V2 + (size_t)k * P::NV2 * Bp + b;
#pragma unroll
                for (int i = 0; i < P::NV2_USED; i++) o2[i * Bp] = v2[i];
            }
        }
    } else {
#pragma unroll
        for (int i = 0; i < P::N_MU_F; i++) mu[i] = w.muF[(size_t)i * Bp + b];
        double cx[P::NX], cxx[P::NQXX];
        ok = P::derivs_final(x, pv, pk, w.T, w.T, w.w_pen_f[b], mu, cx, cxx);
        double *fd = w.FD + b;
#pragma unroll
        for (int i = 0; i < P::NX; i++) fd[i * Bp] = cx[i];
#pragma unroll
        for (int i = 0; i < P::NQXX; i++) fd[(P::NX + i) * Bp] = cxx[i];
    }
    if (!ok && fresh) atomicOr(&w.deriv_fail[b], 1);
}

/* =====================================================================================================================
 * K2: backward pass, one lane per problem, incl. the regularisation retry loop and the gradient exit.
 * ===================================================================================================================== */
/* doubles per (step, problem) the backward pass consumes: time-varying derivative entries, the nominal control
   (gradient measure), and the second-order entries when FULL_DDP */
template <class P, bool FULL> __host__ __device__ constexpr int bp_fields() { return P::NV1 + P::NU + (FULL ? P::NV2_USED : 0); }

template <class P, bool FULL>
__device__ __forceinline__ void bp_issue(const Work &w, double *sm, int k, int stage, int b, int cur)
{
    constexpr int NF = bp_fields<P, FULL>();
    const size_t Bp = w.Bp;
    double *dst = sm + (size_t)stage * NF * BP_BLOCK + threadIdx.x;
    const double *v1 = w.V1 + (size_t)k * P::NV1 * Bp + b;
#pragma unroll
    for (int i = 0; i < P::NV1; i++) cp_async8(dst + i * BP_BLOCK, v1 + i * Bp);
    const double *un = w.XU[cur] + ((size_t)k * Bp + b) * Rec<P>::RXU + P::NX;
#pragma unroll
    for (int i = 0; i < P::NU; i++) cp_async8(dst + (P::NV1 + i) * BP_BLOCK, un + i);
    if (FULL) {
        const double *v2 = w.V2 + (size_t)k * P::NV2 * Bp + b;
#pragma unroll
        for (int i = 0; i < P::NV2_USED; i++) cp_async8(dst + (P::NV1 + P::NU + i) * BP_BLOCK, v2 + i * Bp);
    }
    cp_async_commit();
}

/* MINB = minimum resident blocks per SM the compiler must allow: 8 caps the kernel at 128 registers (16 warps/SM, the
   throughput build for large batches); 1 leaves registers free (no spills, shortest per-step latency, small batches) */
template <class P, bool FULL, int MINB, bool PP>
__global__ void __launch_bounds__(BP_BLOCK, MINB) k_backpass(Work w, Opts o, ParamBlock<P> pb, int iter)
{
    constexpr int NX = P::NX, NU = P::NU, NQXX = P::NQXX, NQUU = P::NQUU, NQXU = P::NQXU;
    constexpr int NF = bp_fields<P, FULL>();
    extern __shared__ double sm[];   /* 2 stages x NF fields x BP_BLOCK columns (dynamic: can exceed 48 KB) */
    /* o.bp_ppw problems per warp (32 = every lane; fewer = the first lanes of more warps: when the batch does not fill the GPU,
       a warp then serialises the divergent box-QP iterations of fewer problems) */
    const int ppw = o.bp_ppw;
    if ((int)(threadIdx.x & 31) >= ppw) return;
    const int b = (blockIdx.x * (BP_BLOCK / 32) + (threadIdx.x >> 5)) * ppw + (threadIdx.x & 31);
    if (b >= w.B) return;
    if (w.status[b] != ST_RUNNING) return;
    ILQG_PARAMS(PP, b)
    if (w.new_deriv[b]) {
        if (w.deriv_fail[b]) { /* "Calculating derivatives failed": break (iLQG.c:248-251) */
            finish(w, b, iter, w.bp_done[b] ? 1 : 0);
            return;
        }
        w.new_deriv[b] = 0;
        w.n_dv[b] += 1;
    }
    const size_t Bp = w.Bp;
    const int T = w.T;
    const int cur = w.cur[b];
    double lambda = w.lambda[b], dlambda = w.dlambda[b];
    Dense<P> D;
    P::consts(pv, D);

    double Vx[NX], Vxx[NQXX];
    double dV0 = 0.0, dV1 = 0.0, g_sum = 0.0;
    int n_bp = w.n_bp[b];
    bool done = false;
    while (!done) {
        n_bp++;
#pragma unroll
        for (int i = 0; i < NX; i++) Vx[i] = w.FD[(size_t)i * Bp + b];
#pragma unroll
        for (int i = 0; i < NQXX; i++) Vxx[i] = w.FD[(size_t)(NX + i) * Bp + b];
        dV0 = 0.0;
        dV1 = 0.0;
        g_sum = 0.0;
        double lk[NU];
#pragma unroll
        for (int i = 0; i < NU; i++) lk[i] = 0.0;
        bool failed = false;

        /* two-stage LDGSTS pipeline: the inputs of step k-1 stream into shared memory while step k is computed.
           Each thread copies and later reads only its own column, so no block barrier is needed. */
        cp_async_wait<0>();
        bp_issue<P, FULL>(w, sm, T - 1, 0, b, cur);
        for (int k = T - 1; k >= 0; k--) {
            const int stage = (T - 1 - k) & 1;
            if (k > 0) bp_issue<P, FULL>(w, sm, k - 1, stage ^ 1, b, cur);
            else cp_async_commit();
            cp_async_wait<1>();
            const double *st = sm + (size_t)stage * NF * BP_BLOCK + threadIdx.x;
            {
                double v1[P::NV1];
#pragma unroll
                for (int i = 0; i < P::NV1; i++) v1[i] = st[i * BP_BLOCK];
                P::unpack(v1, D);
            }
            double Qx[NX], Qu[NU], Qxx[NQXX], Quu[NQUU], Qxu[NQXU], QuuF[NQUU], Qxu_reg[NQXU];
            /* Q-function (back_pass.c:80-131) */
#pragma unroll
            for (int i = 0; i < NU; i++) Qu[i] = D.cu[i];
            add_mul_vec<NX, NU, typename P::Mask_fu>(Qu, Vx, D.fu);
#pragma unroll
            for (int i = 0; i < NX; i++) Qx[i] = D.cx[i];
            add_mul_vec<NX, NX, typename P::Mask_fx>(Qx, Vx, D.fx);
#pragma unroll
            for (int i = 0; i < NQXU; i++) Qxu[i] = D.cxu[i];
            add_mul2_tri<NX, NX, NU, typename P::Mask_fx, typename P::Mask_fu>(Qxu, Vxx, D.fx, D.fu);
#pragma unroll
            for (int i = 0; i < NQUU; i++) Quu[i] = D.cuu[i];
            add_square_tri<NX, NU, typename P::Mask_fu>(Quu, Vxx, D.fu);
#pragma unroll
            for (int i = 0; i < NQXX; i++) Qxx[i] = D.cxx[i];
            add_square_tri<NX, NX, typename P::Mask_fx>(Qxx, Vxx, D.fx);
            if (FULL) {
                double v2[P::NV2];
#pragma unroll
                for (int i = 0; i < P::NV2_USED; i++) v2[i] = st[(P::NV1 + NU + i) * BP_BLOCK];
                P::add2_Qxu(Vx, v2, pv, Qxu);
                P::add2_Quu(Vx, v2, pv, Quu);
                P::add2_Qxx(Vx, v2, pv, Qxx);
            }
            /* regularisation (back_pass.c:134-159) */
#pragma unroll
            for (int i = 0; i < NQUU; i++) QuuF[i] = Quu[i];
#pragma unroll
            for (int i = 0; i < NQXU; i++) Qxu_reg[i] = Qxu[i];
            if (o.regType == 2) {
#pragma unroll
                for (int j = 0; j < NU; j++)
#pragma unroll
                    for (int i = 0; i <= j; i++) {
                        double acc = 0.0;
#pragma unroll
                        for (int c = 0; c < NU; c++)
                            acc += D.fu[symtri(c, i)] * D.fu[symtri(c, j)];
                        QuuF[utri(i, j)] += acc * lambda;
                    }
#pragma unroll
                for (int i = 0; i < NX; i++)
#pragma unroll
                    for (int j = 0; j < NU; j++) {
                        double acc = 0.0;
#pragma unroll
                        for (int c = 0; c < NX; c++)
                            acc += D.fx[c + i * NX] * D.fu[(c + j * NU) < NX * NU ? (c + j * NU) : 0];
                        Qxu_reg[i + j * NX] += acc * lambda;
                    }
            }
            if (o.regType == 1) {
#pragma unroll
                for (int i = 0; i < NU; i++) QuuF[utri(i, i)] += lambda;
            }
            /* box QP, warm-started from step k+1 (back_pass.c:163-171) */
            int clamped[NU], n_free;
            double invH[NQUU];
            const int qp = box_qp<NU>(QuuF, Qu, D.lower, D.upper, lk, clamped, invH, n_free);
            if (w.tr_clamp) {
                int code = (qp & 0xff) << 16;
#pragma unroll
                for (int i = 0; i < NU; i++) code |= clamped[i] << (2 * i);
                w.tr_clamp[(size_t)k * Bp + b] = code;
            }
            if (qp < 1) {
                /* the reference's boxQP iterates on t->l in place (back_pass.c:163-171): a failed QP leaves its last iterate
                   in the trajectory, which is what a solve that ends on this failure returns */
                double *rec = w.Ll[cur] + ((size_t)k * Bp + b) * Rec<P>::RLS;
#pragma unroll
                for (int i = 0; i < NU; i++) rec[i] = lk[i];
                failed = true;
                break;
            }
            /* gains (back_pass.c:173-201) */
            double Lk[NU * NX];
#pragma unroll
            for (int i = 0; i < NU * NX; i++) Lk[i] = 0.0;
#pragma unroll
            for (int i = 0; i < NU; i++) {
                if (clamped[i]) {
                    if (P::HAS_HX) {
#pragma unroll
                        for (int s = 0; s < NX; s++)
                            Lk[i + s * NU] -= (clamped[i] == 1) ? D.lower_sign[i] * D.lower_hx[s + i * NX]
                                                                  : D.upper_sign[i] * D.upper_hx[s + i * NX];
                    }
                    continue;
                }
#pragma unroll
                for (int j = 0; j < NU; j++) {
                    if (!clamped[j]) {
#pragma unroll
                        for (int s = 0; s < NX; s++)
                            Lk[i + s * NU] -= invH[symtri(i, j)] * Qxu_reg[s + j * NX];
                    } else if (P::HAS_HX) {
                        double wgt = 0.0;
#pragma unroll
                        for (int c = 0; c < NU; c++)
                            if (!clamped[c])
                                wgt -= invH[symtri(i, c)] * QuuF[symtri(c, j)];
#pragma unroll
                        for (int s = 0; s < NX; s++)
                            Lk[i + s * NU] -= wgt * ((clamped[j] == 1) ? D.lower_sign[j] * D.lower_hx[s + j * NX]
                                                                         : D.upper_sign[j] * D.upper_hx[s + j * NX]);
                    }
                }
            }
            {
                constexpr int RLM = Rec<P>::RLM, RLS = Rec<P>::RLS;
                double recL[RLM], recl[RLS];
#pragma unroll
                for (int i = 0; i < RLS; i++) recl[i] = (i < NU) ? lk[i] : 0.0;
#pragma unroll
                for (int i = 0; i < RLM; i++) recL[i] = (i < NU * NX) ? Lk[i] : 0.0;
                st_rec<RLM>(w.LL[cur] + ((size_t)k * Bp + b) * RLM, recL);
                st_rec<RLS>(w.Ll[cur] + ((size_t)k * Bp + b) * RLS, recl);
            }
            /* expected reduction (back_pass.c:204-214) */
#pragma unroll
            for (int i = 0; i < NU; i++) dV0 += Qu[i] * lk[i];
#pragma unroll
            for (int i = 0; i < NU; i++) {
                double acc = 0.0;
#pragma unroll
                for (int j = 0; j < NU; j++) acc += lk[j] * Quu[symtri(j, i)];
                dV1 += 0.5 * lk[i] * acc;
            }
            /* value function (back_pass.c:217-241) */
#pragma unroll
            for (int i = 0; i < NX; i++) Vx[i] = Qx[i];
            add_mul2_tri<NU, NX, 1>(Vx, Quu, Lk, lk);
#pragma unroll
            for (int i = 0; i < NX; i++)
#pragma unroll
                for (int j = 0; j < NU; j++) Vx[i] += Lk[j + i * NU] * Qu[j];
#pragma unroll
            for (int i = 0; i < NX; i++)
#pragma unroll
                for (int j = 0; j < NU; j++) Vx[i] += Qxu[i + j * NX] * lk[j];
#pragma unroll
            for (int i = 0; i < NQXX; i++) Vxx[i] = Qxx[i];
            add_square_tri<NU, NX>(Vxx, Quu, Lk);
#pragma unroll
            for (int i = 0; i < NX; i++)
#pragma unroll
                for (int j = 0; j < NX; j++)
#pragma unroll
                    for (int c = 0; c < NU; c++) {
                        double term = Lk[c + i * NU] * Qxu[j + c * NX];
                        if (i == j) term *= 2.0;
                        Vxx[symtri(i, j)] += term;
                    }
            /* gradient measure (back_pass.c:244-251) */
            {
                double gmax = 0.0;
#pragma unroll
                for (int i = 0; i < NU; i++) {
                    const double gi = fabs(lk[i]) / (fabs(st[(P::NV1 + i) * BP_BLOCK]) + 1.0);
                    if (gi > gmax) gmax = gi;
                }
                g_sum += gmax;
            }
        }
        if (failed) {
            if (o.bp_single) break;   /* back_pass(o) on its own: one attempt, the retry loop belongs to iLQG() */
            raise_lambda(o, lambda, dlambda);
            if (lambda > o.lambdaMax) break;
        } else {
            done = true;
        }
    }
    w.n_bp[b] = n_bp;
    w.dV0[b] = dV0;
    w.dV1[b] = dV1;
    w.bp_done[b] = done ? 1 : 0;
    double g_norm = w.g_norm[b];
    if (done) {
        g_norm = g_sum / ((double)(T - 1));
        w.g_norm[b] = g_norm;
    }
    if (o.bp_single) return;
    if (g_norm < o.tolGrad && lambda < 1e-5) { /* iLQG.c:297-303 */
        lower_lambda(o, lambda, dlambda);
        finish(w, b, iter, done ? 1 : 0);
    } else if (!done) {
        finish(w, b, iter, 0);
    }
    w.lambda[b] = lambda;
    w.dlambda[b] = dlambda;
}

/* =====================================================================================================================
 * K2w: backward pass, one WARP per problem (larger state dimensions: the quadrotor has Vxx 78, Qxx 78, fx 144 ...
 * doubles per step).  All matrices live in shared memory; a lane owns OUTPUT ELEMENTS and evaluates each of its dot
 * products serially in the reference's summation order -- there is no cross-lane reduction anywhere, so results are
 * bit-identical to the lane-per-problem kernel and to the reference.  The m x m box-QP runs redundantly in every
 * lane's registers (uniform control flow, no broadcast needed).  The FULL_DDP tensor contractions are data-driven
 * sparse term lists emitted by the generator.
 * ===================================================================================================================== */
constexpr int CW_WARPS = 4;
#ifndef ILQG_CW_MINBLOCKS
#define ILQG_CW_MINBLOCKS 4   /* 128 registers: 16 warps per SM; measured best of 1/3/4/5 on the quadrotor */
#endif

template <class P> struct CoopWS;
template <class P, int LPP> __host__ __device__ constexpr size_t coop_smem_bytes() { return sizeof(CoopWS<P>) * CW_WARPS * (32 / LPP); }
/* leading dimensions of the kernel-private matrices are odd (NX | 1): lanes that walk a column hit distinct banks */
template <class P> struct CoopWS {
    static constexpr int LX = P::NX | 1, LU = P::NU | 1;
    Dense<P> D;
    double Vx[P::NX], VxxF[P::NX * LX], QuuS[P::NU * LU];   /* full symmetric copies: plain row*N+col addressing */
    double Qx[P::NX], Qu[P::NU], Qxx[P::NQXX], Quu[P::NQUU], Qxu[P::NQXU], QuuF[P::NQUU], Qxu_reg[P::NQXU];
    double ba[LX * P::NX], bc[LX * P::NU], bl[LU * P::NX], bv[P::NU];
    double Lk[P::NU * P::NX], lk[P::NU], invH[P::NQUU];
    double v2[P::NV2], c2[P::NC2];
    double un[P::NU];   /* nominal control of the step (gradient measure), fetched one step ahead like the derivative entries */
    double prod[(P::NT2XU + P::NT2UU + P::NT2XX) > 0 ? (P::NT2XU + P::NT2UU + P::NT2XX) : 1];   /* FULL_DDP: products Vx[i] * f??[i][entry], term order xu | uu | xx */
    int clamped[P::NU];
    unsigned char tri_r[P::NQXX], tri_c[P::NQXX];   /* packed upper-triangle index -> (row, col) */
};

__device__ __forceinline__ void tri_rc(int e, int &r, int &c)
{
    c = 0;
    while (((c + 1) * (c + 2)) / 2 <= e) c++;
    r = e - (c * (c + 1)) / 2;
}

template <class P, bool FULL, bool PP, int LPP>
__global__ void __launch_bounds__(CW_WARPS * 32, (ILQG_CW_MINBLOCKS * LPP) / 32) k_backpass_warp(Work w, Opts o, ParamBlock<P> pb, int iter)
{
    static_assert(LPP == 32 || LPP == 16 || LPP == 8, "lanes per problem");
    constexpr int NX = P::NX, NU = P::NU, NQXX = P::NQXX, NQUU = P::NQUU, NQXU = P::NQXU;
    constexpr int LX = CoopWS<P>::LX, LU = CoopWS<P>::LU;
    static_assert(sizeof(Dense<P>) == sizeof(double) * P::DENSE_SIZE, "Dense layout must match the generator's table");
    /* LPP lanes work on one problem, 32 / LPP problems share a warp: the per-problem scalar work (box QP, sparse FULL_DDP term
       lists, short vectors) is issued once for all of them.  Groups never exchange data and synchronise among themselves only
       (their control flow differs: QP iterations, failed passes). */
    constexpr int PPW = 32 / LPP;
    extern __shared__ double cw_smem[];
    CoopWS<P> *ws_all = reinterpret_cast<CoopWS<P> *>(cw_smem);
    const int lane = threadIdx.x & (LPP - 1), grp = (threadIdx.x & 31) / LPP, wid = threadIdx.x >> 5;
    const unsigned gmask = (LPP == 32) ? 0xffffffffu : (((1u << LPP) - 1u) << (grp * LPP));
    const int b = (blockIdx.x * CW_WARPS + wid) * PPW + grp;
    if (b >= w.B) return;
    if (w.status[b] != ST_RUNNING) return;
    ILQG_PARAMS(PP, b)
    CoopWS<P> &ws = ws_all[wid * PPW + grp];
    if (w.new_deriv[b]) {
        if (w.deriv_fail[b]) {
            if (lane == 0) finish(w, b, iter, w.bp_done[b] ? 1 : 0);
            return;
        }
        __syncwarp(gmask);
        if (lane == 0) {
            w.new_deriv[b] = 0;
            w.n_dv[b] += 1;
        }
    }
    const size_t Bp = w.Bp;
    const int T = w.T;
    const int cur = w.cur[b];
    double lambda = w.lambda[b], dlambda = w.dlambda[b];
    double *Dd = reinterpret_cast<double *>(&ws.D);
    if (lane == 0) {
        P::consts(pv, ws.D);
        if (FULL) P::consts2(pv, ws.c2);
    }
    for (int e = lane; e < NQXX; e += LPP) {
        int r, c;
        tri_rc(e, r, c);
        ws.tri_r[e] = (unsigned char)r;
        ws.tri_c[e] = (unsigned char)c;
    }
    __syncwarp(gmask);

    /* FULL_DDP tensor terms (back_pass.c:95-131: Q?? += sum_i Vx[i] * f??[i][entry]): the products of ALL terms are formed lane-parallel
       in phase 1 (term t by lane t % LPP), then the lane that holds slot q of the list of entries that have terms adds its entry's
       products in the reference's order -- one short round instead of a few lanes walking term lists while the others wait.
       Loop-invariant descriptors: terms (index into Vx, source in v2 / c2) and entry slots (matrix, entry, term range). */
    constexpr int NT2 = FULL ? (P::NT2XU + P::NT2UU + P::NT2XX) : 0, NE2 = FULL ? (P::NE2XU + P::NE2UU + P::NE2XX) : 0;
    constexpr int RT = (NT2 + LPP - 1) / LPP, RS = (NE2 + LPP - 1) / LPP;
    /* packed into one register each: term = Vx index | (source + 32768) << 8, -1 = none; slot = matrix (0 xu, 1 uu, 2 xx) | entry << 2 |
       first term << 12 | end term << 22, -1 = none */
    static_assert(NT2 < 512 && NQXX < 1024 && NQXU < 1024, "packed FULL_DDP descriptors");
    int tdesc[RT > 0 ? RT : 1], sdesc[RS > 0 ? RS : 1];
    if (FULL) {
#pragma unroll
        for (int r = 0; r < RT; r++) {
            const int t = lane + LPP * r;
            int vx = -1, src = 0;
            if (t < P::NT2XU) { vx = P::s2xu_vx(t); src = P::s2xu_src(t); }
            else if (t < P::NT2XU + P::NT2UU) { vx = P::s2uu_vx(t - P::NT2XU); src = P::s2uu_src(t - P::NT2XU); }
            else if (t < NT2) { vx = P::s2xx_vx(t - P::NT2XU - P::NT2UU); src = P::s2xx_src(t - P::NT2XU - P::NT2UU); }
            tdesc[r] = vx < 0 ? -1 : (vx | ((src + 32768) << 8));
        }
#pragma unroll
        for (int r = 0; r < RS; r++) sdesc[r] = -1;
        int cnt = 0;
        for (int e = 0; e < NQXU; e++) {
            const int t0 = P::s2xu_start(e), t1 = P::s2xu_start(e + 1);
            if (t1 > t0) {
#pragma unroll
                for (int r = 0; r < RS; r++)
                    if (cnt == lane + LPP * r) sdesc[r] = 0 | (e << 2) | (t0 << 12) | (t1 << 22);
                cnt++;
            }
        }
        for (int e = 0; e < NQUU; e++) {
            const int t0 = P::s2uu_start(e), t1 = P::s2uu_start(e + 1);
            if (t1 > t0) {
#pragma unroll
                for (int r = 0; r < RS; r++)
                    if (cnt == lane + LPP * r) sdesc[r] = 1 | (e << 2) | ((t0 + P::NT2XU) << 12) | ((t1 + P::NT2XU) << 22);
                cnt++;
            }
        }
        for (int e = 0; e < NQXX; e++) {
            const int t0 = P::s2xx_start(e), t1 = P::s2xx_start(e + 1);
            if (t1 > t0) {
#pragma unroll
                for (int r = 0; r < RS; r++)
                    if (cnt == lane + LPP * r) sdesc[r] = 2 | (e << 2) | ((t0 + P::NT2XU + P::NT2UU) << 12) | ((t1 + P::NT2XU + P::NT2UU) << 22);
                cnt++;
            }
        }
    }

    double dV0 = 0.0, dV1 = 0.0, g_sum = 0.0;
    int n_bp = w.n_bp[b];
    bool done = false;
    while (!done) {
        n_bp++;
        for (int e = lane; e < NX; e += LPP) ws.Vx[e] = w.FD[(size_t)e * Bp + b];
        for (int e = lane; e < NQXX; e += LPP) {
            const double v = w.FD[(size_t)(NX + e) * Bp + b];
            ws.VxxF[ws.tri_r[e] * LX + ws.tri_c[e]] = v;
            ws.VxxF[ws.tri_c[e] * LX + ws.tri_r[e]] = v;
        }
        dV0 = 0.0;
        dV1 = 0.0;
        g_sum = 0.0;
        double lk[NU];
#pragma unroll
        for (int i = 0; i < NU; i++) lk[i] = 0.0;
        bool failed = false;
        constexpr int R1 = (P::NV1 + LPP - 1) / LPP, R2 = (P::NV2 + LPP - 1) / LPP;
        constexpr int RU = (NU + LPP - 1) / LPP;
        double pf1[R1], pf2[R2], pfu[RU];
        {
            const double *rec = w.V1 + ((size_t)(T - 1) * Bp + b) * P::NV1;
#pragma unroll
            for (int t = 0; t < R1; t++) {
                const int j = lane + LPP * t;
                pf1[t] = (j < P::NV1) ? rec[j] : 0.0;
            }
            const double *rec2 = w.V2 + ((size_t)(T - 1) * Bp + b) * P::NV2;
#pragma unroll
            for (int t = 0; t < R2; t++) {
                const int j = lane + LPP * t;
                pf2[t] = (FULL && j < P::NV2_USED) ? rec2[j] : 0.0;
            }
            for (int t = 0; t < RU; t++) {
                const int j = lane + LPP * t;
                pfu[t] = (j < NU) ? w.XU[cur][((size_t)(T - 1) * Bp + b) * Rec<P>::RXU + NX + j] : 0.0;
            }
        }

        for (int k = T - 1; k >= 0; k--) {
            /* ---- the time-varying entries of step k were requested one step ahead (registers pf1/pf2, R1/R2 values per
                    lane); scatter them into the dense record, then request step k-1: its HBM latency hides behind
                    the arithmetic of this step ---- */
#pragma unroll
            for (int t = 0; t < R1; t++) {
                const int j = lane + LPP * t;
                if (j < P::NV1) Dd[P::v1_dst(j)] = pf1[t];
            }
            if (FULL) {
#pragma unroll
                for (int t = 0; t < R2; t++) {
                    const int j = lane + LPP * t;
                    if (j < P::NV2_USED) ws.v2[j] = pf2[t];
                }
            }
#pragma unroll
            for (int t = 0; t < RU; t++) {
                const int j = lane + LPP * t;
                if (j < NU) ws.un[j] = pfu[t];
            }
            if (k > 0) {
#pragma unroll
                for (int t = 0; t < RU; t++) {
                    const int j = lane + LPP * t;
                    if (j < NU) pfu[t] = w.XU[cur][((size_t)(k - 1) * Bp + b) * Rec<P>::RXU + NX + j];
                }
                const double *rec = w.V1 + ((size_t)(k - 1) * Bp + b) * P::NV1;
#pragma unroll
                for (int t = 0; t < R1; t++) {
                    const int j = lane + LPP * t;
                    if (j < P::NV1) pf1[t] = rec[j];
                }
                if (FULL) {
                    const double *rec2 = w.V2 + ((size_t)(k - 1) * Bp + b) * P::NV2;
#pragma unroll
                    for (int t = 0; t < R2; t++) {
                        const int j = lane + LPP * t;
                        if (j < P::NV2_USED) pf2[t] = rec2[j];
                    }
                }
            }
            __syncwarp(gmask);
            /* ---- phase 1: Qu, Qx, Vxx*fu, Vxx*fx (back_pass.c:80-92, matMult.c first halves) ---- */
            for (int e = lane; e < NU; e += LPP) {
                double acc = ws.D.cu[e];
#pragma unroll
                for (int r = 0; r < NX; r++) acc += ws.Vx[r] * ws.D.fu[r + e * NX];
                ws.Qu[e] = acc;
            }
            for (int e = lane; e < NX; e += LPP) {
                double acc = ws.D.cx[e];
#pragma unroll
                for (int r = 0; r < NX; r++) acc += ws.Vx[r] * ws.D.fx[r + e * NX];
                ws.Qx[e] = acc;
            }
            for (int e = lane; e < NX * NU; e += LPP) {
                const int r = e % NX, j = e / NX;
                double acc = 0.0;
#pragma unroll
                for (int s = 0; s < NX; s++) acc += ws.VxxF[r * LX + s] * ws.D.fu[s + j * NX];
                ws.bc[r + j * LX] = acc;
            }
            for (int e = lane; e < NX * NX; e += LPP) {
                const int r = e % NX, c = e / NX;
                double acc = 0.0;
#pragma unroll
                for (int s = 0; s < NX; s++) acc += ws.VxxF[r * LX + s] * ws.D.fx[s + c * NX];
                ws.ba[r + c * LX] = acc;
            }
            if (FULL) {
#pragma unroll
                for (int r = 0; r < RT; r++)
                    if (tdesc[r] >= 0) {
                        const int src = (tdesc[r] >> 8) - 32768;
                        ws.prod[lane + LPP * r] = ws.Vx[tdesc[r] & 0xff] * (src >= 0 ? ws.v2[src] : ws.c2[-src - 1]);
                    }
            }
            __syncwarp(gmask);
            /* ---- phase 2: Qxu, Quu, Qxx (first-order parts; the FULL_DDP terms follow in phase 2b) ---- */
            for (int e = lane; e < NQXU; e += LPP) {
                const int i = e % NX, j = e / NX;
                double acc = 0.0;
#pragma unroll
                for (int s = 0; s < NX; s++) acc += ws.D.fx[s + i * NX] * ws.bc[s + j * LX];
                double q = ws.D.cxu[e] + acc;
                ws.Qxu[e] = q;
            }
            for (int e = lane; e < NQUU; e += LPP) {
                const int r = ws.tri_r[e], c = ws.tri_c[e];
                double acc = 0.0;
#pragma unroll
                for (int s = 0; s < NX; s++) acc += ws.D.fu[s + r * NX] * ws.bc[s + c * LX];
                if (r != c) {
#pragma unroll
                    for (int s = 0; s < NX; s++) acc += ws.D.fu[s + c * NX] * ws.bc[s + r * LX];
                    acc *= 0.5;
                }
                double q = ws.D.cuu[e] + acc;
                ws.Quu[e] = q;
                ws.QuuS[r * LU + c] = q;
                ws.QuuS[c * LU + r] = q;
            }
            for (int e = lane; e < NQXX; e += LPP) {
                const int r = ws.tri_r[e], c = ws.tri_c[e];
                double acc = 0.0;
#pragma unroll
                for (int s = 0; s < NX; s++) acc += ws.D.fx[s + r * NX] * ws.ba[s + c * LX];
                if (r != c) {
#pragma unroll
                    for (int s = 0; s < NX; s++) acc += ws.D.fx[s + c * NX] * ws.ba[s + r * LX];
                    acc *= 0.5;
                }
                double q = ws.D.cxx[e] + acc;
                ws.Qxx[e] = q;
            }
            __syncwarp(gmask);
            if (FULL && NE2 > 0) {
                /* ---- phase 2b: Q??[entry] += sum of its products, serial in the reference's term order ---- */
#pragma unroll
                for (int r = 0; r < RS; r++) {
                    if (sdesc[r] < 0) continue;
                    const int kind = sdesc[r] & 3, e = (sdesc[r] >> 2) & 1023, t1 = (sdesc[r] >> 22) & 1023;
                    double d1 = 0.0;
                    for (int t = (sdesc[r] >> 12) & 1023; t < t1; t++) d1 += ws.prod[t];
                    if (kind == 0) ws.Qxu[e] += d1;
                    else if (kind == 2) ws.Qxx[e] += d1;
                    else {
                        const int rr = ws.tri_r[e], cc = ws.tri_c[e];
                        const double q = ws.Quu[e] + d1;
                        ws.Quu[e] = q;
                        ws.QuuS[rr * LU + cc] = q;
                        ws.QuuS[cc * LU + rr] = q;
                    }
                }
                __syncwarp(gmask);
            }
            /* ---- regularisation (back_pass.c:134-159) ---- */
            for (int e = lane; e < NQUU; e += LPP) ws.QuuF[e] = ws.Quu[e];
            for (int e = lane; e < NQXU; e += LPP) ws.Qxu_reg[e] = ws.Qxu[e];
            __syncwarp(gmask);
            if (o.regType == 2 && lane == 0) {
                for (int j = 0; j < NU; j++)
                    for (int i = 0; i <= j; i++) {
                        double acc = 0.0;
                        for (int c = 0; c < NU; c++) acc += ws.D.fu[symtri(c, i)] * ws.D.fu[symtri(c, j)];
                        ws.QuuF[utri(i, j)] += acc * lambda;
                    }
                for (int i = 0; i < NX; i++)
                    for (int j = 0; j < NU; j++) {
                        double acc = 0.0;
                        for (int c = 0; c < NX; c++) acc += ws.D.fx[c + i * NX] * ws.D.fu[(c + j * NU) < NX * NU ? (c + j * NU) : 0];
                        ws.Qxu_reg[i + j * NX] += acc * lambda;
                    }
            }
            if (o.regType == 1)
                for (int e = lane; e < NU; e += LPP) ws.QuuF[utri(e, e)] += lambda;
            __syncwarp(gmask);
            /* ---- box QP in every lane's registers (identical inputs -> identical results, uniform control flow) ---- */
            int clamped[NU], n_free;
            double invH[NQUU];
            int qp;
            {
                double H[NQUU], g[NU], lo[NU], hi[NU];
#pragma unroll
                for (int i = 0; i < NQUU; i++) H[i] = ws.QuuF[i];
#pragma unroll
                for (int i = 0; i < NU; i++) {
                    g[i] = ws.Qu[i];
                    lo[i] = ws.D.lower[i];
                    hi[i] = ws.D.upper[i];
                }
                qp = box_qp<NU, LPP>(H, g, lo, hi, lk, clamped, invH, n_free, lane, gmask, (int)(threadIdx.x & 31) - lane);
            }
            if (lane == 0) {
                if (w.tr_clamp) {
                    int code = (qp & 0xff) << 16;
#pragma unroll
                    for (int i = 0; i < NU; i++) code |= clamped[i] << (2 * i);
                    w.tr_clamp[(size_t)k * Bp + b] = code;
                }
#pragma unroll
                for (int i = 0; i < NU; i++) {
                    ws.clamped[i] = clamped[i];
                    ws.lk[i] = lk[i];
                }
#pragma unroll
                for (int i = 0; i < NQUU; i++) ws.invH[i] = invH[i];
            }
            if (qp < 1) {
                double *rec = w.Ll[cur] + ((size_t)k * Bp + b) * Rec<P>::RLS;   /* the failed QP's last iterate stays in t->l */
                for (int e = lane; e < NU; e += LPP) rec[e] = lk[e];
                failed = true;
                break;
            }
            __syncwarp(gmask);
            /* ---- gains (back_pass.c:173-201), one entry per lane; also the control-law record of step k ---- */
            {
                double *rec = w.LL[cur] + ((size_t)k * Bp + b) * Rec<P>::RLM, *recl = w.Ll[cur] + ((size_t)k * Bp + b) * Rec<P>::RLS;
            for (int e = lane; e < NU * NX; e += LPP) {
                    const int i = e % NU, s = e / NU;
                    double acc = 0.0;
                    if (ws.clamped[i]) {
                        if (P::HAS_HX)
                            acc -= (ws.clamped[i] == 1) ? ws.D.lower_sign[i] * ws.D.lower_hx[s + i * NX] : ws.D.upper_sign[i] * ws.D.upper_hx[s + i * NX];
                    } else {
                        for (int j = 0; j < NU; j++) {
                            if (!ws.clamped[j]) {
                                acc -= ws.invH[symtri(i, j)] * ws.Qxu_reg[s + j * NX];
                            } else if (P::HAS_HX) {
                                double wgt = 0.0;
                                for (int c = 0; c < NU; c++)
                                    if (!ws.clamped[c]) wgt -= ws.invH[symtri(i, c)] * ws.QuuF[symtri(c, j)];
                                acc -= wgt * ((ws.clamped[j] == 1) ? ws.D.lower_sign[j] * ws.D.lower_hx[s + j * NX]
                                                                    : ws.D.upper_sign[j] * ws.D.upper_hx[s + j * NX]);
                            }
                        }
                    }
                    ws.Lk[e] = acc;
                    rec[e] = acc;
                }
                for (int e = NU * NX + lane; e < Rec<P>::RLM; e += LPP) rec[e] = 0.0;
                for (int e = lane; e < Rec<P>::RLS; e += LPP) recl[e] = (e < NU) ? lk[e] : 0.0;
            }
            /* ---- expected reduction (back_pass.c:204-214), every lane keeps the same running sums ---- */
#pragma unroll
            for (int i = 0; i < NU; i++) dV0 += ws.Qu[i] * lk[i];
#pragma unroll
            for (int i = 0; i < NU; i++) {
                double acc = 0.0;
#pragma unroll
                for (int j = 0; j < NU; j++) acc += lk[j] * ws.Quu[symtri(j, i)];
                dV1 += 0.5 * lk[i] * acc;
            }
            __syncwarp(gmask);
            /* ---- phase 3: Quu*l, Quu*L ---- */
            for (int e = lane; e < NU; e += LPP) {
                double acc = 0.0;
#pragma unroll
                for (int s = 0; s < NU; s++) acc += ws.QuuS[e * LU + s] * ws.lk[s];
                ws.bv[e] = acc;
            }
            for (int e = lane; e < NU * NX; e += LPP) {
                const int r = e % NU, c = e / NU;
                double acc = 0.0;
#pragma unroll
                for (int s = 0; s < NU; s++) acc += ws.QuuS[r * LU + s] * ws.Lk[s + c * NU];
                ws.bl[r + c * LU] = acc;
            }
            __syncwarp(gmask);
            /* ---- phase 4: value function (back_pass.c:217-241) ---- */
            for (int e = lane; e < NX; e += LPP) {
                double acc = 0.0;
#pragma unroll
                for (int s = 0; s < NU; s++) acc += ws.Lk[s + e * NU] * ws.bv[s];
                double v = ws.Qx[e] + acc;
#pragma unroll
                for (int j = 0; j < NU; j++) v += ws.Lk[j + e * NU] * ws.Qu[j];
#pragma unroll
                for (int j = 0; j < NU; j++) v += ws.Qxu[e + j * NX] * ws.lk[j];
                ws.Vx[e] = v;
            }
            for (int e = lane; e < NQXX; e += LPP) {
                const int r = ws.tri_r[e], c = ws.tri_c[e];
                double acc = 0.0;
#pragma unroll
                for (int s = 0; s < NU; s++) acc += ws.Lk[s + r * NU] * ws.bl[s + c * LU];
                if (r != c) {
#pragma unroll
                    for (int s = 0; s < NU; s++) acc += ws.Lk[s + c * NU] * ws.bl[s + r * LU];
                    acc *= 0.5;
                }
                double v = ws.Qxx[e] + acc;
                if (r == c) {
#pragma unroll
                    for (int cc = 0; cc < NU; cc++) {
                        double term = ws.Lk[cc + r * NU] * ws.Qxu[r + cc * NX];
                        term *= 2.0;
                        v += term;
                    }
                } else { /* the reference's loop visits (i=r, j=c) before (i=c, j=r) for r < c */
#pragma unroll
                    for (int cc = 0; cc < NU; cc++) v += ws.Lk[cc + r * NU] * ws.Qxu[c + cc * NX];
#pragma unroll
                    for (int cc = 0; cc < NU; cc++) v += ws.Lk[cc + c * NU] * ws.Qxu[r + cc * NX];
                }
                ws.VxxF[r * LX + c] = v;
                ws.VxxF[c * LX + r] = v;
            }
            /* ---- gradient measure (back_pass.c:244-251) ---- */
            {
                double gmax = 0.0;
#pragma unroll
                for (int i = 0; i < NU; i++) {
                    const double gi = fabs(lk[i]) / (fabs(ws.un[i]) + 1.0);
                    if (gi > gmax) gmax = gi;
                }
                g_sum += gmax;
            }
            __syncwarp(gmask);
        }
        __syncwarp(gmask);
        if (failed) {
            if (o.bp_single) break;
            raise_lambda(o, lambda, dlambda);
            if (lambda > o.lambdaMax) break;
        } else {
            done = true;
        }
    }
    if (lane != 0) return;
    w.n_bp[b] = n_bp;
    w.dV0[b] = dV0;
    w.dV1[b] = dV1;
    w.bp_done[b] = done ? 1 : 0;
    double g_norm = w.g_norm[b];
    if (done) {
        g_norm = g_sum / ((double)(T - 1));
        w.g_norm[b] = g_norm;
    }
    if (o.bp_single) return;
    if (g_norm < o.tolGrad && lambda < 1e-5) {
        lower_lambda(o, lambda, dlambda);
        finish(w, b, iter, done ? 1 : 0);
    } else if (!done) {
        finish(w, b, iter, 0);
    }
    w.lambda[b] = lambda;
    w.dlambda[b] = dlambda;
}

} /* namespace ilqg */
#include "ilqg_backpass_split.cuh"
namespace ilqg {

/* =====================================================================================================================
 * K3: rollouts.  MODE 0 = initial rollout of the caller's controls (alpha = 0, clamped; iLQG_mex.c:113-120 and the
 * first lines of iLQG(), iLQG.c:227-237).  MODE 1 = backtracking line search + accept/reject (line_search.c:33-78,
 * iLQG.c:306-361).
 * ===================================================================================================================== */
/* number of time segments a recorded rollout can be replayed in (one per lane of a warp) and their length */
constexpr int LS_SEGS = 32;
__host__ __device__ inline int ls_seg_len(int T) { return (T + LS_SEGS - 1) / LS_SEGS; }

template <class P, bool STORE = true, bool CKPT = false, class PK>
__device__ __forceinline__ bool rollout(const Work &w, const double *pv, const PK &pk, int b, int from, int to, double alpha,
                                        double w_pen_l, double w_pen_f, double &csum, double *ckpt = nullptr)
{
    constexpr int NX = P::NX, NU = P::NU, RXU = Rec<P>::RXU, RLM = Rec<P>::RLM, RLS = Rec<P>::RLS, RLL = NU + RLM;
    const size_t Bp = w.Bp;
    const int T = w.T;
    double xu[RXU], xn[NX], mu[P::N_MU_R + P::N_MU_F + 1];
    double *x = xu, *u = xu + NX;
#pragma unroll
    for (int i = 0; i < RXU; i++) xu[i] = 0.0;
#pragma unroll
    for (int i = 0; i < NX; i++) x[i] = w.x0[(size_t)i * Bp + b];
    csum = 0.0;
    /* software pipeline: the nominal records of step k+1 are requested before step k is computed, so their HBM / L2
       latency hides behind the dynamics and cost arithmetic (they do not depend on the rollout's own state) */
    constexpr bool PF = (RXU + RLL) <= 32;   /* small records only: a second register copy of a large record spills */
    double nom[RXU], ll[RLL], nom_n[PF ? RXU : 1], ll_n[PF ? RLL : 1];
    if (PF) {
        ld_rec<NX + NU>(w.XU[from] + (size_t)b * RXU, nom);
        if (alpha != 0.0) {
            ld_rec<NU>(w.Ll[from] + (size_t)b * RLS, ll);
            ld_rec<NU * NX>(w.LL[from] + (size_t)b * RLM, ll + NU);
        }
    }
    const int seg_len = ls_seg_len(T);
    int next_ck = 0;
    for (int k = 0; k < T; k++) {
        if (CKPT && k == next_ck) { /* state at the start of every segment: k_ls_commit replays the winner segment-parallel */
            double *c = ckpt + ((size_t)(k / seg_len) * Bp + b) * NX;
#pragma unroll
            for (int i = 0; i < NX; i++) c[i] = x[i];
            next_ck += seg_len;
        }
        if (PF) {
            if (k + 1 < T) {
                ld_rec<PF ? NX + NU : 1>(w.XU[from] + ((size_t)(k + 1) * Bp + b) * RXU, nom_n);
                if (alpha != 0.0) {
                    ld_rec<PF ? NU : 1>(w.Ll[from] + ((size_t)(k + 1) * Bp + b) * RLS, ll_n);
                    ld_rec<PF ? NU * NX : 1>(w.LL[from] + ((size_t)(k + 1) * Bp + b) * RLM, ll_n + (PF ? NU : 0));
                }
            }
        } else {
            ld_rec<NX + NU>(w.XU[from] + ((size_t)k * Bp + b) * RXU, nom);
            if (alpha != 0.0) {
                ld_rec<NU>(w.Ll[from] + ((size_t)k * Bp + b) * RLS, ll);
                ld_rec<NU * NX>(w.LL[from] + ((size_t)k * Bp + b) * RLM, ll + NU);
            }
        }
        if (alpha != 0.0) {
#pragma unroll
            for (int j = 0; j < NU; j++) u[j] = nom[NX + j] + ll[j] * alpha;
#pragma unroll
            for (int i = 0; i < NX; i++) {
                const double dx = x[i] - nom[i];
#pragma unroll
                for (int j = 0; j < NU; j++) u[j] += ll[NU + j + i * NU] * dx;
            }
        } else {
#pragma unroll
            for (int j = 0; j < NU; j++) u[j] = nom[NX + j];
        }
#pragma unroll
        for (int i = 0; i < P::N_MU_R; i++) mu[i] = w.muR[((size_t)k * P::N_MU_R + i) * Bp + b];
        double c;
        const bool ok = P::step(x, u, pv, pk, k, T, w_pen_l, mu, xn, c);
        if (STORE) st_rec<RXU>(w.XU[to] + ((size_t)k * Bp + b) * RXU, xu);
        if (!ok) return false;
        csum += c;
#pragma unroll
        for (int i = 0; i < NX; i++) x[i] = xn[i];
        if (PF) {
#pragma unroll
            for (int i = 0; i < (PF ? NX + NU : 0); i++) nom[i] = nom_n[i];
#pragma unroll
            for (int i = 0; i < (PF ? NU + NU * NX : 0); i++) ll[i] = ll_n[i];
        }
    }
#pragma unroll
    for (int j = 0; j < NU; j++) u[j] = 0.0;
    if (STORE) st_rec<RXU>(w.XU[to] + ((size_t)T * Bp + b) * RXU, xu);
#pragma unroll
    for (int i = 0; i < P::N_MU_F; i++) mu[i] = w.muF[(size_t)i * Bp + b];
    double c;
    if (!P::final_cost(x, pv, pk, T, T, w_pen_f, mu, c)) return false;
    csum += c;
    return true;
}

/* cost-only pass over the nominal trajectory (forward_pass with cost_only = 1) */
template <class P, class PK>
__device__ __forceinline__ bool cost_pass(const Work &w, const double *pv, const PK &pk, int b, int buf, double w_pen_l,
                                          double w_pen_f, double &csum)
{
    constexpr int NX = P::NX, NU = P::NU, RXU = Rec<P>::RXU;
    const size_t Bp = w.Bp;
    const int T = w.T;
    double xu[RXU], mu[P::N_MU_R + P::N_MU_F + 1];
    csum = 0.0;
    for (int k = 0; k < T; k++) {
        ld_rec<NX + NU>(w.XU[buf] + ((size_t)k * Bp + b) * RXU, xu);
#pragma unroll
        for (int i = 0; i < P::N_MU_R; i++) mu[i] = w.muR[((size_t)k * P::N_MU_R + i) * Bp + b];
        double c;
        if (!P::step_cost(xu, xu + NX, pv, pk, k, T, w_pen_l, mu, c)) return false;
        csum += c;
    }
    ld_rec<NX>(w.XU[buf] + ((size_t)T * Bp + b) * RXU, xu);
#pragma unroll
    for (int i = 0; i < P::N_MU_F; i++) mu[i] = w.muF[(size_t)i * Bp + b];
    double c;
    if (!P::final_cost(xu, pv, pk, T, T, w_pen_f, mu, c)) return false;
    csum += c;
    return true;
}


/* Steps [k0, k1) of a rollout whose state at step k0 is known (recorded by a checkpointing rollout): the same operations
 * in the same order as rollout(), hence the same bits, always with stores.  The segment that ends at T also writes the
 * final record. */
template <class P, class PK>
__device__ __forceinline__ void rollout_segment(const Work &w, const double *pv, const PK &pk, int b, int from, int to, double alpha,
                                                double w_pen_l, int k0, int k1, const double *xs)
{
    constexpr int NX = P::NX, NU = P::NU, RXU = Rec<P>::RXU, RLM = Rec<P>::RLM, RLS = Rec<P>::RLS, RLL = NU + RLM;
    const size_t Bp = w.Bp;
    const int T = w.T;
    double xu[RXU], xn[NX], mu[P::N_MU_R + P::N_MU_F + 1], nom[RXU], ll[RLL];
    double *x = xu, *u = xu + NX;
#pragma unroll
    for (int i = 0; i < RXU; i++) xu[i] = 0.0;
#pragma unroll
    for (int i = 0; i < NX; i++) x[i] = xs[i];
    for (int k = k0; k < k1; k++) {
        ld_rec<NX + NU>(w.XU[from] + ((size_t)k * Bp + b) * RXU, nom);
        if (alpha != 0.0) {
            ld_rec<NU>(w.Ll[from] + ((size_t)k * Bp + b) * RLS, ll);
            ld_rec<NU * NX>(w.LL[from] + ((size_t)k * Bp + b) * RLM, ll + NU);
#pragma unroll
            for (int j = 0; j < NU; j++) u[j] = nom[NX + j] + ll[j] * alpha;
#pragma unroll
            for (int i = 0; i < NX; i++) {
                const double dx = x[i] - nom[i];
#pragma unroll
                for (int j = 0; j < NU; j++) u[j] += ll[NU + j + i * NU] * dx;
            }
        } else {
#pragma unroll
            for (int j = 0; j < NU; j++) u[j] = nom[NX + j];
        }
#pragma unroll
        for (int i = 0; i < P::N_MU_R; i++) mu[i] = w.muR[((size_t)k * P::N_MU_R + i) * Bp + b];
        double c;
        P::step(x, u, pv, pk, k, T, w_pen_l, mu, xn, c);
        st_rec<RXU>(w.XU[to] + ((size_t)k * Bp + b) * RXU, xu);
#pragma unroll
        for (int i = 0; i < NX; i++) x[i] = xn[i];
    }
    if (k1 == T) {
#pragma unroll
        for (int j = 0; j < NU; j++) u[j] = 0.0;
        st_rec<RXU>(w.XU[to] + ((size_t)T * Bp + b) * RXU, xu);
    }
}

/* update_multipliers(o, init) of one problem (iLQG_func.tem:417-509) on the trajectory in buffer `buf`.  init = 1 only records
 * the constraint values: of step 0 for the running constraints -- the reference's early return sits INSIDE the loop over the
 * steps (iLQG_func.tem:452) -- and of the final ones; it never touches multipliers or penalty weights.  The multiplier
 * updates use the penalty weights the call started with, like the reference's local copies. */
template <class P, class PK>
__device__ __forceinline__ void update_mult(const Work &w, const Opts &o, const double *pv, const PK &pk, int b, int buf, bool init,
                                            double &w_pen_l, double &w_pen_f)
{
    constexpr int NX = P::NX, NU = P::NU, NR = P::N_MU_R, NF = P::N_MU_F;
    const size_t Bp = w.Bp;
    const int T = w.T;
    double x[NX], u[NU], mu[NR + NF + 1], hval[NR + NF + 1], mun[NR + NF + 1];
    if (NR > 0) {
        bool increase = false;
        const int k_end = init ? (T > 0 ? 1 : 0) : T;
        for (int k = 0; k < k_end; k++) {
            double xu[Rec<P>::RXU];
            ld_rec<NX + NU>(w.XU[buf] + ((size_t)k * Bp + b) * Rec<P>::RXU, xu);
#pragma unroll
            for (int i = 0; i < NX; i++) x[i] = xu[i];
#pragma unroll
            for (int j = 0; j < NU; j++) u[j] = xu[NX + j];
#pragma unroll
            for (int i = 0; i < NR; i++) mu[i] = w.muR[((size_t)k * NR + i) * Bp + b];
            P::mult_running(x, u, pv, pk, k, T, w_pen_l, mu, hval, mun);
#pragma unroll
            for (int i = 0; i < NR; i++) {
                double *last = &w.lastR[((size_t)k * NR + i) * Bp + b];
                if (i < P::N_MU_LE) {
                    if (fabs(hval[i]) > o.tolConstraint && o.w_pen_fact1 * fabs(hval[i]) > fabs(*last)) increase = true;
                } else {
                    if (hval[i] > o.tolConstraint && o.w_pen_fact1 * hval[i] > *last) increase = true;
                }
                *last = hval[i];
                if (!init) w.muR[((size_t)k * NR + i) * Bp + b] = mun[i];
            }
        }
        if (!init && increase) w_pen_l = dmin(o.w_pen_max_l, w_pen_l * o.w_pen_fact1);
    }
    if (NF > 0) {
        bool increase = false;
        ld_rec<NX>(w.XU[buf] + ((size_t)T * Bp + b) * Rec<P>::RXU, x);
#pragma unroll
        for (int i = 0; i < NF; i++) mu[i] = w.muF[(size_t)i * Bp + b];
        P::mult_final(x, pv, pk, T, T, w_pen_f, mu, hval, mun);
#pragma unroll
        for (int i = 0; i < NF; i++) {
            double *last = &w.lastF[(size_t)i * Bp + b];
            if (i < P::N_MU_FE) {
                if (fabs(hval[i]) > o.tolConstraint && o.w_pen_fact1 * fabs(hval[i]) > fabs(*last)) increase = true;
            } else {
                if (hval[i] > o.tolConstraint && o.w_pen_fact1 * hval[i] > *last) increase = true;
            }
            *last = hval[i];
            if (!init) w.muF[(size_t)i * Bp + b] = mun[i];
        }
        if (!init && increase) w_pen_f = dmin(o.w_pen_max_f, w_pen_f * o.w_pen_fact1);
    }
}

enum { INIT_MULT = 1, INIT_ROLLOUT = 2, INIT_BEGIN = 4, INIT_ALL = 7 };

template <class P, bool PP, bool TR = false>
__global__ void __launch_bounds__(BP_BLOCK) k_init(Work w, Opts o, ParamBlock<P> pb, int mode)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= w.B) return;
    ILQG_PARAMS(PP, b)
    ILQG_PK(TR, b)
    const size_t Bp = w.Bp;
    const int T = w.T;
    if (mode & INIT_MULT) { /* init_multipliers (iLQG_func.tem:364-400) */
        for (int k = 0; k < T; k++)
#pragma unroll
            for (int i = 0; i < P::N_MU_R; i++) {
                w.muR[((size_t)k * P::N_MU_R + i) * Bp + b] = (i < P::N_MU_LE) ? 0.0 : 1.0;
                w.lastR[((size_t)k * P::N_MU_R + i) * Bp + b] = 0.0;
            }
#pragma unroll
        for (int i = 0; i < P::N_MU_F; i++) {
            w.muF[(size_t)i * Bp + b] = (i < P::N_MU_FE) ? 0.0 : 1.0;
            w.lastF[(size_t)i * Bp + b] = 0.0;
        }
    }
    /* the caller's controls sit in buffer 0; roll them out (clamped) into buffer 1, which becomes nominal.
       The harness-level rollout runs before iLQG() sets the penalty weights, i.e. with whatever the option struct
       holds: w_pen_l/f are still their zero-initialised values at that point (iLQG_mex.c:24,116). */
    bool ok = true;
    if (mode & INIT_ROLLOUT) {
        double csum;
        ok = rollout<P>(w, pv, pk, b, 0, 1, 0.0, 0.0, 0.0, csum);
        w.cur[b] = 1;
        w.cost[b] = csum;
        w.new_cost[b] = csum;
    }
    if (!(mode & INIT_BEGIN)) return;
    const int nb = w.cur[b]; /* nominal buffer */
    w.dcost[b] = 0.0;
    w.expected[b] = 0.0;
    w.g_norm[b] = 0.0;
    w.dV0[b] = 0.0;
    w.dV1[b] = 0.0;
    w.n_ls[b] = 0;
    w.n_bp[b] = 0;
    w.n_dv[b] = 0;
    w.n_roll[b] = 0;
    w.n_tail[b] = 0;
    w.bp_done[b] = 0;
    w.deriv_fail[b] = 0;
    w.post_mode[b] = POST_NONE;
    w.iterations[b] = 0;
    w.result[b] = ok ? 0 : -1;
    w.status[b] = ok ? ST_RUNNING : ST_DONE;
    /* first lines of iLQG() (iLQG.c:226-237) */
    w.lambda[b] = o.lambdaInit;
    w.dlambda[b] = o.dlambdaInit;
    w.w_pen_l[b] = o.w_pen_init_l;
    w.w_pen_f[b] = o.w_pen_init_f;
    w.new_deriv[b] = 1;
    if (ok && (P::N_MU_R + P::N_MU_F) > 0) { /* update_multipliers(o, 1), iLQG.c:236 */
        double wl = o.w_pen_init_l, wf = o.w_pen_init_f;
        update_mult<P>(w, o, pv, pk, b, nb, true, wl, wf);
    }
}

/* forward_pass(candidate, o, alpha, &csum, cost_only) of the single-problem API on its own (iLQG_func.tem:121-185):
 * one rollout from the nominal buffer into the other one (or the cost-only pass over the nominal); csum -> new_cost,
 * success flag -> result.  No solver bookkeeping. */
template <class P, bool PP, bool TR = false>
__global__ void __launch_bounds__(BP_BLOCK) k_rollout_only(Work w, ParamBlock<P> pb, double alpha, int cost_only)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= w.B) return;
    ILQG_PARAMS(PP, b)
    ILQG_PK(TR, b)
    const int cur = w.cur[b];
    double csum;
    const bool ok = cost_only ? cost_pass<P>(w, pv, pk, b, cur, w.w_pen_l[b], w.w_pen_f[b], csum)
                              : rollout<P>(w, pv, pk, b, cur, cur ^ 1, alpha, w.w_pen_l[b], w.w_pen_f[b], csum);
    w.new_cost[b] = csum;
    w.result[b] = ok ? 1 : 0;
}

/* accept / reject bookkeeping of one problem once its line search is decided (iLQG.c:311-361) */
__device__ __forceinline__ void ls_decide(const Work &w, const Opts &o, int b, int iter, int cur, bool accepted, int alpha_idx,
                                          double cnew, double dcost, double w_pen_l, double w_pen_f)
{
    const size_t Bp = w.Bp;
    double lambda = w.lambda[b], dlambda = w.dlambda[b];
    if (w.tr_alpha) w.tr_alpha[(size_t)iter * Bp + b] = alpha_idx;
    if (w.tr_newcost) w.tr_newcost[(size_t)iter * Bp + b] = cnew;
    int post = POST_NONE;
    if (accepted) { /* iLQG.c:311-338 */
        lower_lambda(o, lambda, dlambda);
        w.cur[b] = cur ^ 1;
        w.cost[b] = cnew;
        w.new_deriv[b] = 1;
        if (dcost < o.tolFun)
            finish(w, b, iter, 1);
        else
            post = POST_MULT;
    } else { /* iLQG.c:340-361 */
        raise_lambda(o, lambda, dlambda);
        if (o.w_pen_fact2 > 1.0) {
            w.w_pen_l[b] = dmin(o.w_pen_max_l, w_pen_l * o.w_pen_fact2);
            w.w_pen_f[b] = dmin(o.w_pen_max_f, w_pen_f * o.w_pen_fact2);
            post = POST_COST;
        }
        if (lambda > o.lambdaMax)
            finish(w, b, iter, 1); /* backPassDone is set and iter < max_iter: the reference returns 1 here */
    }
    w.post_mode[b] = post;
    w.lambda[b] = lambda;
    w.dlambda[b] = dlambda;
}

/* K3: line search, one ROUND per launch.  Round r rolls out alpha[r] for every problem that has not accepted a step
 * yet (line_search.c:37-60 tries the alphas in order and takes the first with z > zMin).  Round 0 runs over all
 * running problems with lane == problem; every later round runs over the compacted list of problems the previous
 * round left undecided, so all lanes of a warp do the same amount of work (one full rollout) instead of idling
 * while one neighbour backtracks.  The list keeps the problems of a block in order, which keeps most 32-byte
 * sectors shared between neighbouring lanes.  The problem that accepts, or exhausts the alphas, runs the
 * accept/reject bookkeeping of iLQG.c:311-361 in the same thread. */
template <class P, bool PP, bool TR = false>
__global__ void __launch_bounds__(BP_BLOCK, ILQG_LS_MINBLOCKS)
k_ls_round(Work w, Opts o, ParamBlock<P> pb, int iter, int round)
{
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const size_t Bp = w.Bp;
    int b = -1;
    if (round == 0) {
        if (tid < w.B && w.status[tid] == ST_RUNNING) b = tid;
    } else {
        if (tid < w.ls_count[round]) b = w.ls_list[round & 1][tid];
    }
    bool undecided = false;
    if (b >= 0) {
        ILQG_PARAMS(PP, b)
        ILQG_PK(TR, b)
        const int cur = w.cur[b];
        const double cost = w.cost[b], dV0 = w.dV0[b], dV1 = w.dV1[b];
        double w_pen_l = w.w_pen_l[b], w_pen_f = w.w_pen_f[b];
        double cnew, dcost = w.dcost[b], expected = w.expected[b];
        if (round == 0) {
            if (w.tr_lambda) w.tr_lambda[(size_t)iter * Bp + b] = w.lambda[b];
            w.n_ls[b] += 1;
        }
        w.n_roll[b] += 1;
        const double alpha = o.alpha[round];
        bool accepted = false;
        const bool ok = rollout<P>(w, pv, pk, b, cur, cur ^ 1, alpha, w_pen_l, w_pen_f, cnew);
        if (ok) {
            dcost = cost - cnew;
            expected = -alpha * (dV0 + alpha * dV1);
            const double z = (expected > 0) ? dcost / expected : 0.0;
            accepted = z > o.zMin;
            if (w.tr_z) w.tr_z[(size_t)iter * Bp + b] = z;
        }
        w.new_cost[b] = cnew;
        w.dcost[b] = dcost;
        w.expected[b] = expected;
        if (accepted || round == o.n_alpha - 1) {
            ls_decide(w, o, b, iter, cur, accepted, accepted ? round + 1 : o.n_alpha + 1, cnew, dcost, w_pen_l, w_pen_f);
        } else {
            undecided = true;
        }
    }
    /* ordered compaction of the undecided problems of this block into the next round's list */
    __shared__ int s_warp[BP_BLOCK / 32];
    __shared__ int s_base;
    const unsigned ballot = __ballot_sync(0xffffffffu, undecided);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) s_warp[wid] = __popc(ballot);
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0;
#pragma unroll
        for (int i = 0; i < BP_BLOCK / 32; i++) {
            const int c = s_warp[i];
            s_warp[i] = tot;
            tot += c;
        }
        s_base = tot ? atomicAdd(&w.ls_count[round + 1], tot) : 0;
    }
    __syncthreads();
    if (undecided) {
        w.ls_list[(round + 1) & 1][s_base + s_warp[wid] + __popc(ballot & ((1u << lane) - 1u))] = b;
        w.ls_mask[b] = 0;
    }
}

/* K3 tail (small batches, where a launch is bound by the latency of ONE 500-step rollout, not by throughput): after
 * `from` sequential rounds, all remaining alphas of every undecided problem are rolled out AT ONCE, one lane per
 * (problem, alpha), without storing trajectories; k_ls_commit then replays the reference's sequential decision over
 * the recorded costs (first alpha with z > zMin wins, line_search.c:37-60) and re-runs only the winning rollout with
 * stores.  The line search then costs from + 2 rollout latencies instead of n_alpha; results are bit-identical. */
template <class P, bool PP, bool CKPT, bool TR = false>
__global__ void __launch_bounds__(BP_BLOCK, ILQG_LS_MINBLOCKS) k_ls_tail(Work w, Opts o, ParamBlock<P> pb, int from)
{
    const int nrem = o.n_alpha - from;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = tid / nrem, a = from + tid % nrem;
    int b;
    if (from == 0) { /* no sequential round at all (very small batches): every running problem, every alpha */
        if (i >= w.B || w.status[i] != ST_RUNNING) return;
        b = i;
    } else {
        if (i >= w.ls_count[from]) return;
        b = w.ls_list[from & 1][i];
    }
    ILQG_PARAMS(PP, b)
    ILQG_PK(TR, b)
    const int cur = w.cur[b];
    const double alpha = o.alpha[a];
    double cnew;
    const bool ok = rollout<P, false, CKPT>(w, pv, pk, b, cur, cur ^ 1, alpha, w.w_pen_l[b], w.w_pen_f[b], cnew,
                                            CKPT ? w.ls_ckpt + (size_t)a * LS_SEGS * w.Bp * P::NX : nullptr);
    w.ls_cnew[(size_t)a * w.Bp + b] = cnew;
    if (ok) {
        const double dcost = w.cost[b] - cnew;
        const double expected = -alpha * (w.dV0[b] + alpha * w.dV1[b]);
        const double z = (expected > 0) ? dcost / expected : 0.0;
        atomicOr(&w.ls_mask[b], (1 << a) | ((z > o.zMin) ? (1 << (16 + a)) : 0));   /* low half: rollout ok, high half: accepted */
    }
}

template <class P, bool PP, bool NOROLL, bool TR = false>
__global__ void __launch_bounds__(BP_BLOCK, ILQG_LS_MINBLOCKS) k_ls_commit(Work w, Opts o, ParamBlock<P> pb, int iter, int from)
{
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const size_t Bp = w.Bp;
    int b;
    if (from == 0) {
        if (tid >= w.B || w.status[tid] != ST_RUNNING) return;
        b = tid;
        if (w.tr_lambda) w.tr_lambda[(size_t)iter * Bp + b] = w.lambda[b];
        w.n_ls[b] += 1;
    } else {
        if (tid >= w.ls_count[from]) return;
        b = w.ls_list[from & 1][tid];
    }
    ILQG_PARAMS(PP, b)
    ILQG_PK(TR, b)
    const int cur = w.cur[b];
    const int mask = w.ls_mask[b];
    const double cost = w.cost[b], dV0 = w.dV0[b], dV1 = w.dV1[b];
    double w_pen_l = w.w_pen_l[b], w_pen_f = w.w_pen_f[b];
    double cnew = w.new_cost[b], dcost = w.dcost[b], expected = w.expected[b];
    int win = -1;
    for (int a = from; a < o.n_alpha; a++) { /* the sequential semantics over the recorded rollouts */
        cnew = w.ls_cnew[(size_t)a * Bp + b];
        if (mask & (1 << a)) {
            const double alpha = o.alpha[a];
            dcost = cost - cnew;
            expected = -alpha * (dV0 + alpha * dV1);
            if (w.tr_z) w.tr_z[(size_t)iter * Bp + b] = (expected > 0) ? dcost / expected : 0.0;
        }
        if (mask & (1 << (16 + a))) {
            win = a;
            break;
        }
    }
    w.n_tail[b] += 1;
    w.n_roll[b] += (win >= 0 ? 1 : 0);
    if (win >= 0 && !NOROLL) { /* NOROLL: k_ls_commit_seg has stored the winner's trajectory, its cost is the recorded one */
        double c2;
        rollout<P, true>(w, pv, pk, b, cur, cur ^ 1, o.alpha[win], w_pen_l, w_pen_f, c2); /* same arithmetic -> same cost */
        cnew = c2;
    }
    w.new_cost[b] = cnew;
    w.dcost[b] = dcost;
    w.expected[b] = expected;
    ls_decide(w, o, b, iter, cur, win >= 0, win >= 0 ? win + 1 : o.n_alpha + 1, cnew, dcost, w_pen_l, w_pen_f);
}


/* Segment-parallel re-roll of the winners (with k_ls_tail<.., CKPT = true>): thread (problem, segment) -- blockIdx.y is the
 * segment, lane == position in the problem list exactly as in k_ls_commit, so a warp still reads and writes one contiguous
 * run of records per step -- re-runs steps [s * seg_len, (s + 1) * seg_len) of the winning rollout from the state the tail
 * recorded at the start of that segment, with stores.  The re-roll then costs the latency of T / 32 steps instead of T.
 * Every step repeats the tail's arithmetic on the same inputs, so the stored trajectory is bit-identical to the one the
 * sequential commit writes; k_ls_commit<.., NOROLL = true> follows with the bookkeeping and takes the cost from the tail's
 * record.  This kernel only reads solver state. */
template <class P, bool PP, bool TR = false>
__global__ void __launch_bounds__(BP_BLOCK, ILQG_LS_MINBLOCKS) k_ls_commit_seg(Work w, Opts o, ParamBlock<P> pb, int from)
{
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int seg = blockIdx.y;
    int b;
    if (from == 0) {
        if (tid >= w.B || w.status[tid] != ST_RUNNING) return;
        b = tid;
    } else {
        if (tid >= w.ls_count[from]) return;
        b = w.ls_list[from & 1][tid];
    }
    const int acc = (w.ls_mask[b] >> (16 + from)) & ((1 << (o.n_alpha - from)) - 1);
    if (!acc) return;
    const int win = from + (__ffs(acc) - 1);   /* first acceptable alpha (line_search.c:37-60) */
    const int T = w.T, seg_len = ls_seg_len(T);
    const int k0 = seg * seg_len, k1 = (k0 + seg_len < T) ? k0 + seg_len : T;
    if (k0 >= T) return;
    ILQG_PARAMS(PP, b)
    ILQG_PK(TR, b)
    const int cur = w.cur[b];
    double xs[P::NX];
    const double *c = w.ls_ckpt + (((size_t)win * LS_SEGS + seg) * w.Bp + b) * P::NX;
#pragma unroll
    for (int i = 0; i < P::NX; i++) xs[i] = c[i];
    rollout_segment<P>(w, pv, pk, b, cur, cur ^ 1, o.alpha[win], w.w_pen_l[b], k0, k1, xs);
}

/* K5: update_multipliers(o, 0) and the cost-only pass that follows an accepted step, or the cost-only pass after a
 * rejected step whose penalty weights grew (iLQG.c:337-338, 345-349).  Only launched for problems with multipliers. */
template <class P, bool PP, bool TR = false>
__global__ void __launch_bounds__(BP_BLOCK) k_post(Work w, Opts o, ParamBlock<P> pb)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= w.B) return;
    const int mode = w.post_mode[b];
    if (mode == POST_NONE) return;
    w.post_mode[b] = POST_NONE;
    ILQG_PARAMS(PP, b)
    ILQG_PK(TR, b)
    const int cur = w.cur[b];
    double w_pen_l = w.w_pen_l[b], w_pen_f = w.w_pen_f[b];
    if (mode == POST_MULT) {
        update_mult<P>(w, o, pv, pk, b, cur, false, w_pen_l, w_pen_f);
        w.w_pen_l[b] = w_pen_l;
        w.w_pen_f[b] = w_pen_f;
    }
    double csum;
    cost_pass<P>(w, pv, pk, b, cur, w_pen_l, w_pen_f, csum);
    w.cost[b] = csum;
}


/* update_multipliers(o, init) on its own (iLQG.h:86), for every running problem: the single-problem drop-in's entry point */
template <class P, bool PP, bool TR = false>
__global__ void __launch_bounds__(BP_BLOCK) k_mult(Work w, Opts o, ParamBlock<P> pb, int init)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= w.B || w.status[b] != ST_RUNNING) return;
    ILQG_PARAMS(PP, b)
    ILQG_PK(TR, b)
    double w_pen_l = w.w_pen_l[b], w_pen_f = w.w_pen_f[b];
    update_mult<P>(w, o, pv, pk, b, w.cur[b], init != 0, w_pen_l, w_pen_f);
    w.w_pen_l[b] = w_pen_l;
    w.w_pen_f[b] = w_pen_f;
}

/* The dense per-step record the backward pass works on (fx fu cx cxx cu cuu cxu lower upper lower_sign upper_sign lower_hx
 * upper_hx: the derivative members of trajEl_t, iLQG_problem.tem:23-51), rebuilt from the time-varying entries of the last
 * derivative sweep and the parameters: out[b][k][DENSE_SIZE].  Read-back path of calc_derivs for the drop-in and for tests. */
template <class P, bool PP>
__global__ void __launch_bounds__(DV_BLOCK) k_dense(Work w, ParamBlock<P> pb, double *out)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    const int k = blockIdx.y;
    if (b >= w.B) return;
    ILQG_PARAMS(PP, b)
    const size_t Bp = w.Bp;
    Dense<P> D;
    double *Dd = reinterpret_cast<double *>(&D);
#pragma unroll
    for (int i = 0; i < P::DENSE_SIZE; i++) Dd[i] = 0.0;
    P::consts(pv, D);
    double v1[P::NV1];
    if (use_coop<P>()) {
        const double *r = w.V1 + ((size_t)k * Bp + b) * P::NV1;
#pragma unroll
        for (int i = 0; i < P::NV1; i++) v1[i] = r[i];
    } else {
        const double *r = w.V1 + (size_t)k * P::NV1 * Bp + b;
#pragma unroll
        for (int i = 0; i < P::NV1; i++) v1[i] = r[i * Bp];
    }
    P::unpack(v1, D);
    if (!P::HAS_HX) { /* limitsU also records which side is bounded (iLQG_func.tem:101-118); the solver itself needs the signs only
                         together with state-dependent limits, so they are not part of the stored entries otherwise */
        const double inf = dm_from_bits(0x7ff0000000000000ull);
#pragma unroll
        for (int i = 0; i < P::NU; i++) {
            D.lower_sign[i] = (D.lower[i] == -inf) ? 0.0 : -1.0;
            D.upper_sign[i] = (D.upper[i] == inf) ? 0.0 : 1.0;
        }
    }
    double *o_ = out + ((size_t)b * w.T + k) * P::DENSE_SIZE;
#pragma unroll
    for (int i = 0; i < P::DENSE_SIZE; i++) o_[i] = Dd[i];
}

/* clampU(u, t, k, p, N) (iLQG_func.tem:68-73) for a batch: xu[b] = x | u, the clamped u is written back in place */
template <class P, bool PP, bool TR = false>
__global__ void __launch_bounds__(BP_BLOCK) k_clamp(Work w, ParamBlock<P> pb, double *xu_io, int k)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= w.B) return;
    ILQG_PARAMS(PP, b)
    ILQG_PK(TR, b)
    double x[P::NX], u[P::NU], xn[P::NX], mu[P::N_MU_R + P::N_MU_F + 1], c;
    double *io = xu_io + (size_t)b * (P::NX + P::NU);
#pragma unroll
    for (int i = 0; i < P::NX; i++) x[i] = io[i];
#pragma unroll
    for (int i = 0; i < P::NU; i++) u[i] = io[P::NX + i];
#pragma unroll
    for (int i = 0; i < P::N_MU_R; i++) mu[i] = 0.0;
    P::step(x, u, pv, pk, k, w.T, 0.0, mu, xn, c);   /* the clamp is the first thing a step does to u */
#pragma unroll
    for (int i = 0; i < P::NU; i++) io[P::NX + i] = u[i];
}

/* Single evaluation of the problem functions at one point per problem (the reference's MMex interface, iLQG_MMex.tem:81-226):
 * in[b] = x | u, out[b][...] = the value of `mode` as a FULL column-major array (Hessians with both triangles, second-order
 * dynamics as A(c, j, r) = d2 f_r / d c d j): 0 f, 1 L, 2 F, 3 Fx, 4 Fxx, 5 Lx, 6 Lu, 7 Lxx, 8 Luu, 9 Lxu, 10 fx, 11 fu, 12 fxx,
 * 13 fuu, 14 fxu, 16 clamped u; 17 (not an MMex mode) the user outputs g of calcG (iLQG_func.tem:511-521).  Multipliers are taken as zero and penalty weights as one (problems with folded constraints
 * have no MMex in the reference).  One thread per problem; this is an inspection path, not a hot one. */
template <class P> __host__ __device__ constexpr int eval_size(int mode)
{
    return mode == 0 ? P::NX : (mode == 1 || mode == 2) ? 1 : (mode == 3 || mode == 5) ? P::NX : (mode == 4 || mode == 7 || mode == 10) ? P::NX * P::NX
         : mode == 6 ? P::NU : mode == 8 ? P::NU * P::NU : (mode == 9 || mode == 11) ? P::NX * P::NU : mode == 12 ? P::NX * P::NX * P::NX
         : mode == 13 ? P::NU * P::NU * P::NX : mode == 14 ? P::NX * P::NU * P::NX : mode == 16 ? P::NU : mode == 17 ? P::NG : 0;
}

template <class P, bool PP, bool TR = false>
__global__ void __launch_bounds__(BP_BLOCK) k_eval(Work w, ParamBlock<P> pb, const double *in, double *out, int mode, int k)
{
    constexpr int NX = P::NX, NU = P::NU, NQXX = P::NQXX, NQUU = P::NQUU, NQXU = P::NQXU;
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= w.B) return;
    ILQG_PARAMS(PP, b)
    ILQG_PK(TR, b)
    double x[NX], u[NU], mu[P::N_MU_R + P::N_MU_F + 1];
#pragma unroll
    for (int i = 0; i < NX; i++) x[i] = in[(size_t)b * (NX + NU) + i];
#pragma unroll
    for (int i = 0; i < NU; i++) u[i] = in[(size_t)b * (NX + NU) + NX + i];
#pragma unroll
    for (int i = 0; i < P::N_MU_R + P::N_MU_F + 1; i++) mu[i] = 0.0;
    double *o_ = out + (size_t)b * eval_size<P>(mode);
    const int T = w.T;
    if (mode == 0 || mode == 1) {
        double xn[NX], c;
        P::step_free(x, u, pv, pk, k, T, 1.0, mu, xn, c);
        if (mode == 0) {
#pragma unroll
            for (int i = 0; i < NX; i++) o_[i] = xn[i];
        } else
            o_[0] = c;
    } else if (mode == 2) {
        double c;
        P::final_cost(x, pv, pk, T, T, 1.0, mu, c);
        o_[0] = c;
    } else if (mode == 3 || mode == 4) {
        double cx[NX], cxx[NQXX];
        P::derivs_final(x, pv, pk, T, T, 1.0, mu, cx, cxx);
        if (mode == 3) {
#pragma unroll
            for (int i = 0; i < NX; i++) o_[i] = cx[i];
        } else
            for (int c = 0; c < NX; c++)
                for (int r = 0; r < NX; r++) o_[r + c * NX] = cxx[symtri(r, c)];
    } else if (mode == 17) {
        double g[P::NG + 1];
        P::calc_g(x, u, pv, pk, k, T, 1.0, mu, g);
#pragma unroll
        for (int i = 0; i < P::NG; i++) o_[i] = g[i];
    } else if (mode == 16) {
        double xn[NX], c;
        P::step(x, u, pv, pk, k, T, 1.0, mu, xn, c);
#pragma unroll
        for (int i = 0; i < NU; i++) o_[i] = u[i];
    } else if (mode >= 5 && mode <= 14) {
        Dense<P> D;
        double *Dd = reinterpret_cast<double *>(&D);
        for (int i = 0; i < P::DENSE_SIZE; i++) Dd[i] = 0.0;
        double v1[P::NV1], v2[P::NV2];
        P::consts(pv, D);
        P::derivs_full(x, u, pv, pk, k, T, 1.0, mu, v1, v2);
        P::unpack(v1, D);
        if (mode == 5) for (int i = 0; i < NX; i++) o_[i] = D.cx[i];
        if (mode == 6) for (int i = 0; i < NU; i++) o_[i] = D.cu[i];
        if (mode == 7) for (int c = 0; c < NX; c++) for (int r = 0; r < NX; r++) o_[r + c * NX] = D.cxx[symtri(r, c)];
        if (mode == 8) for (int c = 0; c < NU; c++) for (int r = 0; r < NU; r++) o_[r + c * NU] = D.cuu[symtri(r, c)];
        if (mode == 9) for (int i = 0; i < NQXU; i++) o_[i] = D.cxu[i];
        if (mode == 10) for (int i = 0; i < NX * NX; i++) o_[i] = D.fx[i];
        if (mode == 11) for (int i = 0; i < NX * NU; i++) o_[i] = D.fu[i];
        if (mode >= 12) {
            /* component r of the second-order dynamics = the FULL_DDP contraction with the r-th unit vector for Vx: the sparse
               term lists then reduce to 0 + 1.0 * entry (other terms add 0 * entry = +-0) */
            for (int r = 0; r < NX; r++) {
                double e[NX], q[NQXX > NQXU ? NQXX : NQXU];
                for (int i = 0; i < NX; i++) e[i] = (i == r) ? 1.0 : 0.0;
                for (int i = 0; i < (NQXX > NQXU ? NQXX : NQXU); i++) q[i] = 0.0;
                if (mode == 12) {
                    P::add2_Qxx(e, v2, pv, q);
                    for (int j = 0; j < NX; j++) for (int c = 0; c < NX; c++) o_[c + j * NX + r * NX * NX] = q[symtri(c, j)];
                } else if (mode == 13) {
                    P::add2_Quu(e, v2, pv, q);
                    for (int j = 0; j < NU; j++) for (int c = 0; c < NU; c++) o_[c + j * NU + r * NU * NU] = q[symtri(c, j)];
                } else {
                    P::add2_Qxu(e, v2, pv, q);
                    for (int j = 0; j < NU; j++) for (int c = 0; c < NX; c++) o_[c + j * NX + r * NX * NU] = q[c + j * NX];
                }
            }
        }
    }
}

/* after the last pass: problems still running hit the iteration limit (iLQG.c:365-377) */
__global__ void k_finalize(Work w, int max_iter)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= w.B) return;
    if (w.status[b] == ST_RUNNING) {
        w.status[b] = ST_DONE;
        w.iterations[b] = max_iter;
        w.result[b] = 0;
    }
}

__global__ void k_count_active(Work w, int *out)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    int a = (b < w.B) && (w.status[b] == ST_RUNNING);
    a = __syncthreads_count(a);
    if (threadIdx.x == 0 && a) atomicAdd(out, a);
}

/* Receding horizon (ilqgb_shift / ilqgb_mpc), one thread per problem: log the finished solve (its x0, the applied control
 * u[0], cost, iterations, result), then make its solution the input of the next solve, which is what the reference's caller
 * does between two iLQG_mex calls: the shifted controls go into the u part of buffer 0's records, where ilqgb_upload puts
 * them and k_init's initial rollout reads them, and x[n_shift] (+ w) becomes x0.  Whatever the nominal buffer holds is
 * used, also for a problem whose solve failed.  When cur[b] == 0 the source is the destination: every record is read before
 * it is written because the steps are copied in ascending order, KB of them loaded before any is stored (a copy parallel
 * over (k, b) would not be safe).  Adjacent threads are adjacent problems of the [k][Bp][RXU] records.
 * mpc_log_shift is everything after the next state xn (+ w) is known; k_mpc_advance and k_mpc_plant differ only in how
 * they compute xn. */
template <class P>
__device__ __forceinline__ void mpc_log_shift(const Work &w, const ilqg_mpc_step &a, int b, const double *src, const double *xn)
{
    constexpr int NX = P::NX, NU = P::NU, RXU = Rec<P>::RXU, KB = 8;
    const size_t Bp = w.Bp;
    const int T = w.T, n = a.n_shift;
    const size_t row = (size_t)b * a.n_steps + a.step;
    if (a.x_log) {
        double *xl = a.x_log + ((size_t)b * (a.n_steps + 1) + a.step) * NX;
#pragma unroll
        for (int i = 0; i < NX; i++) xl[i] = w.x0[(size_t)i * Bp + b];
        if (!a.plan)
#pragma unroll
            for (int i = 0; i < NX; i++) xl[NX + i] = xn[i];
    }
    if (a.u_log)
#pragma unroll
        for (int j = 0; j < NU; j++) a.u_log[row * NU + j] = src[(size_t)b * RXU + NX + j];
    if (a.cost_log) a.cost_log[row] = w.cost[b];
    if (a.it_log) a.it_log[row] = w.iterations[b];
    if (a.res_log) a.res_log[row] = w.result[b];
    if (!a.plan) return;
    if (a.set_x0)
#pragma unroll
        for (int i = 0; i < NX; i++) w.x0[(size_t)i * Bp + b] = xn[i];
    double *dst = w.XU[0];
    for (int k0 = 0; k0 < T; k0 += KB) {
        double u[KB][NU];
#pragma unroll
        for (int j = 0; j < KB; j++) {
            const int ks = min(k0 + j + n, T - 1);   /* past the end: the last control, still unwritten (only step T-1 writes it) */
            if (k0 + j < T)
#pragma unroll
                for (int i = 0; i < NU; i++) u[j][i] = src[((size_t)ks * Bp + b) * RXU + NX + i];
        }
#pragma unroll
        for (int j = 0; j < KB; j++)
            if (k0 + j < T)
#pragma unroll
                for (int i = 0; i < NU; i++) dst[((size_t)(k0 + j) * Bp + b) * RXU + NX + i] = u[j][i];
    }
}

template <class P>
__global__ void __launch_bounds__(256) k_mpc_advance(Work w, ilqg_mpc_step a)
{
    constexpr int NX = P::NX, RXU = Rec<P>::RXU;
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= w.B) return;
    const size_t Bp = w.Bp;
    const int n = a.n_shift;
    const double *src = w.XU[w.cur[b]];
    const size_t row = (size_t)b * a.n_steps + a.step;
    double xn[NX];
#pragma unroll
    for (int i = 0; i < NX; i++) {
        xn[i] = src[((size_t)n * Bp + b) * RXU + i];
        if (a.w) xn[i] = xn[i] + a.w[row * NX + i];
    }
    mpc_log_shift<P>(w, a, b, src, xn);
}

/* k_mpc_advance against a plant that differs from the model: the next state is not the solution's prediction x[n_shift] but
 * the plant stepped from the solve's x0 through the n_shift applied controls u[j], each held for pl.n_sub sub-steps.  A sub-step
 * is P::step -- clampU with the plant's limits at the sub-step's own state, then f -- on a fresh copy of the commanded u[j],
 * exactly the reference's forward_pass step (and MMex modes 16 then 0), with zero multipliers and penalty weight as in k_clamp.
 * All sub-steps of control j evaluate at step index j, [k]-indexed parameters from the model (TR: the window of the solve that
 * just finished).  The plant's parameters: the shared block pb_plant, or (PPP) this problem's column of pl.pp.  A non-finite
 * state is passed on as it is; the next solve's initial rollout then fails for that problem alone. */
template <class P, bool PPP, bool TR = false>
__global__ void __launch_bounds__(256) k_mpc_plant(Work w, ilqg_mpc_step a, ParamBlock<P> pb_plant, ilqg_plant pl)
{
    constexpr int NX = P::NX, NU = P::NU, RXU = Rec<P>::RXU;
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= w.B) return;
    const size_t Bp = w.Bp;
    double pl_[PPP ? P::NPF : 1];
    const double *pv = pb_plant.v;
    if (PPP) {
#pragma unroll
        for (int i = 0; i < P::NPF_USED; i++) pl_[i] = pl.pp[(size_t)i * Bp + b];
        pv = pl_;
    }
    ILQG_PK(TR, b)
    const double *src = w.XU[w.cur[b]];
    double xn[NX], x[NX], u[NU], mu[P::N_MU_R + P::N_MU_F + 1], c;
#pragma unroll
    for (int i = 0; i < NX; i++) xn[i] = w.x0[(size_t)i * Bp + b];
#pragma unroll
    for (int i = 0; i < P::N_MU_R; i++) mu[i] = 0.0;
    for (int j = 0; j < a.n_shift; j++)
        for (int s = 0; s < pl.n_sub; s++) {
#pragma unroll
            for (int i = 0; i < NX; i++) x[i] = xn[i];
#pragma unroll
            for (int i = 0; i < NU; i++) u[i] = src[((size_t)j * Bp + b) * RXU + NX + i];
            P::step(x, u, pv, pk, j, w.T, 0.0, mu, xn, c);
        }
    if (a.w) {
        const size_t row = (size_t)b * a.n_steps + a.step;
#pragma unroll
        for (int i = 0; i < NX; i++) xn[i] = xn[i] + a.w[row * NX + i];
    }
    mpc_log_shift<P>(w, a, b, src, xn);
}

/* =====================================================================================================================
 * Feedback policy of a solved batch (ilqgb_policy, ilqgb_policy_rollout, ilqgb_policy_eval).
 * ===================================================================================================================== */
/* ilqgb_policy runs the derivative sweep and one backward pass on every problem, finished or not.  save = 1 (before): keep what
   reaching finished problems changes -- status, new_deriv, deriv_fail, and the iterations / result / counters that the backward
   pass's derivative-failure exit and bookkeeping write -- then mark every problem running with fresh derivatives and no
   successful backward pass.  save = 0 (after): policy_ok = finite derivatives and a successful backward pass; restore. */
__global__ void k_policy_mark(Work w, int *keep /* [7][Bp] */, int *policy_ok, int save)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= w.B) return;
    const size_t Bp = w.Bp;
    if (save) {
        keep[0 * Bp + b] = w.status[b];
        keep[1 * Bp + b] = w.new_deriv[b];
        keep[2 * Bp + b] = w.deriv_fail[b];
        keep[3 * Bp + b] = w.iterations[b];
        keep[4 * Bp + b] = w.result[b];
        keep[5 * Bp + b] = w.n_bp[b];
        keep[6 * Bp + b] = w.n_dv[b];
        w.status[b] = ST_RUNNING;
        w.new_deriv[b] = 1;
        w.deriv_fail[b] = 0;
        w.bp_done[b] = 0;
    } else {
        policy_ok[b] = (!w.deriv_fail[b] && w.bp_done[b]) ? 1 : 0;
        w.status[b] = keep[0 * Bp + b];
        w.new_deriv[b] = keep[1 * Bp + b];
        w.deriv_fail[b] = keep[2 * Bp + b];
        w.iterations[b] = keep[3 * Bp + b];
        w.result[b] = keep[4 * Bp + b];
        w.n_bp[b] = keep[5 * Bp + b];
        w.n_dv[b] = keep[6 * Bp + b];
    }
}

/* u_k(x) = u*_k + 0 * l_k + L_k (x - x*_k): the feedback expression of forward_pass (iLQG_func.tem:121-185) at alpha = 0, in its
   order of operations.  (forward_pass itself takes the open-loop branch when alpha == 0.)  The 0 * l term stays: it decides the
   sign of a zero control.  nom = x* | u* of step k, ll = l | L of step k. */
template <class P>
__device__ __forceinline__ void policy_u(const double *nom, const double *ll, const double *x, double *u)
{
    constexpr int NX = P::NX, NU = P::NU;
#pragma unroll
    for (int j = 0; j < NU; j++) u[j] = nom[NX + j] + ll[j] * 0.0;
#pragma unroll
    for (int i = 0; i < NX; i++) {
        const double dx = x[i] - nom[i];
#pragma unroll
        for (int j = 0; j < NU; j++) u[j] += ll[NU + j + i * NU] * dx;
    }
}

/* the nominal x|u, l and L records of step k of problem b, from the nominal buffer, whose gains ilqgb_policy wrote */
template <class P>
__device__ __forceinline__ void policy_records(const Work &w, int b, int cur, int k, double *nom, double *ll)
{
    const size_t i = (size_t)k * w.Bp + b;
    ld_rec<P::NX + P::NU>(w.XU[cur] + i * Rec<P>::RXU, nom);
    ld_rec<P::NU>(w.Ll[cur] + i * Rec<P>::RLS, ll);
    ld_rec<P::NU * P::NX>(w.LL[cur] + i * Rec<P>::RLM, ll + P::NU);
}

/* Closed-loop rollouts of the feedback policy, one lane per (problem b, sample s), lane b * n_samp + s: forward_pass(candidate, o,
 * 0, &csum, 0) with the gains applied (policy_u), from x0s[b][s], with the final multipliers and penalty weights, clampU at the
 * rollout's own state and, where the handle has a plant, the plant's parameters for the whole step (clampU, f and cost).  The
 * samples of a problem sit in adjacent lanes: a warp reads each nominal record once and broadcasts it to them (one problem per
 * warp from n_samp = 32 on), so the nominal traffic per step is that of one rollout per problem whatever n_samp is.  Nothing is
 * written to the handle's trajectory buffers; x / u rows are stored only when asked for.  A problem without a valid policy, and a
 * rollout that fails, give ok = 0, NaN cost and NaN final state; the stored rows of a failed rollout end with the failing step
 * and the rest are NaN.  PER: parameters from r.pp ([NPF][Bp]); TR: [k]-indexed parameters from the tracks' window. */
template <class P, bool PER, bool TR = false>
__global__ void __launch_bounds__(BP_BLOCK, ILQG_LS_MINBLOCKS) k_policy_rollout(Work w, ParamBlock<P> pb, ilqg_policy r)
{
    constexpr int NX = P::NX, NU = P::NU, RLM = Rec<P>::RLM;
    const size_t row = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int b = (int)(row / (size_t)r.n_samp);
    if (b >= w.B) return;
    const size_t Bp = w.Bp;
    const int T = w.T;
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    double x[NX], xn[NX], u[NU], mu[P::N_MU_R + P::N_MU_F + 1], nom[Rec<P>::RXU], ll[NU + RLM];
#pragma unroll
    for (int i = 0; i < NX; i++) x[i] = r.x0s[row * NX + i];
    double *xs = r.x ? r.x + row * (size_t)(T + 1) * NX : nullptr;
    double *us = r.u ? r.u + row * (size_t)T * NU : nullptr;
    bool ok = r.policy_ok[b] != 0;
    double csum = 0.0;
    int stored = 0;   /* x / u rows written */
    if (ok) {
        double pl_[PER ? P::NPF : 1];
        const double *pv = pb.v;
        if (PER) {
#pragma unroll
            for (int i = 0; i < P::NPF_USED; i++) pl_[i] = r.pp[(size_t)i * Bp + b];
            pv = pl_;
        }
        ILQG_PK(TR, b)
        const int cur = w.cur[b];
        const double w_pen_l = w.w_pen_l[b];
        for (int k = 0; k < T; k++) {
            policy_records<P>(w, b, cur, k, nom, ll);
            policy_u<P>(nom, ll, x, u);
#pragma unroll
            for (int i = 0; i < P::N_MU_R; i++) mu[i] = w.muR[((size_t)k * P::N_MU_R + i) * Bp + b];
            double c;
            ok = P::step(x, u, pv, pk, k, T, w_pen_l, mu, xn, c);
            if (xs) {
#pragma unroll
                for (int i = 0; i < NX; i++) xs[(size_t)k * NX + i] = x[i];
            }
            if (us) {
#pragma unroll
                for (int j = 0; j < NU; j++) us[(size_t)k * NU + j] = u[j];
            }
            stored = k + 1;
            if (!ok) break;
            csum += c;
#pragma unroll
            for (int i = 0; i < NX; i++) x[i] = xn[i];
        }
        if (ok) {
#pragma unroll
            for (int i = 0; i < P::N_MU_F; i++) mu[i] = w.muF[(size_t)i * Bp + b];
            double c;
            ok = P::final_cost(x, pv, pk, T, T, w.w_pen_f[b], mu, c);
            csum += c;
            if (ok && xs) {
#pragma unroll
                for (int i = 0; i < NX; i++) xs[(size_t)T * NX + i] = x[i];
            }
        }
    }
    r.ok[row] = ok ? 1 : 0;
    r.cost[row] = ok ? csum : nan;
#pragma unroll
    for (int i = 0; i < NX; i++) r.x_final[row * NX + i] = ok ? x[i] : nan;
    if (!ok) {
        if (xs)
            for (size_t i = (size_t)stored * NX; i < (size_t)(T + 1) * NX; i++) xs[i] = nan;
        if (us)
            for (size_t i = (size_t)stored * NU; i < (size_t)T * NU; i++) us[i] = nan;
    }
}

/* The policy's control at step k for one state per problem (ilqgb_policy_eval): step k of k_policy_rollout without f, with the
   model's parameters -- policy_u, then clampU at x as in k_clamp.  x [B][NX] in, u [B][NU] out; NaN without a valid policy. */
template <class P, bool PP, bool TR = false>
__global__ void __launch_bounds__(BP_BLOCK) k_policy_eval(Work w, ParamBlock<P> pb, const int *policy_ok, const double *xin, double *uout, int k)
{
    constexpr int NX = P::NX, NU = P::NU;
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= w.B) return;
    double *uo = uout + (size_t)b * NU;
    if (!policy_ok[b]) {
#pragma unroll
        for (int j = 0; j < NU; j++) uo[j] = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    ILQG_PARAMS(PP, b)
    ILQG_PK(TR, b)
    double x[NX], xn[NX], u[NU], mu[P::N_MU_R + P::N_MU_F + 1], nom[Rec<P>::RXU], ll[NU + Rec<P>::RLM], c;
#pragma unroll
    for (int i = 0; i < NX; i++) x[i] = xin[(size_t)b * NX + i];
    policy_records<P>(w, b, w.cur[b], k, nom, ll);
    policy_u<P>(nom, ll, x, u);
#pragma unroll
    for (int i = 0; i < P::N_MU_R; i++) mu[i] = 0.0;
    P::step(x, u, pv, pk, k, w.T, 0.0, mu, xn, c);   /* the clamp is the first thing a step does to u */
#pragma unroll
    for (int j = 0; j < NU; j++) uo[j] = u[j];
}

/* layout changes between the caller's problem-major arrays [B][n_k][n_i] and device arrays addressed as
 * base[(k * stride_k + b) * stride_b + off + i * stride_i]  (records: stride_k = Bp, stride_b = record size, stride_i = 1;
 * structure-of-arrays [k][i][Bp]: handled by the caller passing stride_b = 1, stride_i = Bp, stride_k = n_i * Bp / 1) */
struct Layout {
    long long stride_k, stride_b, stride_i, off;
};

__global__ void k_scatter(const double *src, double *dst, double *dst_alt, const int *sel, int B, int n_k, int n_i, Layout L)
{
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t per = (size_t)n_k * n_i;
    if (e >= per * B) return;
    const size_t i = e % n_i, b = (e / n_i) % B, k = e / ((size_t)n_i * B);
    double *d = (sel && sel[b]) ? dst_alt : dst;
    d[k * L.stride_k + b * L.stride_b + i * L.stride_i + L.off] = src[b * per + k * n_i + i];
}

__global__ void k_gather(const double *src, const double *src_alt, const int *sel, double *dst, int B, int n_k, int n_i, Layout L)
{
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t per = (size_t)n_k * n_i;
    if (e >= per * B) return;
    const size_t i = e % n_i, b = (e / n_i) % B, k = e / ((size_t)n_i * B);
    const double *s = (sel && sel[b]) ? src_alt : src;
    dst[b * per + k * n_i + i] = s[k * L.stride_k + b * L.stride_b + i * L.stride_i + L.off];
}

} /* namespace ilqg */
