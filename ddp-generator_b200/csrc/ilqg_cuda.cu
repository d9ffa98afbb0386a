/* ilqg_cuda.cu -- the CUDA layer under the C host code: kernel instantiation for ONE generated problem
 * (-DILQG_PROBLEM_HEADER=... -DILQG_PROBLEM_STRUCT=... -DFULL_DDP=0|1, like the reference builds one mex per
 * problem and FULL_DDP setting, make_iLQG.m:65-86) and thin extern "C" launch / memory wrappers.
 * No solver logic lives here; see ilqg_host.c.  Build: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false. */
#include <cstdio>
#include <cstring>
#include "ilqg_kernels.cuh"
#include "mod_chol.cuh"
#include ILQG_PROBLEM_HEADER
#include "ilqg_cuda.h"

#ifndef FULL_DDP
#define FULL_DDP 1
#endif

using P = ILQG_PROBLEM_STRUCT;
using namespace ilqg;

static thread_local char g_err[256] = "";
#define ILQGK_MAX_DEVICES 64

static int check(cudaError_t e, const char *what)
{
    if (e == cudaSuccess) return 0;
    snprintf(g_err, sizeof g_err, "%s: %s", what, cudaGetErrorString(e));
    return -1;
}

static ParamBlock<P> make_pb(const double *params)
{
    ParamBlock<P> pb;
    memset(&pb, 0, sizeof pb);
    memcpy(pb.v, params, sizeof(double) * P::NPF_USED);
    return pb;
}

/* the small-batch backward pass exists for problems without state-dependent input limits; the launcher is a class
   template so that the kernel is only instantiated where it applies */
constexpr bool SPLIT_OK = split_supported<P>();
template <class Q, bool PP, bool OK> struct split_launcher {
    static void go(const ilqg_work *, const ilqg_opts *, const double *, int, void *) {}
    static int preload() { return 0; }
};
template <class Q, bool PP> struct split_launcher<Q, PP, true> {
    static void go(const ilqg_work *w, const ilqg_opts *o, const double *params, int iter, void *stream)
    {
        constexpr size_t ssm = split_smem_bytes<Q, 4>();
        static_assert(ssm <= 48 * 1024, "k_backpass_split: workspace exceeds the default shared-memory limit");
        ParamBlock<Q> pb;
        memset(&pb, 0, sizeof pb);
        memcpy(pb.v, params, sizeof(double) * Q::NPF_USED);
        const int ppw = o->bp_ppw < SP_BLOCK / 4 ? (o->bp_ppw < 1 ? 1 : o->bp_ppw) : SP_BLOCK / 4;
        k_backpass_split<Q, FULL_DDP != 0, PP, 4><<<(unsigned)((w->B + ppw - 1) / ppw), SP_BLOCK, ssm, (cudaStream_t)stream>>>(*w, *o, pb, iter);
    }
    static int preload()
    {
        cudaFuncAttributes a;
        return cudaFuncGetAttributes(&a, k_backpass_split<Q, FULL_DDP != 0, PP, 4>) == cudaSuccess ? 0 : -1;
    }
};

/* CUDA loads a kernel lazily at its first launch, and a first launch in the middle of a solve stalls the running streams (measured:
   the running-problem count of the solve engine, first launched in pass 9, cost a 115 ms solve 16 ms).  Every kernel a solve can
   launch is therefore loaded when the first handle of a device is created: querying a function's attributes loads it. */
template <class F> static int preload_one(F *f)
{
    cudaFuncAttributes a;
    return cudaFuncGetAttributes(&a, f) == cudaSuccess ? 0 : -1;
}
/* the kernels that evaluate the problem functions, for shared [k]-indexed parameters or (TR) per-problem tracks */
template <bool PP, bool TR> static int preload_pk()
{
    constexpr bool FULL = FULL_DDP != 0;
    int bad = 0;
    bad |= preload_one(k_init<P, PP, TR>) | preload_one(k_rollout_only<P, PP, TR>) | preload_one(k_derivs<P, FULL, PP, TR>);
    bad |= preload_one(k_ls_round<P, PP, TR>) | preload_one(k_ls_tail<P, PP, true, TR>) | preload_one(k_ls_tail<P, PP, false, TR>);
    bad |= preload_one(k_ls_commit_seg<P, PP, TR>) | preload_one(k_ls_commit<P, PP, true, TR>) | preload_one(k_ls_commit<P, PP, false, TR>);
    bad |= preload_one(k_post<P, PP, TR>) | preload_one(k_mult<P, PP, TR>) | preload_one(k_clamp<P, PP, TR>) | preload_one(k_eval<P, PP, TR>);
    return bad;
}
template <bool PP> static int preload_pp()
{
    constexpr bool FULL = FULL_DDP != 0;
    int bad = preload_pk<PP, false>() | preload_one(k_dense<P, PP>);
    if constexpr (P::NKP > 0) bad |= preload_pk<PP, true>();   /* track variants exist only where there are [k]-indexed parameters */
    if constexpr (use_coop<P>()) {
        bad |= preload_one(k_backpass_warp<P, FULL, PP, 32>) | preload_one(k_backpass_warp<P, FULL, PP, 16>) | preload_one(k_backpass_warp<P, FULL, PP, 8>);
    } else {
        bad |= preload_one(k_backpass<P, FULL, 1, PP>) | preload_one(k_backpass<P, FULL, ILQG_BP_MINBLOCKS, PP>);
    }
    return bad;
}

constexpr bool HAS_KP = P::NKP > 0;

static inline unsigned nblk(int n, int bs) { return (unsigned)((n + bs - 1) / bs); }

/* k_backpass_warp at LPP lanes per problem.  The opt-in to more than 48 KB of dynamic shared memory is a per-device function
   attribute, set for the variant launched only: at 8 lanes per problem the workspace of a large problem can exceed what the device
   gives a block while 32 lanes fit (the handle rejects such a setting, ilqgk_coop_smem) */
template <int LPP> static int cw_launch(const ilqg_work *w, const ilqg_opts *o, const double *params, int iter, void *stream)
{
    constexpr bool FULL = FULL_DDP != 0;
    constexpr int smem = (int)coop_smem_bytes<P, LPP>();
    static unsigned char configured[ILQGK_MAX_DEVICES];
    int dev = 0;
    if (check(cudaGetDevice(&dev), "cudaGetDevice")) return -1;
    if (dev < 0 || dev >= ILQGK_MAX_DEVICES || !configured[dev]) {
        if (check(cudaFuncSetAttribute(k_backpass_warp<P, FULL, false, LPP>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem), "cudaFuncSetAttribute") ||
            check(cudaFuncSetAttribute(k_backpass_warp<P, FULL, true, LPP>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem), "cudaFuncSetAttribute"))
            return -1;
        if (dev >= 0 && dev < ILQGK_MAX_DEVICES) configured[dev] = 1;
    }
    const unsigned grid = nblk(w->B, CW_WARPS * (32 / LPP));
    if (w->pp) k_backpass_warp<P, FULL, true, LPP><<<grid, CW_WARPS * 32, smem, (cudaStream_t)stream>>>(*w, *o, make_pb(params), iter);
    else k_backpass_warp<P, FULL, false, LPP><<<grid, CW_WARPS * 32, smem, (cudaStream_t)stream>>>(*w, *o, make_pb(params), iter);
    return check(cudaGetLastError(), "k_backpass");
}

template <int LPP> static int cw_smem(size_t *need)
{
    cudaFuncAttributes a, b;
    if (check(cudaFuncGetAttributes(&a, k_backpass_warp<P, FULL_DDP != 0, false, LPP>), "cudaFuncGetAttributes") ||
        check(cudaFuncGetAttributes(&b, k_backpass_warp<P, FULL_DDP != 0, true, LPP>), "cudaFuncGetAttributes"))
        return -1;
    *need = coop_smem_bytes<P, LPP>() + (a.sharedSizeBytes > b.sharedSizeBytes ? a.sharedSizeBytes : b.sharedSizeBytes);
    return 0;
}

extern "C" {

const char *ilqgk_last_error(void) { return g_err; }

int ilqgk_preload(void)
{
    static unsigned char loaded[ILQGK_MAX_DEVICES];
    int dev = 0, bad = 0;
    if (check(cudaGetDevice(&dev), "cudaGetDevice")) return -1;
    if (dev >= 0 && dev < ILQGK_MAX_DEVICES && loaded[dev]) return 0;
    bad |= preload_pp<false>() | preload_pp<true>();
    bad |= split_launcher<P, false, SPLIT_OK>::preload() | split_launcher<P, true, SPLIT_OK>::preload();
    bad |= preload_one(k_finalize) | preload_one(k_count_active) | preload_one(k_scatter) | preload_one(k_gather);
    bad |= preload_one(k_mpc_advance<P>);   /* first launched between two steps of a closed loop, while other chunks solve */
    bad |= preload_one(k_mpc_plant<P, false, false>) | preload_one(k_mpc_plant<P, true, false>);
    if constexpr (HAS_KP) bad |= preload_one(k_mpc_plant<P, false, true>) | preload_one(k_mpc_plant<P, true, true>);
    bad |= preload_one(k_policy_mark) | preload_one(k_policy_rollout<P, false, false>) | preload_one(k_policy_rollout<P, true, false>);
    bad |= preload_one(k_policy_eval<P, false, false>) | preload_one(k_policy_eval<P, true, false>);
    if constexpr (HAS_KP) {
        bad |= preload_one(k_policy_rollout<P, false, true>) | preload_one(k_policy_rollout<P, true, true>);
        bad |= preload_one(k_policy_eval<P, false, true>) | preload_one(k_policy_eval<P, true, true>);
    }
    if (bad) { snprintf(g_err, sizeof g_err, "loading the kernels failed: %s", cudaGetErrorString(cudaGetLastError())); return -1; }
    if (dev >= 0 && dev < ILQGK_MAX_DEVICES) loaded[dev] = 1;
    return 0;
}

void ilqgk_dims(ilqgk_dims_t *d)
{
    d->nx = P::NX; d->nu = P::NU; d->nqxx = P::NQXX; d->nquu = P::NQUU; d->nqxu = P::NQXU;
    d->nv1 = P::NV1; d->nv2 = P::NV2; d->npf = P::NPF_USED; d->nkp = P::NKP;
    d->n_mu_r = P::N_MU_R; d->n_mu_f = P::N_MU_F; d->n_mu_le = P::N_MU_LE; d->n_mu_fe = P::N_MU_FE;
    d->full_ddp = FULL_DDP; d->has_hx = P::HAS_HX ? 1 : 0;
    d->bp_split_ok = SPLIT_OK ? 1 : 0;
    d->rxu = Rec<P>::RXU; d->rlm = Rec<P>::RLM; d->rls = Rec<P>::RLS; d->coop = use_coop<P>() ? 1 : 0;
}
const char *ilqgk_problem_name(void) { return P::name(); }
int ilqgk_param_count(void) { return P::param_count(); }
const char *ilqgk_param_name(int i) { return P::param_name(i); }
int ilqgk_param_size(int i) { return P::param_size(i); }

int ilqgk_coop_smem(int dev, int lpp, size_t *need, size_t *limit)
{
    /* queried on device `dev`; the calling thread's current device is restored */
    int prev = 0, optin = 0, rc = 0;
    *need = *limit = 0;
    if constexpr (use_coop<P>()) {
        if (check(cudaGetDevice(&prev), "cudaGetDevice") || check(cudaSetDevice(dev), "cudaSetDevice")) return -1;
        rc = check(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev), "cudaDeviceGetAttribute");
        if (!rc) rc = lpp == 8 ? cw_smem<8>(need) : lpp == 16 ? cw_smem<16>(need) : cw_smem<32>(need);
        *limit = (size_t)optin;
        if (check(cudaSetDevice(prev), "cudaSetDevice")) return -1;
    }
    return rc;
}

int ilqgk_device_count(void) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) return 0; return n; }
int ilqgk_set_device(int dev) { return check(cudaSetDevice(dev), "cudaSetDevice"); }
int ilqgk_malloc(void **p, size_t bytes) { return check(cudaMalloc(p, bytes ? bytes : 8), "cudaMalloc"); }
int ilqgk_free(void *p) { return p ? check(cudaFree(p), "cudaFree") : 0; }
int ilqgk_host_alloc(void **p, size_t bytes) { return check(cudaHostAlloc(p, bytes ? bytes : 8, cudaHostAllocDefault), "cudaHostAlloc"); }
int ilqgk_host_free(void *p) { return p ? check(cudaFreeHost(p), "cudaFreeHost") : 0; }
int ilqgk_memset(void *p, int v, size_t bytes, void *stream) { return check(cudaMemsetAsync(p, v, bytes, (cudaStream_t)stream), "cudaMemsetAsync"); }
int ilqgk_h2d(void *dst, const void *src, size_t bytes, void *stream) { return check(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream), "H2D"); }
int ilqgk_d2h(void *dst, const void *src, size_t bytes, void *stream) { return check(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream), "D2H"); }
int ilqgk_d2d(void *dst, const void *src, size_t bytes, void *stream) { return check(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream), "D2D"); }
int ilqgk_stream_create(void **s) { cudaStream_t st; int r = check(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking), "cudaStreamCreate"); *s = (void *)st; return r; }
int ilqgk_stream_create_prio(void **s, int rank, int n_ranks)
{
    /* rank 0 = most urgent of n_ranks; mapped onto the device's priority range (numerically lower = more urgent) */
    int least = 0, greatest = 0, levels, prio;
    cudaStream_t st;
    if (check(cudaDeviceGetStreamPriorityRange(&least, &greatest), "cudaDeviceGetStreamPriorityRange")) return -1;
    levels = least - greatest + 1;
    if (levels < 1) levels = 1;
    prio = n_ranks > 1 ? greatest + (int)((long long)rank * levels / n_ranks) : least;
    if (prio > least) prio = least;
    int r = check(cudaStreamCreateWithPriority(&st, cudaStreamNonBlocking, prio), "cudaStreamCreateWithPriority");
    *s = (void *)st;
    return r;
}
int ilqgk_stream_destroy(void *s) { return check(cudaStreamDestroy((cudaStream_t)s), "cudaStreamDestroy"); }
int ilqgk_stream_sync(void *s) { return check(cudaStreamSynchronize((cudaStream_t)s), "cudaStreamSynchronize"); }
int ilqgk_event_create(void **e) { cudaEvent_t ev; int r = check(cudaEventCreate(&ev), "cudaEventCreate"); *e = (void *)ev; return r; }
int ilqgk_event_create_notiming(void **e) { cudaEvent_t ev; int r = check(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming), "cudaEventCreate"); *e = (void *)ev; return r; }
int ilqgk_stream_wait_event(void *s, void *e) { return check(cudaStreamWaitEvent((cudaStream_t)s, (cudaEvent_t)e, 0), "cudaStreamWaitEvent"); }
int ilqgk_event_query(void *e)
{
    /* 1 = complete, 0 = still pending, -1 = error */
    const cudaError_t r = cudaEventQuery((cudaEvent_t)e);
    if (r == cudaSuccess) return 1;
    if (r == cudaErrorNotReady) return 0;
    return check(r, "cudaEventQuery");
}
int ilqgk_event_sync(void *e) { return check(cudaEventSynchronize((cudaEvent_t)e), "cudaEventSynchronize"); }
int ilqgk_event_destroy(void *e) { return check(cudaEventDestroy((cudaEvent_t)e), "cudaEventDestroy"); }
int ilqgk_event_record(void *e, void *s) { return check(cudaEventRecord((cudaEvent_t)e, (cudaStream_t)s), "cudaEventRecord"); }
int ilqgk_event_elapsed(void *a, void *b, float *ms) { return check(cudaEventElapsedTime(ms, (cudaEvent_t)a, (cudaEvent_t)b), "cudaEventElapsedTime"); }

/* every solver kernel exists for shared parameters and for per-problem parameter sets */
#define PP_DISPATCH(w_, CALL)          \
    do {                               \
        if ((w_)->pp) { constexpr bool PP = true; CALL; } else { constexpr bool PP = false; CALL; } \
    } while (0)
/* the kernels that evaluate the problem functions also exist, for problems with [k]-indexed parameters, in a variant that
   reads per-problem tracks (TR); without such parameters both branches name the same instantiation */
#define PK_DISPATCH(w_, CALL)                                                                                         \
    do {                                                                                                              \
        if (HAS_KP && (w_)->tr_mask) { constexpr bool TR = HAS_KP; PP_DISPATCH(w_, CALL); }                            \
        else { constexpr bool TR = false; PP_DISPATCH(w_, CALL); }                                                    \
    } while (0)

int ilqgk_launch_init(const ilqg_work *w, const ilqg_opts *o, const double *params, int mode, void *stream)
{
    PK_DISPATCH(w, (k_init<P, PP, TR><<<nblk(w->B, BP_BLOCK), BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, *o, make_pb(params), mode)));
    return check(cudaGetLastError(), "k_init");
}

int ilqgk_launch_rollout(const ilqg_work *w, const double *params, double alpha, int cost_only, void *stream)
{
    PK_DISPATCH(w, (k_rollout_only<P, PP, TR><<<nblk(w->B, BP_BLOCK), BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, make_pb(params), alpha, cost_only)));
    return check(cudaGetLastError(), "k_rollout_only");
}

int ilqgk_launch_derivs(const ilqg_work *w, const double *params, void *stream)
{
    dim3 grid(nblk(w->B, DV_BLOCK), (unsigned)(w->T + 1));
    PK_DISPATCH(w, (k_derivs<P, FULL_DDP != 0, PP, TR><<<grid, DV_BLOCK, 0, (cudaStream_t)stream>>>(*w, make_pb(params))));
    return check(cudaGetLastError(), "k_derivs");
}

int ilqgk_launch_backpass(const ilqg_work *w, const ilqg_opts *o, const double *params, int iter, void *stream)
{
    if constexpr (use_coop<P>()) {
        /* lanes per problem: 32, 16 or 8 (o->cw_lpp); the workspace of all problems of a block sits in dynamic shared memory */
        if (o->cw_lpp == 8) return cw_launch<8>(w, o, params, iter, stream);
        if (o->cw_lpp == 16) return cw_launch<16>(w, o, params, iter, stream);
        return cw_launch<32>(w, o, params, iter, stream);
    }
    else {
        constexpr size_t smem = sizeof(double) * 2 * bp_fields<P, FULL_DDP != 0>() * BP_BLOCK;
        /* the opt-in to > 48 KB dynamic shared memory is a per-device function attribute: applied once on every device
           this process launches on (idempotent, so two threads racing on the same device are harmless) */
        static unsigned char configured[ILQGK_MAX_DEVICES];
        int dev = 0;
        if (check(cudaGetDevice(&dev), "cudaGetDevice")) return -1;
        if (dev < 0 || dev >= ILQGK_MAX_DEVICES || !configured[dev]) {
            if (check(cudaFuncSetAttribute(k_backpass<P, FULL_DDP != 0, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "cudaFuncSetAttribute")) return -1;
            if (check(cudaFuncSetAttribute(k_backpass<P, FULL_DDP != 0, ILQG_BP_MINBLOCKS, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "cudaFuncSetAttribute")) return -1;
            if (check(cudaFuncSetAttribute(k_backpass<P, FULL_DDP != 0, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "cudaFuncSetAttribute")) return -1;
            if (check(cudaFuncSetAttribute(k_backpass<P, FULL_DDP != 0, ILQG_BP_MINBLOCKS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "cudaFuncSetAttribute")) return -1;
            if (dev >= 0 && dev < ILQGK_MAX_DEVICES) configured[dev] = 1;
        }
        if (SPLIT_OK && o->bp_split == 4) {
            PP_DISPATCH(w, (split_launcher<P, PP, SPLIT_OK>::go(w, o, params, iter, stream)));
            return check(cudaGetLastError(), "k_backpass_split");
        }
        const int ppw = (o->bp_ppw >= 1 && o->bp_ppw <= 32) ? o->bp_ppw : 32;
        const unsigned grid = nblk(w->B, ppw * (BP_BLOCK / 32));
        if (ppw != o->bp_ppw) { snprintf(g_err, sizeof g_err, "k_backpass: problems per warp must be 1..32"); return -1; }
        if (o->bp_latency_build)
            PP_DISPATCH(w, (k_backpass<P, FULL_DDP != 0, 1, PP><<<grid, BP_BLOCK, smem, (cudaStream_t)stream>>>(*w, *o, make_pb(params), iter)));
        else
            PP_DISPATCH(w, (k_backpass<P, FULL_DDP != 0, ILQG_BP_MINBLOCKS, PP><<<grid, BP_BLOCK, smem, (cudaStream_t)stream>>>(*w, *o, make_pb(params), iter)));
    }
    return check(cudaGetLastError(), "k_backpass");
}

/* line search = one launch per alpha; rounds > 0 read their problem list and count from device memory, so there is
   no host round trip.  Their grids are sized for the worst case and surplus blocks exit at once. */
int ilqgk_launch_ls_reset(const ilqg_work *w, void *stream)
{
    return check(cudaMemsetAsync(w->ls_count, 0, sizeof(int) * (ILQG_MAX_ALPHA + 2), (cudaStream_t)stream), "memset ls_count");
}

int ilqgk_launch_ls_round(const ilqg_work *w, const ilqg_opts *o, const double *params, int iter, int round, void *stream)
{
    PK_DISPATCH(w, (k_ls_round<P, PP, TR><<<nblk(w->B, BP_BLOCK), BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, *o, make_pb(params), iter, round)));
    return check(cudaGetLastError(), "k_ls_round");
}

int ilqgk_launch_ls_tail(const ilqg_work *w, const ilqg_opts *o, const double *params, int iter, int from, void *stream)
{
    const int nrem = o->n_alpha - from;
    const ParamBlock<P> pb = make_pb(params);
    const bool par = o->ls_commit_par && w->ls_ckpt;
    if (from == 0 && check(cudaMemsetAsync(w->ls_mask, 0, sizeof(int) * w->Bp, (cudaStream_t)stream), "memset ls_mask")) return -1;
    if (par)
        PK_DISPATCH(w, (k_ls_tail<P, PP, true, TR><<<nblk(w->B * nrem, BP_BLOCK), BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, *o, pb, from)));
    else
        PK_DISPATCH(w, (k_ls_tail<P, PP, false, TR><<<nblk(w->B * nrem, BP_BLOCK), BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, *o, pb, from)));
    if (check(cudaGetLastError(), "k_ls_tail")) return -1;
    if (par) {
        dim3 grid(nblk(w->B, BP_BLOCK), LS_SEGS);
        PK_DISPATCH(w, (k_ls_commit_seg<P, PP, TR><<<grid, BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, *o, pb, from)));
        if (check(cudaGetLastError(), "k_ls_commit_seg")) return -1;
        PK_DISPATCH(w, (k_ls_commit<P, PP, true, TR><<<nblk(w->B, BP_BLOCK), BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, *o, pb, iter, from)));
    } else
        PK_DISPATCH(w, (k_ls_commit<P, PP, false, TR><<<nblk(w->B, BP_BLOCK), BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, *o, pb, iter, from)));
    return check(cudaGetLastError(), "k_ls_commit");
}

int ilqgk_launch_post(const ilqg_work *w, const ilqg_opts *o, const double *params, void *stream)
{
    if (P::N_MU_R + P::N_MU_F == 0) return 0;   /* cost does not depend on multipliers/penalties: nothing to redo */
    PK_DISPATCH(w, (k_post<P, PP, TR><<<nblk(w->B, BP_BLOCK), BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, *o, make_pb(params))));
    return check(cudaGetLastError(), "k_post");
}

int ilqgk_launch_mult(const ilqg_work *w, const ilqg_opts *o, const double *params, int init, void *stream)
{
    if (P::N_MU_R + P::N_MU_F == 0) return 0;
    PK_DISPATCH(w, (k_mult<P, PP, TR><<<nblk(w->B, BP_BLOCK), BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, *o, make_pb(params), init)));
    return check(cudaGetLastError(), "k_mult");
}

int ilqgk_dense_size(void) { return P::DENSE_SIZE; }

int ilqgk_launch_dense(const ilqg_work *w, const double *params, double *out, void *stream)
{
    dim3 grid(nblk(w->B, DV_BLOCK), (unsigned)w->T);
    PP_DISPATCH(w, (k_dense<P, PP><<<grid, DV_BLOCK, 0, (cudaStream_t)stream>>>(*w, make_pb(params), out)));
    return check(cudaGetLastError(), "k_dense");
}

int ilqgk_launch_clamp(const ilqg_work *w, const double *params, double *xu_io, int k, void *stream)
{
    PK_DISPATCH(w, (k_clamp<P, PP, TR><<<nblk(w->B, BP_BLOCK), BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, make_pb(params), xu_io, k)));
    return check(cudaGetLastError(), "k_clamp");
}

int ilqgk_eval_size(int mode) { return (mode >= 0 && mode <= 17) ? eval_size<P>(mode) : -1; }

int ilqgk_launch_eval(const ilqg_work *w, const double *params, const double *in, double *out, int mode, int k, void *stream)
{
    PK_DISPATCH(w, (k_eval<P, PP, TR><<<nblk(w->B, BP_BLOCK), BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, make_pb(params), in, out, mode, k)));
    return check(cudaGetLastError(), "k_eval");
}

/* modified Cholesky of `count` packed n x n matrices (host arrays in, host arrays out), one thread per matrix */
int ilqgk_mod_chol(int n, int count, const double *A, const double *b, double *fac, double *E, int *P, double *ret, double *inv, double *H, double *x)
{
    if (n < 1 || n > MC_MAXN || count < 1) { snprintf(g_err, sizeof g_err, "mod_chol: n must be 1..%d and count >= 1", MC_MAXN); return -1; }
    const size_t np = (size_t)(n * (n + 1)) / 2, nA = np * count, nv = (size_t)n * count;
    double *d = NULL;
    int *dP = NULL;
    int rc = -1;
    if (check(cudaMalloc(&d, sizeof(double) * (4 * nA + 3 * nv + count)), "cudaMalloc") || check(cudaMalloc(&dP, sizeof(int) * nv), "cudaMalloc")) goto done;
    {
        double *dA = d, *dfac = dA + nA, *dinv = dfac + nA, *dH = dinv + nA, *db = dH + nA, *dE = db + nv, *dx = dE + nv, *dret = dx + nv;
        if (check(cudaMemcpy(dA, A, sizeof(double) * nA, cudaMemcpyHostToDevice), "H2D") || check(cudaMemcpy(db, b, sizeof(double) * nv, cudaMemcpyHostToDevice), "H2D")) goto done;
        k_mod_chol<<<nblk(count, 64), 64>>>(n, count, dA, db, dfac, dE, dP, dret, dinv, dH, dx);
        if (check(cudaGetLastError(), "k_mod_chol") || check(cudaDeviceSynchronize(), "k_mod_chol")) goto done;
        if (check(cudaMemcpy(fac, dfac, sizeof(double) * nA, cudaMemcpyDeviceToHost), "D2H") || check(cudaMemcpy(inv, dinv, sizeof(double) * nA, cudaMemcpyDeviceToHost), "D2H") ||
            check(cudaMemcpy(H, dH, sizeof(double) * nA, cudaMemcpyDeviceToHost), "D2H") || check(cudaMemcpy(E, dE, sizeof(double) * nv, cudaMemcpyDeviceToHost), "D2H") ||
            check(cudaMemcpy(x, dx, sizeof(double) * nv, cudaMemcpyDeviceToHost), "D2H") || check(cudaMemcpy(ret, dret, sizeof(double) * count, cudaMemcpyDeviceToHost), "D2H") ||
            check(cudaMemcpy(P, dP, sizeof(int) * nv, cudaMemcpyDeviceToHost), "D2H")) goto done;
    }
    rc = 0;
done:
    cudaFree(d);
    cudaFree(dP);
    return rc;
}

int ilqgk_has_post(void) { return (P::N_MU_R + P::N_MU_F) > 0; }

int ilqgk_launch_finalize(const ilqg_work *w, int max_iter, void *stream)
{
    k_finalize<<<nblk(w->B, 256), 256, 0, (cudaStream_t)stream>>>(*w, max_iter);
    return check(cudaGetLastError(), "k_finalize");
}

int ilqgk_launch_count_active(const ilqg_work *w, int *d_counter, void *stream)
{
    if (check(cudaMemsetAsync(d_counter, 0, sizeof(int), (cudaStream_t)stream), "memset")) return -1;
    k_count_active<<<nblk(w->B, 256), 256, 0, (cudaStream_t)stream>>>(*w, d_counter);
    return check(cudaGetLastError(), "k_count_active");
}

int ilqgk_launch_mpc_advance(const ilqg_work *w, const ilqg_mpc_step *a, void *stream)
{
    k_mpc_advance<P><<<nblk(w->B, 256), 256, 0, (cudaStream_t)stream>>>(*w, *a);
    return check(cudaGetLastError(), "k_mpc_advance");
}

int ilqgk_launch_mpc_plant(const ilqg_work *w, const ilqg_mpc_step *a, const double *params_plant, const ilqg_plant *pl, void *stream)
{
    /* PPP: per-problem plant table; TR: the model's [k]-indexed parameters from the tracks */
    const ParamBlock<P> pb = make_pb(params_plant);
    const unsigned grid = nblk(w->B, 256);
    if (HAS_KP && w->tr_mask) {
        constexpr bool TR = HAS_KP;
        if (pl->pp) k_mpc_plant<P, true, TR><<<grid, 256, 0, (cudaStream_t)stream>>>(*w, *a, pb, *pl);
        else k_mpc_plant<P, false, TR><<<grid, 256, 0, (cudaStream_t)stream>>>(*w, *a, pb, *pl);
    } else {
        if (pl->pp) k_mpc_plant<P, true, false><<<grid, 256, 0, (cudaStream_t)stream>>>(*w, *a, pb, *pl);
        else k_mpc_plant<P, false, false><<<grid, 256, 0, (cudaStream_t)stream>>>(*w, *a, pb, *pl);
    }
    return check(cudaGetLastError(), "k_mpc_plant");
}

int ilqgk_launch_policy_mark(const ilqg_work *w, int *keep, int *policy_ok, int save, void *stream)
{
    k_policy_mark<<<nblk(w->B, 256), 256, 0, (cudaStream_t)stream>>>(*w, keep, policy_ok, save);
    return check(cudaGetLastError(), "k_policy_mark");
}

int ilqgk_launch_policy_rollout(const ilqg_work *w, const double *params, const ilqg_policy *r, void *stream)
{
    /* PER: per-problem parameter table r->pp; TR: [k]-indexed parameters from the tracks */
    const ParamBlock<P> pb = make_pb(params);
    const long long lanes = (long long)w->B * r->n_samp;
    const unsigned grid = (unsigned)((lanes + BP_BLOCK - 1) / BP_BLOCK);
    if (HAS_KP && w->tr_mask) {
        constexpr bool TR = HAS_KP;
        if (r->pp) k_policy_rollout<P, true, TR><<<grid, BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, pb, *r);
        else k_policy_rollout<P, false, TR><<<grid, BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, pb, *r);
    } else {
        if (r->pp) k_policy_rollout<P, true, false><<<grid, BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, pb, *r);
        else k_policy_rollout<P, false, false><<<grid, BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, pb, *r);
    }
    return check(cudaGetLastError(), "k_policy_rollout");
}

int ilqgk_launch_policy_eval(const ilqg_work *w, const double *params, const int *policy_ok, const double *x, double *u, int k, void *stream)
{
    PK_DISPATCH(w, (k_policy_eval<P, PP, TR><<<nblk(w->B, BP_BLOCK), BP_BLOCK, 0, (cudaStream_t)stream>>>(*w, make_pb(params), policy_ok, x, u, k)));
    return check(cudaGetLastError(), "k_policy_eval");
}

int ilqgk_launch_scatter(const double *src, double *dst, double *dst_alt, const int *sel, int B, int n_k, int n_i, long long stride_k,
                         long long stride_b, long long stride_i, long long off, void *stream)
{
    const size_t n = (size_t)B * n_k * n_i;
    if (!n) return 0;
    const Layout L = {stride_k, stride_b, stride_i, off};
    k_scatter<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(src, dst, dst_alt, sel, B, n_k, n_i, L);
    return check(cudaGetLastError(), "k_scatter");
}

int ilqgk_launch_gather(const double *src, const double *src_alt, const int *sel, double *dst, int B, int n_k, int n_i,
                        long long stride_k, long long stride_b, long long stride_i, long long off, void *stream)
{
    const size_t n = (size_t)B * n_k * n_i;
    if (!n) return 0;
    const Layout L = {stride_k, stride_b, stride_i, off};
    k_gather<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(src, src_alt, sel, dst, B, n_k, n_i, L);
    return check(cudaGetLastError(), "k_gather");
}

} /* extern "C" */
