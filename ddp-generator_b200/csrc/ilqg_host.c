/* ilqg_host.c -- C host side of the B200 batched iLQG solver (implements include/ilqg_b200.h).
 *
 * Plain C, no CUDA headers: device work goes through the thin layer declared in ilqg_cuda.h.  The solve loop of
 * the reference (iLQG.c:239-363) becomes a fixed launch sequence per pass -- derivative kernel, backward-pass
 * kernel, line-search kernel, (multiplier/cost kernel) -- over the whole batch; the per-problem control flow
 * (lambda schedule, accept/reject, termination) lives in per-problem device state, so ragged convergence needs no
 * host round trip per pass.  All problems that are still running are at the same pass index `iter`.
 */
#define _POSIX_C_SOURCE 200809L
#include <stdio.h>
#include <stdlib.h>
#include <time.h>
#include <string.h>
#include <math.h>

#include "ilqg_b200.h"
#include "ilqg_cuda.h"

#define ACTIVE_CHECK_EVERY 8
#define POLL_RING 4          /* progress polls a chunk may have in flight (engine look-ahead is 2 blocks of passes) */
#define ENGINE_BLOCK 8       /* passes issued per chunk between two progress polls */
#define ENGINE_LOOKAHEAD 2
enum { TC_DERIVS = 0, TC_BACKPASS = 1, TC_LINESEARCH = 2, TC_POST = 3, TC_N = 4 };

typedef struct {
    void *start, *stop;
    int cls;
} ev_pair;

typedef struct chunk chunk;
struct chunk {
    int device, B, Bp, T, flags;
    ilqgk_dims_t d;
    ilqg_work w;
    ilqg_opts o;
    double *params;        /* flat, time-invariant */
    double *d_kp[16];      /* [k]-indexed parameters: device arrays of n_hor + 1 doubles, in parameter order */
    double **d_pk;         /* device table of those pointers (ilqg_work.pk); a parameter with a track points to the track */
    double *d_tr[16];      /* per-problem tracks [tr_len][Bp] of [k]-indexed parameters (ilqgb_set_param_track), or null;
                              their window offset is w.tr_off and their bits are w.tr_mask */
    int tr_len[16];
    double *d_pp;          /* per-problem parameter sets [npf][Bp] (ilqg_work.pp), allocated on first use */
    /* plant of the closed loops (ilqgb_set_plant_*): per flat parameter entry, where its value comes from; the plant's shared
       values; its per-problem values [npf][Bp]; and the table k_mpc_plant reads, rebuilt when anything it depends on changed */
    int plant_on, plant_n_sub, plant_dirty;
    unsigned char *plant_src;   /* [npf] PLANT_MODEL, PLANT_SHARED or PLANT_BATCH */
    double *plant_val;          /* [npf] shared plant values */
    double *d_plant_pp;         /* [npf][Bp] per-problem plant values (rows of PLANT_BATCH entries), allocated on first use */
    double *plant_params;       /* [npf] effective shared set (when neither the model nor the plant is per-problem) */
    double *d_plant_eff;        /* [npf][Bp] effective per-problem set, allocated on first use */
    int plant_per;              /* the effective set is d_plant_eff (else plant_params) */
    /* feedback policy (ilqgb_policy): per problem, whether its gains are valid; what k_policy_mark keeps while the policy's
       passes run; whether the nominal buffers still hold the gains ilqgb_policy computed (cleared by anything that may move them) */
    int *d_policy_ok, *d_policy_keep;
    int policy_valid;
    void *stream;          /* the stream all work of this chunk is enqueued on (stream_main, or stream_io during an end-to-end solve) */
    void *stream_main, *stream_io;
    int owns_stream;
    int prio_rank, prio_n; /* position of this chunk among the chunks of its device (stream_io priority) */
    int iter;              /* pass index of the running problems */
    /* asynchronous solve engine (run_engine): progress polls in flight, early stop, gating */
    int *h_poll;           /* pinned ring of POLL_RING running-problem counts */
    void *ev_poll[4];
    int poll_issued, poll_seen, stop, phase, mpc_step;
    ilqg_mpc_step mpc;     /* closed loop (ilqgb_mpc): this chunk's step and its w / log arrays in the staging buffer */
    void *ev_gate;
    int gate_recorded;
    int ls_tail_from;      /* -1 = choose by batch size */
    int bp_latency;        /* -1 = choose by batch size */
    int bp_ppw;            /* backward pass: problems per warp, -1 = choose by batch size */
    int bp_split;          /* lanes per problem of the small-batch backward pass (0 = lane per problem, 4), -1 = choose by batch size */
    int cw_lpp;            /* warp-cooperative backward pass: lanes per problem */
    int total_B;           /* problems of the whole handle (all chunks run concurrently on one GPU) */
    int started;
    int trace_cap;         /* max_iter the trace arrays were sized for */
    void **allocs;
    int n_allocs, cap_allocs;
    double *d_stage;       /* device staging for layout changes */
    size_t stage_doubles;
    int *d_counter;
    int *h_counter;        /* pinned */
    ev_pair *ev;
    int n_ev, cap_ev, n_ev_created;
    double t_ms[TC_N];
    long t_n[TC_N];
    long n_launches;       /* kernels launched since creation */
    char err[256];
};

enum { PLANT_MODEL = 0, PLANT_SHARED = 1, PLANT_BATCH = 2 };

static char g_create_err[256] = "";
#define fail_create(msg) (snprintf(g_create_err, sizeof g_create_err, "%s", msg), (void)0)

static int fail(chunk *h, const char *msg)
{
    snprintf(h ? h->err : g_create_err, 256, "%s", msg);
    return -1;
}

static int failk(chunk *h) { return fail(h, ilqgk_last_error()); }

#define BP_SPLIT_MAX_B 6144    /* problems on one GPU up to which the backward pass runs four lanes per problem, four problems per
                                  warp (measured on B200, scripts/gpu_probe_split.sh, car, 50 passes, ms per backward pass: 4096 problems
                                  2.38 one lane per problem, 1.89 the same with 8 problems per warp, 1.82 split; 16 384: 2.44 / 3.9) */

static int env_int(const char *name, int dflt)
{
    const char *v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

/* The warp-cooperative backward pass keeps the workspace of every problem of a block in shared memory, 32 / lpp problems per warp:
   a lanes-per-problem count whose workspace the device cannot give a block is refused here, not in the middle of a solve */
static int coop_fits(const chunk *h, int lpp, char *err, size_t n)
{
    size_t need = 0, limit = 0;
    if (!h->d.coop) return 1;
    if (ilqgk_coop_smem(h->device, lpp, &need, &limit)) {
        snprintf(err, n, "%s", ilqgk_last_error());
        return 0;
    }
    if (need <= limit) return 1;
    snprintf(err, n, "cw_lpp %d: the warp-cooperative backward pass needs %zu bytes of shared memory per block, the device allows %zu", lpp, need, limit);
    return 0;
}

static void *dalloc(chunk *h, size_t bytes)
{
    void *p = NULL;
    if (ilqgk_malloc(&p, bytes)) {
        failk(h);
        return NULL;
    }
    if (h->n_allocs == h->cap_allocs) {
        const int cap = h->cap_allocs ? 2 * h->cap_allocs : 64;
        void **a = (void **)realloc(h->allocs, sizeof(void *) * cap);
        if (!a) {
            ilqgk_free(p);
            fail(h, "out of host memory");
            return NULL;
        }
        h->allocs = a;
        h->cap_allocs = cap;
    }
    h->allocs[h->n_allocs++] = p;
    return p;
}

/* release one device allocation made by dalloc before the handle goes away */
static void dfree(chunk *h, void *p)
{
    int i;
    if (!p) return;
    for (i = 0; i < h->n_allocs; i++)
        if (h->allocs[i] == p) {
            h->allocs[i] = h->allocs[--h->n_allocs];
            break;
        }
    ilqgk_free(p);
}

/* ---- static facts -------------------------------------------------------------------------------------------------- */
const char *ilqgb_problem_name(void) { return ilqgk_problem_name(); }
int ilqgb_nx(void) { ilqgk_dims_t d; ilqgk_dims(&d); return d.nx; }
int ilqgb_nu(void) { ilqgk_dims_t d; ilqgk_dims(&d); return d.nu; }
int ilqgb_full_ddp(void) { ilqgk_dims_t d; ilqgk_dims(&d); return d.full_ddp; }
int ilqgb_n_params(void) { return ilqgk_param_count(); }
const char *ilqgb_param_name(int i) { return ilqgk_param_name(i); }
int ilqgb_param_size(int i) { return ilqgk_param_size(i); }
int ilqgb_device_count(void) { return ilqgk_device_count(); }
void ilqgb_mult_counts(int *n_running_eq, int *n_final_eq)
{
    ilqgk_dims_t d;
    ilqgk_dims(&d);
    if (n_running_eq) *n_running_eq = d.n_mu_le;
    if (n_final_eq) *n_final_eq = d.n_mu_fe;
}
int ilqgb_deriv_doubles_per_step(void) { ilqgk_dims_t d; ilqgk_dims(&d); return d.nv1 + (d.full_ddp ? d.nv2 : 0); }

static void ck_destroy(chunk *h);
static int ensure_stage(chunk *h, size_t doubles);

/* ---- options (reference: standard_parameters iLQG.c:57-78, setOptParam iLQG.c:91-216) ----------------------------------- */
static const double k_alpha_default[8] = {1.0, 0.3727594, 0.1389495, 0.0517947, 0.0193070, 0.0071969, 0.0026827, 0.0010000};

static void ck_standard_parameters(chunk *h)
{
    ilqg_opts *o = &h->o;
    memset(o, 0, sizeof *o);
    memcpy(o->alpha, k_alpha_default, sizeof k_alpha_default);
    o->n_alpha = 8;
    o->tolFun = 1e-7;
    o->tolConstraint = 1e-7;
    o->tolGrad = 1e-5;
    o->max_iter = 20;
    o->lambdaInit = 1;
    o->dlambdaInit = 1;
    o->lambdaFactor = 1.6;
    o->lambdaMax = 1e10;
    o->lambdaMin = 1e-6;
    o->regType = 1;
    o->zMin = 0.0;
    o->w_pen_init_l = 1.0;
    o->w_pen_init_f = 1.0;
    o->w_pen_max_l = INFINITY;
    o->w_pen_max_f = INFINITY;
    o->w_pen_fact1 = 4.0;
    o->w_pen_fact2 = 1.0;
}

typedef enum { V_POSITIVE, V_NONNEG, V_GE_ONE, V_ONE_TWO, V_ZERO_ONE, V_DEBUG } vrule;
typedef struct {
    const char *name;
    size_t offset;
    int is_int;
    vrule rule;
} opt_desc;

#define OPT_D(field, rule) {#field, offsetof(ilqg_opts, field), 0, rule}
#define OPT_I(field, rule) {#field, offsetof(ilqg_opts, field), 1, rule}
static const opt_desc k_opts[] = {
    OPT_D(tolFun, V_POSITIVE),      OPT_D(tolConstraint, V_POSITIVE), OPT_D(tolGrad, V_POSITIVE),
    OPT_I(max_iter, V_NONNEG),      OPT_D(lambdaInit, V_NONNEG),      OPT_D(dlambdaInit, V_NONNEG),
    OPT_D(lambdaFactor, V_GE_ONE),  OPT_D(lambdaMax, V_NONNEG),       OPT_D(lambdaMin, V_NONNEG),
    OPT_I(regType, V_ONE_TWO),      OPT_D(zMin, V_ZERO_ONE),          OPT_D(w_pen_init_l, V_NONNEG),
    OPT_D(w_pen_init_f, V_NONNEG),  OPT_D(w_pen_max_l, V_NONNEG),     OPT_D(w_pen_max_f, V_NONNEG),
    OPT_D(w_pen_fact1, V_GE_ONE),   OPT_D(w_pen_fact2, V_GE_ONE),
};

static const char *rule_message(vrule r, double v)
{
    switch (r) {
    case V_POSITIVE: return v <= 0.0 ? "parameter must be positive" : NULL;
    case V_NONNEG: return v < 0.0 ? "parameter must be positive" : NULL;
    case V_GE_ONE: return v < 1.0 ? "parameter must be > 1" : NULL;
    case V_ONE_TWO: return (v < 1.0 || v > 2.0) ? "parameter must be in range [1..2]" : NULL;
    case V_ZERO_ONE: return (v < 0.0 || v >= 1.0) ? "parameter must be in range [0..1)" : NULL;
    case V_DEBUG: return (v < 0.0 || v > 6.0) ? "parameter must be in range [0..6]" : NULL;
    }
    return NULL;
}

/* validation only (no handle, no device): NULL = acceptable, otherwise the reference's message */
const char *ilqgb_validate_opt(const char *name, const double *value, int n)
{
    size_t i;
    if (strcmp(name, "alpha") == 0) {
        int k;
        for (k = 0; k < n; k++) {
            if (value[k] < 0.0 || value[k] > 1.0) return "all alpha must be in the range [1.0..0.0)";
            if (k > 0 && value[k] >= value[k - 1]) return "all alpha must be monotonically decreasing";
        }
        if (n > ILQG_MAX_ALPHA) return "at most 16 alpha values are supported";
        return NULL;
    }
    if (strcmp(name, "debug_level") == 0) { /* accepted and validated; the batched solver prints nothing */
        if (n != 1) return "parameter must be scalar";
        return rule_message(V_DEBUG, value[0]);
    }
    for (i = 0; i < sizeof k_opts / sizeof k_opts[0]; i++) {
        if (strcmp(name, k_opts[i].name) != 0) continue;
        if (n != 1) return "parameter must be scalar";
        return rule_message(k_opts[i].rule, value[0]);
    }
    return "no such parameter";
}

static const char *ck_set_opt(chunk *h, const char *name, const double *value, int n)
{
    size_t i;
    const char *msg = ilqgb_validate_opt(name, value, n);
    if (msg) return msg;
    if (strcmp(name, "alpha") == 0) {
        memcpy(h->o.alpha, value, sizeof(double) * n);
        h->o.n_alpha = n;
        return NULL;
    }
    for (i = 0; i < sizeof k_opts / sizeof k_opts[0]; i++) {
        const opt_desc *d = &k_opts[i];
        if (strcmp(name, d->name) != 0) continue;
        if (d->is_int)
            *(int *)((char *)&h->o + d->offset) = (int)value[0];
        else
            *(double *)((char *)&h->o + d->offset) = value[0];
        return NULL;
    }
    return NULL; /* debug_level */
}

static int param_offset(int index)
{
    int i, off = 0;
    for (i = 0; i < index; i++)
        if (ilqgk_param_size(i) > 0) off += ilqgk_param_size(i);
    return off;
}

/* one device row [Bp] = the same value for every problem */
static int fill_row(chunk *h, double *dst, double v)
{
    size_t b;
    double *tmp = (double *)malloc(sizeof(double) * h->Bp);
    int rc;
    if (!tmp) return fail(h, "out of host memory");
    for (b = 0; b < (size_t)h->Bp; b++) tmp[b] = v;
    rc = ilqgk_h2d(dst, tmp, sizeof(double) * h->Bp, h->stream) || ilqgk_stream_sync(h->stream);
    free(tmp);
    return rc ? failk(h) : 0;
}

/* one row of the per-problem table = the same value for every problem */
static int pp_fill_row(chunk *h, int row, double v) { return fill_row(h, h->d_pp + (size_t)row * h->Bp, v); }

/* parameter `index` for every problem of the chunk: value[b][n] (a batch of independent reference calls, each with
   its own parameter struct).  The first call switches the chunk to per-problem parameters, seeded from the shared set. */
static int ck_set_param_batch(chunk *h, int index, const double *value, int n)
{
    int i, off;
    size_t b;
    double *tmp;
    if (index < 0 || index >= ilqgk_param_count()) return fail(h, "parameter index out of range");
    if (ilqgk_param_size(index) == -1) return fail(h, "[k]-indexed parameters are shared by the batch");
    if (n != ilqgk_param_size(index)) return fail(h, "wrong parameter length");
    if (ilqgk_set_device(h->device)) return failk(h);
    h->plant_dirty = 1;   /* plant entries that follow the model follow this change */
    if (!h->d_pp) {
        h->d_pp = (double *)dalloc(h, sizeof(double) * (size_t)(h->d.npf > 0 ? h->d.npf : 1) * h->Bp);
        if (!h->d_pp) return -1;
        for (i = 0; i < h->d.npf; i++)
            if (pp_fill_row(h, i, h->params[i])) return -1;
        h->w.pp = h->d_pp;
    }
    off = param_offset(index);
    tmp = (double *)calloc((size_t)h->Bp, sizeof(double));
    if (!tmp) return fail(h, "out of host memory");
    for (i = 0; i < n; i++) {
        for (b = 0; b < (size_t)h->B; b++) tmp[b] = value[b * n + i];
        if (ilqgk_h2d(h->d_pp + (size_t)(off + i) * h->Bp, tmp, sizeof(double) * h->Bp, h->stream) || ilqgk_stream_sync(h->stream)) {
            free(tmp);
            return failk(h);
        }
    }
    free(tmp);
    return 0;
}

/* position of parameter `index` among the [k]-indexed ones */
static int kp_index(int index)
{
    int i, kidx = 0;
    for (i = 0; i < index; i++)
        if (ilqgk_param_size(i) == -1) kidx++;
    return kidx;
}

/* entry kidx of the device pointer table: the track if there is one, else the shared array */
static int ck_point_pk(chunk *h, int kidx)
{
    const double *p = h->d_tr[kidx] ? h->d_tr[kidx] : h->d_kp[kidx];
    if (ilqgk_h2d(h->d_pk + kidx, &p, sizeof p, h->stream) || ilqgk_stream_sync(h->stream)) return failk(h);
    return 0;
}

static int ck_drop_track(chunk *h, int kidx)
{
    dfree(h, h->d_tr[kidx]);   /* cudaFree waits for the work that still reads it */
    h->d_tr[kidx] = NULL;
    h->tr_len[kidx] = 0;
    h->w.tr_mask &= ~(1u << kidx);
    return ck_point_pk(h, kidx);
}

/* the track of [k]-indexed parameter kidx for every problem of the chunk: value[b][len] (checked by the caller), moved to
   [len][Bp] through the staging buffer by one layout kernel */
static int ck_set_param_track(chunk *h, int kidx, const double *value, int len)
{
    const size_t n = (size_t)h->B * len;
    if (ilqgk_set_device(h->device)) return failk(h);
    if (h->d_tr[kidx] && h->tr_len[kidx] != len) {
        dfree(h, h->d_tr[kidx]);
        h->d_tr[kidx] = NULL;
    }
    if (!h->d_tr[kidx]) {
        h->d_tr[kidx] = (double *)dalloc(h, sizeof(double) * (size_t)len * h->Bp);
        if (!h->d_tr[kidx]) return -1;
        h->tr_len[kidx] = len;
    }
    if (ensure_stage(h, n)) return -1;
    if (ilqgk_h2d(h->d_stage, value, sizeof(double) * n, h->stream)) return failk(h);
    if (ilqgk_launch_scatter(h->d_stage, h->d_tr[kidx], NULL, NULL, h->B, len, 1, h->Bp, 1, 0, 0, h->stream)) return failk(h);
    h->n_launches++;
    h->w.tr_mask |= 1u << kidx;
    return ck_point_pk(h, kidx);
}

static int ck_set_param(chunk *h, int index, const double *value, int n)
{
    int i, off = 0;
    if (index < 0 || index >= ilqgk_param_count()) return fail(h, "parameter index out of range");
    if (ilqgk_param_size(index) == -1) { /* one value per timestep, name[k] in the problem file */
        const int kidx = kp_index(index);
        if (n != h->T + 1) return fail(h, "wrong parameter length (n_hor + 1 expected)");
        if (ilqgk_set_device(h->device)) return failk(h);
        if (ilqgk_h2d(h->d_kp[kidx], value, sizeof(double) * n, h->stream) || ilqgk_stream_sync(h->stream)) return failk(h);
        return h->d_tr[kidx] ? ck_drop_track(h, kidx) : 0;   /* shared and fixed again */
    }
    if (n != ilqgk_param_size(index)) return fail(h, "wrong parameter length");
    for (i = 0; i < index; i++)
        if (ilqgk_param_size(i) > 0) off += ilqgk_param_size(i);
    memcpy(h->params + off, value, sizeof(double) * n);
    h->plant_dirty = 1;
    if (h->d_pp) /* per-problem table in use: a shared value overwrites every problem's entry */
        for (i = 0; i < n; i++)
            if (pp_fill_row(h, off + i, value[i])) return -1;
    return 0;
}

/* ---- plant of the closed loops (see ilqg_b200.h); index, value and length are checked by the caller ---- */
static void ck_set_plant_param(chunk *h, int index, const double *value, int n)
{
    const int off = param_offset(index);
    int i;
    for (i = 0; i < n; i++) {
        h->plant_src[off + i] = PLANT_SHARED;
        h->plant_val[off + i] = value[i];
    }
    h->plant_on = 1;
    h->plant_dirty = 1;
}

static int ck_set_plant_param_batch(chunk *h, int index, const double *value, int n)
{
    const int off = param_offset(index);
    int i;
    size_t b;
    double *tmp;
    if (ilqgk_set_device(h->device)) return failk(h);
    if (!h->d_plant_pp) {
        h->d_plant_pp = (double *)dalloc(h, sizeof(double) * (size_t)h->d.npf * h->Bp);
        if (!h->d_plant_pp) return -1;
    }
    tmp = (double *)calloc((size_t)h->Bp, sizeof(double));
    if (!tmp) return fail(h, "out of host memory");
    for (i = 0; i < n; i++) {
        for (b = 0; b < (size_t)h->B; b++) tmp[b] = value[b * n + i];
        if (ilqgk_h2d(h->d_plant_pp + (size_t)(off + i) * h->Bp, tmp, sizeof(double) * h->Bp, h->stream) || ilqgk_stream_sync(h->stream)) {
            free(tmp);
            return failk(h);
        }
        h->plant_src[off + i] = PLANT_BATCH;
    }
    free(tmp);
    h->plant_on = 1;
    h->plant_dirty = 1;
    return 0;
}

static void ck_clear_plant(chunk *h)
{
    ilqgk_set_device(h->device);
    dfree(h, h->d_plant_pp);   /* cudaFree waits for the work that still reads it */
    dfree(h, h->d_plant_eff);
    h->d_plant_pp = h->d_plant_eff = NULL;
    memset(h->plant_src, PLANT_MODEL, (size_t)(h->d.npf > 0 ? h->d.npf : 1));
    h->plant_on = h->plant_per = 0;
    h->plant_n_sub = 1;
    h->plant_dirty = 1;
}

/* The one table k_mpc_plant reads, entry by entry the plant's own value where it has one and the model's current value
   (shared, or this problem's under per-problem model parameters) elsewhere.  A shared set when neither the model nor the
   plant is per-problem, else [npf][Bp] built on the device.  Rebuilt only after a change (plant_dirty). */
static int ck_plant_prepare(chunk *h)
{
    const size_t Bp = (size_t)h->Bp;
    int i, per = h->d_pp != NULL;
    if (!h->plant_dirty) return 0;
    for (i = 0; i < h->d.npf; i++) {
        h->plant_params[i] = h->plant_src[i] == PLANT_SHARED ? h->plant_val[i] : h->params[i];
        if (h->plant_src[i] == PLANT_BATCH) per = 1;
    }
    if (per) {
        if (ilqgk_set_device(h->device)) return failk(h);
        if (!h->d_plant_eff) {
            h->d_plant_eff = (double *)dalloc(h, sizeof(double) * (size_t)h->d.npf * Bp);
            if (!h->d_plant_eff) return -1;
        }
        for (i = 0; i < h->d.npf; i++) {
            double *dst = h->d_plant_eff + (size_t)i * Bp;
            if (h->plant_src[i] == PLANT_BATCH) {
                if (ilqgk_d2d(dst, h->d_plant_pp + (size_t)i * Bp, sizeof(double) * Bp, h->stream)) return failk(h);
            } else if (h->plant_src[i] == PLANT_MODEL && h->d_pp) {
                if (ilqgk_d2d(dst, h->d_pp + (size_t)i * Bp, sizeof(double) * Bp, h->stream)) return failk(h);
            } else if (fill_row(h, dst, h->plant_params[i]))
                return -1;
        }
        if (ilqgk_stream_sync(h->stream)) return failk(h);
    }
    h->plant_per = per;
    h->plant_dirty = 0;
    return 0;
}

/* x0 of the next solve from the solution's prediction (k_mpc_advance) or, with a plant, from the plant (k_mpc_plant) */
static int launch_advance(chunk *h, const ilqg_mpc_step *a)
{
    if (h->plant_on && a->set_x0) {
        ilqg_plant pl;
        if (ck_plant_prepare(h)) return -1;
        pl.n_sub = h->plant_n_sub;
        pl.pp = h->plant_per ? h->d_plant_eff : NULL;
        if (ilqgk_launch_mpc_plant(&h->w, a, h->plant_params, &pl, h->stream)) return failk(h);
    } else if (ilqgk_launch_mpc_advance(&h->w, a, h->stream))
        return failk(h);
    h->n_launches++;
    return 0;
}

/* ---- lifecycle ------------------------------------------------------------------------------------------------------------- */
#define DALLOC(dst, type, count)                                   \
    do {                                                           \
        (dst) = (type *)dalloc(h, sizeof(type) * (size_t)(count)); \
        if (!(dst)) goto oom;                                      \
    } while (0)

static chunk *ck_create(int device, int batch, int n_hor, int flags, void *stream, int prio_rank, int prio_n)
{
    chunk *h;
    size_t Bp, T = (size_t)n_hor;
    if (batch < 1 || n_hor < 1) {
        fail(NULL, "batch and n_hor must be >= 1");
        return NULL;
    }
    if (ilqgk_device_count() < 1) {
        fail(NULL, "no CUDA device available: this library has no CPU fallback");
        return NULL;
    }
    if (ilqgk_set_device(device)) {
        failk(NULL);
        return NULL;
    }
    h = (chunk *)calloc(1, sizeof *h);
    if (!h) {
        fail(NULL, "out of host memory");
        return NULL;
    }
    h->device = device;
    h->B = batch;
    h->total_B = batch;
    h->Bp = (batch + 31) / 32 * 32;
    h->T = n_hor;
    h->flags = flags;
    h->ls_tail_from = getenv("ILQG_LS_TAIL_FROM") ? atoi(getenv("ILQG_LS_TAIL_FROM")) : -1;
    h->bp_latency = getenv("ILQG_BP_LATENCY") ? atoi(getenv("ILQG_BP_LATENCY")) : -1;
    h->cw_lpp = env_int("ILQG_CW_LPP", 32);
    h->bp_split = env_int("ILQG_BP_SPLIT", -1);
    h->bp_ppw = env_int("ILQG_BP_PPW", -1);
    ilqgk_dims(&h->d);
    if (ilqgk_set_device(device) || ilqgk_preload()) {   /* no lazily loaded kernel inside a later solve */
        fail(NULL, ilqgk_last_error());
        free(h);
        return NULL;
    }
    if (h->d.nkp > 16) {
        fail(NULL, "too many [k]-indexed parameters");
        free(h);
        return NULL;
    }
    if (!coop_fits(h, 32, g_create_err, sizeof g_create_err) || !coop_fits(h, h->cw_lpp, g_create_err, sizeof g_create_err)) {
        free(h);
        return NULL;
    }
    h->params = (double *)calloc((size_t)(h->d.npf > 0 ? h->d.npf : 1), sizeof(double));
    if (!h->params) {
        fail(NULL, "out of host memory");
        free(h);
        return NULL;
    }
    h->plant_src = (unsigned char *)calloc((size_t)(h->d.npf > 0 ? h->d.npf : 1), 1);
    h->plant_val = (double *)calloc((size_t)(h->d.npf > 0 ? h->d.npf : 1), sizeof(double));
    h->plant_params = (double *)calloc((size_t)(h->d.npf > 0 ? h->d.npf : 1), sizeof(double));
    if (!h->plant_src || !h->plant_val || !h->plant_params) {
        fail(NULL, "out of host memory");
        free(h->plant_src);
        free(h->plant_val);
        free(h->plant_params);
        free(h->params);
        free(h);
        return NULL;
    }
    h->plant_n_sub = 1;
    h->plant_dirty = 1;
    ck_standard_parameters(h);
    h->prio_rank = prio_rank;
    h->prio_n = prio_n;
    if (stream) {
        h->stream_main = stream;
    } else {
        if (ilqgk_stream_create(&h->stream_main)) goto oom;
        h->owns_stream = 1;
    }
    h->stream = h->stream_main;
    Bp = (size_t)h->Bp;
    {
        const ilqgk_dims_t *d = &h->d;
        ilqg_work *w = &h->w;
        int i;
        w->B = batch;
        w->Bp = h->Bp;
        w->T = n_hor;
        for (i = 0; i < 2; i++) {
            DALLOC(w->XU[i], double, (T + 1) * Bp * d->rxu);
            ilqgk_memset(w->XU[i], 0, sizeof(double) * (T + 1) * Bp * d->rxu, h->stream);
        }
        DALLOC(w->x0, double, d->nx * Bp);
        for (i = 0; i < 2; i++) {
            DALLOC(w->LL[i], double, T * Bp * d->rlm);
            DALLOC(w->Ll[i], double, T * Bp * d->rls);
        }
        DALLOC(w->V1, double, T * d->nv1 * Bp);
        DALLOC(w->V2, double, d->full_ddp ? T * d->nv2 * Bp : 1);
        DALLOC(w->FD, double, (d->nx + d->nqxx) * Bp);
        DALLOC(w->muR, double, T * (d->n_mu_r ? d->n_mu_r : 0) * Bp + 1);
        DALLOC(w->lastR, double, T * (d->n_mu_r ? d->n_mu_r : 0) * Bp + 1);
        DALLOC(w->muF, double, d->n_mu_f * Bp + 1);
        DALLOC(w->lastF, double, d->n_mu_f * Bp + 1);
        w->pk = NULL;
        if (d->nkp > 0) {
            for (i = 0; i < d->nkp; i++) {
                DALLOC(h->d_kp[i], double, T + 1);
                ilqgk_memset(h->d_kp[i], 0, sizeof(double) * (T + 1), h->stream);
            }
            DALLOC(h->d_pk, double *, d->nkp);
            if (ilqgk_h2d(h->d_pk, h->d_kp, sizeof(double *) * d->nkp, h->stream) || ilqgk_stream_sync(h->stream)) goto oom;
            w->pk = (const double *const *)h->d_pk;
        }
        DALLOC(w->cost, double, Bp);
        DALLOC(w->new_cost, double, Bp);
        DALLOC(w->dcost, double, Bp);
        DALLOC(w->expected, double, Bp);
        DALLOC(w->lambda, double, Bp);
        DALLOC(w->dlambda, double, Bp);
        DALLOC(w->g_norm, double, Bp);
        DALLOC(w->dV0, double, Bp);
        DALLOC(w->dV1, double, Bp);
        DALLOC(w->w_pen_l, double, Bp);
        DALLOC(w->w_pen_f, double, Bp);
        DALLOC(w->cur, int, Bp);
        DALLOC(w->status, int, Bp);
        DALLOC(w->new_deriv, int, Bp);
        DALLOC(w->deriv_fail, int, Bp);
        DALLOC(w->iterations, int, Bp);
        DALLOC(w->result, int, Bp);
        DALLOC(w->n_ls, int, Bp);
        DALLOC(w->n_bp, int, Bp);
        DALLOC(w->bp_done, int, Bp);
        DALLOC(w->post_mode, int, Bp);
        DALLOC(w->ls_list[0], int, Bp);
        DALLOC(w->ls_list[1], int, Bp);
        DALLOC(w->ls_count, int, ILQG_MAX_ALPHA + 2);
        DALLOC(w->ls_cnew, double, (size_t)ILQG_MAX_ALPHA * Bp);
        DALLOC(w->ls_mask, int, Bp);
        if (env_int("ILQG_LS_COMMIT_PAR", 1)) DALLOC(w->ls_ckpt, double, (size_t)ILQG_MAX_ALPHA * 32 * Bp * d->nx);
        DALLOC(w->n_dv, int, Bp);
        DALLOC(w->n_roll, int, Bp);
        DALLOC(w->n_tail, int, Bp);
        ilqgk_memset(w->status, 0, sizeof(int) * Bp, h->stream);
        ilqgk_memset(w->cur, 0, sizeof(int) * Bp, h->stream);
        if (flags & ILQGB_TRACE) {
            DALLOC(w->tr_clamp, int, T * Bp);
            ilqgk_memset(w->tr_clamp, 0, sizeof(int) * T * Bp, h->stream);
        }
        DALLOC(h->d_counter, int, 1);
        DALLOC(h->d_policy_ok, int, Bp);
        DALLOC(h->d_policy_keep, int, 7 * Bp);
        ilqgk_memset(h->d_policy_ok, 0, sizeof(int) * Bp, h->stream);
    }
    if (ilqgk_host_alloc((void **)&h->h_counter, sizeof(int))) goto oom;
    if (ilqgk_host_alloc((void **)&h->h_poll, sizeof(int) * POLL_RING)) goto oom;
    {
        int i;
        for (i = 0; i < POLL_RING; i++)
            if (ilqgk_event_create_notiming(&h->ev_poll[i])) goto oom;
        if (ilqgk_event_create_notiming(&h->ev_gate)) goto oom;
    }
    return h;
oom:
    snprintf(g_create_err, sizeof g_create_err, "%s", h->err[0] ? h->err : ilqgk_last_error());
    ck_destroy(h);
    return NULL;
}

static void ck_destroy(chunk *h)
{
    int i;
    if (!h) return;
    ilqgk_set_device(h->device);
    if (h->stream_main) ilqgk_stream_sync(h->stream_main);
    if (h->stream_io) ilqgk_stream_sync(h->stream_io);
    for (i = 0; i < POLL_RING; i++)
        if (h->ev_poll[i]) ilqgk_event_destroy(h->ev_poll[i]);
    if (h->ev_gate) ilqgk_event_destroy(h->ev_gate);
    if (h->h_poll) ilqgk_host_free(h->h_poll);
    for (i = 0; i < h->n_allocs; i++) ilqgk_free(h->allocs[i]);
    free(h->allocs);
    for (i = 0; i < h->n_ev_created; i++) {
        ilqgk_event_destroy(h->ev[i].start);
        ilqgk_event_destroy(h->ev[i].stop);
    }
    free(h->ev);
    if (h->h_counter) ilqgk_host_free(h->h_counter);
    if (h->stream_io) ilqgk_stream_destroy(h->stream_io);
    if (h->owns_stream && h->stream_main) ilqgk_stream_destroy(h->stream_main);
    free(h->params);
    free(h->plant_src);
    free(h->plant_val);
    free(h->plant_params);
    free(h);
}

static int ensure_stage(chunk *h, size_t doubles)
{
    if (doubles <= h->stage_doubles) return 0;
    if (h->d_stage) { /* work that still reads the old buffer is ordered before its release (cudaFree synchronises) */
        if (ilqgk_stream_sync(h->stream)) return failk(h);
        dfree(h, h->d_stage);
        h->d_stage = NULL;
        h->stage_doubles = 0;
    }
    h->d_stage = (double *)dalloc(h, sizeof(double) * doubles);
    if (!h->d_stage) {
        h->stage_doubles = 0;
        return -1;
    }
    h->stage_doubles = doubles;
    return 0;
}

static int ensure_traces(chunk *h)
{
    size_t n, n_old;
    const int need = h->o.max_iter > 0 ? h->o.max_iter : 1;
    double *lam, *nc, *z;
    int *al;
    if (!(h->flags & ILQGB_TRACE) || need <= h->trace_cap) return 0;
    n = (size_t)need * h->Bp;
    n_old = (size_t)h->trace_cap * h->Bp;
    lam = (double *)dalloc(h, sizeof(double) * n);
    nc = (double *)dalloc(h, sizeof(double) * n);
    al = (int *)dalloc(h, sizeof(int) * n);
    z = (double *)dalloc(h, sizeof(double) * n);
    if (!lam || !nc || !al || !z) return -1;
    if (n_old) { /* max_iter was raised after the traces were sized (possibly mid-solve): keep what has been recorded */
        if (ilqgk_d2d(lam, h->w.tr_lambda, sizeof(double) * n_old, h->stream) || ilqgk_d2d(nc, h->w.tr_newcost, sizeof(double) * n_old, h->stream) ||
            ilqgk_d2d(al, h->w.tr_alpha, sizeof(int) * n_old, h->stream) || ilqgk_d2d(z, h->w.tr_z, sizeof(double) * n_old, h->stream) ||
            ilqgk_stream_sync(h->stream))
            return failk(h);
        dfree(h, h->w.tr_lambda);
        dfree(h, h->w.tr_newcost);
        dfree(h, h->w.tr_alpha);
        dfree(h, h->w.tr_z);
    }
    h->w.tr_lambda = lam;
    h->w.tr_newcost = nc;
    h->w.tr_alpha = al;
    h->w.tr_z = z;
    h->trace_cap = need;
    return 0;
}

/* ---- data movement ------------------------------------------------------------------------------------------------------------ */
static int ck_upload(chunk *h, const double *x0, const double *u_nom)
{
    const size_t B = (size_t)h->B, T = (size_t)h->T, nx = (size_t)h->d.nx, nu = (size_t)h->d.nu;
    if (ilqgk_set_device(h->device)) return failk(h);
    if (ensure_stage(h, B * T * nu + B * nx)) return -1;
    if (ilqgk_h2d(h->d_stage, u_nom, sizeof(double) * B * T * nu, h->stream)) return failk(h);
    if (ilqgk_h2d(h->d_stage + B * T * nu, x0, sizeof(double) * B * nx, h->stream)) return failk(h);
    /* controls into the u part of buffer 0's records; x0 into its own [NX][Bp] array */
    if (ilqgk_launch_scatter(h->d_stage, h->w.XU[0], NULL, NULL, h->B, h->T, h->d.nu, (long long)h->Bp * h->d.rxu, h->d.rxu, 1, h->d.nx, h->stream)) return failk(h);
    h->n_launches += 2;
    if (ilqgk_launch_scatter(h->d_stage + B * T * nu, h->w.x0, NULL, NULL, h->B, 1, h->d.nx, 0, 1, h->Bp, 0, h->stream)) return failk(h);
    h->started = 0;
    h->policy_valid = 0;
    return 0;
}

/* ---- receding horizon -------------------------------------------------------------------------------------------------------- */
/* the solution becomes the next solve's input: controls shifted by n_shift, x0 from the host or x[n_shift] (+ w [B][nx]) */
static int ck_shift(chunk *h, int n_shift, const double *x0, const double *w)
{
    const size_t B = (size_t)h->B, nx = (size_t)h->d.nx;
    ilqg_mpc_step a;
    if (ilqgk_set_device(h->device)) return failk(h);
    if ((x0 || w) && ensure_stage(h, B * nx)) return -1;
    memset(&a, 0, sizeof a);
    a.n_shift = n_shift;
    a.set_x0 = !x0;
    a.plan = 1;
    a.n_steps = 1;
    if (w) {
        if (ilqgk_h2d(h->d_stage, w, sizeof(double) * B * nx, h->stream)) return failk(h);
        a.w = h->d_stage;
    }
    if (launch_advance(h, &a)) return -1;
    if (x0) { /* into its own [NX][Bp] array, as ck_upload does */
        if (ilqgk_h2d(h->d_stage, x0, sizeof(double) * B * nx, h->stream)) return failk(h);
        if (ilqgk_launch_scatter(h->d_stage, h->w.x0, NULL, NULL, h->B, 1, h->d.nx, 0, 1, h->Bp, 0, h->stream)) return failk(h);
        h->n_launches++;
    }
    h->started = 0;
    h->policy_valid = 0;
    return 0;
}

/* a closed loop of n_steps (ilqgb_mpc): host w [B][n_steps][nx] (may be NULL) and log arrays (any may be NULL) of the caller */
typedef struct {
    int n_steps;
    const double *w;
    double *x, *u, *cost;
    int *iterations, *result;
} mpc_t;

/* w and the logs of one closed loop live in the staging buffer, problem-major, so that they go to and from the caller's
   arrays in one copy each; w (the chunk's slice) is uploaded here */
static int ck_mpc_begin(chunk *h, const mpc_t *m, const double *w)
{
    const size_t B = (size_t)h->B, S = (size_t)m->n_steps, nx = (size_t)h->d.nx, nu = (size_t)h->d.nu, ints = (B * S + 1) / 2;
    const size_t n_w = w ? B * S * nx : 0, n_x = m->x ? B * (S + 1) * nx : 0, n_u = m->u ? B * S * nu : 0, n_c = m->cost ? B * S : 0;
    const size_t n_it = m->iterations ? ints : 0, n_res = m->result ? ints : 0;
    double *s;
    if (ilqgk_set_device(h->device)) return failk(h);
    if (h->plant_on && ck_plant_prepare(h)) return -1;   /* here, not between two steps of the loop */
    if (ensure_stage(h, n_w + n_x + n_u + n_c + n_it + n_res)) return -1;
    s = h->d_stage;
    memset(&h->mpc, 0, sizeof h->mpc);
    h->mpc.n_shift = 1;
    h->mpc.set_x0 = 1;
    h->mpc.n_steps = m->n_steps;
    if (w) {
        if (ilqgk_h2d(s, w, sizeof(double) * n_w, h->stream)) return failk(h);
        h->mpc.w = s;
    }
    s += n_w;
    h->mpc.x_log = m->x ? s : NULL;
    s += n_x;
    h->mpc.u_log = m->u ? s : NULL;
    s += n_u;
    h->mpc.cost_log = m->cost ? s : NULL;
    s += n_c;
    h->mpc.it_log = m->iterations ? (int *)s : NULL;
    s += n_it;
    h->mpc.res_log = m->result ? (int *)s : NULL;
    return 0;
}

/* after the solve of step `step`: log it; unless it was the last one, its solution becomes the next step's input */
static int ck_mpc_advance(chunk *h, int step)
{
    h->mpc.step = step;
    h->mpc.plan = step + 1 < h->mpc.n_steps;
    if (launch_advance(h, &h->mpc)) return -1;
    if (h->mpc.plan) {
        h->started = 0;   /* the input has been replaced */
        h->w.tr_off++;    /* the tracks move with the plan: every later launch of this chunk passes the next window */
    }
    return 0;
}

/* the chunk's logs into the caller's arrays (problem `first` of the handle is row 0 of this chunk) */
static int ck_mpc_logs(chunk *h, const mpc_t *m, size_t first)
{
    const size_t B = (size_t)h->B, S = (size_t)m->n_steps, nx = (size_t)h->d.nx, nu = (size_t)h->d.nu;
    const ilqg_mpc_step *a = &h->mpc;
    if (ilqgk_set_device(h->device)) return failk(h);
    if (m->x && ilqgk_d2h(m->x + first * (S + 1) * nx, a->x_log, sizeof(double) * B * (S + 1) * nx, h->stream)) return failk(h);
    if (m->u && ilqgk_d2h(m->u + first * S * nu, a->u_log, sizeof(double) * B * S * nu, h->stream)) return failk(h);
    if (m->cost && ilqgk_d2h(m->cost + first * S, a->cost_log, sizeof(double) * B * S, h->stream)) return failk(h);
    if (m->iterations && ilqgk_d2h(m->iterations + first * S, a->it_log, sizeof(int) * B * S, h->stream)) return failk(h);
    if (m->result && ilqgk_d2h(m->result + first * S, a->res_log, sizeof(int) * B * S, h->stream)) return failk(h);
    return 0;
}

typedef struct {
    long long stride_k, stride_b, stride_i, off;
} lay_t;

static lay_t lay_rec(const chunk *h, int rec, int off) { lay_t l = {(long long)h->Bp * rec, rec, 1, off}; return l; }
static lay_t lay_soa(const chunk *h, int n_i) { lay_t l = {(long long)h->Bp * n_i, 1, h->Bp, 0}; return l; }

static int gather_to_host(chunk *h, const double *src, const double *alt, const int *sel, int n_k, int n_i, lay_t L, double *out)
{
    const size_t n = (size_t)h->B * n_k * n_i;
    if (!n) return 0;
    if (ensure_stage(h, n)) return -1;
    if (ilqgk_launch_gather(src, alt, sel, h->d_stage, h->B, n_k, n_i, L.stride_k, L.stride_b, L.stride_i, L.off, h->stream)) return failk(h);
    h->n_launches++;
    if (ilqgk_d2h(out, h->d_stage, sizeof(double) * n, h->stream)) return failk(h);
    return 0;
}

/* download without intermediate synchronisation: x and u are staged in disjoint halves of the staging buffer */
static int ck_download_async(chunk *h, double *x, double *u, double *cost, int *iterations, int *result, int *n_linesearch)
{
    const size_t B = (size_t)h->B, nxs = B * (h->T + 1) * h->d.nx, nus = B * h->T * h->d.nu;
    if (ilqgk_set_device(h->device)) return failk(h);
    if (ensure_stage(h, nxs + nus)) return -1;
    if (x) {
        const lay_t L = lay_rec(h, h->d.rxu, 0);
        if (ilqgk_launch_gather(h->w.XU[0], h->w.XU[1], h->w.cur, h->d_stage, h->B, h->T + 1, h->d.nx, L.stride_k, L.stride_b, L.stride_i, L.off, h->stream)) return failk(h);
        if (ilqgk_d2h(x, h->d_stage, sizeof(double) * nxs, h->stream)) return failk(h);
        h->n_launches++;
    }
    if (u) {
        const lay_t L = lay_rec(h, h->d.rxu, h->d.nx);
        if (ilqgk_launch_gather(h->w.XU[0], h->w.XU[1], h->w.cur, h->d_stage + nxs, h->B, h->T, h->d.nu, L.stride_k, L.stride_b, L.stride_i, L.off, h->stream)) return failk(h);
        if (ilqgk_d2h(u, h->d_stage + nxs, sizeof(double) * nus, h->stream)) return failk(h);
        h->n_launches++;
    }
    if (cost && ilqgk_d2h(cost, h->w.cost, sizeof(double) * B, h->stream)) return failk(h);
    if (iterations && ilqgk_d2h(iterations, h->w.iterations, sizeof(int) * B, h->stream)) return failk(h);
    if (result && ilqgk_d2h(result, h->w.result, sizeof(int) * B, h->stream)) return failk(h);
    if (n_linesearch && ilqgk_d2h(n_linesearch, h->w.n_ls, sizeof(int) * B, h->stream)) return failk(h);
    return 0;
}

static int ck_download(chunk *h, double *x, double *u, double *cost, int *iterations, int *result, int *n_linesearch)
{
    const size_t B = (size_t)h->B;
    if (ilqgk_set_device(h->device)) return failk(h);
    /* the staging buffer is reused: serialise x and u through the stream (stream order keeps this correct) */
    if (x) {
        if (gather_to_host(h, h->w.XU[0], h->w.XU[1], h->w.cur, h->T + 1, h->d.nx, lay_rec(h, h->d.rxu, 0), x)) return -1;
        if (ilqgk_stream_sync(h->stream)) return failk(h);
    }
    if (u) {
        if (gather_to_host(h, h->w.XU[0], h->w.XU[1], h->w.cur, h->T, h->d.nu, lay_rec(h, h->d.rxu, h->d.nx), u)) return -1;
        if (ilqgk_stream_sync(h->stream)) return failk(h);
    }
    if (cost && ilqgk_d2h(cost, h->w.cost, sizeof(double) * B, h->stream)) return failk(h);
    if (iterations && ilqgk_d2h(iterations, h->w.iterations, sizeof(int) * B, h->stream)) return failk(h);
    if (result && ilqgk_d2h(result, h->w.result, sizeof(int) * B, h->stream)) return failk(h);
    if (n_linesearch && ilqgk_d2h(n_linesearch, h->w.n_ls, sizeof(int) * B, h->stream)) return failk(h);
    if (ilqgk_stream_sync(h->stream)) return failk(h);
    return 0;
}

/* ---- timing -------------------------------------------------------------------------------------------------------------------- */
static ev_pair *timing_begin(chunk *h, int cls)
{
    ev_pair *p;
    if (!(h->flags & ILQGB_TIMING)) return NULL;
    if (h->n_ev == h->cap_ev) {
        const int cap = h->cap_ev ? 2 * h->cap_ev : 256;
        ev_pair *e = (ev_pair *)realloc(h->ev, sizeof(ev_pair) * cap);
        if (!e) return NULL; /* out of host memory: this launch goes untimed */
        h->ev = e;
        h->cap_ev = cap;
    }
    p = &h->ev[h->n_ev];
    if (h->n_ev == h->n_ev_created) {
        if (ilqgk_event_create(&p->start) || ilqgk_event_create(&p->stop)) return NULL;
        h->n_ev_created++;
    }
    h->n_ev++;
    p->cls = cls;
    ilqgk_event_record(p->start, h->stream);
    return p;
}

static void timing_end(chunk *h, ev_pair *p)
{
    if (p) ilqgk_event_record(p->stop, h->stream);
}

static int ck_timing(chunk *h, double *ms, long *launches, int reset)
{
    int i;
    if (ilqgk_set_device(h->device)) return failk(h);
    if (ilqgk_stream_sync(h->stream)) return failk(h);
    for (i = 0; i < h->n_ev; i++) {
        float t = 0.f;
        if (ilqgk_event_elapsed(h->ev[i].start, h->ev[i].stop, &t) == 0) {
            h->t_ms[h->ev[i].cls] += t;
            h->t_n[h->ev[i].cls] += 1;
        }
    }
    h->n_ev = 0;
    for (i = 0; i < TC_N; i++) {
        if (ms) ms[i] = h->t_ms[i];
        if (launches) launches[i] = h->t_n[i];
        if (reset) {
            h->t_ms[i] = 0.0;
            h->t_n[i] = 0;
        }
    }
    return 0;
}

/* ---- the solve ------------------------------------------------------------------------------------------------------------------ */
static int ck_start(chunk *h)
{
    if (ilqgk_set_device(h->device)) return failk(h);
    if (ensure_traces(h)) return -1;
    if (h->flags & ILQGB_TRACE) { /* parity mode: control-law records start from zero like a calloc'ed trajectory */
        int i;
        for (i = 0; i < 2; i++)
            if (ilqgk_memset(h->w.LL[i], 0, sizeof(double) * (size_t)h->T * h->Bp * h->d.rlm, h->stream) ||
                ilqgk_memset(h->w.Ll[i], 0, sizeof(double) * (size_t)h->T * h->Bp * h->d.rls, h->stream))
                return failk(h);
    }
    if (ilqgk_launch_init(&h->w, &h->o, h->params, 7, h->stream)) return failk(h);
    h->n_launches++;
    h->policy_valid = 0;
    h->iter = 0;
    h->started = 1;
    return 0;
}

static int launch_pass(chunk *h, int do_derivs, int do_back, int do_ls)
{
    ev_pair *p;
    h->policy_valid = 0;   /* passes move the trajectories and gains (ck_policy sets it again after its own) */
    if (ensure_traces(h)) return -1;   /* max_iter may have been raised since the solve started */
    if (do_derivs) {
        p = timing_begin(h, TC_DERIVS);
        if (ilqgk_launch_derivs(&h->w, h->params, h->stream)) return failk(h);
        h->n_launches++;
        timing_end(h, p);
    }
    if (do_back) {
        p = timing_begin(h, TC_BACKPASS);
        h->o.bp_latency_build = h->bp_latency >= 0 ? h->bp_latency : (h->total_B <= 40000);
        h->o.cw_lpp = h->cw_lpp;
        /* few problems on the GPU: four lanes per problem (a quarter of the matrix work per lane, box-QP iterations diverge over
           8 problems instead of 32); threshold measured on B200 (scripts/gpu_probe_split.sh) */
        h->o.bp_split = !h->d.bp_split_ok ? 0 : (h->bp_split >= 0 ? (h->bp_split == 4 ? 4 : 0) : (h->total_B <= BP_SPLIT_MAX_B ? 4 : 0));
        h->o.bp_ppw = h->bp_ppw >= 1 ? h->bp_ppw : (h->o.bp_split ? 4 : 32);
        if (h->o.bp_split && h->o.bp_ppw > 8) h->o.bp_ppw = 8;
        if (ilqgk_launch_backpass(&h->w, &h->o, h->params, h->iter, h->stream)) return failk(h);
        h->n_launches++;
        timing_end(h, p);
    }
    if (do_ls) {
        int r;
        if (ilqgk_launch_ls_reset(&h->w, h->stream)) return failk(h);
        {
            /* small batches: one sequential round, then all remaining alphas at once (latency-bound regime);
               large batches: one alpha per launch over the shrinking list of undecided problems (throughput-bound) */
            /* thresholds measured on B200 (scripts/gpu_probe.py with ILQG_LS_TAIL_FROM), by problems resident on the GPU */
            int from = h->ls_tail_from >= 0 ? h->ls_tail_from
                                            : (h->total_B <= 17000 ? 0 : (h->total_B <= 24000 ? 1 : (h->total_B <= 50000 ? 2 : (h->total_B <= 140000 ? 3 : 4))));
            if (from > h->o.n_alpha || h->o.n_alpha - from < 2) from = h->o.n_alpha;
            h->o.ls_tail_from = from;
            h->o.ls_commit_par = h->w.ls_ckpt != NULL;
            for (r = 0; r < from; r++) {
                p = timing_begin(h, TC_LINESEARCH);
                if (ilqgk_launch_ls_round(&h->w, &h->o, h->params, h->iter, r, h->stream)) return failk(h);
                h->n_launches++;
                timing_end(h, p);
            }
            if (from < h->o.n_alpha) {
                p = timing_begin(h, TC_LINESEARCH);
                if (ilqgk_launch_ls_tail(&h->w, &h->o, h->params, h->iter, from, h->stream)) return failk(h);
                h->n_launches += h->o.ls_commit_par ? 3 : 2;
                timing_end(h, p);
            }
        }
        if (ilqgk_has_post()) {
            p = timing_begin(h, TC_POST);
            if (ilqgk_launch_post(&h->w, &h->o, h->params, h->stream)) return failk(h);
            h->n_launches++;
            timing_end(h, p);
        }
    }
    return 0;
}

static int ck_active(chunk *h)
{
    if (ilqgk_set_device(h->device)) return failk(h);
    if (ilqgk_launch_count_active(&h->w, h->d_counter, h->stream)) return failk(h);
    h->n_launches++;
    if (ilqgk_d2h(h->h_counter, h->d_counter, sizeof(int), h->stream)) return failk(h);
    if (ilqgk_stream_sync(h->stream)) return failk(h);
    return *h->h_counter;
}

static int ck_finish(chunk *h)
{
    if (ilqgk_set_device(h->device)) return failk(h);
    /* problems that are still running after max_iter passes: iLQG.c:365-377 */
    if (h->iter >= h->o.max_iter && ilqgk_launch_finalize(&h->w, h->o.max_iter, h->stream)) return failk(h);
    return 0;
}

static long ck_launch_count(const chunk *h) { return h->n_launches; }

static int ck_sync(chunk *h)
{
    if (ilqgk_set_device(h->device)) return failk(h);
    return ilqgk_stream_sync(h->stream) ? failk(h) : 0;
}

static int ck_phase_backpass_once(chunk *h)
{
    int rc;
    if (ilqgk_set_device(h->device)) return failk(h);
    h->o.bp_single = 1;
    rc = launch_pass(h, 0, 1, 0);
    h->o.bp_single = 0;
    return rc;
}

/* ---- feedback policy of a solved batch (see ilqg_b200.h) ---- */
/* calc_derivs(o); back_pass(o) on every problem: the derivative sweep and one backward pass at the final lambda, through the
   solver's own launch sequence (ilqgb_phase_derivs + ilqgb_phase_backpass_once); k_policy_mark reaches the finished problems
   and puts back what that changes */
static int ck_policy(chunk *h)
{
    int rc;
    if (ilqgk_set_device(h->device)) return failk(h);
    if (ilqgk_launch_policy_mark(&h->w, h->d_policy_keep, h->d_policy_ok, 1, h->stream)) return failk(h);
    h->n_launches++;
    h->o.bp_single = 1;
    rc = launch_pass(h, 1, 1, 0);
    h->o.bp_single = 0;
    if (rc) return -1;
    if (ilqgk_launch_policy_mark(&h->w, h->d_policy_keep, h->d_policy_ok, 0, h->stream)) return failk(h);
    h->n_launches++;
    h->policy_valid = 1;
    return 0;
}

/* doubles of the staging buffer one sample of a rollout group needs: x0, cost, final state, ok (as a double), trajectories */
static size_t policy_sample_doubles(const chunk *h, int traj_x, int traj_u)
{
    const size_t nx = (size_t)h->d.nx, nu = (size_t)h->d.nu, T = (size_t)h->T;
    return 2 * nx + 2 + (traj_x ? (T + 1) * nx : 0) + (traj_u ? T * nu : 0);
}

/* samples s0 .. s0+g-1 of every problem of the chunk: inputs in, kernel launched.  The group's arrays sit in the staging buffer,
   [B][g][..] each; a group of all M samples copies straight from the caller's rows, a smaller one is packed on the host. */
typedef struct {
    int M, s0, g;
    const double *x0s;
    double *cost, *x_final, *x, *u;
    int *ok;
} prollout_t;

static void policy_stage_layout(chunk *h, const prollout_t *q, ilqg_policy *r)
{
    const size_t Bg = (size_t)h->B * q->g, nx = (size_t)h->d.nx, T = (size_t)h->T;
    double *s = h->d_stage;
    r->n_samp = q->g;
    r->x0s = s;
    s += Bg * nx;
    r->cost = s;
    s += Bg;
    r->x_final = s;
    s += Bg * nx;
    r->ok = (int *)s;
    s += Bg;
    r->x = q->x ? s : NULL;
    s += q->x ? Bg * (T + 1) * nx : 0;
    r->u = q->u ? s : NULL;
}

/* copy [B][g][n] between the caller's [B][M][n] rows (from sample s0 on) and a packed host buffer */
static void policy_pack(const prollout_t *q, int B, size_t n, const double *src, double *dst, int to_packed)
{
    int b;
    for (b = 0; b < B; b++) {
        const size_t caller = ((size_t)b * q->M + q->s0) * n, packed = (size_t)b * q->g * n;
        if (to_packed) memcpy(dst + packed, src + caller, sizeof(double) * q->g * n);
        else memcpy(dst + caller, src + packed, sizeof(double) * q->g * n);
    }
}

static int ck_policy_rollout_launch(chunk *h, const prollout_t *q, double *tmp)
{
    const size_t Bg = (size_t)h->B * q->g, nx = (size_t)h->d.nx;
    ilqg_policy r;
    const double *table = h->params;
    if (ilqgk_set_device(h->device)) return failk(h);
    memset(&r, 0, sizeof r);
    r.pp = h->w.pp;
    if (h->plant_on) {   /* the plant's effective set: its own entries, the model's elsewhere */
        if (ck_plant_prepare(h)) return -1;
        table = h->plant_params;
        r.pp = h->plant_per ? h->d_plant_eff : NULL;
    }
    r.policy_ok = h->d_policy_ok;
    if (ensure_stage(h, Bg * policy_sample_doubles(h, q->x != NULL, q->u != NULL))) return -1;
    policy_stage_layout(h, q, &r);
    if (q->g == q->M) {
        if (ilqgk_h2d((double *)r.x0s, q->x0s, sizeof(double) * Bg * nx, h->stream)) return failk(h);
    } else {
        policy_pack(q, h->B, nx, q->x0s, tmp, 1);
        if (ilqgk_h2d((double *)r.x0s, tmp, sizeof(double) * Bg * nx, h->stream) || ilqgk_stream_sync(h->stream)) return failk(h);
    }
    if (ilqgk_launch_policy_rollout(&h->w, table, &r, h->stream)) return failk(h);
    h->n_launches++;
    return 0;
}

static int ck_policy_rollout_collect(chunk *h, const prollout_t *q, double *tmp)
{
    const size_t Bg = (size_t)h->B * q->g, nx = (size_t)h->d.nx, nu = (size_t)h->d.nu, T = (size_t)h->T;
    ilqg_policy r;
    if (ilqgk_set_device(h->device)) return failk(h);
    policy_stage_layout(h, q, &r);
    if (q->g == q->M) {
        if (ilqgk_d2h(q->cost, r.cost, sizeof(double) * Bg, h->stream) || ilqgk_d2h(q->x_final, r.x_final, sizeof(double) * Bg * nx, h->stream) ||
            ilqgk_d2h(q->ok, r.ok, sizeof(int) * Bg, h->stream) || (q->x && ilqgk_d2h(q->x, r.x, sizeof(double) * Bg * (T + 1) * nx, h->stream)) ||
            (q->u && ilqgk_d2h(q->u, r.u, sizeof(double) * Bg * T * nu, h->stream)))
            return failk(h);
        return 0;
    }
    {
        /* a group: through the host buffer, one array at a time */
        const double *dsrc[4] = {r.cost, r.x_final, r.x, r.u};
        double *hdst[4] = {q->cost, q->x_final, q->x, q->u};
        const size_t n[4] = {1, nx, (T + 1) * nx, T * nu};
        int i, b;
        for (i = 0; i < 4; i++) {
            if (!hdst[i]) continue;
            if (ilqgk_d2h(tmp, dsrc[i], sizeof(double) * Bg * n[i], h->stream) || ilqgk_stream_sync(h->stream)) return failk(h);
            policy_pack(q, h->B, n[i], tmp, hdst[i], 0);
        }
        if (ilqgk_d2h(tmp, r.ok, sizeof(int) * Bg, h->stream) || ilqgk_stream_sync(h->stream)) return failk(h);
        for (b = 0; b < h->B; b++) memcpy(q->ok + (size_t)b * q->M + q->s0, (const int *)tmp + (size_t)b * q->g, sizeof(int) * q->g);
    }
    return 0;
}

static int ck_policy_eval(chunk *h, int k, const double *x, double *u)
{
    const size_t B = (size_t)h->B, nx = (size_t)h->d.nx, nu = (size_t)h->d.nu;
    if (ilqgk_set_device(h->device)) return failk(h);
    if (ensure_stage(h, B * (nx + nu))) return -1;
    if (ilqgk_h2d(h->d_stage, x, sizeof(double) * B * nx, h->stream) ||
        ilqgk_launch_policy_eval(&h->w, h->params, h->d_policy_ok, h->d_stage, h->d_stage + B * nx, k, h->stream) ||
        ilqgk_d2h(u, h->d_stage + B * nx, sizeof(double) * B * nu, h->stream) || ilqgk_stream_sync(h->stream))
        return failk(h);
    h->n_launches++;
    return 0;
}

static int ck_phase_multipliers(chunk *h, int init)
{
    if (ilqgk_set_device(h->device)) return failk(h);
    if (ilqgk_launch_mult(&h->w, &h->o, h->params, init, h->stream)) return failk(h);
    h->n_launches++;
    h->policy_valid = 0;
    return 0;
}

static int ck_clamp_u(chunk *h, int k, const double *x, double *u)
{
    const size_t B = (size_t)h->B, nx = (size_t)h->d.nx, nu = (size_t)h->d.nu;
    size_t b;
    double *tmp;
    if (ilqgk_set_device(h->device)) return failk(h);
    if (ensure_stage(h, B * (nx + nu))) return -1;
    tmp = (double *)malloc(sizeof(double) * B * (nx + nu));
    if (!tmp) return fail(h, "out of host memory");
    for (b = 0; b < B; b++) {
        memcpy(tmp + b * (nx + nu), x + b * nx, sizeof(double) * nx);
        memcpy(tmp + b * (nx + nu) + nx, u + b * nu, sizeof(double) * nu);
    }
    if (ilqgk_h2d(h->d_stage, tmp, sizeof(double) * B * (nx + nu), h->stream) || ilqgk_launch_clamp(&h->w, h->params, h->d_stage, k, h->stream) ||
        ilqgk_d2h(tmp, h->d_stage, sizeof(double) * B * (nx + nu), h->stream) || ilqgk_stream_sync(h->stream)) {
        free(tmp);
        return failk(h);
    }
    h->n_launches++;
    for (b = 0; b < B; b++) memcpy(u + b * nu, tmp + b * (nx + nu) + nx, sizeof(double) * nu);
    free(tmp);
    return 0;
}

static int ck_eval(chunk *h, int mode, int k, const double *x, const double *u, double *out)
{
    const size_t B = (size_t)h->B, nx = (size_t)h->d.nx, nu = (size_t)h->d.nu, no = (size_t)ilqgk_eval_size(mode);
    size_t b;
    double *tmp;
    if (ilqgk_set_device(h->device)) return failk(h);
    if (!no) return 0;
    if (ensure_stage(h, B * (nx + nu + no))) return -1;
    tmp = (double *)malloc(sizeof(double) * B * (nx + nu));
    if (!tmp) return fail(h, "out of host memory");
    for (b = 0; b < B; b++) {
        memcpy(tmp + b * (nx + nu), x + b * nx, sizeof(double) * nx);
        memcpy(tmp + b * (nx + nu) + nx, u + b * nu, sizeof(double) * nu);
    }
    if (ilqgk_h2d(h->d_stage, tmp, sizeof(double) * B * (nx + nu), h->stream) ||
        ilqgk_launch_eval(&h->w, h->params, h->d_stage, h->d_stage + B * (nx + nu), mode, k, h->stream) ||
        ilqgk_d2h(out, h->d_stage + B * (nx + nu), sizeof(double) * B * no, h->stream) || ilqgk_stream_sync(h->stream)) {
        free(tmp);
        return failk(h);
    }
    h->n_launches++;
    free(tmp);
    return 0;
}

static int ck_phase_derivs(chunk *h) { return ilqgk_set_device(h->device) ? failk(h) : launch_pass(h, 1, 0, 0); }
static int ck_phase_backpass(chunk *h) { return ilqgk_set_device(h->device) ? failk(h) : launch_pass(h, 0, 1, 0); }
static int ck_phase_linesearch(chunk *h) { return ilqgk_set_device(h->device) ? failk(h) : launch_pass(h, 0, 0, 1); }

/* ---- read-back -------------------------------------------------------------------------------------------------------------------- */
typedef struct {
    double *scal;             /* per-problem scalar array, or */
    double *src, *alt;        /* trajectory-like field (alt = second buffer, chosen by sel) */
    const int *sel;
    int n_k, n_i;
    lay_t L;
} field_t;

static int find_field(chunk *h, const char *f, field_t *o)
{
    ilqg_work *w = &h->w;
    const ilqgk_dims_t *d = &h->d;
    memset(o, 0, sizeof *o);
    if (!strcmp(f, "cost")) o->scal = w->cost;
    else if (!strcmp(f, "new_cost")) o->scal = w->new_cost;
    else if (!strcmp(f, "dcost")) o->scal = w->dcost;
    else if (!strcmp(f, "expected")) o->scal = w->expected;
    else if (!strcmp(f, "lambda")) o->scal = w->lambda;
    else if (!strcmp(f, "dlambda")) o->scal = w->dlambda;
    else if (!strcmp(f, "g_norm")) o->scal = w->g_norm;
    else if (!strcmp(f, "dV0")) o->scal = w->dV0;
    else if (!strcmp(f, "dV1")) o->scal = w->dV1;
    else if (!strcmp(f, "w_pen_l")) o->scal = w->w_pen_l;
    else if (!strcmp(f, "w_pen_f")) o->scal = w->w_pen_f;
    if (o->scal) return 0;
    if (!strcmp(f, "x")) { o->src = w->XU[0]; o->alt = w->XU[1]; o->sel = w->cur; o->n_k = h->T + 1; o->n_i = d->nx; o->L = lay_rec(h, d->rxu, 0); }
    else if (!strcmp(f, "u")) { o->src = w->XU[0]; o->alt = w->XU[1]; o->sel = w->cur; o->n_k = h->T; o->n_i = d->nu; o->L = lay_rec(h, d->rxu, d->nx); }
    else if (!strcmp(f, "x_cand")) { o->src = w->XU[1]; o->alt = w->XU[0]; o->sel = w->cur; o->n_k = h->T + 1; o->n_i = d->nx; o->L = lay_rec(h, d->rxu, 0); }
    else if (!strcmp(f, "u_cand")) { o->src = w->XU[1]; o->alt = w->XU[0]; o->sel = w->cur; o->n_k = h->T; o->n_i = d->nu; o->L = lay_rec(h, d->rxu, d->nx); }
    else if (!strcmp(f, "x0")) { o->src = w->x0; o->n_k = 1; o->n_i = d->nx; o->L = lay_soa(h, d->nx); }
    else if (!strcmp(f, "l")) { o->src = w->Ll[0]; o->alt = w->Ll[1]; o->sel = w->cur; o->n_k = h->T; o->n_i = d->nu; o->L = lay_rec(h, d->rls, 0); }
    else if (!strcmp(f, "L")) { o->src = w->LL[0]; o->alt = w->LL[1]; o->sel = w->cur; o->n_k = h->T; o->n_i = d->nu * d->nx; o->L = lay_rec(h, d->rlm, 0); }
    else if (!strcmp(f, "v1")) { o->src = w->V1; o->n_k = h->T; o->n_i = d->nv1; o->L = d->coop ? lay_rec(h, d->nv1, 0) : lay_soa(h, o->n_i); }
    else if (!strcmp(f, "v2") && d->full_ddp) { o->src = w->V2; o->n_k = h->T; o->n_i = d->nv2; o->L = d->coop ? lay_rec(h, d->nv2, 0) : lay_soa(h, o->n_i); }
    else if (!strcmp(f, "fd")) { o->src = w->FD; o->n_k = 1; o->n_i = d->nx + d->nqxx; o->L = lay_soa(h, o->n_i); }
    else if (!strcmp(f, "mu_f")) { o->src = w->muF; o->n_k = 1; o->n_i = d->n_mu_f; o->L = lay_soa(h, o->n_i); }
    else if (!strcmp(f, "last_f")) { o->src = w->lastF; o->n_k = 1; o->n_i = d->n_mu_f; o->L = lay_soa(h, o->n_i); }
    else if (!strcmp(f, "mu_r")) { o->src = w->muR; o->n_k = h->T; o->n_i = d->n_mu_r; o->L = lay_soa(h, o->n_i); }
    else if (!strcmp(f, "last_r")) { o->src = w->lastR; o->n_k = h->T; o->n_i = d->n_mu_r; o->L = lay_soa(h, o->n_i); }
    else if (!strcmp(f, "tr_lambda") && w->tr_lambda) { o->src = w->tr_lambda; o->n_k = h->trace_cap; o->n_i = 1; o->L = lay_soa(h, 1); }
    else if (!strcmp(f, "tr_newcost") && w->tr_newcost) { o->src = w->tr_newcost; o->n_k = h->trace_cap; o->n_i = 1; o->L = lay_soa(h, 1); }
    else if (!strcmp(f, "tr_z") && w->tr_z) { o->src = w->tr_z; o->n_k = h->trace_cap; o->n_i = 1; o->L = lay_soa(h, 1); }
    else return fail(h, "unknown field");
    return 0;
}

static long ck_get(chunk *h, const char *f, double *out)
{
    const size_t B = (size_t)h->B;
    field_t fd;
    if (ilqgk_set_device(h->device)) return failk(h);
    if (!strcmp(f, "dense")) { /* computed field: the dense per-step derivative record, rebuilt on the device */
        const size_t n = B * (size_t)h->T * (size_t)ilqgk_dense_size();
        if (ensure_stage(h, n)) return -1;
        if (ilqgk_launch_dense(&h->w, h->params, h->d_stage, h->stream) || ilqgk_d2h(out, h->d_stage, sizeof(double) * n, h->stream) ||
            ilqgk_stream_sync(h->stream))
            return failk(h);
        h->n_launches++;
        return (long)n;
    }
    if (!strcmp(f, "plant")) { /* computed field: the effective plant parameter set of every problem [B][npf] */
        const size_t npf = (size_t)h->d.npf;
        size_t b;
        if (ck_plant_prepare(h)) return -1;
        if (!h->plant_per) {
            for (b = 0; b < B; b++) memcpy(out + b * npf, h->plant_params, sizeof(double) * npf);
            return (long)(B * npf);
        }
        if (gather_to_host(h, h->d_plant_eff, NULL, NULL, 1, h->d.npf, lay_soa(h, h->d.npf), out)) return -1;
        if (ilqgk_stream_sync(h->stream)) return failk(h);
        return (long)(B * npf);
    }
    if (find_field(h, f, &fd)) return -1;
    if (fd.scal) {
        if (ilqgk_d2h(out, fd.scal, sizeof(double) * B, h->stream) || ilqgk_stream_sync(h->stream)) return failk(h);
        return (long)B;
    }
    if (gather_to_host(h, fd.src, fd.alt, fd.sel, fd.n_k, fd.n_i, fd.L, out)) return -1;
    if (ilqgk_stream_sync(h->stream)) return failk(h);
    return (long)(B * fd.n_k * fd.n_i);
}

/* host -> device write of one field (same names and shapes as ck_get) */
static long ck_put(chunk *h, const char *f, const double *in)
{
    const size_t B = (size_t)h->B;
    field_t fd;
    size_t n;
    if (ilqgk_set_device(h->device)) return failk(h);
    if (find_field(h, f, &fd)) return -1;
    h->policy_valid = 0;
    if (fd.scal) {
        if (ilqgk_h2d(fd.scal, in, sizeof(double) * B, h->stream) || ilqgk_stream_sync(h->stream)) return failk(h);
        return (long)B;
    }
    n = B * fd.n_k * fd.n_i;
    if (!n) return 0;
    if (ensure_stage(h, n)) return -1;
    if (ilqgk_h2d(h->d_stage, in, sizeof(double) * n, h->stream)) return failk(h);
    if (ilqgk_launch_scatter(h->d_stage, fd.src, fd.alt, fd.sel, h->B, fd.n_k, fd.n_i, fd.L.stride_k, fd.L.stride_b, fd.L.stride_i, fd.L.off, h->stream)) return failk(h);
    h->n_launches++;
    if (ilqgk_stream_sync(h->stream)) return failk(h);
    return (long)n;
}

static long ck_get_int(chunk *h, const char *f, int *out)
{
    const ilqg_work *w = &h->w;
    const size_t B = (size_t)h->B, Bp = (size_t)h->Bp;
    const int *scal = NULL, *arr = NULL;
    size_t n_k = 0;
    if (ilqgk_set_device(h->device)) return failk(h);
    if (!strcmp(f, "iterations")) scal = w->iterations;
    else if (!strcmp(f, "result")) scal = w->result;
    else if (!strcmp(f, "status")) scal = w->status;
    else if (!strcmp(f, "n_linesearch")) scal = w->n_ls;
    else if (!strcmp(f, "n_backpass")) scal = w->n_bp;
    else if (!strcmp(f, "cur")) scal = w->cur;
    else if (!strcmp(f, "n_derivs")) scal = w->n_dv;
    else if (!strcmp(f, "n_rollouts")) scal = w->n_roll;
    else if (!strcmp(f, "n_tails")) scal = w->n_tail;
    else if (!strcmp(f, "bp_done")) scal = w->bp_done;
    else if (!strcmp(f, "deriv_fail")) scal = w->deriv_fail;
    else if (!strcmp(f, "policy_ok")) scal = h->d_policy_ok;
    {
        /* test hooks: the kernel variant the last backward pass and line search of this chunk ran with.  bp_split: lanes per
           problem of the small-batch backward pass (4) or 0; cw_lpp: lanes per problem of the warp-cooperative backward pass, 0
           for problems that do not use it; bp_latency: register build of k_backpass; ls_tail_from: sequential rounds before
           the parallel-alpha tail (n_alpha = no tail); ls_commit_par: checkpointed segment-parallel commit (1) or sequential */
        int v = 0, is_hook = 1;
        size_t b;
        if (!strcmp(f, "bp_split")) v = h->o.bp_split;
        else if (!strcmp(f, "cw_lpp")) v = h->d.coop ? h->o.cw_lpp : 0;
        else if (!strcmp(f, "bp_latency")) v = h->o.bp_latency_build;
        else if (!strcmp(f, "ls_tail_from")) v = h->o.ls_tail_from;
        else if (!strcmp(f, "ls_commit_par")) v = h->o.ls_commit_par;
        else is_hook = 0;
        if (is_hook) {
            for (b = 0; b < B; b++) out[b] = v;
            return (long)B;
        }
    }
    if (scal) {
        if (ilqgk_d2h(out, scal, sizeof(int) * B, h->stream) || ilqgk_stream_sync(h->stream)) return failk(h);
        return (long)B;
    }
    if (!strcmp(f, "tr_alpha") && w->tr_alpha) { arr = w->tr_alpha; n_k = (size_t)h->trace_cap; }
    else if (!strcmp(f, "tr_clamp") && w->tr_clamp) { arr = w->tr_clamp; n_k = (size_t)h->T; }
    else return fail(h, "unknown field");
    {
        /* small, test-only path: copy [n_k][Bp] and transpose on the host */
        int *tmp = (int *)malloc(sizeof(int) * n_k * Bp);
        size_t b, k;
        if (!tmp) return fail(h, "out of host memory");
        if (ilqgk_d2h(tmp, arr, sizeof(int) * n_k * Bp, h->stream) || ilqgk_stream_sync(h->stream)) {
            free(tmp);
            return failk(h);
        }
        for (b = 0; b < B; b++)
            for (k = 0; k < n_k; k++) out[b * n_k + k] = tmp[k * Bp + b];
        free(tmp);
        return (long)(B * n_k);
    }
}


static long ck_put_int(chunk *h, const char *f, const int *in)
{
    const size_t B = (size_t)h->B;
    int *dst = NULL;
    if (ilqgk_set_device(h->device)) return failk(h);
    if (!strcmp(f, "cur")) dst = h->w.cur;
    else if (!strcmp(f, "status")) dst = h->w.status;
    else if (!strcmp(f, "new_deriv")) dst = h->w.new_deriv;
    else if (!strcmp(f, "deriv_fail")) dst = h->w.deriv_fail;
    else if (!strcmp(f, "bp_done")) dst = h->w.bp_done;
    else return fail(h, "unknown field");
    h->policy_valid = 0;
    if (ilqgk_h2d(dst, in, sizeof(int) * B, h->stream) || ilqgk_stream_sync(h->stream)) return failk(h);
    return (long)B;
}

/* start of a solve on imported state (nominal trajectory, cost, multipliers already on the device): only the first
   lines of iLQG() run (iLQG.c:226-237) -- used by the single-problem drop-in iLQG(tOptSet*) */
static int ck_begin(chunk *h)
{
    if (ilqgk_set_device(h->device)) return failk(h);
    if (ensure_traces(h)) return -1;
    if (ilqgk_launch_init(&h->w, &h->o, h->params, 4, h->stream)) return failk(h);
    h->n_launches++;
    h->policy_valid = 0;
    h->iter = 0;
    h->started = 1;
    return 0;
}

static int ck_rollout(chunk *h, double alpha, int cost_only)
{
    if (ilqgk_set_device(h->device)) return failk(h);
    if (ilqgk_launch_rollout(&h->w, h->params, alpha, cost_only, h->stream)) return failk(h);
    h->n_launches++;
    h->policy_valid = 0;
    return 0;
}

/* =====================================================================================================================
 * Public handle: the batch is split into contiguous chunks, each a complete single-stream solver (above) on its own
 * CUDA stream.  Chunks are independent (problems never interact), so the GPU overlaps the latency-bound tails of
 * one chunk (late line-search rounds with few undecided problems) with the wide kernels of another, and uploads /
 * downloads of one chunk with the compute of the others.  Work enqueued by one API call is ordered in the handle's
 * main stream: chunk streams fork from it at entry and join it at exit.
 *
 * A handle may span several GPUs (ilqgb_create_multi): the batch is cut into one contiguous shard per device
 * (SURVEY 8e: no exchange step, one final host-side gather) and every shard into chunks as above; one host thread
 * drives all devices, which works because nothing below ever blocks on a single chunk.
 * ===================================================================================================================== */
#define MAX_CHUNKS 64
#define MAX_DEVICES 16
struct ilqgb_handle {
    int n, device, B, T, flags;
    int n_dev, devices[MAX_DEVICES];
    chunk *c[MAX_CHUNKS];
    int first[MAX_CHUNKS];
    void *stream;      /* main stream (caller's or owned), on devices[0] */
    int owns_stream;
    void *ev_fork, *ev_join[MAX_CHUNKS];
    int e2e_prio, e2e_stagger;   /* end-to-end solve: chunk streams with descending priority; start gate in passes */
    ilqgk_dims_t d;
    int tr_off;        /* window offset of the parameter tracks (every chunk's w.tr_off between two calls) */
    char err[256];
};

static int auto_chunks(int batch)
{
    /* measured on B200 (scripts/gpu_probe_e2e.py, car, 20 passes, 262 144 problems; resident s / end-to-end s): 2 chunks 0.656 / 0.763,
       4 chunks 0.645 / 0.711, 8 chunks 0.673 / 0.718, 16 chunks 0.679 / 0.720 (end to end on prioritised streams; with equal
       priorities 4 chunks 0.729, 8 chunks 0.734).  32 768 problems: 1 chunk 0.121 / 0.142, 2 chunks 0.118-0.120 / 0.133, 4 chunks
       0.119-0.121 / 0.132-0.134, 8 chunks 0.131 / 0.138.  So: chunks of about 65 536 problems, at most four, and two from 16 384
       problems on, so that an end-to-end solve has something to overlap its copies with. */
    int n = batch / 65536;
    if (n < 2) n = batch >= 16384 ? 2 : 1;
    if (n > 4) n = 4;
    return n;
}

static int hfail(ilqgb_handle *h, const chunk *c)
{
    snprintf(h->err, sizeof h->err, "%s", c ? c->err : ilqgk_last_error());
    return -1;
}

static int fork_streams(ilqgb_handle *h)
{
    int i;
    if (h->n == 1 && h->c[0]->stream == h->stream) return 0;
    if (ilqgk_set_device(h->device)) return hfail(h, NULL);
    if (ilqgk_event_record(h->ev_fork, h->stream)) return hfail(h, NULL);
    for (i = 0; i < h->n; i++) {
        if (ilqgk_set_device(h->c[i]->device)) return hfail(h, NULL);
        if (ilqgk_stream_wait_event(h->c[i]->stream, h->ev_fork)) return hfail(h, NULL);
    }
    return 0;
}

static int join_streams(ilqgb_handle *h)
{
    int i;
    if (h->n == 1 && h->c[0]->stream == h->stream) return 0;
    for (i = 0; i < h->n; i++) {
        if (ilqgk_set_device(h->c[i]->device)) return hfail(h, NULL);
        if (ilqgk_event_record(h->ev_join[i], h->c[i]->stream)) return hfail(h, NULL);
    }
    if (ilqgk_set_device(h->device)) return hfail(h, NULL);
    for (i = 0; i < h->n; i++)
        if (ilqgk_stream_wait_event(h->stream, h->ev_join[i])) return hfail(h, NULL);
    return 0;
}

const char *ilqgb_last_error(const ilqgb_handle *h) { return h ? h->err : g_create_err; }

ilqgb_handle *ilqgb_create_multi(int n_devices, const int *devices, int batch, int n_hor, int flags, void *stream)
{
    ilqgb_handle *h;
    int d, n_req = (flags >> 8) & 0xff, n_total = 0;
    if (batch < 1 || n_hor < 1) {
        fail_create("batch and n_hor must be >= 1");
        return NULL;
    }
    if (n_devices < 1 || n_devices > MAX_DEVICES) {
        fail_create("n_devices out of range");
        return NULL;
    }
    if (ilqgk_device_count() < 1) {
        fail_create("no CUDA device available: this library has no CPU fallback");
        return NULL;
    }
    for (d = 0; d < n_devices; d++)
        if ((devices ? devices[d] : d) < 0 || (devices ? devices[d] : d) >= ilqgk_device_count()) {
            fail_create("device index out of range");
            return NULL;
        }
    if (n_devices > batch) n_devices = batch;
    if (ilqgk_set_device(devices ? devices[0] : 0)) {
        fail_create(ilqgk_last_error());
        return NULL;
    }
    h = (ilqgb_handle *)calloc(1, sizeof *h);
    if (!h) {
        fail_create("out of host memory");
        return NULL;
    }
    h->n_dev = n_devices;
    for (d = 0; d < n_devices; d++) h->devices[d] = devices ? devices[d] : d;
    h->device = h->devices[0];
    h->B = batch; h->T = n_hor; h->flags = flags;
    h->e2e_prio = env_int("ILQG_E2E_PRIO", 1);
    h->e2e_stagger = env_int("ILQG_E2E_STAGGER", 0);
    ilqgk_dims(&h->d);
    if (stream) {
        h->stream = stream;
    } else {
        if (ilqgk_stream_create(&h->stream)) { fail_create(ilqgk_last_error()); free(h); return NULL; }
        h->owns_stream = 1;
    }
    for (d = 0; d < n_devices; d++) {
        /* contiguous shard of device d, then its chunks (sizes are multiples of a warp; the final chunk count is fixed
           before any chunk is created, so a single chunk runs on the handle's own stream) */
        const int sfirst = (int)((long long)batch * d / n_devices), scount = (int)((long long)batch * (d + 1) / n_devices) - sfirst;
        int n = n_req ? n_req : auto_chunks(scount), per, i, made = 0;
        if (n > scount) n = scount;
        per = ((scount + n - 1) / n + 31) / 32 * 32;
        n = (scount + per - 1) / per;
        if (n_total + n > MAX_CHUNKS) n = MAX_CHUNKS - n_total;
        if (n < 1) { fail_create("too many chunks"); ilqgb_destroy(h); return NULL; }
        per = ((scount + n - 1) / n + 31) / 32 * 32;
        for (i = 0; i < n; i++) {
            const int first = i * per;
            const int cnt = scount - first < per ? scount - first : per;
            chunk *c;
            if (cnt <= 0) break;
            c = ck_create(h->devices[d], cnt, n_hor, flags & 0xff, (n == 1 && n_devices == 1) ? h->stream : NULL, i, n);
            if (!c) { ilqgb_destroy(h); return NULL; }
            c->total_B = scount;
            h->first[n_total + made] = sfirst + first;
            h->c[n_total + made] = c;
            made++;
        }
        n_total += made;
    }
    h->n = n_total;
    if (ilqgk_set_device(h->device) || ilqgk_event_create_notiming(&h->ev_fork)) { fail_create(ilqgk_last_error()); ilqgb_destroy(h); return NULL; }
    for (d = 0; d < h->n; d++)
        if (ilqgk_set_device(h->c[d]->device) || ilqgk_event_create_notiming(&h->ev_join[d])) { fail_create(ilqgk_last_error()); ilqgb_destroy(h); return NULL; }
    ilqgk_set_device(h->device);
    return h;
}

ilqgb_handle *ilqgb_create(int device, int batch, int n_hor, int flags, void *stream)
{
    if (device < 0) {
        fail_create("device index out of range");
        return NULL;
    }
    return ilqgb_create_multi(1, &device, batch, n_hor, flags, stream);
}

void ilqgb_destroy(ilqgb_handle *h)
{
    int i;
    if (!h) return;
    for (i = 0; i < MAX_CHUNKS; i++) {
        if (h->c[i]) ilqgk_set_device(h->c[i]->device);
        if (h->ev_join[i]) ilqgk_event_destroy(h->ev_join[i]);
        if (h->c[i]) ck_destroy(h->c[i]);
    }
    ilqgk_set_device(h->device);
    if (h->ev_fork) ilqgk_event_destroy(h->ev_fork);
    if (h->owns_stream && h->stream) ilqgk_stream_destroy(h->stream);
    free(h);
}

int ilqgb_devices(const ilqgb_handle *h) { return h->n_dev; }

void ilqgb_standard_parameters(ilqgb_handle *h) { int i; for (i = 0; i < h->n; i++) ck_standard_parameters(h->c[i]); }

const char *ilqgb_set_opt(ilqgb_handle *h, const char *name, const double *value, int n)
{
    int i;
    const char *msg = ilqgb_validate_opt(name, value, n);
    if (msg) return msg;
    for (i = 0; i < h->n; i++) ck_set_opt(h->c[i], name, value, n);
    return NULL;
}

int ilqgb_set_param(ilqgb_handle *h, int index, const double *value, int n)
{
    int i;
    for (i = 0; i < h->n; i++)
        if (ck_set_param(h->c[i], index, value, n)) return hfail(h, h->c[i]);
    return 0;
}

int ilqgb_set_param_batch(ilqgb_handle *h, int index, const double *value, int n)
{
    int i;
    for (i = 0; i < h->n; i++)
        if (ck_set_param_batch(h->c[i], index, value + (size_t)h->first[i] * n, n)) return hfail(h, h->c[i]);
    return 0;
}

/* ---- time-indexed parameter tracks (see ilqg_b200.h) ---- */
/* length of the shortest track, 0 without tracks (every chunk holds the same tracks) */
static int track_min_len(const ilqgb_handle *h)
{
    const chunk *c = h->c[0];
    int j, m = 0;
    for (j = 0; j < 16; j++)
        if (c->d_tr[j] && (!m || c->tr_len[j] < m)) m = c->tr_len[j];
    return m;
}

/* a window starting at `off` lies inside every track */
static int window_fits(const ilqgb_handle *h, long long off)
{
    const int m = track_min_len(h);
    return !m || off + h->T + 1 <= m;
}

static void set_track_offset(ilqgb_handle *h, int off)
{
    int i;
    h->tr_off = off;
    for (i = 0; i < h->n; i++) h->c[i]->w.tr_off = off;
}

int ilqgb_set_param_track(ilqgb_handle *h, int index, const double *value, int len)
{
    int i, kidx;
    const int off = track_min_len(h) ? h->tr_off : 0;
    if (index < 0 || index >= ilqgk_param_count()) { snprintf(h->err, sizeof h->err, "parameter index out of range"); return -1; }
    if (ilqgk_param_size(index) != -1) { snprintf(h->err, sizeof h->err, "only [k]-indexed parameters have tracks"); return -1; }
    if (!value) { snprintf(h->err, sizeof h->err, "no track values"); return -1; }
    if ((long long)len < (long long)off + h->T + 1) {
        snprintf(h->err, sizeof h->err, "track too short: len >= offset + n_hor + 1 = %lld expected", (long long)off + h->T + 1);
        return -1;
    }
    kidx = kp_index(index);
    set_track_offset(h, off);
    for (i = 0; i < h->n; i++)
        if (ck_set_param_track(h->c[i], kidx, value + (size_t)h->first[i] * len, len)) return hfail(h, h->c[i]);
    return 0;
}

int ilqgb_set_track_offset(ilqgb_handle *h, int offset)
{
    if (offset < 0) { snprintf(h->err, sizeof h->err, "the track offset must be >= 0"); return -1; }
    if (!window_fits(h, offset)) { snprintf(h->err, sizeof h->err, "offset + n_hor + 1 exceeds the length of a track"); return -1; }
    set_track_offset(h, offset);
    return 0;
}

int ilqgb_track_offset(const ilqgb_handle *h) { return h->tr_off; }

/* ---- plant of the closed loops (see ilqg_b200.h) ---- */
static int plant_param_ok(ilqgb_handle *h, int index, const double *value, int n)
{
    const char *msg = NULL;
    if (index < 0 || index >= ilqgk_param_count()) msg = "parameter index out of range";
    else if (ilqgk_param_size(index) == -1) msg = "[k]-indexed parameters of the plant are the model's: they cannot be set";
    else if (n != ilqgk_param_size(index)) msg = "wrong parameter length";
    else if (!value) msg = "no parameter values";
    if (msg) snprintf(h->err, sizeof h->err, "%s", msg);
    return !msg;
}

int ilqgb_set_plant_param(ilqgb_handle *h, int index, const double *value, int n)
{
    int i;
    if (!plant_param_ok(h, index, value, n)) return -1;
    for (i = 0; i < h->n; i++) ck_set_plant_param(h->c[i], index, value, n);
    return 0;
}

int ilqgb_set_plant_param_batch(ilqgb_handle *h, int index, const double *value, int n)
{
    int i;
    if (!plant_param_ok(h, index, value, n)) return -1;
    for (i = 0; i < h->n; i++)
        if (ck_set_plant_param_batch(h->c[i], index, value + (size_t)h->first[i] * n, n)) return hfail(h, h->c[i]);
    return 0;
}

int ilqgb_set_plant_substeps(ilqgb_handle *h, int n_sub)
{
    int i;
    if (n_sub < 1 || n_sub > 64) { snprintf(h->err, sizeof h->err, "n_sub must be in 1..64"); return -1; }
    for (i = 0; i < h->n; i++) {
        h->c[i]->plant_n_sub = n_sub;
        h->c[i]->plant_on = 1;
    }
    return 0;
}

int ilqgb_clear_plant(ilqgb_handle *h)
{
    int i;
    for (i = 0; i < h->n; i++) ck_clear_plant(h->c[i]);
    return 0;
}

int ilqgb_upload(ilqgb_handle *h, const double *x0, const double *u_nom)
{
    int i;
    if (fork_streams(h)) return -1;
    for (i = 0; i < h->n; i++)
        if (ck_upload(h->c[i], x0 + (size_t)h->first[i] * h->d.nx, u_nom + (size_t)h->first[i] * h->T * h->d.nu)) return hfail(h, h->c[i]);
    return join_streams(h);
}

int ilqgb_download(ilqgb_handle *h, double *x, double *u, double *cost, int *iterations, int *result, int *n_linesearch)
{
    int i;
    if (fork_streams(h)) return -1;
    for (i = 0; i < h->n; i++) {
        const size_t f = (size_t)h->first[i];
        if (ck_download(h->c[i], x ? x + f * (h->T + 1) * h->d.nx : NULL, u ? u + f * h->T * h->d.nu : NULL, cost ? cost + f : NULL,
                        iterations ? iterations + f : NULL, result ? result + f : NULL, n_linesearch ? n_linesearch + f : NULL))
            return hfail(h, h->c[i]);
    }
    return join_streams(h);
}

int ilqgb_start(ilqgb_handle *h)
{
    int i;
    if (fork_streams(h)) return -1;
    for (i = 0; i < h->n; i++)
        if (ck_start(h->c[i])) return hfail(h, h->c[i]);
    return join_streams(h);
}

int ilqgb_active(ilqgb_handle *h)
{
    int i, tot = 0;
    for (i = 0; i < h->n; i++) {
        const int a = ck_active(h->c[i]);
        if (a < 0) return hfail(h, h->c[i]);
        tot += a;
    }
    return tot;
}

/* passes of the loop for every chunk in lock step (the stepwise API: a caller can look at the state between calls) */
int ilqgb_iterate(ilqgb_handle *h, int n_passes)
{
    int done = 0, i;
    for (i = 0; i < h->n; i++)
        if (!h->c[i]->started) { snprintf(h->err, sizeof h->err, "ilqgb_start has not been called"); return -1; }
    if (fork_streams(h)) return -1;
    while (done < n_passes) {
        int launched = 0;
        for (i = 0; i < h->n; i++) {   /* issue pass p of every chunk before pass p+1 of any: streams advance together */
            chunk *c = h->c[i];
            if (c->iter >= c->o.max_iter) continue;
            if (ilqgk_set_device(c->device)) return hfail(h, NULL);
            if (launch_pass(c, 1, 1, 1)) return hfail(h, c);
            c->iter++;
            launched = 1;
        }
        if (!launched) break;
        done++;
        if (done % ACTIVE_CHECK_EVERY == 0 && done < n_passes) {
            const int a = ilqgb_active(h);
            if (a < 0) return -1;
            if (a == 0) break;
        }
    }
    if (join_streams(h)) return -1;
    return done;
}

int ilqgb_finish(ilqgb_handle *h)
{
    int i;
    if (fork_streams(h)) return -1;
    for (i = 0; i < h->n; i++)
        if (ck_finish(h->c[i])) return hfail(h, h->c[i]);
    return join_streams(h);
}

/* ---- asynchronous solve engine -----------------------------------------------------------------------------------------
 * Every chunk runs its whole solve (optionally framed by its upload and its download) on its own stream; the host
 * never waits for a particular chunk.  Passes are issued in blocks of ENGINE_BLOCK per chunk, at most ENGINE_LOOKAHEAD
 * blocks ahead of the last block known to have completed; each block ends with a count of the problems still
 * running, copied to pinned memory and polled with cudaEventQuery, so a chunk whose problems have all finished stops
 * being issued (ragged convergence) without a host synchronisation.
 * End to end (`io`): uploads are queued first, in chunk order; with e2e_prio the chunk streams carry descending
 * priorities, so the chunks FINISH one after the other instead of all at once and the result copies of chunk i
 * overlap the passes of chunks i+1.. (the copy engines and both PCIe directions stay busy while the SMs do);
 * e2e_stagger additionally holds chunk i back until chunk i-1 of its device has issued that many passes. */
typedef struct {
    const double *x0, *u_nom;
    double *x, *u, *cost;
    int *iterations, *result, *n_linesearch;
} io_t;

static int engine_poll(chunk *c)
{
    while (c->poll_seen < c->poll_issued) {
        const int slot = c->poll_seen % POLL_RING;
        const int q = ilqgk_event_query(c->ev_poll[slot]);
        if (q < 0) return failk(c);
        if (q == 0) break;
        if (c->h_poll[slot] == 0) c->stop = 1;
        c->poll_seen++;
    }
    return 0;
}

static int run_engine(ilqgb_handle *h, const io_t *io, const mpc_t *mpc)
{
    int i, remaining, rc = 0;
    const int prio = io && h->e2e_prio && h->n > 1;
    struct timespec nap = {0, 20000};
    if (fork_streams(h)) return -1;
    if (prio) { /* the end-to-end solve runs on prioritised streams; they fork from the main stream like the others */
        for (i = 0; i < h->n; i++) {
            chunk *c = h->c[i];
            if (ilqgk_set_device(c->device)) return hfail(h, NULL);
            if (!c->stream_io && ilqgk_stream_create_prio(&c->stream_io, c->prio_rank, c->prio_n)) return hfail(h, NULL);
            if (ilqgk_stream_wait_event(c->stream_io, h->ev_fork)) return hfail(h, NULL);
            c->stream = c->stream_io;
        }
    }
    for (i = 0; i < h->n; i++) {
        chunk *c = h->c[i];
        c->poll_issued = c->poll_seen = c->stop = c->phase = c->gate_recorded = c->mpc_step = 0;
        if (io && ck_upload(c, io->x0 + (size_t)h->first[i] * h->d.nx, io->u_nom + (size_t)h->first[i] * h->T * h->d.nu)) { rc = hfail(h, c); goto out; }
        if (mpc && ck_mpc_begin(c, mpc, mpc->w ? mpc->w + (size_t)h->first[i] * mpc->n_steps * h->d.nx : NULL)) { rc = hfail(h, c); goto out; }
    }
    remaining = h->n;
    while (remaining > 0) {
        int progressed = 0;
        for (i = 0; i < h->n; i++) {
            chunk *c = h->c[i];
            const int max_iter = c->o.max_iter;
            if (c->phase == 3) continue;
            if (ilqgk_set_device(c->device)) { rc = hfail(h, NULL); goto out; }
            if (c->phase == 0) { /* start, possibly gated on the previous chunk of the same device */
                if (io && h->e2e_stagger > 0 && c->prio_rank > 0) {
                    chunk *prev = h->c[i - 1];
                    if (!prev->gate_recorded) continue;
                    if (ilqgk_stream_wait_event(c->stream, prev->ev_gate)) { rc = hfail(h, NULL); goto out; }
                }
                if (ck_start(c)) { rc = hfail(h, c); goto out; }
                c->phase = 1;
                progressed = 1;
            }
            if (engine_poll(c)) { rc = hfail(h, c); goto out; }
            if (c->phase == 1 && !c->stop && c->iter < max_iter && c->poll_issued - c->poll_seen < ENGINE_LOOKAHEAD) {
                int n = max_iter - c->iter < ENGINE_BLOCK ? max_iter - c->iter : ENGINE_BLOCK;
                while (n-- > 0) {
                    if (launch_pass(c, 1, 1, 1)) { rc = hfail(h, c); goto out; }
                    c->iter++;
                    if (io && h->e2e_stagger > 0 && !c->gate_recorded && c->iter >= h->e2e_stagger) {
                        if (ilqgk_event_record(c->ev_gate, c->stream)) { rc = hfail(h, NULL); goto out; }
                        c->gate_recorded = 1;
                    }
                }
                if (c->iter < max_iter) {
                    const int slot = c->poll_issued % POLL_RING;
                    if (ilqgk_launch_count_active(&c->w, c->d_counter, c->stream) || ilqgk_d2h(&c->h_poll[slot], c->d_counter, sizeof(int), c->stream) ||
                        ilqgk_event_record(c->ev_poll[slot], c->stream)) { rc = hfail(h, NULL); goto out; }
                    c->n_launches++;
                    c->poll_issued++;
                }
                progressed = 1;
            }
            if (c->phase == 1 && (c->stop || c->iter >= max_iter)) { /* iteration limit bookkeeping (iLQG.c:365-377), results out */
                if (!c->gate_recorded) {
                    if (ilqgk_event_record(c->ev_gate, c->stream)) { rc = hfail(h, NULL); goto out; }
                    c->gate_recorded = 1;
                }
                if (ilqgk_launch_finalize(&c->w, max_iter, c->stream)) { rc = hfail(h, NULL); goto out; }
                c->n_launches++;
                if (mpc) { /* closed loop: log the step and, until the last one, solve again from the shifted solution */
                    if (ck_mpc_advance(c, c->mpc_step)) { rc = hfail(h, c); goto out; }
                    progressed = 1;
                    if (++c->mpc_step < mpc->n_steps) {
                        /* polls still in flight belong to the finished solve: a zero among them must not stop the next one.
                           They are dropped; their slots are recorded again before they are read. */
                        c->poll_issued = c->poll_seen = c->stop = 0;
                        c->phase = 0;
                        continue;
                    }
                }
                if (io) {
                    const size_t f = (size_t)h->first[i];
                    if (ck_download_async(c, io->x ? io->x + f * (h->T + 1) * h->d.nx : NULL, io->u ? io->u + f * h->T * h->d.nu : NULL,
                                          io->cost ? io->cost + f : NULL, io->iterations ? io->iterations + f : NULL,
                                          io->result ? io->result + f : NULL, io->n_linesearch ? io->n_linesearch + f : NULL)) { rc = hfail(h, c); goto out; }
                }
                c->phase = 3;
                remaining--;
                progressed = 1;
            }
        }
        if (!progressed) nanosleep(&nap, NULL);
    }
    if (mpc) /* the logs of every chunk, once all of them have finished their last step */
        for (i = 0; i < h->n; i++)
            if (ck_mpc_logs(h->c[i], mpc, (size_t)h->first[i])) { rc = hfail(h, h->c[i]); goto out; }
out:
    if (join_streams(h)) rc = -1;
    if (prio) {
        if (ilqgb_sync(h)) rc = -1;
        for (i = 0; i < h->n; i++) h->c[i]->stream = h->c[i]->stream_main;
    }
    return rc;
}

int ilqgb_solve(ilqgb_handle *h) { return run_engine(h, NULL, NULL); }

/* End to end from and to host buffers (pinned for full overlap); same results as upload + solve + download. */
int ilqgb_solve_host(ilqgb_handle *h, const double *x0, const double *u_nom, double *x, double *u, double *cost,
                     int *iterations, int *result, int *n_linesearch)
{
    io_t io = {x0, u_nom, x, u, cost, iterations, result, n_linesearch};
    if (!x0 || !u_nom) { snprintf(h->err, sizeof h->err, "x0 and u_nom are required"); return -1; }
    if (run_engine(h, &io, NULL)) return -1;
    return ilqgb_sync(h);
}

/* Receding horizon (the reference's caller shifts u between two iLQG_mex calls; SURVEY.md:211): see ilqg_b200.h */
int ilqgb_shift(ilqgb_handle *h, int n_shift, const double *x0, const double *w)
{
    int i;
    if (n_shift < 0 || n_shift > h->T) { snprintf(h->err, sizeof h->err, "n_shift must be in 0..n_hor"); return -1; }
    if (x0 && w) { snprintf(h->err, sizeof h->err, "w is added to the solution's state: it cannot go with x0"); return -1; }
    for (i = 0; i < h->n; i++)
        if (!h->c[i]->started) { snprintf(h->err, sizeof h->err, "ilqgb_start has not been called since the last upload or shift"); return -1; }
    if (!window_fits(h, (long long)h->tr_off + n_shift)) {
        snprintf(h->err, sizeof h->err, "offset + n_shift + n_hor + 1 exceeds the length of a track");
        return -1;
    }
    if (fork_streams(h)) return -1;
    for (i = 0; i < h->n; i++) {
        const size_t f = (size_t)h->first[i] * h->d.nx;
        if (ck_shift(h->c[i], n_shift, x0 ? x0 + f : NULL, w ? w + f : NULL)) return hfail(h, h->c[i]);
    }
    set_track_offset(h, h->tr_off + n_shift);
    return join_streams(h);
}

/* Every chunk runs its own closed loop in the solve engine: when a solve of the chunk finishes, k_mpc_advance logs it and
   shifts it into the next input, and the chunk starts again at once -- a chunk that converged early does not wait for the
   others, which a host loop of ilqgb_shift + ilqgb_solve would make it do at every step. */
int ilqgb_mpc(ilqgb_handle *h, int n_steps, const double *x0, const double *u_nom, const double *w, double *x_cl, double *u_cl,
              double *cost, int *iterations, int *result)
{
    const mpc_t m = {n_steps, w, x_cl, u_cl, cost, iterations, result};
    int i, rc;
    if (n_steps < 1) { snprintf(h->err, sizeof h->err, "n_steps must be >= 1"); return -1; }
    if (!x0 != !u_nom) { snprintf(h->err, sizeof h->err, "x0 and u_nom go together (neither: continue from the current input)"); return -1; }
    if (!x0)
        for (i = 0; i < h->n; i++)
            if (h->c[i]->started) { snprintf(h->err, sizeof h->err, "no input to continue from: ilqgb_upload or ilqgb_shift since the last start"); return -1; }
    if (!window_fits(h, (long long)h->tr_off + n_steps - 1)) {
        snprintf(h->err, sizeof h->err, "offset + (n_steps - 1) + n_hor + 1 exceeds the length of a track");
        return -1;
    }
    if (x0 && ilqgb_upload(h, x0, u_nom)) return -1;
    /* each chunk moves its own offset as it shifts (ck_mpc_advance); all of them end n_steps - 1 further */
    rc = run_engine(h, NULL, &m);
    set_track_offset(h, rc ? h->tr_off : h->tr_off + n_steps - 1);
    if (rc) return -1;
    return ilqgb_sync(h);
}

int ilqgb_sync(ilqgb_handle *h)
{
    int i;
    for (i = 0; i < h->n; i++)
        if (ck_sync(h->c[i])) return hfail(h, h->c[i]);
    if (ilqgk_set_device(h->device)) return hfail(h, NULL);
    return ilqgk_stream_sync(h->stream) ? hfail(h, NULL) : 0;
}

#define FANOUT_PHASE(NAME)                                             \
    int ilqgb_phase_##NAME(ilqgb_handle *h)                            \
    {                                                                  \
        int i;                                                         \
        if (fork_streams(h)) return -1;                                \
        for (i = 0; i < h->n; i++)                                     \
            if (ck_phase_##NAME(h->c[i])) return hfail(h, h->c[i]);    \
        return join_streams(h);                                        \
    }
FANOUT_PHASE(derivs)
FANOUT_PHASE(backpass)
FANOUT_PHASE(linesearch)
FANOUT_PHASE(backpass_once)

int ilqgb_phase_multipliers(ilqgb_handle *h, int init)
{
    int i;
    if (fork_streams(h)) return -1;
    for (i = 0; i < h->n; i++)
        if (ck_phase_multipliers(h->c[i], init)) return hfail(h, h->c[i]);
    return join_streams(h);
}

int ilqgb_clamp_u(ilqgb_handle *h, int k, const double *x, double *u)
{
    int i;
    if (ilqgb_sync(h)) return -1;
    for (i = 0; i < h->n; i++)
        if (ck_clamp_u(h->c[i], k, x + (size_t)h->first[i] * h->d.nx, u + (size_t)h->first[i] * h->d.nu)) return hfail(h, h->c[i]);
    return 0;
}

/* ---- feedback policy of a solved batch (see ilqg_b200.h) ---- */
/* staging of one rollout group per chunk: 2^26 doubles (512 MB), so requested trajectories go in groups of samples;
   ILQG_POLICY_STAGE (doubles) lowers it, which is how the tests reach the grouped path at small sizes */
#define POLICY_STAGE_DOUBLES ((size_t)1 << 26)

int ilqgb_policy(ilqgb_handle *h)
{
    int i;
    if (fork_streams(h)) return -1;
    for (i = 0; i < h->n; i++)
        if (ck_policy(h->c[i])) return hfail(h, h->c[i]);
    return join_streams(h);
}

static int policy_ready(ilqgb_handle *h)
{
    int i;
    for (i = 0; i < h->n; i++)
        if (!h->c[i]->policy_valid) {
            snprintf(h->err, sizeof h->err, "no current feedback policy: call ilqgb_policy after the solve (an upload, start, begin, shift, "
                                            "closed loop, solve, pass, rollout or put since then discards it)");
            return 0;
        }
    return 1;
}

int ilqgb_policy_rollout(ilqgb_handle *h, int M, const double *x0s, double *cost, double *x_final, int *ok, double *x, double *u)
{
    const size_t nx = (size_t)h->d.nx, nu = (size_t)h->d.nu, T = (size_t)h->T;
    size_t G, maxB = 0, per;
    double *tmp = NULL;
    int i, s0, rc = 0;
    if (M < 1) { snprintf(h->err, sizeof h->err, "M must be >= 1"); return -1; }
    if (!x0s || !cost || !x_final || !ok) { snprintf(h->err, sizeof h->err, "x0s, cost, x_final and ok are required"); return -1; }
    if (h->c[0]->plant_on && h->c[0]->plant_n_sub > 1) {
        snprintf(h->err, sizeof h->err, "policy rollouts step the plant once per control: n_sub > 1 is not supported");
        return -1;
    }
    if (!policy_ready(h)) return -1;
    for (i = 0; i < h->n; i++)
        if ((size_t)h->c[i]->B > maxB) maxB = (size_t)h->c[i]->B;
    per = policy_sample_doubles(h->c[0], x != NULL, u != NULL);
    {
        const long cap = env_int("ILQG_POLICY_STAGE", 0);
        G = (cap > 0 && (size_t)cap < POLICY_STAGE_DOUBLES ? (size_t)cap : POLICY_STAGE_DOUBLES) / (maxB * per);
    }
    if (G < 1) G = 1;
    if (G > (size_t)M) G = (size_t)M;
    if (G < (size_t)M && !(tmp = (double *)malloc(sizeof(double) * maxB * G * per))) { snprintf(h->err, sizeof h->err, "out of host memory"); return -1; }
    if (fork_streams(h)) { free(tmp); return -1; }
    for (s0 = 0; s0 < M && !rc; s0 += (int)G) {
        /* every chunk's group is launched before any is collected, so that the chunks' rollouts run concurrently */
        for (i = 0; i < h->n && !rc; i++) {
            const size_t f = (size_t)h->first[i] * M;
            const prollout_t q = {M, s0, (int)(M - s0 < (int)G ? M - s0 : (int)G), x0s + f * nx, cost + f, x_final + f * nx,
                                  x ? x + f * (T + 1) * nx : NULL, u ? u + f * T * nu : NULL, ok + f};
            if (ck_policy_rollout_launch(h->c[i], &q, tmp)) rc = hfail(h, h->c[i]);
        }
        for (i = 0; i < h->n && !rc; i++) {
            const size_t f = (size_t)h->first[i] * M;
            const prollout_t q = {M, s0, (int)(M - s0 < (int)G ? M - s0 : (int)G), x0s + f * nx, cost + f, x_final + f * nx,
                                  x ? x + f * (T + 1) * nx : NULL, u ? u + f * T * nu : NULL, ok + f};
            if (ck_policy_rollout_collect(h->c[i], &q, tmp)) rc = hfail(h, h->c[i]);
        }
    }
    if (join_streams(h)) rc = -1;
    if (!rc && ilqgb_sync(h)) rc = -1;
    free(tmp);
    return rc;
}

int ilqgb_policy_eval(ilqgb_handle *h, int k, const double *x, double *u)
{
    int i;
    if (k < 0 || k >= h->T) { snprintf(h->err, sizeof h->err, "k must be in 0..n_hor-1"); return -1; }
    if (!x || !u) { snprintf(h->err, sizeof h->err, "x and u are required"); return -1; }
    if (!policy_ready(h)) return -1;
    if (ilqgb_sync(h)) return -1;
    for (i = 0; i < h->n; i++)
        if (ck_policy_eval(h->c[i], k, x + (size_t)h->first[i] * h->d.nx, u + (size_t)h->first[i] * h->d.nu)) return hfail(h, h->c[i]);
    return 0;
}

int ilqgb_dense_size(void) { return ilqgk_dense_size(); }

int ilqgb_mod_chol(int device, int n, int count, const double *A, const double *b, double *factor, double *E, int *P, double *shift, double *inverse,
                   double *H, double *x)
{
    if (ilqgk_device_count() < 1) { fail_create("no CUDA device available: this library has no CPU fallback"); return -1; }
    if (ilqgk_set_device(device) || ilqgk_mod_chol(n, count, A, b, factor, E, P, shift, inverse, H, x)) { fail_create(ilqgk_last_error()); return -1; }
    return 0;
}

int ilqgb_eval_size(int mode) { return ilqgk_eval_size(mode); }

int ilqgb_eval(ilqgb_handle *h, int mode, int k, const double *x, const double *u, double *out)
{
    int i;
    const int no = ilqgk_eval_size(mode);
    if (no < 0) { snprintf(h->err, sizeof h->err, "no such evaluation mode"); return -1; }
    if (k < 0 || k > h->T) { snprintf(h->err, sizeof h->err, "k out of range"); return -1; }
    if (ilqgb_sync(h)) return -1;
    for (i = 0; i < h->n; i++)
        if (ck_eval(h->c[i], mode, k, x + (size_t)h->first[i] * h->d.nx, u + (size_t)h->first[i] * h->d.nu, out + (size_t)h->first[i] * no))
            return hfail(h, h->c[i]);
    return 0;
}

/* run-time tuning knobs (the defaults are chosen from the batch size): "ls_tail_from" (sequential line-search rounds before the
   parallel-alpha tail, >= n_alpha = all sequential), "bp_latency" (0/1: register-unconstrained back-pass build), and
   "pass_index" (the loop index `iter` the next single phase runs as: row of the traces) */
int ilqgb_set_tuning(ilqgb_handle *h, const char *name, int value)
{
    int i;
    if (!strcmp(name, "cw_lpp"))
        for (i = 0; i < h->n; i++)
            if ((value == 32 || value == 16 || value == 8) && !coop_fits(h->c[i], value, h->err, sizeof h->err)) return -1;
    for (i = 0; i < h->n; i++) {
        if (!strcmp(name, "ls_tail_from")) h->c[i]->ls_tail_from = value;
        else if (!strcmp(name, "pass_index")) { h->c[i]->iter = value; h->c[i]->started = 1; }
        else if (!strcmp(name, "bp_latency")) h->c[i]->bp_latency = value;
        else if (!strcmp(name, "bp_ppw") && value >= -1 && value <= 32 && value != 0) h->c[i]->bp_ppw = value;
        else if (!strcmp(name, "bp_split") && (value == -1 || value == 0 || value == 4)) h->c[i]->bp_split = value;
        else if (!strcmp(name, "cw_lpp") && (value == 32 || value == 16 || value == 8)) h->c[i]->cw_lpp = value;
        else { snprintf(h->err, sizeof h->err, "unknown tuning knob"); return -1; }
    }
    return 0;
}

long ilqgb_get(ilqgb_handle *h, const char *field, double *out)
{
    int i;
    long per = -1, tot = 0;
    if (ilqgb_sync(h)) return -1;
    for (i = 0; i < h->n; i++) {
        long n = ck_get(h->c[i], field, out + (per < 0 ? 0 : (size_t)h->first[i] * per));
        if (n < 0) return hfail(h, h->c[i]);
        if (per < 0) per = n / h->c[i]->B;
        tot += n;
    }
    return tot;
}

long ilqgb_get_int(ilqgb_handle *h, const char *field, int *out)
{
    int i;
    long per = -1, tot = 0;
    if (ilqgb_sync(h)) return -1;
    for (i = 0; i < h->n; i++) {
        long n = ck_get_int(h->c[i], field, out + (per < 0 ? 0 : (size_t)h->first[i] * per));
        if (n < 0) return hfail(h, h->c[i]);
        if (per < 0) per = n / h->c[i]->B;
        tot += n;
    }
    return tot;
}

int ilqgb_timing(ilqgb_handle *h, double *ms, long *launches, int reset)
{
    int i, k;
    double m[TC_N];
    long l[TC_N];
    for (k = 0; k < TC_N; k++) {
        if (ms) ms[k] = 0.0;
        if (launches) launches[k] = 0;
    }
    for (i = 0; i < h->n; i++) {
        if (ck_timing(h->c[i], m, l, reset)) return hfail(h, h->c[i]);
        for (k = 0; k < TC_N; k++) {
            if (ms) ms[k] += m[k];
            if (launches) launches[k] += l[k];
        }
    }
    return 0;
}

long ilqgb_launch_count(const ilqgb_handle *h)
{
    int i;
    long n = 0;
    for (i = 0; i < h->n; i++) n += ck_launch_count(h->c[i]);
    return n;
}

int ilqgb_chunks(const ilqgb_handle *h) { return h->n; }


long ilqgb_put(ilqgb_handle *h, const char *field, const double *in)
{
    int i;
    long per = -1, tot = 0;
    if (ilqgb_sync(h)) return -1;
    for (i = 0; i < h->n; i++) {
        long n = ck_put(h->c[i], field, in + (per < 0 ? 0 : (size_t)h->first[i] * per));
        if (n < 0) return hfail(h, h->c[i]);
        if (per < 0) per = n / h->c[i]->B;
        tot += n;
    }
    return tot;
}

long ilqgb_put_int(ilqgb_handle *h, const char *field, const int *in)
{
    int i;
    long tot = 0;
    if (ilqgb_sync(h)) return -1;
    for (i = 0; i < h->n; i++) {
        long n = ck_put_int(h->c[i], field, in + h->first[i]);
        if (n < 0) return hfail(h, h->c[i]);
        tot += n;
    }
    return tot;
}

int ilqgb_begin(ilqgb_handle *h)
{
    int i;
    if (fork_streams(h)) return -1;
    for (i = 0; i < h->n; i++)
        if (ck_begin(h->c[i])) return hfail(h, h->c[i]);
    return join_streams(h);
}

int ilqgb_rollout(ilqgb_handle *h, double alpha, int cost_only)
{
    int i;
    if (fork_streams(h)) return -1;
    for (i = 0; i < h->n; i++)
        if (ck_rollout(h->c[i], alpha, cost_only)) return hfail(h, h->c[i]);
    return join_streams(h);
}
