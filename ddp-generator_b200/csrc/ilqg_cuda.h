/* ilqg_cuda.h -- C declarations of the thin CUDA layer (ilqg_cuda.cu) used by the C host code (ilqg_host.c).
 * Plain pointers and sizes only; `stream` is a cudaStream_t passed as void*. All functions return 0 on success. */
#ifndef ILQG_CUDA_H
#define ILQG_CUDA_H
#include <stddef.h>
#include "ilqg_work.h"
#ifdef __cplusplus
extern "C" {
#endif

typedef struct ilqgk_dims_t {
    int nx, nu, nqxx, nquu, nqxu, nv1, nv2, npf, nkp, n_mu_r, n_mu_f, n_mu_le, n_mu_fe, full_ddp, has_hx, rxu, rlm, rls, coop, bp_split_ok;
} ilqgk_dims_t;

const char *ilqgk_last_error(void);
void ilqgk_dims(ilqgk_dims_t *d);
const char *ilqgk_problem_name(void);
int ilqgk_param_count(void);
const char *ilqgk_param_name(int i);
int ilqgk_param_size(int i);

int ilqgk_preload(void); /* load every solver kernel on the current device (idempotent) */
int ilqgk_device_count(void);
int ilqgk_set_device(int dev);
int ilqgk_malloc(void **p, size_t bytes);
int ilqgk_free(void *p);
int ilqgk_host_alloc(void **p, size_t bytes);
int ilqgk_host_free(void *p);
int ilqgk_memset(void *p, int v, size_t bytes, void *stream);
int ilqgk_h2d(void *dst, const void *src, size_t bytes, void *stream);
int ilqgk_d2h(void *dst, const void *src, size_t bytes, void *stream);
int ilqgk_d2d(void *dst, const void *src, size_t bytes, void *stream);
int ilqgk_stream_create(void **s);
int ilqgk_stream_create_prio(void **s, int rank, int n_ranks); /* rank 0 = most urgent of n_ranks */
int ilqgk_stream_destroy(void *s);
int ilqgk_stream_sync(void *s);
int ilqgk_event_create(void **e);
int ilqgk_event_create_notiming(void **e);
int ilqgk_stream_wait_event(void *s, void *e);
int ilqgk_event_query(void *e); /* 1 complete, 0 pending, -1 error */
int ilqgk_event_sync(void *e);
int ilqgk_event_destroy(void *e);
int ilqgk_event_record(void *e, void *s);
int ilqgk_event_elapsed(void *a, void *b, float *ms);

/* mode bits: 1 init multipliers, 2 initial rollout of buffer 0 into buffer 1, 4 first lines of iLQG() */
int ilqgk_launch_init(const ilqg_work *w, const ilqg_opts *o, const double *params, int mode, void *stream);
int ilqgk_launch_rollout(const ilqg_work *w, const double *params, double alpha, int cost_only, void *stream);
int ilqgk_launch_derivs(const ilqg_work *w, const double *params, void *stream);
int ilqgk_launch_backpass(const ilqg_work *w, const ilqg_opts *o, const double *params, int iter, void *stream);
int ilqgk_launch_ls_reset(const ilqg_work *w, void *stream);
int ilqgk_launch_ls_round(const ilqg_work *w, const ilqg_opts *o, const double *params, int iter, int round, void *stream);
int ilqgk_launch_ls_tail(const ilqg_work *w, const ilqg_opts *o, const double *params, int iter, int from, void *stream);
int ilqgk_launch_post(const ilqg_work *w, const ilqg_opts *o, const double *params, void *stream);
int ilqgk_launch_mult(const ilqg_work *w, const ilqg_opts *o, const double *params, int init, void *stream);
int ilqgk_dense_size(void);
int ilqgk_launch_dense(const ilqg_work *w, const double *params, double *out /* [B][T][dense_size] */, void *stream);
int ilqgk_launch_clamp(const ilqg_work *w, const double *params, double *xu_io /* [B][nx+nu] */, int k, void *stream);
int ilqgk_eval_size(int mode); /* doubles per problem mode 0..16 of ilqgk_launch_eval returns, -1 = no such mode */
int ilqgk_launch_eval(const ilqg_work *w, const double *params, const double *in /* [B][nx+nu] */, double *out, int mode, int k, void *stream);
int ilqgk_mod_chol(int n, int count, const double *A, const double *b, double *fac, double *E, int *P, double *ret, double *inv, double *H, double *x);
int ilqgk_has_post(void);
int ilqgk_launch_finalize(const ilqg_work *w, int max_iter, void *stream);
int ilqgk_launch_count_active(const ilqg_work *w, int *d_counter, void *stream);
/* log the finished solve of every problem and shift its solution into the input of the next one (k_mpc_advance) */
int ilqgk_launch_mpc_advance(const ilqg_work *w, const ilqg_mpc_step *a, void *stream);
/* the same with the next state from the plant (k_mpc_plant): params_plant = the shared plant set (used when pl->pp is null) */
int ilqgk_launch_mpc_plant(const ilqg_work *w, const ilqg_mpc_step *a, const double *params_plant, const ilqg_plant *pl, void *stream);
/* feedback policy of a solved batch: k_policy_mark (save = 1 before, 0 after the derivative sweep and backward pass of
   ilqgb_policy), k_policy_rollout (params = the shared set, used when r->pp is null), k_policy_eval (x [B][nx] -> u [B][nu]) */
int ilqgk_launch_policy_mark(const ilqg_work *w, int *keep /* [7][Bp] */, int *policy_ok, int save, void *stream);
int ilqgk_launch_policy_rollout(const ilqg_work *w, const double *params, const ilqg_policy *r, void *stream);
int ilqgk_launch_policy_eval(const ilqg_work *w, const double *params, const int *policy_ok, const double *x, double *u, int k, void *stream);
/* [B][n_k][n_i] (host order) <-> device element (k, b, i) at base[k*stride_k + b*stride_b + i*stride_i + off] */
int ilqgk_launch_scatter(const double *src, double *dst, double *dst_alt, const int *sel, int B, int n_k, int n_i, long long stride_k,
                         long long stride_b, long long stride_i, long long off, void *stream);
int ilqgk_launch_gather(const double *src, const double *src_alt, const int *sel, double *dst, int B, int n_k, int n_i,
                        long long stride_k, long long stride_b, long long stride_i, long long off, void *stream);

#ifdef __cplusplus
}
#endif
#endif
