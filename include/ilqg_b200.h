/* ilqg_b200.h -- C ABI of the B200 batched iLQG / control-limited DDP solver.
 *
 * One shared library per generated problem and FULL_DDP setting (libilqg_b200_<problem>_ddp<0|1>.so), exactly as
 * the reference builds one mex per problem (make_iLQG.m:65-86).  All entry points are extern "C", take plain
 * pointers and sizes, and run on the GPU: there is no CPU fallback -- creation fails if no CUDA device is usable.
 *
 * What each entry point replaces in the reference (file:line in jgeisler0303/DDP-Generator):
 *   ilqgb_create / ilqgb_destroy   allocation of trajectories/multipliers by the caller, iLQG_mex.c:100-103, 141-143
 *   ilqgb_create_multi             the same for a batch sharded over several GPUs (no counterpart in the reference, which
 *                                  solves one problem per call; SURVEY.md 8b/8e)
 *   ilqgb_standard_parameters      standard_parameters(), iLQG.c:57-78
 *   ilqgb_set_opt                  setOptParam(), iLQG.c:91-216 (same names, validation and messages)
 *   ilqgb_set_param                binding of the parameter struct by name, iLQG_mex.c:70-84 / paramdesc, iLQG.h:97-99
 *   ilqgb_upload                   o.x0, copy of u_nom into the nominal trajectory, iLQG_mex.c:55-56, 113-115
 *   ilqgb_start                    init_opt + initial rollout + makeCandidateNominal, iLQG_mex.c:108-120, and the
 *                                  first lines of iLQG(), iLQG.c:226-237
 *   ilqgb_iterate                  passes of the iLQG() loop, iLQG.c:239-363, for every problem of the batch
 *   ilqgb_finish                   iLQG.c:365-378 (iteration-limit bookkeeping)
 *   ilqgb_solve                    = start + iterate(max_iter) + finish: the whole iLQG() call for B problems
 *   ilqgb_download                 copy-out of x, u, cost, iLQG_mex.c:127-137, plus iterations / return value
 *   ilqgb_shift / ilqgb_mpc        what a receding-horizon caller does between two iLQG_mex calls (SURVEY.md:211: the
 *                                  previous u, shifted, is the next u_nom), on the device; ilqgb_mpc runs whole closed loops
 *   ilqgb_set_plant_*              the plant of such a loop, which the caller steps with iLQG<Name>MMex modes 16 and 0 and
 *                                  the plant's parameter struct (iLQG_MMex.tem:81-226)
 *   ilqgb_policy / _policy_rollout calc_derivs + back_pass on the tOptSet iLQG() left behind, then forward_pass's feedback step
 *   / _policy_eval                 from other initial states: the solved controller's local feedback law, rolled out on the device
 *   ilqgb_phase_*                  calc_derivs / back_pass / line_search on their own (iLQG.h:83, back_pass.h:7,
 *                                  line_search.h:6) for phase-level parity tests
 *   ilqgb_get / ilqgb_get_int      read-back of any per-problem field (tOptSet / trajEl_t members)
 * The single-problem drop-in (iLQG(tOptSet*) etc., include/ilqg_compat.h) is layered on these.
 */
#ifndef ILQG_B200_H
#define ILQG_B200_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct ilqgb_handle ilqgb_handle;

enum {
    ILQGB_TRACE = 1,  /* keep per-iteration lambda / alpha / cost and per-step active sets (parity tests) */
    ILQGB_TIMING = 2  /* record CUDA events around every kernel launch (bench roofline) */
    /* bits 8..15 of `flags`: number of chunks (concurrent streams) the batch is split into; 0 = automatic */
};
#define ILQGB_CHUNKS(n) (((n) & 0xff) << 8)

/* static facts of this library build */
const char *ilqgb_problem_name(void);
int ilqgb_nx(void);
int ilqgb_nu(void);
int ilqgb_full_ddp(void);
int ilqgb_n_params(void);
const char *ilqgb_param_name(int i);
int ilqgb_param_size(int i); /* 1, k > 1, or -1: one value per timestep (n_hor + 1) */
int ilqgb_device_count(void);
void ilqgb_mult_counts(int *n_running_eq, int *n_final_eq); /* equality constraints among the running / final multipliers */
int ilqgb_deriv_doubles_per_step(void); /* time-varying derivative doubles the derivative kernel stores per step */

/* lifecycle; `stream` may be NULL (the handle then owns a stream) or a cudaStream_t of the caller */
ilqgb_handle *ilqgb_create(int device, int batch, int n_hor, int flags, void *stream);
/* one handle over several GPUs of this process (SURVEY.md 8b "new batched entry ... n_gpus", 8e): the batch is cut into one
 * contiguous shard per device, every call below fans out over all of them, host buffers are indexed by the global problem
 * number, so ilqgb_download / ilqgb_solve_host gather the results of all devices into the caller's single arrays.  No
 * collective and no peer access are involved.  devices = NULL means 0..n_devices-1; `stream` (optional) belongs to
 * devices[0]; ILQGB_CHUNKS(n) counts chunks per device. */
ilqgb_handle *ilqgb_create_multi(int n_devices, const int *devices, int batch, int n_hor, int flags, void *stream);
int ilqgb_devices(const ilqgb_handle *h);
void ilqgb_destroy(ilqgb_handle *h);
const char *ilqgb_last_error(const ilqgb_handle *h); /* h may be NULL for creation errors */

/* options and parameters (shared by the whole batch) */
void ilqgb_standard_parameters(ilqgb_handle *h);
const char *ilqgb_set_opt(ilqgb_handle *h, const char *name, const double *value, int n); /* NULL = ok */
const char *ilqgb_validate_opt(const char *name, const double *value, int n);               /* same check, no handle */
int ilqgb_set_param(ilqgb_handle *h, int index, const double *value, int n);
/* one value set per problem: value[batch][n].  A batch is then B independent reference calls, each with its own parameter
 * struct (iLQG_mex.c:70-84); parameters never set this way keep the shared value.  Not for [k]-indexed parameters. */
int ilqgb_set_param_batch(ilqgb_handle *h, int index, const double *value, int n);
/* Time-indexed parameter tracks.  A [k]-indexed parameter (ilqgb_param_size(index) == -1) gets one track per problem,
 * value[batch][len] (problem-major, global problem index for multi-device handles), len >= n_hor + 1.  A solve reads
 * name[k] = track[b][offset + k], k = 0..n_hor.  The handle has ONE window offset for all its tracks: 0 after the first
 * ilqgb_set_param_track; ilqgb_set_track_offset sets it; ilqgb_shift(n) adds n; ilqgb_mpc adds 1 per shift (n_steps - 1 in
 * all: the handle keeps the last step's unshifted solution).  ilqgb_upload does not move it.  Any call that would leave a
 * window past the end of a track fails before doing anything.  ilqgb_set_param on the same index drops the track: the
 * parameter is shared and fixed again, exactly as today.  [k]-indexed parameters without a track keep today's behaviour. */
int ilqgb_set_param_track(ilqgb_handle *h, int index, const double *value, int len);
int ilqgb_set_track_offset(ilqgb_handle *h, int offset);
int ilqgb_track_offset(const ilqgb_handle *h);

/* host -> device: x0 [batch][nx], u_nom [batch][n_hor][nu] (problem-major, as a caller holds them) */
int ilqgb_upload(ilqgb_handle *h, const double *x0, const double *u_nom);

/* the solve, asynchronous on the handle's stream */
int ilqgb_start(ilqgb_handle *h);
int ilqgb_iterate(ilqgb_handle *h, int n_passes); /* returns passes actually launched (stops when none is running) */
int ilqgb_finish(ilqgb_handle *h);
int ilqgb_solve(ilqgb_handle *h);
int ilqgb_sync(ilqgb_handle *h);
/* upload + solve + download in one call (host buffers should be pinned); same results as ilqgb_upload + ilqgb_solve +
 * ilqgb_download.  Chunks run on streams of descending priority, so they finish one after the other and the result copies
 * of one chunk overlap the passes of the next ones (ILQG_E2E_PRIO=0 in the environment turns that off).  Any output pointer
 * may be NULL.  Synchronises. */
int ilqgb_solve_host(ilqgb_handle *h, const double *x0, const double *u_nom, double *x, double *u, double *cost,
                     int *iterations, int *result, int *n_linesearch);
int ilqgb_active(ilqgb_handle *h); /* problems still running (synchronises) */

/* Receding horizon.  One closed-loop step is one reference call (upload + solve, every counter, lambda, penalty weight and
 * multiplier re-initialised); [k]-indexed parameters are not shifted unless they have a track (ilqgb_set_param_track), whose
 * window then moves with the plan.  A problem whose solve failed (result 0 or -1) goes on
 * with whatever its nominal trajectory holds, as a host loop over ilqgb_solve would.
 * The current solution of every problem becomes the input of the next solve (the reference's caller does this by hand between
 * two iLQG_mex calls): u[k] <- u[k+n_shift] (k < n_hor-n_shift), u[n_hor-1] after that; x0 <- x0 (host [batch][nx]) if given,
 * else the solution's state x[n_shift] (+ w[batch][nx] if w != NULL; w requires x0 == NULL).  0 <= n_shift <= n_hor; requires
 * ilqgb_start since the last upload / shift.  Asynchronous. */
int ilqgb_shift(ilqgb_handle *h, int n_shift, const double *x0, const double *w);
/* n_steps >= 1 closed-loop steps entirely on the device: solve, log, apply u[0], x0 <- x[1] + w[step], shift by one.
 * x0 / u_nom: as ilqgb_upload, or both NULL = start from the handle's current input (last upload or shift).
 * w [batch][n_steps][nx] or NULL.  Logs (any may be NULL): x_cl [batch][n_steps+1][nx], u_cl [batch][n_steps][nu],
 * cost / iterations / result [batch][n_steps].  Afterwards the handle holds the LAST step's solution (not shifted), so
 * ilqgb_download / ilqgb_get return the final plan.  Every chunk advances through the steps on its own.  Synchronises. */
int ilqgb_mpc(ilqgb_handle *h, int n_steps, const double *x0, const double *u_nom, const double *w,
              double *x_cl, double *u_cl, double *cost, int *iterations, int *result);
/* A plant that differs from the model (Monte-Carlo robustness of one controller over sampled plants).  The plant is the same
 * generated problem with its own parameter values, stepped n_sub times per control interval.  With a plant, wherever
 * ilqgb_shift (without a host x0) and ilqgb_mpc set x0 <- x[n] (+ w), they instead step xp = the finished solve's x0 through the
 * n applied controls u[j], j = 0..n-1, each held for n_sub sub-steps: xp <- f(xp, clampU(u[j])) with the plant's parameters,
 * clampU at each sub-step's own state on a fresh copy of u[j] (the reference's forward_pass step; MMex modes 16 then 0), then
 * x0 <- xp (+ w).  u[j] are the solution's controls, which is also what u_cl logs.  n = 0 leaves x0 (+ w); a host x0 ignores
 * the plant.  All sub-steps of control j evaluate at step index k = j, and [k]-indexed parameters are the model's (its shared
 * array, or the window of the solve that just finished).  A non-finite plant state is passed on: the next solve of that problem
 * fails its initial rollout (result -1), as a host loop would.
 * Only non-[k]-indexed parameters can be set for the plant (ilqgb_set_param / ilqgb_set_param_batch shapes; batch rows by
 * global problem index).  An entry never set FOLLOWS THE MODEL: it is, for every problem, the model's current value, shared
 * or per-problem, including later ilqgb_set_param / ilqgb_set_param_batch calls.  n_sub (1..64) rescales nothing: set the
 * plant's time-step parameter (h of the car, dt of the quadrotor and the pendulum) to the model's divided by n_sub yourself,
 * the library does not know which parameter is the time step.  Any of the three setters gives the handle a plant
 * (ilqgb_set_plant_substeps(h, 1) alone: a plant equal to the model).  ilqgb_clear_plant removes it: x0 <- x[n] (+ w) again,
 * bit for bit.  ilqgb_get(h, "plant", out) returns the effective plant set of every problem [batch][sum of parameter sizes]
 * (the "follow the model" rule applied).  Bad index, [k]-indexed parameter, wrong length or n_sub: -1, nothing changed. */
int ilqgb_set_plant_param(ilqgb_handle *h, int index, const double *value, int n);
int ilqgb_set_plant_param_batch(ilqgb_handle *h, int index, const double *value, int n);  /* value[batch][n] */
int ilqgb_set_plant_substeps(ilqgb_handle *h, int n_sub);
int ilqgb_clear_plant(ilqgb_handle *h);

/* Feedback policy of a solved batch.  A solve leaves a plan (x*, u*) and a local feedback law u_k(x) = u*_k + L_k (x - x*_k).
 * ilqgb_policy computes the gains at the final trajectory: for every problem, finished or not, exactly calc_derivs(o); back_pass(o)
 * on the tOptSet iLQG(o) left behind (iLQG.h:83, back_pass.h:7) -- one derivative sweep and ONE backward pass at the final lambda,
 * with the final multipliers and penalty weights, no regularisation retry, no gradient exit.  Afterwards "l" "L" "dV0" "dV1"
 * "g_norm" "v1" "v2" "fd" and "bp_done" hold what back_pass writes; x, u, cost, iterations, result, status, lambda, dlambda, cur
 * and the multipliers are unchanged.  ilqgb_get_int(h, "policy_ok") = derivatives finite and backward pass successful
 * (bp_done).  Asynchronous.  The policy stays valid until the next ilqgb_upload, _start, _begin, _shift, _mpc, _solve*,
 * _iterate, _phase_*, _rollout or ilqgb_put*; after those ilqgb_policy_rollout and ilqgb_policy_eval fail. */
int ilqgb_policy(ilqgb_handle *h);
/* M >= 1 closed-loop rollouts of the policy per problem from x0s [batch][M][nx]: sample (b, i) is forward_pass(candidate, o, alpha,
 * &csum, 0) (iLQG_func.tem:121-185) with alpha's feedback branch taken at alpha = 0 -- u = u*_k + 0 * l_k + L_k (x - x*_k), then
 * clampU at the rollout's own state, then f -- from o.x0 = x0s[b][i].  (forward_pass skips the gains when alpha == 0 exactly;
 * a rollout here always applies them.)  With a plant (ilqgb_set_plant_*), o.p is problem b's effective plant set (ilqgb_get
 * "plant") for the whole step; otherwise the model's.  [k]-indexed parameters: the model's, through the solve's track window.
 * cost [batch][M] = csum (running and final cost with the final multipliers and penalty weights), ok [batch][M] = forward_pass's
 * return value, x_final [batch][M][nx]; x [batch][M][n_hor+1][nx] and u [batch][M][n_hor][nu] (the clamped controls) are
 * optional (NULL).  A problem with policy_ok == 0, and a rollout that fails, give ok = 0 and NaN cost and final state (logged rows
 * after the failing step: NaN).  Nothing of the handle changes: its trajectories, download and get stay as they were.  Needs
 * ilqgb_policy since the last solve; plant sub-steps (n_sub > 1) are rejected.  Rows by global problem index.  Synchronises. */
int ilqgb_policy_rollout(ilqgb_handle *h, int M, const double *x0s, double *cost, double *x_final, int *ok, double *x, double *u);
/* the policy's control at step k (0 <= k < n_hor) for one state per problem, x [batch][nx] -> u [batch][nu]: step k of a policy
 * rollout without f, with the model's parameters (the controller's own limits).  NaN for problems with policy_ok == 0.  For
 * callers that step their own simulator.  Synchronises. */
int ilqgb_policy_eval(ilqgb_handle *h, int k, const double *x, double *u);

/* device -> host; any pointer may be NULL. x [batch][n_hor+1][nx], u [batch][n_hor][nu] */
int ilqgb_download(ilqgb_handle *h, double *x, double *u, double *cost, int *iterations, int *result,
                   int *n_linesearch);

/* single phases on the current nominal trajectories of all running problems */
int ilqgb_phase_derivs(ilqgb_handle *h);
int ilqgb_phase_backpass(ilqgb_handle *h);
int ilqgb_phase_linesearch(ilqgb_handle *h);
/* back_pass(o) exactly (back_pass.h:7): ONE attempt at the current lambda -- no regularisation retry (iLQG.c:261-284), no
 * gradient exit (iLQG.c:297-303); success = ilqgb_get_int "bp_done".  update_multipliers(o, init) (iLQG.h:86) and
 * clampU(u, t, k, p, N) (iLQG_func.tem:68) for every problem of the batch: x [batch][nx], u [batch][nu] clamped in place. */
int ilqgb_phase_backpass_once(ilqgb_handle *h);
int ilqgb_phase_multipliers(ilqgb_handle *h, int init);
int ilqgb_clamp_u(ilqgb_handle *h, int k, const double *x, double *u);
/* single evaluations of the generated problem functions at one point per problem, the reference's MMex interface
 * (iLQG_MMex.tem:81-226; mex/iLQG_MMex_b200.c is the gateway): x [batch][nx], u [batch][nu], 0-based step k; out
 * [batch][ilqgb_eval_size(mode)] as FULL column-major arrays.  mode: 0 f, 1 L, 2 F, 3 Fx, 4 Fxx, 5 Lx, 6 Lu, 7 Lxx, 8 Luu, 9 Lxu,
 * 10 fx, 11 fu, 12 fxx (nx x nx x nx: A(c,j,r) = d2 f_r / dx_c dx_j), 13 fuu (nu x nu x nx), 14 fxu (nx x nu x nx), 15 y (empty),
 * 16 clamped u; 17 (beyond MMex) the user outputs g[] of calcG (iLQG_func.tem:511-521), ilqgb_eval_size(17) = get_g_size().
 * Multipliers are zero and penalty weights one here. */
int ilqgb_eval_size(int mode);
int ilqgb_eval(ilqgb_handle *h, int mode, int k, const double *x, const double *u, double *out);
/* The reference's modified-Cholesky family (mod_chol, mod_chol_inv, perm_tri_square, mod_chol_solve: cholesky.c:129-356) as a
 * device unit, for `count` packed upper-triangular n x n matrices A (n <= 16) and right-hand sides b [count][n]: factor
 * [count][n(n+1)/2], E [count][n] (diagonal shift), P [count][n] (pivot order), shift [count] (return value), inverse and H
 * (= P L'L P', the regularised matrix) [count][n(n+1)/2], x [count][n] = (A + E)^-1 b.  Bit-identical to the reference's
 * functions; not used by the solver (its call site in the reference, boxQP.c:69-72 under -DMOD_CHOL, is inconsistent).
 * Errors are reported through ilqgb_last_error(NULL). */
int ilqgb_mod_chol(int device, int n, int count, const double *A, const double *b, double *factor, double *E, int *P, double *shift,
                   double *inverse, double *H, double *x);
/* "dense" field of ilqgb_get: [batch][n_hor][ilqgb_dense_size()] = fx fu cx cxx cu cuu cxu lower upper lower_sign upper_sign
 * lower_hx upper_hx of every step (the derivative members of trajEl_t) as the backward pass sees them */
int ilqgb_dense_size(void);
/* run-time tuning knobs, otherwise chosen from the batch size: "ls_tail_from" (sequential line-search rounds before the
 * parallel-alpha tail; >= n_alpha: all rounds sequential, every tried rollout is stored as in the reference), "bp_latency";
 * "bp_split": lanes per problem of the backward pass, 4 = the small-batch kernel k_backpass_split (problems without state-dependent input
 * limits; ignored otherwise), 0 = one lane per problem, -1 = by batch size; "cw_lpp";
 * "pass_index": the loop index the next ilqgb_phase_* call runs as (row of the traces) */
int ilqgb_set_tuning(ilqgb_handle *h, const char *name, int value);

/* field read-back (synchronises). Per-problem scalars: "cost" "new_cost" "dcost" "expected" "lambda" "dlambda"
 * "g_norm" "dV0" "dV1" "w_pen_l" "w_pen_f" -> [batch].  Trajectory fields, problem-major [batch][k][i]:
 * "x" "u" (nominal), "l" "L" "v1" (time-varying derivative entries) "v2" "fd" (final cx,cxx) "mu_f" "mu_r";
 * traces (ILQGB_TRACE): "tr_lambda" "tr_newcost" -> [batch][max_iter].  Returns doubles written, <0 on error.
 * "v1" "v2" "fd" hold the derivatives of the last sweep that covered the problem; for a problem that has finished they may
 * have been re-evaluated at its final trajectory by a later sweep (they are never read again by the solver). */
long ilqgb_get(ilqgb_handle *h, const char *field, double *out);
/* "iterations" "result" "status" "n_linesearch" "n_backpass" "n_derivs" "n_rollouts" "n_tails" "cur" "bp_done" "deriv_fail" -> [batch]; "tr_alpha" -> [batch][max_iter];
 * "tr_clamp" -> [batch][n_hor] (2 bits per input: 0 free, 1 lower, 2 upper; QP return code in bits 16..23);
 * the kernel variants the last pass ran with, the same value for every problem of a chunk -> [batch]: "bp_split" (4 or 0),
 * "cw_lpp" (lanes per problem of the warp-cooperative backward pass, 0 where the problem does not use it), "bp_latency"
 * (register build of the lane-per-problem backward pass), "ls_tail_from" (sequential line-search rounds before the tail,
 * n_alpha = none), "ls_commit_par" (1 = checkpointed segment-parallel commit, 0 = sequential; ILQG_LS_COMMIT_PAR) */
long ilqgb_get_int(ilqgb_handle *h, const char *field, int *out);

/* host -> device write of a field (names and shapes of ilqgb_get, plus "x0" "x_cand" "u_cand" "last_r" "last_f";
 * ints: "cur" "status" "new_deriv" "deriv_fail" "bp_done"), a solve start on imported state (only the first lines of iLQG(), iLQG.c:226-237, run), and a
 * bare rollout = forward_pass(candidates[0] or nominal, o, alpha, &csum, cost_only) of iLQG.h:82: csum -> "new_cost",
 * its return value -> "result".  These carry the single-problem drop-in (csrc/ilqg_dropin.c). */
long ilqgb_put(ilqgb_handle *h, const char *field, const double *in);
long ilqgb_put_int(ilqgb_handle *h, const char *field, const int *in);
int ilqgb_begin(ilqgb_handle *h);
int ilqgb_rollout(ilqgb_handle *h, double alpha, int cost_only);

/* accumulated device time per kernel class since the last reset (ILQGB_TIMING): ms[4] / launches[4] in the
 * order derivs, backpass, linesearch, post */
int ilqgb_timing(ilqgb_handle *h, double *ms, long *launches, int reset);
/* kernels launched by this handle since creation (all classes, incl. layout and bookkeeping kernels) */
long ilqgb_launch_count(const ilqgb_handle *h);
int ilqgb_chunks(const ilqgb_handle *h); /* number of chunks / streams this handle runs on */

#ifdef __cplusplus
}
#endif
#endif
