/* ilqg_work.h -- plain-C descriptors shared by the C host layer (ilqg_host.c) and the CUDA layer (ilqg_cuda.cu).
 * Everything a kernel needs travels by value in these two structs (kernel parameter space), never via globals. */
#ifndef ILQG_WORK_H
#define ILQG_WORK_H

#define ILQG_MAX_ALPHA 16

/* run-time options: the numeric subset of tOptSet the solve loop reads (reference iLQG.h:45-68) */
typedef struct ilqg_opts {
    double alpha[ILQG_MAX_ALPHA];
    int n_alpha;
    double lambdaMax, lambdaMin, lambdaInit, dlambdaInit, lambdaFactor;
    double tolGrad, tolFun, tolConstraint, zMin;
    double w_pen_init_l, w_pen_init_f, w_pen_max_l, w_pen_max_f, w_pen_fact1, w_pen_fact2;
    int regType, max_iter;
    int bp_latency_build; /* backward pass: 1 = register-unconstrained build (small batches), 0 = 128-register build */
    int ls_tail_from;   /* line search: rounds [0, ls_tail_from) run one alpha per launch, the remaining alphas all at once;
                           >= n_alpha: purely sequential rounds (large batches) */
    int cw_lpp;         /* warp-cooperative backward pass: lanes per problem (32, 16 or 8; 32 / cw_lpp problems share a warp) */
    int bp_split;       /* backward pass: lanes per problem of the small-batch kernel k_backpass_split (4), 0 = lane per problem */
    int bp_ppw;         /* backward pass (lane per problem and split kernels): problems per warp; 32 (8 for the split kernel) = all
                           lanes, fewer = sparse warps for small batches */
    int bp_single;      /* backward pass: 1 = one attempt at the current lambda, no retry, no exit test (back_pass(o) on its own) */
    int ls_commit_par;  /* 1: the tail records the state at the start of 32 time segments and the commit replays the
                           winner segment-parallel (one warp per problem); 0: the commit re-rolls the winner sequentially */
} ilqg_opts;

/* device workspace of one batch; all arrays are [..][Bp] with the problem index fastest */
typedef struct ilqg_work {
    int B, Bp, T;
    double *XU[2];             /* two trajectory buffers of records [T+1][Bp][RXU] = x|u|pad; cur[b] says which is nominal */
    double *x0;                /* [NX][Bp] */
    double *Ll[2];             /* feed-forward records [T][Bp][RLS] = l | pad, one per trajectory buffer like LL */
    double *LL[2];             /* gain records [T][Bp][RLM] = L | pad, one per trajectory buffer: like the
                                  reference, where l and L are members of the trajectory element (iLQG_problem.tem:33-34) */
    double *V1, *V2, *FD;      /* time-varying derivative entries [T][NV1][Bp], [T][NV2][Bp]; final cx,cxx [NX+NQXX][Bp] */
    double *muR, *lastR, *muF, *lastF;
    const double *const *pk;   /* [k]-indexed parameters (device pointers), or null */
    const double *pp;          /* per-problem parameter sets [NPF][Bp], or null = one shared set (kernel argument) */
    double *cost, *new_cost, *dcost, *expected, *lambda, *dlambda, *g_norm, *dV0, *dV1, *w_pen_l, *w_pen_f;
    int *cur, *status, *new_deriv, *deriv_fail, *iterations, *result, *n_ls, *n_bp, *bp_done, *post_mode;
    int *ls_list[2], *ls_count; /* line search: compacted lists of undecided problems (ping-pong), per-round counts */
    double *ls_cnew;            /* [MAX_ALPHA][Bp] rollout cost per alpha (parallel tail of the line search) */
    int *ls_mask;               /* [Bp] bit a: rollout of alpha a finite; bit 16+a: alpha a acceptable */
    double *ls_ckpt;            /* [MAX_ALPHA][32][Bp][NX] state at the start of each time segment of the tail's rollouts
                                   (null: the commit re-rolls the winner sequentially) */
    int *n_dv, *n_roll, *n_tail; /* work counters (bench roofline accounting): derivative sweeps consumed, rollouts that
                                  stored a trajectory, parallel-alpha tails (one shared read of the nominal, no stores) */
    /* optional traces for parity tests (null when disabled) */
    double *tr_lambda, *tr_newcost, *tr_z; /* [max_iter][Bp]: lambda at the line search, last rollout cost, last z */
    int *tr_alpha;                  /* [max_iter][Bp] */
    int *tr_clamp;                  /* [T][Bp]: is_clamped of the last back pass, 2 bits per input, QP code << 16 */
    /* time-indexed parameter tracks (appended: the kernel-argument offsets of the fields above do not move) */
    unsigned tr_mask;               /* bit j: pk[j] is a track [len][Bp] read at step tr_off + k; clear: shared [n_hor + 1] */
    int tr_off;                     /* window offset of this chunk's tracks */
} ilqg_work;

/* one receding-horizon step of every problem (k_mpc_advance).  The disturbance and the logs are problem-major
 * ([B][n_steps][..], x_log [B][n_steps + 1][NX]) so that they copy to and from the caller's arrays without a layout change. */
typedef struct ilqg_mpc_step {
    int n_shift;        /* u[k] <- u[k + n_shift] for k < T - n_shift, u[T-1] after that */
    int set_x0;         /* 1: x0 <- x[n_shift] (+ w); 0: x0 is left to the caller */
    int plan;           /* 0: log only (the last step of a closed loop): the solution stays in place */
    int step, n_steps;  /* row of w and of the logs */
    const double *w;    /* [B][n_steps][NX] disturbance added to x[n_shift], or null */
    double *x_log, *u_log, *cost_log;   /* x0 of the solve (and, log only, the next state), u[0], cost; null = not logged */
    int *it_log, *res_log;              /* iterations, result */
} ilqg_mpc_step;

/* the plant of a closed loop (k_mpc_plant): the same problem with its own parameter values, stepped n_sub times per applied
 * control.  It travels in k_mpc_plant's own arguments so that ilqg_work and ilqg_mpc_step, which other kernels take by
 * value, keep their layout. */
typedef struct ilqg_plant {
    int n_sub;          /* 1..64 sub-steps per control interval */
    const double *pp;   /* per-problem plant parameter sets [NPF][Bp], or null = one shared set (kernel argument) */
} ilqg_plant;

/* one launch of k_policy_rollout: n_samp closed-loop rollouts of the feedback policy per problem, lane b * n_samp + s.  The
 * arrays are problem-major ([B][n_samp][..]) so that they copy to and from the caller's arrays without a layout change.  Like
 * ilqg_plant it travels in the kernel's own arguments. */
typedef struct ilqg_policy {
    int n_samp;             /* samples per problem in this launch */
    const int *policy_ok;   /* [Bp] the problem's gains are valid (ilqgb_policy) */
    const double *pp;       /* per-problem parameter sets [NPF][Bp] (the model's or the plant's), or null = one shared set */
    const double *x0s;      /* [B][n_samp][NX] initial states */
    double *cost, *x_final; /* [B][n_samp], [B][n_samp][NX] */
    int *ok;                /* [B][n_samp] forward_pass's return value */
    double *x, *u;          /* [B][n_samp][T+1][NX], [B][n_samp][T][NU], or null = not stored */
} ilqg_policy;

#endif
