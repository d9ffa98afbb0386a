/* tests/policy_oracle_shim.c -- TEST INFRASTRUCTURE for tests/policy_util.py, compiled per problem at test time against the
 * reference's structure layout (include/ilqg_compat.h + the problem's iLQG_problem.h).  The oracle's HSolver begins with its
 * tOptSet (oracle/harness.c), so an oracle handle is also a tOptSet pointer.  ps_sizeof_trajEl lets the caller check that this
 * build and the oracle library agree on the layout before it touches anything. */
#include <string.h>

#include "iLQG.h"

int ps_sizeof_trajEl(void) { return (int)sizeof(trajEl_t); }

/* o.x0 <- x0 without re-initialising: the next forward_pass starts from another state */
void ps_set_x0(tOptSet *o, const double *x0) { memcpy(o->x0, x0, sizeof(double) * N_X); }

/* l <- l * f on every step of the nominal trajectory: after f = 0, forward_pass(alpha = 1) computes u + (0 * l) * 1 + L dx, the
   feedback branch at alpha = 0 with its signs of zero (forward_pass itself skips the gains when alpha == 0) */
void ps_scale_l(tOptSet *o, double f)
{
    int k, j;
    for (k = 0; k < o->n_hor; k++)
        for (j = 0; j < N_U; j++) o->nominal->t[k].l[j] *= f;
}
