/*
 * tests/sens/rti_sens.c — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Reference for qmpc_eval_sens_x0 (acados eval_param_sens "ex"): the derivatives of one RTI step's result w.r.t. x0,
 * computed with the oracle's own routines (linearize and riccati of oracle/qmpc_oracle.c, compiled in unchanged) along
 * a route deliberately different from the kernel's: 13 independent LQR solves instead of one factorisation and a
 * 13-column sweep.  Built by tests/sens/sens_ref.py into a library of its own.
 */
#include "../../oracle/qmpc_oracle.c"

/* Derivatives of one RTI step's result (x, u) w.r.t. x0 at the explicit active set act[N*4] (0 free, 1/2 pinned):
   the linearisation of orc_rti_step at the PRE-solve iterate xit/uit (it does not depend on x0), then 13 independent
   homogeneous LQR solves (riccati with the pinned inputs at 0, no offsets, no linear costs) from x0 = e_i.
   sens_x [(n_stages+1)][13][13] (may be NULL), sens_u [n_stages][4][13]; column i = derivative w.r.t. x0[i].
   returns 1 when every factorisation was positive definite. */
int orc_rti_sens(const double *quad, double dt, int N,
                 int M, const double *gpX, const double *gpth, const double *alpha,
                 const double *Wd, const double *Wed, const double *xit, const double *uit,
                 const unsigned char *act, int n_stages, double *sens_x, double *sens_u)
{
    model_t m = mk_model(quad, M, gpX, gpth, alpha);
    double *A = (double *)malloc(sizeof(double) * N * NX * NX);
    double *B = (double *)malloc(sizeof(double) * N * NX * NU);
    double *zx = (double *)calloc((size_t)(N + 1) * NX, sizeof(double));
    double *zu = (double *)calloc((size_t)N * NU, sizeof(double));
    double *xs = (double *)malloc(sizeof(double) * (N + 1) * NX);
    double *us = (double *)malloc(sizeof(double) * N * NU);
    for (int k = 0; k < N; ++k) {
        double Phi[NX];
        linearize(&m, xit + k * NX, uit + k * NU, dt, Phi, A + k * NX * NX, B + k * NX * NU);
    }
    qp_t qp; qp.N = N; qp.A = A; qp.B = B; qp.c = zx; qp.q = zx; qp.r = zu; qp.lb = 0; qp.ub = 0;
    for (int i = 0; i < NX; ++i) { qp.Qd[i] = dt * Wd[i]; qp.QNd[i] = Wed[i]; }
    for (int a = 0; a < NU; ++a) qp.Rd[a] = dt * Wd[NX + a];
    int ok = 1;
    for (int c = 0; c < NX; ++c) {
        double e[NX] = {0};
        e[c] = 1.0;
        qp.x0 = e;
        ok &= riccati(&qp, NULL, zu, act, zu, xs, us);
        for (int k = 0; k <= n_stages; ++k)
            for (int i = 0; i < NX; ++i) if (sens_x) sens_x[(k * NX + i) * NX + c] = xs[k * NX + i];
        for (int k = 0; k < n_stages; ++k)
            for (int a = 0; a < NU; ++a) sens_u[(k * NU + a) * NX + c] = us[k * NU + a];
    }
    free(A); free(B); free(zx); free(zu); free(xs); free(us);
    return ok;
}
