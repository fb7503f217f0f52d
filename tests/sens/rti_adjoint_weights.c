/*
 * tests/sens/rti_adjoint_weights.c — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Reference for the cost-weight outputs of qmpc_eval_adjoint_weights, computed with the oracle's own routines
 * (linearize and riccati of oracle/qmpc_oracle.c, compiled in unchanged).  Built by tests/sens/adjoint_weights_ref.py
 * into a library of its own.
 */
#include "../../oracle/qmpc_oracle.c"

/* The gradients of <x_bar, x> + <u_bar, u> (cotangents x_bar [(N+1)][13], u_bar [N][4], either may be NULL = zero) w.r.t.
   the cost weights Wd [17] and Wed [13], at the explicit active set act[N*4].  The linearisation does not read the
   weights, so on the active set the solution z = (x, u) of the QP
   min sum_k 1/2 (z_k - yref_k)' dt W (z_k - yref_k) + 1/2 (x_N - yref_e)' W_e (x_N - yref_e) is a smooth function of
   them; differentiating its optimality conditions gives, with (xh, uh) the minimiser of the homogeneous pinned LQR with
   linear costs q = -x_bar, r = -u_bar from xh_0 = 0 (the oracle's riccati, as orc_rti_adjoint builds it):
   w_bar[i] = -dt sum_k (xh_k, uh_k)_i (z_k - yref_k)_i and we_bar[i] = -xh_N,i (x_N - yref_e)_i.
   xit, uit: the PRE-solve iterate (the linearisation point); x [(N+1)][13], u [N][4]: the step's solution (rti_step's
   output); yref [N][17], yref_e [13] its reference.  Either output may be NULL.
   returns 1 when every factorisation was positive definite. */
int orc_rti_adjoint_weights(const double *quad, double dt, int N,
                            int M, const double *gpX, const double *gpth, const double *alpha,
                            const double *Wd, const double *Wed, const double *xit, const double *uit,
                            const unsigned char *act, const double *x_bar, const double *u_bar,
                            const double *x, const double *u, const double *yref, const double *yref_e,
                            double *w_bar, double *we_bar)
{
    model_t m = mk_model(quad, M, gpX, gpth, alpha);
    double *A = (double *)malloc(sizeof(double) * N * NX * NX);
    double *B = (double *)malloc(sizeof(double) * N * NX * NU);
    double *zx = (double *)calloc((size_t)N * NX, sizeof(double));
    double *zu = (double *)calloc((size_t)N * NU, sizeof(double));
    double *q = (double *)calloc((size_t)(N + 1) * NX, sizeof(double));
    double *r = (double *)calloc((size_t)N * NU, sizeof(double));
    double *xs = (double *)malloc(sizeof(double) * (N + 1) * NX);
    double *us = (double *)malloc(sizeof(double) * N * NU);
    for (int k = 0; k < N; ++k) {
        double Phi[NX];
        linearize(&m, xit + k * NX, uit + k * NU, dt, Phi, A + k * NX * NX, B + k * NX * NU);
    }
    if (x_bar) for (int i = 0; i < (N + 1) * NX; ++i) q[i] = -x_bar[i];
    if (u_bar) for (int i = 0; i < N * NU; ++i) r[i] = -u_bar[i];
    qp_t qp; qp.N = N; qp.A = A; qp.B = B; qp.c = zx; qp.q = q; qp.r = r; qp.lb = 0; qp.ub = 0;
    double x0[NX] = {0};
    qp.x0 = x0;
    for (int i = 0; i < NX; ++i) { qp.Qd[i] = dt * Wd[i]; qp.QNd[i] = Wed[i]; }
    for (int a = 0; a < NU; ++a) qp.Rd[a] = dt * Wd[NX + a];
    int ok = riccati(&qp, NULL, r, act, zu, xs, us);
    if (w_bar) {
        for (int i = 0; i < NX + NU; ++i) w_bar[i] = 0.0;
        for (int k = 0; k < N; ++k) {
            for (int i = 0; i < NX; ++i) w_bar[i] += xs[k * NX + i] * (x[k * NX + i] - yref[k * (NX + NU) + i]);
            for (int a = 0; a < NU; ++a)
                w_bar[NX + a] += us[k * NU + a] * (u[k * NU + a] - yref[k * (NX + NU) + NX + a]);
        }
        for (int i = 0; i < NX + NU; ++i) w_bar[i] *= -dt;
    }
    if (we_bar) for (int i = 0; i < NX; ++i) we_bar[i] = -xs[N * NX + i] * (x[N * NX + i] - yref_e[i]);
    free(A); free(B); free(zx); free(zu); free(q); free(r); free(xs); free(us);
    return ok;
}
