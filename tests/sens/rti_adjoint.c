/*
 * tests/sens/rti_adjoint.c — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Reference for qmpc_eval_adjoint (reverse mode of one RTI step w.r.t. x0 and the reference), computed with the oracle's
 * own routines (linearize and riccati of oracle/qmpc_oracle.c, compiled in unchanged) along a route deliberately
 * different from the kernel's.  Built by tests/sens/adjoint_ref.py into a library of its own.
 */
#include "../../oracle/qmpc_oracle.c"

/* The reverse mode of one RTI step's result w.r.t. x0 and the reference, for the cotangents
   x_bar [(N+1)][13] and u_bar [N][4] (either may be NULL = zero), at the explicit active set act[N*4].  The minimiser
   (xh, uh) of the homogeneous pinned LQR with linear costs q = -x_bar, r = -u_bar from xh_0 = 0 (the oracle's riccati),
   then yref_bar [N][17] = (Qd xh_k, Rd uh_k), yref_e_bar [13] = QNd xh_N and x0_bar [13] = pi_0 of the explicit costate
   recursion pi_N = x_bar_N - QNd xh_N, pi_k = x_bar_k - Qd xh_k + A_k' pi_{k+1} (not the kernel's route, -p_0).
   Any output may be NULL.  returns 1 when every factorisation was positive definite. */
int orc_rti_adjoint(const double *quad, double dt, int N,
                    int M, const double *gpX, const double *gpth, const double *alpha,
                    const double *Wd, const double *Wed, const double *xit, const double *uit,
                    const unsigned char *act, const double *x_bar, const double *u_bar,
                    double *x0_bar, double *yref_bar, double *yref_e_bar)
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
    if (yref_bar)
        for (int k = 0; k < N; ++k) {
            for (int i = 0; i < NX; ++i) yref_bar[k * (NX + NU) + i] = qp.Qd[i] * xs[k * NX + i];
            for (int a = 0; a < NU; ++a) yref_bar[k * (NX + NU) + NX + a] = qp.Rd[a] * us[k * NU + a];
        }
    if (yref_e_bar) for (int i = 0; i < NX; ++i) yref_e_bar[i] = qp.QNd[i] * xs[N * NX + i];
    double pi[NX], pn[NX];
    for (int i = 0; i < NX; ++i) pi[i] = (x_bar ? x_bar[N * NX + i] : 0.0) - qp.QNd[i] * xs[N * NX + i];
    for (int k = N - 1; k >= 0; --k) {
        const double *Ak = A + k * NX * NX;
        for (int i = 0; i < NX; ++i) {
            double s = (x_bar ? x_bar[k * NX + i] : 0.0) - qp.Qd[i] * xs[k * NX + i];
            for (int l = 0; l < NX; ++l) s += Ak[l * NX + i] * pi[l];
            pn[i] = s;
        }
        memcpy(pi, pn, sizeof(pi));
    }
    if (x0_bar) memcpy(x0_bar, pi, sizeof(pi));
    free(A); free(B); free(zx); free(zu); free(q); free(r); free(xs); free(us);
    return ok;
}
