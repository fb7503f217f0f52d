/*
 * tests/sens/rti_jvp.c — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Reference for qmpc_eval_jvp (forward mode of one RTI step w.r.t. x0, the reference and the cost weights), computed
 * with the oracle's own routines (linearize and riccati of oracle/qmpc_oracle.c, compiled in unchanged).  Built by
 * tests/sens/jvp_ref.py into a library of its own.
 */
#include "../../oracle/qmpc_oracle.c"

/* The tangent (dx [(N+1)][13], du [N][4]) of one RTI step's result for the tangents dx0 [13], dyref [N][17],
   dyref_e [13], dw [17] (of Wd) and dwe [13] (of Wed), any of them NULL = zero, at the explicit active set act[N*4].
   The linearisation does not read x0, the reference or the weights, so on the active set the step is linear in them and
   (dx, du) is the minimiser of the pinned LQR (the oracle's riccati) with the Hessian of the step's QP, x_0 = dx0 and
   the linear costs obtained by differentiating the QP's gradient dt W (z_k - yref_k), W_e (x_N - yref_e):
   q_k = -dt Wd[0:13] dyref_k + dt dw[0:13] (x_k - yref_k),   r_k = -dt Wd[13:17] dyref_k + dt dw[13:17] (u_k - yref_k),
   q_N = -Wed dyref_e + dwe (x_N - yref_e).
   xit, uit: the PRE-solve iterate (the linearisation point); x [(N+1)][13], u [N][4]: the step's solution (rti_step's
   output); yref [N][17], yref_e [13] its reference.  dx may be NULL.
   returns 1 when every factorisation was positive definite. */
int orc_rti_jvp(const double *quad, double dt, int N,
                int M, const double *gpX, const double *gpth, const double *alpha,
                const double *Wd, const double *Wed, const double *xit, const double *uit,
                const unsigned char *act, const double *x, const double *u, const double *yref, const double *yref_e,
                const double *dx0, const double *dyref, const double *dyref_e, const double *dw, const double *dwe,
                double *dx, double *du)
{
    model_t m = mk_model(quad, M, gpX, gpth, alpha);
    double *A = (double *)malloc(sizeof(double) * N * NX * NX);
    double *B = (double *)malloc(sizeof(double) * N * NX * NU);
    double *zx = (double *)calloc((size_t)N * NX, sizeof(double));
    double *zu = (double *)calloc((size_t)N * NU, sizeof(double));
    double *q = (double *)calloc((size_t)(N + 1) * NX, sizeof(double));
    double *r = (double *)calloc((size_t)N * NU, sizeof(double));
    double *xs = (double *)malloc(sizeof(double) * (N + 1) * NX);
    for (int k = 0; k < N; ++k) {
        double Phi[NX];
        linearize(&m, xit + k * NX, uit + k * NU, dt, Phi, A + k * NX * NX, B + k * NX * NU);
    }
    for (int k = 0; k < N; ++k) {
        const double *yk = yref + k * (NX + NU);
        for (int i = 0; i < NX; ++i)
            q[k * NX + i] = (dyref ? -dt * Wd[i] * dyref[k * (NX + NU) + i] : 0.0)
                          + (dw ? dt * dw[i] * (x[k * NX + i] - yk[i]) : 0.0);
        for (int a = 0; a < NU; ++a)
            r[k * NU + a] = (dyref ? -dt * Wd[NX + a] * dyref[k * (NX + NU) + NX + a] : 0.0)
                          + (dw ? dt * dw[NX + a] * (u[k * NU + a] - yk[NX + a]) : 0.0);
    }
    for (int i = 0; i < NX; ++i)
        q[N * NX + i] = (dyref_e ? -Wed[i] * dyref_e[i] : 0.0) + (dwe ? dwe[i] * (x[N * NX + i] - yref_e[i]) : 0.0);
    qp_t qp; qp.N = N; qp.A = A; qp.B = B; qp.c = zx; qp.q = q; qp.r = r; qp.lb = 0; qp.ub = 0;
    double x0[NX] = {0};
    if (dx0) memcpy(x0, dx0, sizeof(x0));
    qp.x0 = x0;
    for (int i = 0; i < NX; ++i) { qp.Qd[i] = dt * Wd[i]; qp.QNd[i] = Wed[i]; }
    for (int a = 0; a < NU; ++a) qp.Rd[a] = dt * Wd[NX + a];
    int ok = riccati(&qp, NULL, r, act, zu, xs, du);
    if (dx) memcpy(dx, xs, sizeof(double) * (N + 1) * NX);
    free(A); free(B); free(zx); free(zu); free(q); free(r); free(xs);
    return ok;
}
