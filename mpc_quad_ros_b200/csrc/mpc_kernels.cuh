// mpc_kernels.cuh — the two kernels behind qmpc_solve (one SQP-RTI iteration per vehicle).
//
//   K1  qmpc_linearize_kernel : RK4 + forward sensitivities (incl. GP Jacobian) at the N nodes of every
//       vehicle.  Two phases: the primal (with the GP term) once per node, then one sensitivity column per lane on
//       cached Jacobian blocks (see LIN_NB below).  Replaces CasADi expl_vde_forw +
//       acados ERK inside AcadosOcpSolver.solve() (reference src/quad_opt.py:333, model :164-262).
//   K2  qmpc_ipm_kernel       : Gauss-Newton QP (LINEAR_LS cost scaled by dt, x0 pinned, box on u) solved by a
//       Mehrotra predictor-corrector IPM whose Newton systems are Riccati recursions; one OCP per warp.
//       Replaces acados SQP_RTI + full condensing + HPIPM (reference src/quad_opt.py:146-151,333;
//       src/_acados_ocp.json:2082-2110).  Full step, un-shifted persistent iterate, objective at the new
//       iterate (SURVEY.md App. A.3).
//   qmpc_sens_kernel      : behind qmpc_eval_sens_x0, not part of a solve: derivatives of the last solve's x[k], u[k] with
//       respect to x0 (acados eval_param_sens "ex"), one OCP per warp from the tiles and the active set the solve left.
//   qmpc_adjoint_kernel   : behind qmpc_eval_adjoint, not part of a solve: reverse mode of the same map, the gradients w.r.t.
//       x0, yref and yref_e of <x_bar, x> + <u_bar, u> for given cotangents, one OCP per warp; its WGT instantiation
//       (qmpc_eval_adjoint_weights) adds the gradients w.r.t. the cost weights w_diag / we_diag.
//   qmpc_jvp_kernel       : behind qmpc_eval_jvp, not part of a solve: forward mode of the same map w.r.t. x0, yref,
//       yref_e and the cost weights, K tangent directions per vehicle on one pinned factorisation, one OCP per warp.
//
// Per-stage tile written by K1 and streamed by K2 (HBM/L2, `real`):   W[13 rows][16 cols], row stride WR
//   cols 0..3  = B = dPhi/du            cols 4..13 = dPhi/dx_s for s = 3..12 (q,v,r)
//   col 14     = b = Phi(x_k,u_k) - x_{k+1}  (QP in increments)        col 15 = q = dt*W_x (x_k - xref_k)
// The three position columns of A are unit vectors (f does not depend on p) and are never stored.
#pragma once
#include "common.cuh"
#include "model.cuh"

namespace qmpc {

constexpr int QMPC_STATUS_OK_ = 0, QMPC_STATUS_MAXITER_ = 1, QMPC_STATUS_NAN_ = 2;
#ifndef QMPC_WR
#define QMPC_WR 18               // row stride of a stage tile in reals (18: rows 144 B apart, bank-conflict-free row reads from shared memory)
#endif
#ifndef QMPC_RING
#define QMPC_RING 2              // Riccati kernel: stage tiles staged through a shared-memory ring of this many slots by TMA bulk copies (0: read from L2/L1)
#endif
constexpr int WR = QMPC_WR;
constexpr int WT = 13 * WR;  // reals per stage tile
constexpr int FAC = 72;      // reals per stage factor record: Lx[13][4], lg[4], Lam[10], lgc[4], pad[2]

// real = arithmetic of the RK4 / sensitivity propagation, treal = storage type of the stage tiles.  fp32 handles run
// <double, float>: the defect b = Phi - x_{k+1} and the gradient q = dt W (x - xref) are differences of O(10) quantities -
// formed in fp32 they carry 1e-6 absolute noise that the feedback gains turn into 1e-4..1e-2 of control error; formed in
// fp64 and rounded once, their error is relative to their own (small) size.
template <typename real, typename treal = real>
struct LinArgs {
    int B, N;
    real dt;
    ModelParams<real> mp;
    real Qd[13];          // dt * w_diag[0:13]
    const double* xit;    // [B][N+1][13]
    const double* uit;    // [B][N][4]
    const double* yref;   // [B][N][17]
    const double* alpha;  // [B][3][M]  (unused when mp.M == 0)
    int alpha_stride;     // doubles between vehicles: 3*M, or 0 when one shared model serves every vehicle
    const double* gpX;    // [3][M]
    treal* W;             // [B][N][13][16]
};

// K1 runs in two phases per block of LIN_NB nodes (the primal is evaluated ONCE per node, not once per sensitivity column):
//   phase A, lane = node:   RK4 of the nominal + GP dynamics; at each of the four stage points the lane leaves what the
//                           tangent needs (q, r and the velocity-row Jacobian blocks: LIN_SF reals) in shared memory,
//                           field-major so that the stores are conflict-free, and finally Phi(x_k, u_k);
//   phase B, 16 lanes/node: lane j carries tile column j (one unit seed) through the four cached stage points with the
//                           hand-written tangent jvp_cached - every read of a stage field is a broadcast - and stores its column.
// No shuffles, one block barrier.  The 3M kernel evaluations of the GP are spread over the lanes by construction (each
// lane owns a node), so nothing is reduced across lanes either.
constexpr int LIN_NB = 32;                 // nodes per block
constexpr int LIN_THREADS = 64;
constexpr int LIN_SF = 31;                 // q4 r3 Cq12 Cv9 Rz3 (model.cuh velocity_jacobian)
constexpr int LIN_NF = 4 * LIN_SF + NX;    // four stage points + Phi

template <typename real>
__device__ __forceinline__ void gp_eval(const ModelParams<real>& mp, const double* __restrict__ gpX, const double* __restrict__ alpha,
                                        const real* vb, real* mu, real* dmu)
{
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const real il2 = mp.iL2[d], sf2 = mp.sf2[d], v = vb[d];
        const double* X = gpX + d * mp.M;
        const double* al = alpha + d * mp.M;
        real s = 0, ds = 0;
        if (mp.gdx[d] > real(0)) {
            // equispaced axis: k_m = exp(-(v - X_m)^2 / 2L^2) obeys k_{m+-1} = k_m rho_m, rho_{m+-1} = rho_m exp(-dx^2 / L^2).
            // Started at the basis point nearest to v and run outwards, every factor is <= 1: the values decay
            // monotonically (no overflow; underflow is the correct limit).  3 exps per axis instead of M.
            const real dx = mp.gdx[d], g = dx * il2, cc = mp.gcc[d];
            real t = (v - mp.gx0[d]) * mp.gidx[d];
            t = fmin(fmax(t, real(0)), real(mp.M - 1));
            const int ms = int(rint(t));
            const real es = v - real(__ldg(X + ms));
            const real ks = rexp<real>(real(-0.5) * es * il2 * es);
            real q = real(__ldg(al + ms)) * ks;
            s = q; q *= es;
            real k = ks, rho = rexp<real>((es - real(0.5) * dx) * g), e = es;
#pragma unroll 4
            for (int m = ms + 1; m < mp.M; ++m) {
                k *= rho; rho *= cc; e -= dx;
                const real ka = real(__ldg(al + m)) * k;
                s += ka; q = fma(ka, e, q);
            }
            k = ks; rho = rexp<real>(-(es + real(0.5) * dx) * g); e = es;
#pragma unroll 4
            for (int m = ms - 1; m >= 0; --m) {
                k *= rho; rho *= cc; e += dx;
                const real ka = real(__ldg(al + m)) * k;
                s += ka; q = fma(ka, e, q);
            }
            s *= sf2; ds = -sf2 * il2 * q;
        } else {
#pragma unroll 4
            for (int i = 0; i < mp.M; ++i) {
                const real e = v - real(__ldg(X + i));
                const real ka = sf2 * real(__ldg(al + i)) * rexp<real>(real(-0.5) * e * il2 * e);
                s += ka; ds -= ka * e * il2;
            }
        }
        mu[d] = s; dmu[d] = ds;
    }
}

// phase A for one node: o = field 0 of the node inside its chunk of LIN_NB nodes (fields LIN_NB reals apart)
template <typename real, typename treal>
__device__ __forceinline__ void lin_primal(const LinArgs<real, treal>& a, int node, real* o)
{
    const int b = node / a.N, k = node - b * a.N;
    const double* xk = a.xit + ((size_t)b * (a.N + 1) + k) * NX;
    const double* uk = a.uit + ((size_t)b * a.N + k) * NU;
    const double* al = a.alpha + (size_t)b * a.alpha_stride;
    real x[NX], u[NU], kprev[NX], accx[NX];
#pragma unroll
    for (int i = 0; i < NX; ++i) { x[i] = real(__ldg(xk + i)); accx[i] = x[i]; kprev[i] = 0; }
#pragma unroll
    for (int i = 0; i < NU; ++i) u[i] = real(__ldg(uk + i));
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        const real as = s == 0 ? real(0) : (s == 3 ? a.dt : a.dt * real(0.5));
        const real ws = (s == 0 || s == 3) ? a.dt / real(6) : a.dt / real(3);
        real xs[NX], kk[NX], mu[3] = {0, 0, 0}, dmu[3] = {0, 0, 0};
#pragma unroll
        for (int i = 0; i < NX; ++i) xs[i] = x[i] + as * kprev[i];
        if (a.mp.M > 0) {
            real vb[3];
            body_velocity(xs, vb);
            gp_eval(a.mp, a.gpX, al, vb, mu, dmu);
        }
        EvalPoint<real> e;
        eval_f(a.mp, xs, u, mu, dmu, e, kk);
        real Cq[12], Cv[9];
        velocity_jacobian(e, Cq, Cv);
        real* os = o + (size_t)s * LIN_SF * LIN_NB;
#pragma unroll
        for (int i = 0; i < 4; ++i) os[i * LIN_NB] = e.q[i];
#pragma unroll
        for (int i = 0; i < 3; ++i) { os[(4 + i) * LIN_NB] = e.r[i]; os[(28 + i) * LIN_NB] = e.R[3 * i + 2]; }
#pragma unroll
        for (int i = 0; i < 12; ++i) os[(7 + i) * LIN_NB] = Cq[i];
#pragma unroll
        for (int i = 0; i < 9; ++i) os[(19 + i) * LIN_NB] = Cv[i];
#pragma unroll
        for (int i = 0; i < NX; ++i) { accx[i] += ws * kk[i]; kprev[i] = kk[i]; }
    }
#pragma unroll
    for (int i = 0; i < NX; ++i) o[(size_t)(4 * LIN_SF + i) * LIN_NB] = accx[i];
}

// phase B for tile column j of one node
template <typename real, typename treal>
__device__ __forceinline__ void lin_tangent(const LinArgs<real, treal>& a, int node, int j, const real* o)
{
    const int sj = (j >= 4 && j < 14) ? j - 1 : -1;    // state index of this lane's x-direction
    const int b = node / a.N, k = node - b * a.N;
    if (j >= 12) {       // columns 14 / 15 read x_k, x_{k+1}, yref_k from global memory after the tangent columns: warm L1 now
        const double* late = j < 14 ? a.xit + ((size_t)b * (a.N + 1) + k) * NX : a.yref + ((size_t)b * a.N + k) * NY;
        prefetch_l1(late + (j & 1) * 16);
    }
    real dkprev[NX], accd[NX];
#pragma unroll
    for (int i = 0; i < NX; ++i) { dkprev[i] = 0; accd[i] = (i == sj) ? real(1) : real(0); }
    if (j < 14) {
        // input columns (j < 4): thrust enters v_dot through R[:,2] T/m, the body torques are constants of the column
        const real usel = j < 4 ? a.mp.thrust_over_mass : real(0);
        const int ju = j < 4 ? j : 0;
        const real tq[3] = {j < 4 ? a.mp.T * a.mp.yf[ju] * a.mp.invJ[0] : real(0), j < 4 ? -a.mp.T * a.mp.xf[ju] * a.mp.invJ[1] : real(0),
                            j < 4 ? a.mp.T * a.mp.zt[ju] * a.mp.invJ[2] : real(0)};
        const real kr[3] = {a.mp.Jc[0] * a.mp.invJ[0], a.mp.Jc[1] * a.mp.invJ[1], a.mp.Jc[2] * a.mp.invJ[2]};
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const real as = s == 0 ? real(0) : (s == 3 ? a.dt : a.dt * real(0.5));
            const real ws = (s == 0 || s == 3) ? a.dt / real(6) : a.dt / real(3);
            const real* os = o + (size_t)s * LIN_SF * LIN_NB;
            real q[4], r[3], Cq[12], Cv[9], uz[3];
#pragma unroll
            for (int i = 0; i < 4; ++i) q[i] = os[i * LIN_NB];
#pragma unroll
            for (int i = 0; i < 3; ++i) { r[i] = os[(4 + i) * LIN_NB]; uz[i] = usel * os[(28 + i) * LIN_NB]; }
#pragma unroll
            for (int i = 0; i < 12; ++i) Cq[i] = os[(7 + i) * LIN_NB];
#pragma unroll
            for (int i = 0; i < 9; ++i) Cv[i] = os[(19 + i) * LIN_NB];
            real dxs[NX], dk[NX];
#pragma unroll
            for (int i = 0; i < NX; ++i) dxs[i] = ((i == sj) ? real(1) : real(0)) + as * dkprev[i];
            jvp_cached(q, r, Cq, Cv, uz, kr, tq, dxs, dk);
#pragma unroll
            for (int i = 0; i < NX; ++i) { accd[i] += ws * dk[i]; dkprev[i] = dk[i]; }
        }
    } else if (j == 14) {                              // b = Phi - x_{k+1}
        const double* xn = a.xit + ((size_t)b * (a.N + 1) + k + 1) * NX;
#pragma unroll
        for (int i = 0; i < NX; ++i) accd[i] = o[(size_t)(4 * LIN_SF + i) * LIN_NB] - real(__ldg(xn + i));
    } else {                                           // q = dt W_x (x_k - xref_k)
        const double* xk = a.xit + ((size_t)b * (a.N + 1) + k) * NX;
        const double* yr = a.yref + ((size_t)b * a.N + k) * NY;
#pragma unroll
        for (int i = 0; i < NX; ++i) accd[i] = a.Qd[i] * (real(__ldg(xk + i)) - real(__ldg(yr + i)));
    }
    treal* Wt = a.W + (size_t)node * WT;
#pragma unroll
    for (int i = 0; i < NX; ++i) Wt[i * WR + j] = treal(accd[i]);
}

template <typename real, typename treal = real>
__global__ void __launch_bounds__(LIN_THREADS) qmpc_linearize_kernel(LinArgs<real, treal> a)
{
    QMPC_STATIC_SMEM(real, sd, LIN_NF * LIN_NB);       // [field][node of the block]
    const int tid = threadIdx.x;
    const int total = a.B * a.N, base = blockIdx.x * LIN_NB;
    if (tid < LIN_NB && base + tid < total) lin_primal(a, base + tid, sd + tid);
    __syncthreads();
    const int j = tid & 15;
    for (int it = 0; it < LIN_NB * 16 / LIN_THREADS; ++it) {
        const int nl = it * (LIN_THREADS / 16) + (tid >> 4), node = base + nl;
        if (node < total) lin_tangent(a, node, j, sd + nl);
    }
}

// ------------------------------------------------------------------------------------------ K2

template <typename real>
struct IpmArgs {
    int B, N;
    real Qd[13], QNd[13], Rd[4];   // dt*W_x, W_e, dt*W_u
    real dt, lb, ub, mu_tol;
    real lam0_scale, lam0_min, lam0_max;   // initial multipliers of the cold IPM: clip(scale * mean|dJ/du(centre)|, min, max)
    real mu_switch;                // complementarity at which the IPM hands over to the active-set refinement
    real refine_gtol;              // sign tolerance on the multipliers of pinned inputs
    real resfac_final;             // an IPM-only exit also needs the initial stationarity residual reduced to this fraction
    int max_iter;
    int max_iter_failed;           // iteration limit of a vehicle whose last two solves failed (fail_streak >= 2)
    const int* fail_streak;        // [B] consecutive failed solves, or null
    int max_refine;                // refinement rounds after the IPM; 0 = pure IPM down to mu_tol
    int warm_rounds;               // refinement rounds tried FIRST from the previous solve's active set; 0 = off
    int dense_warm_rounds;         // dense kernel: active-set rounds from the handed-over guess before the IPM; 0 = IPM first
    int warm_rounds_busy;          // screening mode: round limit of a busy step (see unsettled_prev); 0 = warm_rounds
    int bail_round_busy;           // bail_round of a busy step
    int bail_to_ipm;               // screening mode: an OCP whose rounds gave up (cycle, not contracting) skips the dense kernel's warm rounds
    int skip_screen_iters;         // screening mode: previous-solve IPM iterations from which an OCP skips the rounds (0 = never)
    int busy_threshold;            // a step is busy when the previous step left more than this many OCPs unsettled after warm_rounds
    const int* unsettled_prev;     // device counters (previous / this step) of OCPs not settled after warm_rounds rounds, or null
    int* unsettled_cur;
    int bail_round;                // rounds (0-based) from which a non-contracting change count ends the attempt (default 2)
    int bail_changed;              // a round that still moves more inputs than this ends the attempt at once (default: never)
    int final_rollout;             // 1: always roll the horizon out at the end (A/B knob)
    int post_bail;                 // 1: the rounds after the IPM may give up early too (fp32: rounding noise can keep them busy)
    int smem_per_warp;             // reals
    int refine_off;                // fp32 handles: offset (reals) of the fp64 scratch of the iterative refinement, 0 = none
    int ring_off;                  // offset (reals) of the tile ring + its mbarriers inside the per-warp block (QMPC_RING builds)
    const double* x0;              // [B][13]
    const double* yref;            // [B][N][17]
    const double* yref_e;          // [B][13]
    double* xit;                   // [B][N+1][13]  in/out
    double* uit;                   // [B][N][4]     in/out
    const real* W;                 // [B][N][13][16] (+1 padding tile)
    real* fac;                     // [B][N][FAC]
    unsigned char* act;            // [B][4N] active set of the previous solve: 0 free, 1 lower, 2 upper, 255 unknown
    double* u0;                    // [B][4]
    double* cost;                  // [B]
    int* status;                   // [B]
    int* iters;                    // [B]  IPM iterations
    int* rounds;                   // [B]  active-set refinement rounds (warm + after the IPM)
    long long* timeline;           // [B][2] %globaltimer at start / end of each OCP, or null (measurement hook)
    int* hard_list;                // screening mode (hard_count != null): an OCP whose warm-started rounds do not settle is
    int* hard_count;               // appended here for the dense kernel instead of running the IPM in this warp
};

// IPM iteration limit of this solve: a vehicle whose last two or more solves failed gets a bounded attempt, except every
// eighth failure in a row, which gets the full limit again (a reset problem that needs more than max_iter_failed
// iterations must not stay failed for ever)
template <typename real>
__device__ __forceinline__ int iter_limit(const IpmArgs<real>& a, int ocp)
{
    if (!a.fail_streak) return a.max_iter;
    const int s = a.fail_streak[ocp];
    return (s >= 2 && (s & 7) != 0) ? a.max_iter_failed : a.max_iter;
}

__device__ __forceinline__ long long global_ns()
{
#ifdef QMPC_EMU
    return 0;
#else
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
#endif
}

template <typename real> struct Vec2;
template <> struct Vec2<double> { typedef double2 type; };
template <> struct Vec2<float> { typedef float2 type; };

// two consecutive reals with one load (p must be aligned to 2 reals)
template <typename real>
__device__ __forceinline__ void ld2(const real* p, real& a, real& b)
{
    const typename Vec2<real>::type v = *reinterpret_cast<const typename Vec2<real>::type*>(p);
    a = v.x; b = v.y;
}
template <typename real>
__device__ __forceinline__ void ldg2(const real* p, real& a, real& b)
{
    const typename Vec2<real>::type v = __ldg(reinterpret_cast<const typename Vec2<real>::type*>(p));
    a = v.x; b = v.y;
}

template <typename real>
__device__ __forceinline__ void st2(real* p, real a, real b)
{
    typename Vec2<real>::type v;
    v.x = a; v.y = b;
    *reinterpret_cast<typename Vec2<real>::type*>(p) = v;
}

template <typename real>
struct Chol4 {   // Lam = chol(M_uu) with reciprocal diagonal; inputs / outputs of any floating type, arithmetic in `real`
    real l10, l20, l21, l30, l31, l32, i0, i1, i2, i3;
    // NOBRANCH (double only): reciprocal square roots without the library's special-case branch (common.cuh rsqrt_nobranch)
    template <typename T, bool NOBRANCH = false>
    __device__ __forceinline__ void factor(const T* M /* 4x4 row-major, lower used */)
    {
        auto rs = [](real x) -> real {
            if constexpr (NOBRANCH && sizeof(real) == 8) return real(rsqrt_nobranch(double(x)));
            else return rrsqrt<real>(x);
        };
        i0 = rs(real(M[0]));
        l10 = real(M[4]) * i0; l20 = real(M[8]) * i0; l30 = real(M[12]) * i0;
        i1 = rs(real(M[5]) - l10 * l10);
        l21 = (real(M[9]) - l20 * l10) * i1; l31 = (real(M[13]) - l30 * l10) * i1;
        i2 = rs(real(M[10]) - l20 * l20 - l21 * l21);
        l32 = (real(M[14]) - l30 * l20 - l31 * l21) * i2;
        i3 = rs(real(M[15]) - l30 * l30 - l31 * l31 - l32 * l32);
    }
    // Keeps the factorisation where it is written: without it the compiler sinks factor() into each of the divergent
    // branches that use the result (tile rows / right-hand side / diagonal), and a warp then runs the 4x4 Cholesky's
    // dependent chain once per branch, one after the other (seen in the SASS of the dense kernel: three copies).
    __device__ __forceinline__ void pin()
    {
#ifndef QMPC_EMU
        if constexpr (sizeof(real) == 8)
            asm volatile("" : "+d"(l10), "+d"(l20), "+d"(l21), "+d"(l30), "+d"(l31), "+d"(l32), "+d"(i0), "+d"(i1), "+d"(i2), "+d"(i3));
        else
            asm volatile("" : "+f"(l10), "+f"(l20), "+f"(l21), "+f"(l30), "+f"(l31), "+f"(l32), "+f"(i0), "+f"(i1), "+f"(i2), "+f"(i3));
#endif
    }
    template <typename TI, typename TO>
    __device__ __forceinline__ void fsolve(const TI* v, TO* z) const   // Lam z = v
    {
        const real z0 = real(v[0]) * i0;
        const real z1 = (real(v[1]) - l10 * z0) * i1;
        const real z2 = (real(v[2]) - l20 * z0 - l21 * z1) * i2;
        const real z3 = (real(v[3]) - l30 * z0 - l31 * z1 - l32 * z2) * i3;
        z[0] = TO(z0); z[1] = TO(z1); z[2] = TO(z2); z[3] = TO(z3);
    }
    template <typename TI, typename TO>
    __device__ __forceinline__ void bsolve_neg(const TI* v, TO* u) const   // Lam^T u = -v
    {
        const real u3 = -real(v[3]) * i3;
        const real u2 = (-real(v[2]) - l32 * u3) * i2;
        const real u1 = (-real(v[1]) - l21 * u2 - l31 * u3) * i1;
        const real u0 = (-real(v[0]) - l10 * u1 - l20 * u2 - l30 * u3) * i0;
        u[0] = TO(u0); u[1] = TO(u1); u[2] = TO(u2); u[3] = TO(u3);
    }
    template <typename TO>
    __device__ __forceinline__ void store(TO* p) const
    {
        p[0] = TO(l10); p[1] = TO(l20); p[2] = TO(l21); p[3] = TO(l30); p[4] = TO(l31); p[5] = TO(l32);
        p[6] = TO(i0); p[7] = TO(i1); p[8] = TO(i2); p[9] = TO(i3);
    }
    template <typename TI>
    __device__ __forceinline__ void load(const TI* p)
    {
        TI a, b;
        ld2(p, a, b); l10 = real(a); l20 = real(b);
        ld2(p + 2, a, b); l21 = real(a); l30 = real(b);
        ld2(p + 4, a, b); l31 = real(a); l32 = real(b);
        ld2(p + 6, a, b); i0 = real(a); i1 = real(b);
        ld2(p + 8, a, b); i2 = real(a); i3 = real(b);
    }
};

// ---- cycle detection of the primal-dual active-set rounds: 64-bit fingerprint of an active set (sum over the inputs of
// a per-(input, state) odd multiplier; lanes add their elements, warp_sum completes it) and the last few fingerprints.
template <typename real>
__device__ __forceinline__ unsigned long long active_set_term(int e, real f)
{
    const unsigned long long k = (unsigned long long)(e + 1) * 0x9E3779B97F4A7C15ull;
    return f == real(0) ? 0ull : (f == real(1) ? (k | 1ull) : (k * 0xC2B2AE3D27D4EB4Full) | 1ull);
}
struct ActiveSetHistory {      // storage in shared memory (registers are the scarce resource of both solver kernels)
    static constexpr int DEPTH = 6;
    unsigned long long* h;
    int n;
    __device__ __forceinline__ void init(void* storage) { h = reinterpret_cast<unsigned long long*>(storage); n = 0; }
    __device__ __forceinline__ void clear() { n = 0; }
    // warp-collective: every lane passes the same fingerprint; returns whether it was met before, then records it
    __device__ __forceinline__ bool seen_then_push(unsigned long long fp, int lane)
    {
        bool hit = false;
        const int m = n < DEPTH ? n : DEPTH;
        for (int i = 0; i < m; ++i) hit = hit || h[i] == fp;
        __syncwarp();
        if (lane == 0) h[n % DEPTH] = fp;
        __syncwarp();
        ++n;
        return hit;
    }
};

template <typename real>
__device__ __forceinline__ real dot4(const real* a, const real* b)
{
    return a[0] * b[0] + a[1] * b[1] + a[2] * b[2] + a[3] * b[3];
}
template <typename real>
__device__ __forceinline__ real sel4(const real* v, int i)   // v[i] for a register array and a run-time i
{
    return i == 0 ? v[0] : (i == 1 ? v[1] : (i == 2 ? v[2] : v[3]));
}

// per-warp shared-memory carve-up (offsets in reals; every block starts on an even offset)
constexpr int PS = 14;         // row stride of P (even: rows are read two reals at a time)
constexpr int SM_P = 0;        // 14 x 14 (row 13 stays zero)
constexpr int SM_PV = 200;     // 16  costate offset p
constexpr int SM_WV = 216;     // 16  forward vector: u(4), z(10), one, zero
constexpr int SM_XP = 232;     // 16  position part of the forward state
constexpr int SM_HV = 248;     // 16  h = P b + p
constexpr int SM_LS = 264;     // 64  l_j per tile column
constexpr int SM_CS = 328;     // 32  Muu(16) Mpu(12) gu(4)
constexpr int SM_VEC = 360;    // 13 vectors of 4N, then the state trajectory (N+1) x 13 of the refinement
constexpr int SM_NVEC = 13;

template <typename real> __host__ __device__ constexpr int HIST_REALS() { return 64 / (int)sizeof(real); }   // 64 bytes

// One tangent direction of qmpc_eval_jvp and what its linear costs are formed from (WarpCtx::backward_cotangent<true>):
// the tangents of the reference and the cost weights (any may be null = zero) and the last solve's solution and reference.
struct TanDir {
    const double *dyref, *dyref_e, *dw, *dwe;   // [N][17], [13], [17], [13]
    const double *xs, *us, *yr, *yre;           // [(N+1)][13], [N][4], [N][17], [13]
};

template <typename real>
struct WarpCtx {
    const IpmArgs<real>& a;
    int lane, h, j, sidx, ocp, N, E;
    unsigned hmask;
    real *P, *pv, *wv, *xp, *hv, *Ls, *cs;
    real *rt, *dR, *usol, *ua, *ucur, *ll, *lu, *ubar, *rdel, *cl, *cu, *tl, *tu, *xtr;
    real *fx, *fv, *grad;          // aliases of cl, cu, ua while the active set is refined
    const real* Wv;
    real* facv;
    const double *x0, *yref, *yref_e;
    double *xit, *uit;

    // ---- stage tiles.  RING (fp64 builds with QMPC_RING > 0): a sweep streams its tiles through RING shared-memory slots;
    // lane 0 issues one TMA bulk copy per stage (cp.async.bulk + mbarrier, RING - 1 stages ahead of the compute), the warp
    // waits on the slot's barrier and reads the tile with LDS.  Otherwise the tile is read in place (L2/L1, __ldg).
    static constexpr int RING = (sizeof(real) == 8) ? QMPC_RING : 0;
    bool gave_up;                    // the last refine_rounds ended on a cycle / a non-contracting change count (not on its round limit)
    void* hist_store;                // 6 x 8 bytes: active-set fingerprints of the running attempt (cycle detection)
    real* ring;                      // RING slots of WT reals
    unsigned long long* rbar;        // one mbarrier per slot
    unsigned rphase;                 // bit s: parity of the next completion of slot s

    __device__ __forceinline__ static real tld(const real* p) { return RING ? *p : __ldg(p); }
    __device__ __forceinline__ static void tld2(const real* p, real& x, real& y) { if (RING) ld2(p, x, y); else ldg2(p, x, y); }

    __device__ __forceinline__ void ring_issue(int slot, int k) const
    {
        if (lane == 0) {
            mbar_expect(rbar + slot, (unsigned)(WT * sizeof(real)));
            bulk_g2s(ring + slot * WT, Wv + (size_t)k * WT, (unsigned)(WT * sizeof(real)), rbar + slot);
        }
    }
    // start of a sweep over stages k0, k0 + dir, ...: fill the ring
    __device__ __forceinline__ void sweep_begin(int k0, int dir) const
    {
        if (RING) {
            __syncwarp();            // the slots' last readers are done
#pragma unroll
            for (int s = 0; s < RING; ++s) { const int k = k0 + s * dir; if (k >= 0 && k < N) ring_issue(s, k); }
        }
    }
    // tile of the i-th stage of the sweep (stage index k)
    __device__ __forceinline__ const real* tile_at(int i, int k)
    {
        if (RING) {
            const int s = i % (RING ? RING : 1);
            bulk_wait_warp(rbar + s, (rphase >> s) & 1u);
            rphase ^= 1u << s;
            return ring + s * WT;
        }
        return Wv + (size_t)k * WT;
    }
    // call after a warp barrier that follows the last read of the i-th tile: refills its slot with stage knext
    __device__ __forceinline__ void tile_done(int i, int knext) const
    {
        if (RING) { if (knext >= 0 && knext < N) ring_issue(i % (RING ? RING : 1), knext); }
    }

    __device__ __forceinline__ void load_col(const real* tile, real* w) const
    {
        const real* t = tile + j;
#pragma unroll
        for (int i = 0; i < NX; ++i) w[i] = tld(t + i * WR);
    }

    // L1 prefetch of the tile (13 lines) and factor record (<= 6 lines) of the stage the sweep visits next
    __device__ __forceinline__ void prefetch_stage(int k, bool with_fac) const
    {
        if (k < 0 || k >= N) return;
        if (!RING && lane < NX) prefetch_l1(Wv + (size_t)k * WT + lane * WR);
        else if (with_fac && lane >= NX && lane < NX + 6) prefetch_l1(reinterpret_cast<const char*>(facv + (size_t)k * FAC) + (lane - NX) * 128);
    }

    // Backward Riccati sweep with factorisation.  Gradient: rt (inputs), q column (states), b column (offset).
    // FIXED: inputs flagged in fx are pinned at fv (exact elimination: their rows/columns of M_uu, M_ux become
    // identity/zero and M[:,a] fv_a moves into the gradient); rt = rdel and dR = 0 in that mode.
    //
    // lane = (h, j): tile column j (0..3 B, 4..13 A', 14 b, 15 q); half h owns rows 7h..7h+6 of y = P w_j and
    // rows 8h..8h+7 of this column of M = W^T P W.
    template <bool FIXED>
    __device__ void backward_full()
    {
        for (int idx = lane; idx < 196; idx += 32) P[idx] = 0;
        __syncwarp();
        if (lane < NX) {
            P[lane * PS + lane] = a.QNd[lane];
            pv[lane] = a.QNd[lane] * real(xit[(size_t)N * NX + lane] - yref_e[lane]);
        }
        __syncwarp();
        const int r0 = 7 * h, o0 = 7 - r0, cb = 8 * h;
        sweep_begin(N - 1, -1);
        for (int k = N - 1; k >= 0; --k) {
            const real* tile = tile_at(N - 1 - k, k);
            real w[NX];
            load_col(tile, w);
            prefetch_stage(k - 1, false);
            const real qj = sidx >= 0 ? tld(tile + sidx * WR + 15) : real(0);
            // y = P w: rows r0..r0+6 here, rows o0..o0+6 from the partner lane (row 13 is the zero padding row)
            real ym[7], yo[7];
#pragma unroll
            for (int ii = 0; ii < 7; ++ii) {
                const real* pr = P + (r0 + ii) * PS;
                real s0 = 0, s1 = 0;
#pragma unroll
                for (int c = 0; c < 12; c += 2) {
                    real p0, p1;
                    ld2(pr + c, p0, p1);
                    s0 += p0 * w[c]; s1 += p1 * w[c + 1];
                }
                ym[ii] = s0 + s1 + pr[12] * w[12];
            }
#pragma unroll
            for (int ii = 0; ii < 7; ++ii) yo[ii] = __shfl_xor_sync(FULL, ym[ii], 16);
            if (lane == 14) {                      // h = P b + p  (lane 14: r0 = 0, o0 = 7)
#pragma unroll
                for (int ii = 0; ii < 7; ++ii) hv[ii] = ym[ii] + pv[ii];
#pragma unroll
                for (int ii = 0; ii < 6; ++ii) hv[7 + ii] = yo[ii] + pv[7 + ii];
            }
            // rows cb..cb+7 of this lane's column of M:  M[i][j] = sum_r W[r][i] y[r]
            real m[8];
#pragma unroll
            for (int ii = 0; ii < 8; ++ii) m[ii] = 0;
#pragma unroll
            for (int kk = 0; kk < 7; ++kk) {
                const real* tr = tile + (r0 + kk < NX ? r0 + kk : NX - 1) * WR + cb;   // y is 0 on the padding row
#pragma unroll
                for (int c = 0; c < 8; c += 2) {
                    real t0, t1;
                    tld2(tr + c, t0, t1);
                    m[c] += t0 * ym[kk]; m[c + 1] += t1 * ym[kk];
                }
            }
#pragma unroll
            for (int kk = 0; kk < 7; ++kk) {
                const real* tr = tile + (o0 + kk < NX ? o0 + kk : NX - 1) * WR + cb;
#pragma unroll
                for (int c = 0; c < 8; c += 2) {
                    real t0, t1;
                    tld2(tr + c, t0, t1);
                    m[c] += t0 * yo[kk]; m[c + 1] += t1 * yo[kk];
                }
            }
            // cost diagonal of this column (added where the diagonal entry is consumed)
            const real dg = j < 4 ? a.Rd[j] + (FIXED ? real(0) : dR[k * 4 + j]) : (j < 14 ? a.Qd[j - 1] : real(0));
            __syncwarp();                          // hv visible; every read of the old P and of the tile is done
            tile_done(N - 1 - k, k - RING);
            real g = 0;
#pragma unroll
            for (int c = 0; c < 12; c += 2) {
                real h0, h1;
                ld2(hv + c, h0, h1);
                g += w[c] * h0 + w[c + 1] * h1;
            }
            g += w[12] * hv[12];
            g += (j < 4) ? (FIXED ? rdel[k * 4 + j] : rt[k * 4 + j]) : qj;
            real mu4[4];                           // rows 0..3 (inputs) of this lane's column; they live in the h=0 half
#pragma unroll
            for (int aa = 0; aa < 4; ++aa) mu4[aa] = __shfl_sync(FULL, m[aa], j);
            // pinned inputs: fva is 0 for free inputs, keep is the 0/1 mask of the free ones
            real keep[4] = {1, 1, 1, 1}, fva[4] = {0, 0, 0, 0};
            if (FIXED) {
#pragma unroll
                for (int aa = 0; aa < 4; ++aa) { keep[aa] = fx[k * 4 + aa] != real(0) ? real(0) : real(1); fva[aa] = fv[k * 4 + aa]; }
#pragma unroll
                for (int aa = 0; aa < 4; ++aa) g = fma(mu4[aa], fva[aa], g);            // M[:,a] fv_a -> gradient
            }
            if (lane < 4) {
                const real kme = FIXED ? sel4(keep, lane) : real(1);
#pragma unroll
                for (int aa = 0; aa < 4; ++aa) cs[aa * 4 + lane] = FIXED ? m[aa] * (keep[aa] * kme) : m[aa];
#pragma unroll
                for (int pi = 0; pi < 3; ++pi) cs[16 + pi * 4 + lane] = ym[pi];    // M[p_i][a] = (P w_a)[p_i]
                cs[28 + lane] = g * kme;
                // diagonal: cost + barrier term; a pinned input keeps an identity row/column
                cs[lane * 5] = (kme != real(0)) ? cs[lane * 5] + dg : real(1);
            }
            __syncwarp();
            Chol4<double> L;               // fp32 handles too: cond(M_uu) ~ 1e3, its inverse carries the whole feedback gain
            real lg[4], lp[3][4], lj[4], lpme[4];
            real gpme = 0;                         // gradient correction of "my" position row from pinned inputs
            {
                real Muu[16];
#pragma unroll
                for (int t = 0; t < 16; t += 2) ld2(cs + t, Muu[t], Muu[t + 1]);
#if QMPC_RSQRT_NOBRANCH
                L.template factor<real, true>(Muu);
#else
                L.factor(Muu);
#endif
                real gu[4];
                ld2(cs + 28, gu[0], gu[1]); ld2(cs + 30, gu[2], gu[3]);
                L.fsolve(gu, lg);
#pragma unroll
                for (int pi = 0; pi < 3; ++pi) {
                    real mpu[4];
                    ld2(cs + 16 + pi * 4, mpu[0], mpu[1]); ld2(cs + 18 + pi * 4, mpu[2], mpu[3]);
                    if (FIXED) {
#pragma unroll
                        for (int aa = 0; aa < 4; ++aa) mpu[aa] *= keep[aa];
                    }
                    L.fsolve(mpu, lp[pi]);
                }
                // the same for "my" position state (lanes 0..2), addressed with the lane index instead of selects
                real mpu[4];
                const int pme = lane < 3 ? lane : 2;
                ld2(cs + 16 + pme * 4, mpu[0], mpu[1]); ld2(cs + 18 + pme * 4, mpu[2], mpu[3]);
                if (FIXED) {
#pragma unroll
                    for (int aa = 0; aa < 4; ++aa) { gpme = fma(mpu[aa], fva[aa], gpme); mpu[aa] *= keep[aa]; }
                }
                L.fsolve(mpu, lpme);
            }
            if (FIXED) {
#pragma unroll
                for (int aa = 0; aa < 4; ++aa) mu4[aa] *= keep[aa];
            }
            L.fsolve(mu4, lj);
            if (h == 0) {
#pragma unroll
                for (int aa = 0; aa < 4; ++aa) Ls[j * 4 + aa] = lj[aa];
            }
            __syncwarp();
            if (k > 0) {
                if (j >= 4 && j < 14) {
                    const int sj = j - 1;
#pragma unroll
                    for (int ii = 0; ii < 8; ++ii) {
                        const int i = cb + ii;
                        if (i >= 4 && i < 14) {
                            real l0, l1, l2, l3;
                            ld2(Ls + i * 4, l0, l1); ld2(Ls + i * 4 + 2, l2, l3);
                            real v = fma(-l0, lj[0], m[ii]);
                            v = fma(-l1, lj[1], v); v = fma(-l2, lj[2], v); v = fma(-l3, lj[3], v);
                            P[(i - 1) * PS + sj] = v;
                        }
                    }
                    if ((j >> 3) == h) P[sj * PS + sj] += dg;          // state cost on the diagonal (own write above)
                    if (h == 0) {
#pragma unroll
                        for (int pi = 0; pi < 3; ++pi) {
                            const real v = ym[pi] - dot4(lp[pi], lj);
                            P[pi * PS + sj] = v;
                            P[sj * PS + pi] = v;
                        }
                        pv[sj] = g - dot4(lj, lg);
                    }
                }
                if (lane < 3) {
#pragma unroll
                    for (int pi = 0; pi < 3; ++pi) P[pi * PS + lane] -= dot4(lp[pi], lpme);
                    P[lane * PS + lane] += a.Qd[lane];
                    pv[lane] = hv[lane] + qj + gpme - dot4(lpme, lg);
                }
            }
            if (h == 0) {
                real* f = facv + (size_t)k * FAC;
                if (j >= 4 && j < 14) {
#pragma unroll
                    for (int aa = 0; aa < 4; ++aa) f[(j - 1) * 4 + aa] = lj[aa];
                } else if (j < 3) {
#pragma unroll
                    for (int aa = 0; aa < 4; ++aa) f[j * 4 + aa] = lpme[aa];
                } else if (j == 14) {
#pragma unroll
                    for (int aa = 0; aa < 4; ++aa) f[52 + aa] = lg[aa];
                } else if (j == 15) {
                    L.store(f + 56);
                }
            }
            __syncwarp();
        }
    }

    // backward sweep of the gradient only (corrector): zero offset/terminal, input gradient rt
    // PINNED: the factors in `fac` come from a pinned round (backward_full<true>): pinned inputs take no gradient
    template <bool PINNED = false>
    __device__ void backward_vec()
    {
        if (lane < 16) pv[lane] = 0;
        __syncwarp();
        sweep_begin(N - 1, -1);
        for (int k = N - 1; k >= 0; --k) {
            real w[NX];
            load_col(tile_at(N - 1 - k, k), w);
            prefetch_stage(k - 1, true);
            const real* f = facv + (size_t)k * FAC;
            Chol4<double> L;
            L.load(f + 56);
            real lx[4] = {0, 0, 0, 0};
            if (sidx >= 0) { ld2(f + sidx * 4, lx[0], lx[1]); ld2(f + sidx * 4 + 2, lx[2], lx[3]); }
            real g = 0;
#pragma unroll
            for (int c = 0; c < 12; c += 2) {
                real h0, h1;
                ld2(pv + c, h0, h1);
                g += w[c] * h0 + w[c + 1] * h1;
            }
            g += w[12] * pv[12];
            if (j < 4) g += rt[k * 4 + j];
            real gu[4], lgc[4];
#pragma unroll
            for (int aa = 0; aa < 4; ++aa) gu[aa] = __shfl_sync(FULL, g, aa);
            if (PINNED) {
#pragma unroll
                for (int aa = 0; aa < 4; ++aa) if (fx[k * 4 + aa] != real(0)) gu[aa] = 0;
            }
            L.fsolve(gu, lgc);
            const real pold = j < 3 ? pv[j] : real(0);
            __syncwarp();
            tile_done(N - 1 - k, k - RING);
            if (h == 0) {
                if (j >= 4 && j < 14) pv[j - 1] = g - dot4(lx, lgc);
                else if (j < 3) pv[j] = pold - dot4(lx, lgc);
                else if (j == 14) {
#pragma unroll
                    for (int aa = 0; aa < 4; ++aa) facv[(size_t)k * FAC + 66 + aa] = lgc[aa];
                }
            }
            __syncwarp();
        }
    }

    // adjoint sweep at the point (xtr, usol): grad[e] = d(objective)/d(u_e) through the linearised dynamics
    __device__ void backward_adjoint()
    {
        if (lane < NX) pv[lane] = a.QNd[lane] * (xtr[(size_t)N * NX + lane] + real(xit[(size_t)N * NX + lane] - yref_e[lane]));
        __syncwarp();
        sweep_begin(N - 1, -1);
        for (int k = N - 1; k >= 0; --k) {
            real w[NX];
            const real* tile = tile_at(N - 1 - k, k);
            load_col(tile, w);
            prefetch_stage(k - 1, false);
            const real qj = sidx >= 0 ? tld(tile + sidx * WR + 15) : real(0);
            real g = 0;
#pragma unroll
            for (int c = 0; c < 12; c += 2) {
                real h0, h1;
                ld2(pv + c, h0, h1);
                g += w[c] * h0 + w[c + 1] * h1;
            }
            g += w[12] * pv[12];
            const real xk = sidx >= 0 ? xtr[k * NX + sidx] : real(0);
            const real pold = j < 3 ? pv[j] : real(0);
            __syncwarp();
            tile_done(N - 1 - k, k - RING);
            if (h == 0) {
                if (j < 4) grad[k * 4 + j] = g + a.Rd[j] * usol[k * 4 + j] + rdel[k * 4 + j];
                if (j >= 4 && j < 14) pv[j - 1] = g + a.Qd[j - 1] * xk + qj;
                else if (j < 3) pv[j] = pold + a.Qd[j] * xk + qj;
            }
            __syncwarp();
        }
    }

    // ---- fp32 handles only: one step of iterative refinement of the solution of the last pinned round.
    // The fp32 Riccati recursion leaves 1e-5..1e-4 of relative error in du (cancellation in P <- M_xx - l'l).  The residual
    // of the stationarity condition is evaluated in fp64 (state increments rolled out in double, adjoint swept back in
    // double; the tiles themselves are fp32-rounded fp64 values, worth ~1e-6), the correction is solved with the fp32
    // factors already in `fac` (backward_vec + forward<1>, the IPM's corrector path), and the states are re-rolled.
    // dxd: (N+1) x 13 doubles, pvd: 16 doubles of per-warp shared memory.
    __device__ void rollout_fp64(double* dxd, const double* dud) const
    {
        if (lane < NX) dxd[lane] = x0[lane] - xit[lane];
        __syncwarp();
        const int i = lane < NX ? lane : NX - 1;
        for (int k = 0; k < N; ++k) {
            const real* row = Wv + (size_t)k * WT + i * WR;
            const double* dx = dxd + k * NX;
            double acc = double(__ldg(row + 14)) + (i < 3 ? dx[i] : 0.0);
#pragma unroll
            for (int c = 0; c < 4; ++c) acc = fma(double(__ldg(row + c)), dud[k * 4 + c], acc);
#pragma unroll
            for (int s_ = 3; s_ < NX; ++s_) acc = fma(double(__ldg(row + 1 + s_)), dx[s_], acc);
            if (lane < NX) dxd[(k + 1) * NX + lane] = acc;
            __syncwarp();
        }
    }
    // adjoint sweep in double at the inputs usol / states dxd: stationarity residual of every input into rt (fp32 storage;
    // for a pinned input this is its multiplier).  lane j < 16 = tile column (0-3 inputs, 4-13 states 3..12).
    __device__ void adjoint_fp64(const double* dxd, const double* dud, double* pvd)
    {
        if (lane < NX) pvd[lane] = double(a.QNd[lane]) * (dxd[N * NX + lane] + (xit[(size_t)N * NX + lane] - yref_e[lane]));
        __syncwarp();
        for (int k = N - 1; k >= 0; --k) {
            const real* tile = Wv + (size_t)k * WT;
            double g = 0;
            if (lane < 14) {
#pragma unroll
                for (int r = 0; r < NX; ++r) g = fma(double(__ldg(tile + r * WR + lane)), pvd[r], g);
            }
            const double pold = lane < 3 ? pvd[lane] : 0.0;
            const int st = lane < 3 ? lane : lane - 1;                    // state index of lanes 0-2 (positions) and 4-13
            double pn = 0;
            if (lane < 3 || (lane >= 4 && lane < 14))
                pn = (lane < 3 ? pold : g) + double(a.Qd[st]) * dxd[k * NX + st] + double(__ldg(tile + st * WR + 15));
            __syncwarp();
            if (lane < 4) {
                const int e = k * 4 + lane;
                rt[e] = real(g + double(a.Rd[lane]) * dud[e] + double(rdel[e]));
            }
            if (lane < 3 || (lane >= 4 && lane < 14)) pvd[st] = pn;
            __syncwarp();
        }
    }
    // one refinement step, then the active set is CHECKED with the fp64 gradient of the refined point: fp32 multipliers
    // carry ~1e-4 of relative noise, enough to mis-sign a weakly active bound (and a wrong active set is a 1e-2 error).
    // Returns the number of inputs whose status it changed in fx (0: the active set is verified).
    __device__ int refine_solution_fp64(double* dxd, double* pvd, real lb, real ub)
    {
        double* dud = pvd + 16;                      // the input increments in double: fp32 storage of du alone is worth
        for (int e = lane; e < E; e += 32) dud[e] = double(usol[e]);      // |H| * 6e-8 |du| ~ 1e-5 of gradient noise
        __syncwarp();
        for (int step = 0; ; ++step) {
            rollout_fp64(dxd, dud);
            adjoint_fp64(dxd, dud, pvd);
            real rmax = 0;
            for (int e = lane; e < E; e += 32) if (fx[e] == real(0)) rmax = fmax(rmax, fabs(rt[e]));
            rmax = warp_max(rmax);
            if (step == 3 || (step > 0 && rmax < real(2e-7))) break;       // refined: rt holds the gradient at the final point
            for (int e = lane; e < E; e += 32) if (fx[e] != real(0)) rt[e] = 0;
            __syncwarp();
            backward_vec<true>();
            forward<1>();
            __syncwarp();
            for (int e = lane; e < E; e += 32) if (fx[e] == real(0)) dud[e] += double(usol[e]);
            __syncwarp();
        }
        for (int e = lane; e < E; e += 32) usol[e] = real(dud[e]);
        for (int idx = lane; idx < (N + 1) * NX; idx += 32) xtr[idx] = real(dxd[idx]);
        int changed = 0;
        const real gtol = real(1e-6);         // the fp32-rounded tiles themselves are worth ~1e-6 of gradient accuracy
        for (int e = lane; e < E; e += 32) {
            const real f = fx[e], gr = rt[e];
            const double un = double(ubar[e]) + dud[e];
            if (f == real(1)) { if (gr < -gtol) { fx[e] = 0; ++changed; } }
            else if (f == real(2)) { if (gr > gtol) { fx[e] = 0; ++changed; } }
            else if (un < double(lb) - 1e-7) { fx[e] = 1; ++changed; }
            else if (un > double(ub) + 1e-7) { fx[e] = 2; ++changed; }
        }
        changed = warp_sum(changed);
        __syncwarp();
#ifdef QMPC_EMU_TRACE
        if (lane == 0) { double m = 0; int np_ = 0; for (int e = 0; e < E; ++e) { if (fx[e] == real(0)) m = fmax(m, fabs((double)rt[e])); else ++np_; }
            printf("  [trace ocp %d] fp64 check: changed %d, max |residual(free)| after refinement %.3e, pinned %d\n", ocp, changed, m, np_); }
        __syncwarp();
#endif
        return changed;
    }

    // Primal-dual active-set rounds from the active set in fx.  Each round solves the LQR with the active inputs
    // pinned (one factorisation + one forward sweep) and checks the multipliers with an adjoint sweep.
    // Returns true when the active set is self-consistent: usol then holds the exact minimiser of the box-QP.
    // may_bail: give up early when the change count stops contracting (warm start only: the IPM is the fall-back there;
    // after the IPM the rounds run to max_rounds, because giving up means an IPM-accurate instead of an exact answer)
    // mark_round / mark_counter (screening): an OCP still unsettled after mark_round rounds is counted once
    __device__ bool refine_rounds(real lb, real ub, int max_rounds, int& rounds, bool may_bail, int bail_round,
                                  int mark_round = -1, int* mark_counter = nullptr)
    {
        int prev_changed = 1 << 30;
        gave_up = false;
        ActiveSetHistory hist;
        hist.init(hist_store);
        for (int round = 0; round < max_rounds; ++round) {
            int pinned = 0;
            for (int e = lane; e < E; e += 32) {
                fv[e] = fx[e] == real(1) ? lb - ubar[e] : (fx[e] == real(2) ? ub - ubar[e] : real(0));
                pinned += fx[e] != real(0);
            }
            pinned = warp_sum(pinned);
            __syncwarp();
            backward_full<true>();
            forward<0, true>();
            __syncwarp();
            if (pinned) backward_adjoint();       // multipliers are only looked at for pinned inputs
            __syncwarp();
            ++rounds;
            int changed = 0;
            unsigned long long fp = 0;
#ifdef QMPC_EMU_TRACE
            int tr_kmax = -1;
#endif
            for (int e = lane; e < E; e += 32) {
                const real f = fx[e], un = ubar[e] + usol[e], gr = grad[e];
                if (f == real(1)) { if (gr < -a.refine_gtol) { fx[e] = 0; ++changed; } }
                else if (f == real(2)) { if (gr > a.refine_gtol) { fx[e] = 0; ++changed; } }
                else if (un < lb) { fx[e] = 1; ++changed; }
                else if (un > ub) { fx[e] = 2; ++changed; }
                fp += active_set_term(e, fx[e]);
#ifdef QMPC_EMU_TRACE
                if (fx[e] != f) tr_kmax = (e >> 2) > tr_kmax ? (e >> 2) : tr_kmax;
#endif
            }
#ifdef QMPC_EMU_TRACE
            tr_kmax = warp_max(tr_kmax);
#endif
            changed = warp_sum(changed);
            fp = warp_sum(fp);
#ifdef QMPC_EMU_TRACE
            if (lane == 0) {
                int kmax = -1, kmin = 1 << 20, np_ = 0;
                for (int e = 0; e < E; ++e) { if (fx[e] != real(0)) ++np_; }
                printf("  [trace ocp %d] riccati round %d: changed %d pinned %d kmax %d\n", ocp, round + 1, changed, np_, tr_kmax);
            }
#endif
            if (!changed) return true;
            const bool cycling = hist.seen_then_push(fp, lane);   // the deterministic iteration met this active set before: it cycles
            if ((round + 1 == mark_round || (cycling && round + 1 < mark_round)) && mark_counter && lane == 0) atomicAdd(mark_counter, 1);
            if (cycling) { gave_up = true; return false; }
            if (may_bail && round >= bail_round && changed >= prev_changed) { gave_up = true; return false; }   // not contracting: leave it to the IPM
            if (may_bail && round >= 1 && changed > a.bail_changed) { gave_up = true; return false; }
            prev_changed = changed;
        }
        return false;
    }

    // forward sweep.  MODE 0: feedback with lg and offset b (predictor, writes usol)
    //                 MODE 1: feedback with lgc, homogeneous (corrector increment, writes usol)
    //                 MODE 2: open loop with usol, offset b; writes the new iterate and returns the objective
    //                 FIXED (with MODE 0): pinned inputs take fv; the state trajectory is kept in xtr for the adjoint
    // lane = (h, i): row i of the tile (state i), half h multiplies tile columns 8h..8h+7.
    template <int MODE, bool FIXED = false>
    __device__ real forward()
    {
        if (lane < NX) {
            const real v = MODE == 1 ? real(0) : real(x0[lane] - xit[lane]);
            if (lane < 3) xp[lane] = v; else wv[lane + 1] = v;
            if (FIXED) xtr[lane] = v;
        } else if (lane == 14) wv[14] = MODE == 1 ? real(0) : real(1);
        else if (lane == 15) wv[15] = 0;
        real cost = 0;
        if (MODE == 2 && h == 0 && j < NX) {
            const real e0 = real(x0[j] - yref[j]);
            cost = real(0.5) * a.Qd[j] * e0 * e0;
            xit[j] = x0[j];
        }
        __syncwarp();
        const int irow = j < NX ? j : NX - 1;
        sweep_begin(0, 1);
        for (int k = 0; k < N; ++k) {
            const real* tr = tile_at(k, k) + irow * WR + h * 8;
            real wr[8];
#pragma unroll
            for (int c = 0; c < 8; c += 2) tld2(tr + c, wr[c], wr[c + 1]);
            prefetch_stage(k + 1, MODE != 2);
            real u[4];
            if (MODE != 2) {
                const real* f = facv + (size_t)k * FAC;
                Chol4<double> L;
                L.load(f + 56);
                const real xo = j < 3 ? xp[j] : (j < NX ? wv[j + 1] : real(0));
                real v[4] = {0, 0, 0, 0};
                const int src = j < NX ? j * 4 : (MODE == 0 ? 52 : 66);
                if (j <= NX) { ld2(f + src, v[0], v[1]); ld2(f + src + 2, v[2], v[3]); }
                const real sc = j < NX ? xo : real(1);
#pragma unroll
                for (int aa = 0; aa < 4; ++aa) v[aa] = half_sum(hmask, v[aa] * sc);
                L.bsolve_neg(v, u);
                if (FIXED) {
#pragma unroll
                    for (int aa = 0; aa < 4; ++aa) if (fx[k * 4 + aa] != real(0)) u[aa] = fv[k * 4 + aa];
                }
            } else {
                ld2(usol + k * 4, u[0], u[1]); ld2(usol + k * 4 + 2, u[2], u[3]);
            }
            __syncwarp();                       // everyone has read the old state (and its part of the tile)
            tile_done(k, k + RING);
            if (lane < 4) {
                const real ul = sel4(u, lane);
                wv[lane] = ul;
                if (MODE != 2) usol[k * 4 + lane] = ul;
            }
            __syncwarp();
            real acc0 = 0, acc1 = 0;
#pragma unroll
            for (int c = 0; c < 8; c += 2) {
                real v0, v1;
                ld2(wv + h * 8 + c, v0, v1);
                acc0 += wr[c] * v0; acc1 += wr[c + 1] * v1;
            }
            real acc = acc0 + acc1;
            acc += __shfl_xor_sync(FULL, acc, 16);
            if (j < 3) acc += xp[j];
            __syncwarp();
            if (h == 0 && j < NX) {
                if (j < 3) xp[j] = acc; else wv[j + 1] = acc;
                if (FIXED) xtr[(k + 1) * NX + j] = acc;
                if (MODE == 2) {
                    double* xo = xit + (size_t)(k + 1) * NX + j;
                    const double xnew = *xo + double(acc);
                    *xo = xnew;
                    const real wgt = (k + 1 < N) ? a.Qd[j] : a.QNd[j];
                    const double ref = (k + 1 < N) ? yref[(size_t)(k + 1) * NY + j] : yref_e[j];
                    const real e = real(xnew - ref);
                    cost += real(0.5) * wgt * e * e;
                }
            } else if (MODE == 2 && h == 1 && j < 4) {
                const real e = real(double(ubar[k * 4 + j]) + double(sel4(u, j)) - yref[(size_t)k * NY + NX + j]);
                cost += real(0.5) * a.Rd[j] * e * e;
            }
            __syncwarp();
        }
        return cost;
    }

    // Sensitivity sweep w.r.t. x0 of the pinned LQR whose factors backward_full<true>() left in `fac`: the 13 columns of
    // dx_0 = I go through the stages with the algebra of forward<0, true> without offsets, du = -Lam^-T Lx^T dx (pinned
    // rows 0), dx+ = A dx + B du.  Lane c < 13 carries column c in registers; tile rows, factor records and fx are
    // broadcasts.  Stores du_k to su[k][4][13] and dx_k to sx[k][13][13] (sx may be null), lanes c < 13 writing
    // consecutive doubles of every row.  Covers stages 0..N-1 of the context (the caller may shorten N).
    __device__ void forward_sens(double* sx, double* su)
    {
        const int c = lane < NX ? lane : NX - 1;     // lanes 13..31 follow column 12 and store nothing
        real dx[NX];
#pragma unroll
        for (int i = 0; i < NX; ++i) dx[i] = i == c ? real(1) : real(0);
        if (sx && lane < NX) {
#pragma unroll
            for (int i = 0; i < NX; ++i) sx[i * NX + lane] = double(dx[i]);
        }
        sweep_begin(0, 1);
        for (int k = 0; k < N; ++k) {
            const real* t = tile_at(k, k);
            const real* f = facv + (size_t)k * FAC;
            Chol4<double> L;
            L.load(f + 56);
            real v[4] = {0, 0, 0, 0};
#pragma unroll
            for (int s_ = 0; s_ < NX; ++s_) {
                real l0, l1, l2, l3;
                ld2(f + s_ * 4, l0, l1); ld2(f + s_ * 4 + 2, l2, l3);
                v[0] = fma(l0, dx[s_], v[0]); v[1] = fma(l1, dx[s_], v[1]);
                v[2] = fma(l2, dx[s_], v[2]); v[3] = fma(l3, dx[s_], v[3]);
            }
            real du[4];
            L.bsolve_neg(v, du);
#pragma unroll
            for (int aa = 0; aa < 4; ++aa) if (fx[k * 4 + aa] != real(0)) du[aa] = 0;
            real xn[NX];
#pragma unroll
            for (int i = 0; i < NX; ++i) {
                const real* row = t + i * WR;
                real acc = i < 3 ? dx[i] : real(0);             // position columns of A: unit vectors, not stored
#pragma unroll
                for (int aa = 0; aa < 4; ++aa) acc = fma(tld(row + aa), du[aa], acc);
#pragma unroll
                for (int s_ = 3; s_ < NX; ++s_) acc = fma(tld(row + 1 + s_), dx[s_], acc);
                xn[i] = acc;
            }
            __syncwarp();                       // every lane has read the tile
            tile_done(k, k + RING);
            if (lane < NX) {
#pragma unroll
                for (int aa = 0; aa < 4; ++aa) su[(k * NU + aa) * NX + lane] = double(du[aa]);
                if (sx) {
#pragma unroll
                    for (int i = 0; i < NX; ++i) sx[((k + 1) * NX + i) * NX + lane] = double(xn[i]);
                }
            }
#pragma unroll
            for (int i = 0; i < NX; ++i) dx[i] = xn[i];
        }
    }

    // Backward half of the adjoint (reverse mode) of the pinned LQR whose factors backward_full<true>() left in `fac`:
    // the gradient sweep of backward_vec<true> with the cotangents as linear costs, q_k = -xb_k on the states, r_k = -ub_k
    // on the inputs (pinned inputs take none), p_N = -xb_N, no offsets.  Unlike backward_vec it carries the state terms
    // and updates p at stage 0 as well: on return pv[0..12] = p_0, the costate of x_0, and x0_bar = -p_0.  lgc goes to
    // fac[66..69] for forward_cotangent.  xb [(N+1)][13], ub [N][4]; either may be null (zero cotangent).
    // TAN (qmpc_eval_jvp): the linear costs are those of the forward mode for the direction t instead (xb, ub unused),
    // formed per stage:  c_k = -(Qd, Rd) dyref_k + dt dw (z_k - yref_k),  c_N = -QNd dyref_e + dwe (x_N - yref_e)
    // (DESIGN.md §4), i.e. the cotangents xb = -c_x, ub = -c_u.
    template <bool TAN = false>
    __device__ void backward_cotangent(const double* xb, const double* ub, const TanDir* t = nullptr)
    {
        real qd = 0, dq = 0, rd = 0, dr = 0;        // TAN: this lane's Hessian and dt dw entries of state sidx / input j
        if constexpr (TAN) {
            if (lane < 16) {
                real pn = 0;
                if (lane < NX) {
                    if (t->dyref_e) pn = -a.QNd[lane] * real(t->dyref_e[lane]);
                    if (t->dwe) pn = fma(real(t->dwe[lane]), real(t->xs[(size_t)N * NX + lane] - t->yre[lane]), pn);
                }
                pv[lane] = pn;
            }
            if (sidx >= 0) { qd = a.Qd[sidx]; if (t->dw) dq = a.dt * real(t->dw[sidx]); }
            if (j < 4) { rd = a.Rd[j]; if (t->dw) dr = a.dt * real(t->dw[NX + j]); }
        } else {
            if (lane < 16) pv[lane] = (xb && lane < NX) ? real(-xb[(size_t)N * NX + lane]) : real(0);
        }
        __syncwarp();
        sweep_begin(N - 1, -1);
        for (int k = N - 1; k >= 0; --k) {
            real w[NX];
            load_col(tile_at(N - 1 - k, k), w);
            prefetch_stage(k - 1, true);
            const real* f = facv + (size_t)k * FAC;
            Chol4<double> L;
            L.load(f + 56);
            real lx[4] = {0, 0, 0, 0};
            if (sidx >= 0) { ld2(f + sidx * 4, lx[0], lx[1]); ld2(f + sidx * 4 + 2, lx[2], lx[3]); }
            real g = 0;
#pragma unroll
            for (int c = 0; c < 12; c += 2) {
                real h0, h1;
                ld2(pv + c, h0, h1);
                g += w[c] * h0 + w[c + 1] * h1;
            }
            g += w[12] * pv[12];
            real qs;
            if constexpr (TAN) {
                qs = 0;
                const double* yk = t->yr + (size_t)k * NY;
                if (j < 4) {
                    real cu = 0;
                    if (t->dyref) cu = -rd * real(t->dyref[(size_t)k * NY + NX + j]);
                    if (t->dw) cu = fma(dr, real(t->us[k * 4 + j] - yk[NX + j]), cu);
                    g += cu;
                }
                if (sidx >= 0) {
                    if (t->dyref) qs = -qd * real(t->dyref[(size_t)k * NY + sidx]);
                    if (t->dw) qs = fma(dq, real(t->xs[(size_t)k * NX + sidx] - yk[sidx]), qs);
                }
            } else {
                if (j < 4 && ub) g -= real(ub[k * 4 + j]);
                qs = (sidx >= 0 && xb) ? real(-xb[(size_t)k * NX + sidx]) : real(0);
            }
            real gu[4], lgc[4];
#pragma unroll
            for (int aa = 0; aa < 4; ++aa) gu[aa] = __shfl_sync(FULL, g, aa);
#pragma unroll
            for (int aa = 0; aa < 4; ++aa) if (fx[k * 4 + aa] != real(0)) gu[aa] = 0;
            L.fsolve(gu, lgc);
            const real pold = j < 3 ? pv[j] : real(0);
            __syncwarp();
            tile_done(N - 1 - k, k - RING);
            if (h == 0) {
                if (j >= 4 && j < 14) pv[j - 1] = g + qs - dot4(lx, lgc);
                else if (j < 3) pv[j] = pold + qs - dot4(lx, lgc);
                else if (j == 14) {
#pragma unroll
                    for (int aa = 0; aa < 4; ++aa) facv[(size_t)k * FAC + 66 + aa] = lgc[aa];
                }
            }
            __syncwarp();
        }
    }

    // Forward half of the adjoint: the minimiser of that LQR from x_0 = 0, du_k = -Lam^-T (Lx dx_k + lgc_k) (pinned
    // entries 0), dx_{k+1} = A dx_k + B du_k, contracted with the cost weights as it goes: yb[k] = (Qd dx_k, Rd du_k),
    // yeb = QNd dx_N.  Every lane carries the whole state (tile rows and factor records are broadcasts, as in
    // forward_sens); lanes 0..16 store one entry of yb[k] each, lanes 0..12 one of yeb.  yb [N][17], yeb [13] or null.
    // WGT (qmpc_eval_adjoint_weights): also the gradients w.r.t. the cost weights, from the last solve's solution xs
    // [(N+1)][13], us [N][4] and the reference yr [N][17], yre [13]: lane i < 17 accumulates (dx_k, du_k)_i (z_k - yref_k)_i
    // over k and stores wb[i] = -dt acc, lanes 0..12 store web[i] = -dx_N,i (x_N - yref_e)_i.  wb [17], web [13] or null.
    // Each lane owns its entries: no cross-lane reduction, so the result is bit-reproducible.
    // TAN (qmpc_eval_jvp): the roll-out starts from dx_0 = dx0 [13] (null = 0) and stores the tangent itself, dx_k to
    // dxo [(N+1)][13] (or null) and du_k to duo [N][4]; yb, yeb must be null.
    template <bool WGT = false, bool TAN = false>
    __device__ void forward_cotangent(double* yb, double* yeb, const double* xs = nullptr, const double* us = nullptr,
                                      const double* yr = nullptr, const double* yre = nullptr, double* wb = nullptr,
                                      double* web = nullptr, const double* dx0 = nullptr, double* dxo = nullptr,
                                      double* duo = nullptr)
    {
        real dx[NX];
#pragma unroll
        for (int i = 0; i < NX; ++i) dx[i] = 0;
        if constexpr (TAN) {
            if (dx0) {
#pragma unroll
                for (int i = 0; i < NX; ++i) dx[i] = real(dx0[i]);
            }
            if (dxo) {
                real mine = 0;
#pragma unroll
                for (int i = 0; i < NX; ++i) if (lane == i) mine = dx[i];
                if (lane < NX) dxo[lane] = double(mine);
            }
        }
        real wacc = 0;
        sweep_begin(0, 1);
        for (int k = 0; k < N; ++k) {
            const real* t = tile_at(k, k);
            const real* f = facv + (size_t)k * FAC;
            Chol4<double> L;
            L.load(f + 56);
            real v[4];
            ld2(f + 66, v[0], v[1]); ld2(f + 68, v[2], v[3]);
#pragma unroll
            for (int s_ = 0; s_ < NX; ++s_) {
                real l0, l1, l2, l3;
                ld2(f + s_ * 4, l0, l1); ld2(f + s_ * 4 + 2, l2, l3);
                v[0] = fma(l0, dx[s_], v[0]); v[1] = fma(l1, dx[s_], v[1]);
                v[2] = fma(l2, dx[s_], v[2]); v[3] = fma(l3, dx[s_], v[3]);
            }
            real du[4];
            L.bsolve_neg(v, du);
#pragma unroll
            for (int aa = 0; aa < 4; ++aa) if (fx[k * 4 + aa] != real(0)) du[aa] = 0;
            real xn[NX];
#pragma unroll
            for (int i = 0; i < NX; ++i) {
                const real* row = t + i * WR;
                real acc = i < 3 ? dx[i] : real(0);             // position columns of A: unit vectors, not stored
#pragma unroll
                for (int aa = 0; aa < 4; ++aa) acc = fma(tld(row + aa), du[aa], acc);
#pragma unroll
                for (int s_ = 3; s_ < NX; ++s_) acc = fma(tld(row + 1 + s_), dx[s_], acc);
                xn[i] = acc;
            }
            __syncwarp();                       // every lane has read the tile
            tile_done(k, k + RING);
            if (yb) {
                real mine = 0;                  // selects on the lane index, not a run-time index into the register arrays
#pragma unroll
                for (int i = 0; i < NX; ++i) if (lane == i) mine = a.Qd[i] * dx[i];
#pragma unroll
                for (int aa = 0; aa < 4; ++aa) if (lane == NX + aa) mine = a.Rd[aa] * du[aa];
                if (lane < NY) yb[k * NY + lane] = double(mine);
            }
            if constexpr (WGT) {
                real mine = 0, res = 0;
#pragma unroll
                for (int i = 0; i < NX; ++i) if (lane == i) mine = dx[i];
#pragma unroll
                for (int aa = 0; aa < 4; ++aa) if (lane == NX + aa) mine = du[aa];
                if (lane < NX) res = real(xs[k * NX + lane] - yr[k * NY + lane]);
                else if (lane < NY) res = real(us[k * 4 + lane - NX] - yr[k * NY + lane]);
                wacc = fma(mine, res, wacc);
            }
            if constexpr (TAN) {
                real mu = 0, mx = 0;
#pragma unroll
                for (int aa = 0; aa < 4; ++aa) if (lane == aa) mu = du[aa];
                if (lane < NU) duo[k * NU + lane] = double(mu);
                if (dxo) {
#pragma unroll
                    for (int i = 0; i < NX; ++i) if (lane == i) mx = xn[i];
                    if (lane < NX) dxo[(size_t)(k + 1) * NX + lane] = double(mx);
                }
            }
#pragma unroll
            for (int i = 0; i < NX; ++i) dx[i] = xn[i];
        }
        if (yeb) {
            real mine = 0;
#pragma unroll
            for (int i = 0; i < NX; ++i) if (lane == i) mine = a.QNd[i] * dx[i];
            if (lane < NX) yeb[lane] = double(mine);
        }
        if constexpr (WGT) {
            if (wb && lane < NY) wb[lane] = -double(a.dt * wacc);
            if (web) {
                real mine = 0;
#pragma unroll
                for (int i = 0; i < NX; ++i) if (lane == i) mine = dx[i];
                if (lane < NX) web[lane] = -double(mine * real(xs[(size_t)N * NX + lane] - yre[lane]));
            }
        }
    }
};

#ifndef QMPC_IPM_MIN_WARPS
#define QMPC_IPM_MIN_WARPS 16      // resident warps per SM the register allocation is sized for
#endif

template <typename real, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, QMPC_IPM_MIN_WARPS / WARPS) qmpc_ipm_kernel(IpmArgs<real> a)
{
    QMPC_DYN_SMEM(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ocp = blockIdx.x * WARPS + warp;
    if (ocp >= a.B) return;
    const int N = a.N, E = 4 * N;
    real* sm = reinterpret_cast<real*>(smem_raw) + (size_t)warp * a.smem_per_warp;
    WarpCtx<real> c{a};
    c.lane = lane; c.h = lane >> 4; c.j = lane & 15; c.ocp = ocp; c.N = N; c.E = E;
    c.hmask = 0xffffu << (lane & 16);
    c.sidx = (c.j < 3) ? c.j : ((c.j >= 4 && c.j < 14) ? c.j - 1 : -1);
    c.P = sm + SM_P; c.pv = sm + SM_PV; c.wv = sm + SM_WV; c.xp = sm + SM_XP; c.hv = sm + SM_HV;
    c.Ls = sm + SM_LS; c.cs = sm + SM_CS;
    real* v = sm + SM_VEC;
    if (a.hard_count) {
        // screening mode never enters the IPM: only the 6 vectors of the active-set rounds are laid out (the new inputs
        // of the epilogue reuse the multiplier vector, which is dead by then): 12.8 KB per OCP with the tile ring,
        // 16 warps per SM
        c.usol = v; c.ua = v + E; c.ucur = v + E; c.ubar = v + 2 * E; c.rdel = v + 3 * E; c.cl = v + 4 * E; c.cu = v + 5 * E;
        c.xtr = v + 6 * E;
        c.rt = c.dR = c.ll = c.lu = c.tl = c.tu = v;
    } else {
        c.rt = v; c.dR = v + E; c.usol = v + 2 * E; c.ua = v + 3 * E; c.ucur = v + 4 * E; c.ll = v + 5 * E;
        c.lu = v + 6 * E; c.ubar = v + 7 * E; c.rdel = v + 8 * E; c.cl = v + 9 * E; c.cu = v + 10 * E;
        c.tl = v + 11 * E; c.tu = v + 12 * E; c.xtr = v + 13 * E;
    }
    c.fx = c.cl; c.fv = c.cu; c.grad = c.ua;
    c.hist_store = sm + a.ring_off;                      // 48 bytes, then the ring (offsets stay 16-byte aligned)
    c.ring = sm + a.ring_off + HIST_REALS<real>();
    c.rbar = reinterpret_cast<unsigned long long*>(c.ring + WarpCtx<real>::RING * WT);
    c.rphase = 0;
    c.gave_up = false;
    if (WarpCtx<real>::RING) {
        if (lane == 0) for (int s_ = 0; s_ < WarpCtx<real>::RING; ++s_) mbar_init(c.rbar + s_, 1);
        __syncwarp();
    }
    c.Wv = a.W + (size_t)ocp * N * WT;
    c.facv = a.fac + (size_t)ocp * N * FAC;
    c.x0 = a.x0 + (size_t)ocp * NX;
    c.yref = a.yref + (size_t)ocp * N * NY;
    c.yref_e = a.yref_e + (size_t)ocp * NX;
    c.xit = a.xit + (size_t)ocp * (N + 1) * NX;
    c.uit = a.uit + (size_t)ocp * N * NU;
    unsigned char* act = a.act + (size_t)ocp * E;
    if (a.timeline && lane == 0) a.timeline[2 * ocp] = global_ns();

    const real lb = a.lb, ub = a.ub;
    for (int e = lane; e < E; e += 32) {
        const real ub_ = real(c.uit[e]);
        c.ubar[e] = ub_;
        c.rdel[e] = a.Rd[e & 3] * (ub_ - real(c.yref[(size_t)(e >> 2) * NY + NX + (e & 3)]));
    }
    __syncwarp();

    int it = 0, rounds = 0, status = QMPC_STATUS_MAXITER_;
    bool exact = false;
    // screening mode: an OCP whose previous solve needed a long interior-point run (a vehicle far off its reference, most
    // inputs saturated) will need it again.  It skips the rounds and enters the hard list at once, i.e. near its head: the
    // dense launch starts its longest items first.
    const bool long_ipm_last_time = a.hard_count && a.skip_screen_iters > 0 && a.iters[ocp] >= a.skip_screen_iters;
    // ---- 1. warm start: the active set of the previous solve is usually still right (RTI does not shift the horizon)
    if (a.warm_rounds > 0 && !long_ipm_last_time) {
        int known = 1;
        for (int e = lane; e < E; e += 32) { const unsigned char f = act[e]; if (f > 2) known = 0; c.fx[e] = real(f <= 2 ? f : 0); }
        known = -warp_max(-known);
        // busy step (the previous step left many OCPs unsettled, the dense launch would need several waves): keep the
        // contracting ones here for more rounds - a Riccati round costs a quarter of the dense kernel's condensing
        const bool busy = a.unsettled_prev && a.warm_rounds_busy > a.warm_rounds && *a.unsettled_prev > a.busy_threshold;
        if (known && c.refine_rounds(lb, ub, busy ? a.warm_rounds_busy : a.warm_rounds, rounds, true,
                                     busy ? a.bail_round_busy : a.bail_round, a.warm_rounds, a.unsettled_cur)) {
            exact = true; status = QMPC_STATUS_OK_;
        }
        if (!known && a.unsettled_cur && lane == 0) atomicAdd(a.unsettled_cur, 1);
    } else if (long_ipm_last_time && a.unsettled_cur && lane == 0) atomicAdd(a.unsettled_cur, 1);
    if (!exact && a.hard_count) {
        // screening mode: hand the OCP to the dense kernel together with the active-set guess the rounds ended on
        if (a.warm_rounds > 0 && !long_ipm_last_time) {
            bool was_known = true;
            for (int e = lane; e < E; e += 32) was_known = was_known && act[e] <= 2;
            was_known = warp_max(int(!was_known)) == 0;
            if (was_known) for (int e = lane; e < E; e += 32) act[e] = c.fx[e] == real(1) ? 1 : (c.fx[e] == real(2) ? 2 : 0);
        }
        // the dense kernel continues the rounds from the guess they ended on - unless they ended on a cycle or stopped
        // contracting (or last step's solve was a long IPM run): more rounds will not settle, it starts its IPM at once
        if (long_ipm_last_time || (a.bail_to_ipm && c.gave_up)) for (int e = lane; e < E; e += 32) act[e] = 255;
        if (lane == 0) { a.rounds[ocp] = rounds; a.hard_list[atomicAdd(a.hard_count, 1)] = ocp; }
        return;
    }
    // ---- 2. Mehrotra predictor-corrector IPM (cold start), handing over to the active-set refinement at mu_switch
    if (!exact) {
        // initial multipliers scaled with the problem: lam0 = clip(0.01 * mean |dJ/du| at the box centre, 0.1, 100)
        // (one open-loop roll-out + one adjoint sweep; heavily saturated problems otherwise spend many iterations
        //  growing the multipliers)
        for (int e = lane; e < E; e += 32) { c.fx[e] = 1; c.fv[e] = real(0.5) * (lb + ub) - c.ubar[e]; }
        __syncwarp();
        c.template forward<0, true>();
        __syncwarp();
        c.backward_adjoint();
        __syncwarp();
        real gs = 0;
        for (int e = lane; e < E; e += 32) gs += fabs(c.grad[e]);
        gs = warp_sum(gs) / real(E);
        const real lam0 = rfinite(gs) ? fmin(fmax(a.lam0_scale * gs, a.lam0_min), a.lam0_max) : a.lam0_min;
        for (int e = lane; e < E; e += 32) {
            const real u0 = real(0.5) * (lb + ub);
            c.ucur[e] = u0; c.tl[e] = u0 - lb; c.tu[e] = ub - u0;     // slacks are carried, never recomputed from u
            c.ll[e] = lam0; c.lu[e] = lam0;
        }
        real resfac = 1;                  // fraction of the initial stationarity residual still present
        int attempts = 0;                 // hand-overs to the active-set rounds so far
        bool refine = a.max_refine > 0;
        real target = refine ? a.mu_switch : a.mu_tol;
        const real inv2E = real(1) / real(2 * E);
        while (true) {
            real s = 0;
            for (int e = lane; e < E; e += 32) s += c.ll[e] * c.tl[e] + c.lu[e] * c.tu[e];
            const real mu = warp_sum(s) * inv2E;
            if (!rfinite(mu)) { status = QMPC_STATUS_NAN_; break; }
            if (mu < target && resfac < (refine ? real(1e-3) : a.resfac_final)) {
                if (refine) {
                    for (int e = lane; e < E; e += 32)
                        c.fx[e] = c.tl[e] < c.ll[e] ? real(1) : (c.tu[e] < c.lu[e] ? real(2) : real(0));
                    if (c.refine_rounds(lb, ub, a.max_refine, rounds, a.post_bail != 0, a.bail_round)) { status = QMPC_STATUS_OK_; exact = true; break; }
                    // inconsistent active set: one more attempt from a 100x sharper IPM point.  fp64: then a last one from
                    // the IPM point at mu_tol; if that does not settle either, the IPM point is returned flagged MAXITER,
                    // never as status 0 (it is not the minimiser: its distance grows as the dt-scaled multipliers shrink,
                    // 3e-4 at N = 256).  fp32: the IPM alone to mu_tol, then the fp64-checked rounds below.
                    if (++attempts < 2) target *= real(1e-2);
                    else if (sizeof(real) == 8 && attempts == 2) target = a.mu_tol;
                    else if (sizeof(real) == 8) break;
                    else { refine = false; target = a.mu_tol; }
                    if (!refine && mu < target) { status = QMPC_STATUS_OK_; break; }
                } else { status = QMPC_STATUS_OK_; break; }
            }
            if (it >= iter_limit(a, ocp)) break;
            // predictor
            for (int e = lane; e < E; e += 32) {
                const real d = c.ll[e] / c.tl[e] + c.lu[e] / c.tu[e];
                c.dR[e] = d;
                c.rt[e] = c.rdel[e] - d * (c.ucur[e] - c.ubar[e]);
            }
            __syncwarp();
            c.template backward_full<false>();
            c.template forward<0>();
            __syncwarp();
            // predictor step lengths: primal (slacks) and dual (multipliers) separately
            real apm = 1, adm = 1;
            for (int e = lane; e < E; e += 32) {
                const real tl = c.tl[e], tu = c.tu[e];
                const real du = c.ubar[e] + c.usol[e] - c.ucur[e];
                const real dl = -c.ll[e] - c.ll[e] / tl * du;
                const real dv = -c.lu[e] + c.lu[e] / tu * du;
                c.ua[e] = c.usol[e];
                c.cl[e] = du * dl; c.cu[e] = -du * dv;
                c.rt[e] = dl; c.dR[e] = dv;
                if (du < 0) apm = fmin(apm, -tl / du);
                if (du > 0) apm = fmin(apm, tu / du);
                if (dl < 0) adm = fmin(adm, -c.ll[e] / dl);
                if (dv < 0) adm = fmin(adm, -c.lu[e] / dv);
            }
            const real apa = warp_min(apm), ada = warp_min(adm);
            s = 0;
            for (int e = lane; e < E; e += 32) {
                const real du = c.ubar[e] + c.ua[e] - c.ucur[e];
                s += (c.ll[e] + ada * c.rt[e]) * (c.tl[e] + apa * du) + (c.lu[e] + ada * c.dR[e]) * (c.tu[e] - apa * du);
            }
            const real muaff = warp_sum(s) * inv2E;
            real sigma = muaff / mu; sigma = sigma * sigma * sigma;
            // corrector (increment on top of the predictor solution).  Safeguard: if the Mehrotra step is blocked
            // (step length < 1/2) it is recomputed once as a centring step without the second-order term.
            real so = 1, ap = 1, ad = 1;
            for (int pass = 0; pass < 2; ++pass) {
                const real smu = sigma * mu;
                for (int e = lane; e < E; e += 32)
                    c.rt[e] = -(smu - so * c.cl[e]) / c.tl[e] + (smu - so * c.cu[e]) / c.tu[e];
                __syncwarp();
                c.template backward_vec<false>();
                c.template forward<1>();
                __syncwarp();
                real apx = real(1e30), adx = real(1e30);
                for (int e = lane; e < E; e += 32) {
                    const real tl = c.tl[e], tu = c.tu[e];
                    const real du = c.ubar[e] + c.ua[e] + c.usol[e] - c.ucur[e];
                    const real dl = (smu - so * c.cl[e]) / tl - c.ll[e] - c.ll[e] / tl * du;
                    const real dv = (smu - so * c.cu[e]) / tu - c.lu[e] + c.lu[e] / tu * du;
                    c.usol[e] = du; c.rt[e] = dl; c.dR[e] = dv;
                    if (du < 0) apx = fmin(apx, -tl / du);
                    if (du > 0) apx = fmin(apx, tu / du);
                    if (dl < 0) adx = fmin(adx, -c.ll[e] / dl);
                    if (dv < 0) adx = fmin(adx, -c.lu[e] / dv);
                }
                ap = warp_min(apx); ad = warp_min(adx);
                if (pass == 1 || fmin(ap, ad) >= real(0.5)) break;
                so = 0; sigma = fmax(sigma, real(0.5));
                __syncwarp();
            }
            ap = fmin(real(1), real(0.995) * ap); ad = fmin(real(1), real(0.995) * ad);
            for (int e = lane; e < E; e += 32) {
                const real du = ap * c.usol[e];
                c.ucur[e] += du; c.tl[e] += du; c.tu[e] -= du;
                c.ll[e] += ad * c.rt[e];
                c.lu[e] += ad * c.dR[e];
            }
            resfac *= real(1) - fmin(ap, ad);
            ++it;
        }
    }
    {   // a solve that ended with a non-finite control is a breakdown too (never hand NaN to the plant or the RGP)
        real chk = 0;
        for (int e = lane; e < E; e += 32) {
            const real un = exact ? c.usol[e] : c.ucur[e];
            chk += un - un;
        }
        chk = warp_sum(chk);
        if (!(chk == real(0))) status = QMPC_STATUS_NAN_;
    }
    if (status == QMPC_STATUS_NAN_) {
        // numerical breakdown (e.g. a vehicle that has already crashed): keep the previous iterate, hold its first control
        for (int e = lane; e < E; e += 32) act[e] = 255;
        if (lane < 4) a.u0[(size_t)ocp * 4 + lane] = double(fmin(fmax(c.ubar[lane], lb), ub));
        if (lane == 0) { a.cost[ocp] = nan(""); a.status[ocp] = status; a.iters[ocp] = it; a.rounds[ocp] = rounds; }
        if (a.timeline && lane == 0) a.timeline[2 * ocp + 1] = global_ns();
        return;
    }
    if (sizeof(real) == 4 && a.refine_off > 0 && (exact || status == QMPC_STATUS_OK_)) {
        // fp32 handles: refine the fp32 solution with an fp64 residual and VERIFY its active set with the fp64 gradient.
        // Where the check moves the active set (or the fp32 rounds never settled and the IPM point is all there is), the
        // rounds continue here with the fp64 check as their update rule: pinned solve in fp32, refinement, check.
        double* dxd = reinterpret_cast<double*>(sm + a.refine_off);
        if (!exact) {
            for (int e = lane; e < E; e += 32) c.fx[e] = c.tl[e] < c.ll[e] ? real(1) : (c.tu[e] < c.lu[e] ? real(2) : real(0));
        }
        bool solved = exact;                 // usol / fac hold the pinned solve of the active set in fx
        exact = false;
        for (int pass = 0; pass < 10 && !exact; ++pass) {
            if (!solved) {
                for (int e = lane; e < E; e += 32)
                    c.fv[e] = c.fx[e] == real(1) ? lb - c.ubar[e] : (c.fx[e] == real(2) ? ub - c.ubar[e] : real(0));
                __syncwarp();
                c.template backward_full<true>();
                c.template forward<0, true>();
                __syncwarp();
                ++rounds;
            }
            exact = c.refine_solution_fp64(dxd, dxd + (N + 1) * NX, lb, ub) == 0;
            solved = false;
        }
        if (!exact) { exact = true; status = QMPC_STATUS_MAXITER_; }      // unverified: the last refined point is returned, flagged
        else status = QMPC_STATUS_OK_;
    }
    // ---- 3. full step: new iterate = solution of the QP, states re-rolled through the linearised dynamics
    for (int e = lane; e < E; e += 32) {
        real un;
        unsigned char f;
        if (exact) {
            f = c.fx[e] == real(1) ? 1 : (c.fx[e] == real(2) ? 2 : 0);
            un = f == 1 ? lb : (f == 2 ? ub : c.ubar[e] + c.usol[e]);
        } else {
            un = fmin(fmax(c.ucur[e], lb), ub);
            f = status == QMPC_STATUS_OK_ ? (c.tl[e] < c.ll[e] ? 1 : (c.tu[e] < c.lu[e] ? 2 : 0)) : 255;
        }
        act[e] = f;
        c.ucur[e] = un;
    }
    for (int e = lane; e < E; e += 32) c.usol[e] = c.ucur[e] - c.ubar[e];
    __syncwarp();
    real cost = 0;
    if (exact && !a.final_rollout) {
        // the pinned forward sweep of the last active-set round already holds the state increments of this solution
        // (xtr): add them and evaluate the objective element-wise instead of rolling the horizon out once more
        for (int idx = lane; idx < (N + 1) * NX; idx += 32) {
            const int k = idx / NX, r = idx - k * NX;
            const double xnew = k == 0 ? c.x0[r] : c.xit[idx] + double(c.xtr[idx]);
            c.xit[idx] = xnew;
            const real w = k < N ? a.Qd[r] : a.QNd[r];
            const real e_ = real(xnew - (k < N ? c.yref[(size_t)k * NY + r] : c.yref_e[r]));
            cost += real(0.5) * w * e_ * e_;
        }
        for (int e = lane; e < E; e += 32) {
            const real e_ = real(double(c.ucur[e]) - c.yref[(size_t)(e >> 2) * NY + NX + (e & 3)]);
            cost += real(0.5) * a.Rd[e & 3] * e_ * e_;
        }
    } else {
        cost = c.template forward<2>();
    }
    cost = warp_sum(cost);
    for (int e = lane; e < E; e += 32) c.uit[e] = double(c.ucur[e]);
    if (lane < 4) a.u0[(size_t)ocp * 4 + lane] = double(c.ucur[lane]);
    if (lane == 0) { a.cost[ocp] = double(cost); a.status[ocp] = status; a.iters[ocp] = it; a.rounds[ocp] = rounds; }
    if (a.timeline && lane == 0) a.timeline[2 * ocp + 1] = global_ns();
}

// ------------------------------------------------------------------------------------------ sensitivities w.r.t. x0

template <typename real>
struct SensArgs {
    IpmArgs<real> b;        // read: B, N, weights, W, fac (scratch between solves, rewritten here), act, xit, yref_e,
                            // smem_per_warp / ring_off of the screening layout
    int n_stages;           // 1..N: stages 0..n_stages-1 are swept
    double* sens_x;         // [B][n_stages+1][13][13] or null
    double* sens_u;         // [B][n_stages][4][13]
};

// RTI never reads x0 in K1, so x0 -> (x, u) is the box-QP's solution map: piecewise affine, and on the active set the
// solve ended on its Jacobian is the closed loop of the LQR with those inputs pinned.  One warp per OCP: the pinned
// factorisation of the active-set rounds (backward_full<true>), then forward_sens.  A vehicle whose active set is
// unknown (any entry 255) gets NaN everywhere.
// resident warps per SM the register allocation is sized for: at 16 (the solver kernel's) the fp64 factorisation spills;
// 12 leaves it 167 registers and no spill
constexpr int SENS_MIN_WARPS = 12;

template <typename real, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, SENS_MIN_WARPS / WARPS) qmpc_sens_kernel(SensArgs<real> s)
{
    QMPC_DYN_SMEM(smem_raw);
    const IpmArgs<real>& a = s.b;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ocp = blockIdx.x * WARPS + warp;
    if (ocp >= a.B) return;
    const int N = a.N, E = 4 * N, ns = s.n_stages;
    const unsigned char* act = a.act + (size_t)ocp * E;
    double* sx = s.sens_x ? s.sens_x + (size_t)ocp * (ns + 1) * NX * NX : nullptr;
    double* su = s.sens_u + (size_t)ocp * ns * NU * NX;
    int known = 1;
    for (int e = lane; e < E; e += 32) if (act[e] > 2) known = 0;
    if (!warp_min(known)) {
        const double qnan = nan("");
        if (sx) for (int i = lane; i < (ns + 1) * NX * NX; i += 32) sx[i] = qnan;
        for (int i = lane; i < ns * NU * NX; i += 32) su[i] = qnan;
        return;
    }
    // the set-up of qmpc_ipm_kernel in its screening layout (kept separate: that kernel's code is tuned); the sweeps used
    // here read the per-warp work space, rdel, fx, fv, the tiles, `fac`, and xit / yref_e for the (unused) costate offset
    real* sm = reinterpret_cast<real*>(smem_raw) + (size_t)warp * a.smem_per_warp;
    WarpCtx<real> c{a};
    c.lane = lane; c.h = lane >> 4; c.j = lane & 15; c.ocp = ocp; c.N = N; c.E = E;
    c.hmask = 0xffffu << (lane & 16);
    c.sidx = (c.j < 3) ? c.j : ((c.j >= 4 && c.j < 14) ? c.j - 1 : -1);
    c.P = sm + SM_P; c.pv = sm + SM_PV; c.wv = sm + SM_WV; c.xp = sm + SM_XP; c.hv = sm + SM_HV;
    c.Ls = sm + SM_LS; c.cs = sm + SM_CS;
    real* v = sm + SM_VEC;
    c.usol = c.ua = c.ucur = c.ubar = c.grad = v; c.rdel = v + 3 * E; c.cl = v + 4 * E; c.cu = v + 5 * E;
    c.xtr = v + 6 * E;
    c.rt = c.dR = c.ll = c.lu = c.tl = c.tu = v;
    c.fx = c.cl; c.fv = c.cu;
    c.hist_store = sm + a.ring_off;
    c.ring = sm + a.ring_off + HIST_REALS<real>();
    c.rbar = reinterpret_cast<unsigned long long*>(c.ring + WarpCtx<real>::RING * WT);
    c.rphase = 0;
    c.gave_up = false;
    if (WarpCtx<real>::RING) {
        if (lane == 0) for (int s_ = 0; s_ < WarpCtx<real>::RING; ++s_) mbar_init(c.rbar + s_, 1);
        __syncwarp();
    }
    c.Wv = a.W + (size_t)ocp * N * WT;
    c.facv = a.fac + (size_t)ocp * N * FAC;
    c.x0 = nullptr; c.yref = nullptr; c.uit = nullptr;
    c.yref_e = a.yref_e + (size_t)ocp * NX;
    c.xit = a.xit + (size_t)ocp * (N + 1) * NX;
    // homogeneous problem: pinned inputs at 0, no input gradient (the offsets only reach lg / p, never the factors)
    for (int e = lane; e < E; e += 32) { c.fx[e] = real(act[e]); c.fv[e] = 0; c.rdel[e] = 0; }
    __syncwarp();
    c.template backward_full<true>();
    c.N = ns;              // the sweep streams stages 0..ns-1 only: no tile copy is in flight when the warp exits
    c.forward_sens(sx, su);
}

// ------------------------------------------------------------------------------------------ adjoint sensitivities

// Set-up of qmpc_adjoint_kernel for one OCP, the same as qmpc_sens_kernel's (that kernel keeps its inline copy: moved into
// this function it compiles to a different register allocation): the warp context of qmpc_ipm_kernel in its screening
// layout, then the pinned factorisation of the active-set rounds (backward_full<true>) on the active set `act` of the
// last solve.  The sweeps that follow read the per-warp work space, rdel, fx, fv, the tiles, `fac`, and xit / yref_e
// for the (unused) costate offset.
template <typename real>
__device__ __forceinline__ void sens_factorise(WarpCtx<real>& c, unsigned char* smem_raw, int warp, int lane, int ocp,
                                               const unsigned char* act)
{
    const IpmArgs<real>& a = c.a;
    const int N = a.N, E = 4 * N;
    real* sm = reinterpret_cast<real*>(smem_raw) + (size_t)warp * a.smem_per_warp;
    c.lane = lane; c.h = lane >> 4; c.j = lane & 15; c.ocp = ocp; c.N = N; c.E = E;
    c.hmask = 0xffffu << (lane & 16);
    c.sidx = (c.j < 3) ? c.j : ((c.j >= 4 && c.j < 14) ? c.j - 1 : -1);
    c.P = sm + SM_P; c.pv = sm + SM_PV; c.wv = sm + SM_WV; c.xp = sm + SM_XP; c.hv = sm + SM_HV;
    c.Ls = sm + SM_LS; c.cs = sm + SM_CS;
    real* v = sm + SM_VEC;
    c.usol = c.ua = c.ucur = c.ubar = c.grad = v; c.rdel = v + 3 * E; c.cl = v + 4 * E; c.cu = v + 5 * E;
    c.xtr = v + 6 * E;
    c.rt = c.dR = c.ll = c.lu = c.tl = c.tu = v;
    c.fx = c.cl; c.fv = c.cu;
    c.hist_store = sm + a.ring_off;
    c.ring = sm + a.ring_off + HIST_REALS<real>();
    c.rbar = reinterpret_cast<unsigned long long*>(c.ring + WarpCtx<real>::RING * WT);
    c.rphase = 0;
    c.gave_up = false;
    if (WarpCtx<real>::RING) {
        if (lane == 0) for (int s_ = 0; s_ < WarpCtx<real>::RING; ++s_) mbar_init(c.rbar + s_, 1);
        __syncwarp();
    }
    c.Wv = a.W + (size_t)ocp * N * WT;
    c.facv = a.fac + (size_t)ocp * N * FAC;
    c.x0 = nullptr; c.yref = nullptr; c.uit = nullptr;
    c.yref_e = a.yref_e + (size_t)ocp * NX;
    c.xit = a.xit + (size_t)ocp * (N + 1) * NX;
    // homogeneous problem: pinned inputs at 0, no input gradient (the offsets only reach lg / p, never the factors)
    for (int e = lane; e < E; e += 32) { c.fx[e] = real(act[e]); c.fv[e] = 0; c.rdel[e] = 0; }
    __syncwarp();
    c.template backward_full<true>();
}

template <typename real>
struct AdjArgs {
    IpmArgs<real> b;           // as SensArgs::b
    const double* x_bar;       // [B][N+1][13] cotangent of the states, or null (zero)
    const double* u_bar;       // [B][N][4] cotangent of the inputs, or null (zero)
    double* x0_bar;            // [B][13] or null
    double* yref_bar;          // [B][N][17] or null
    double* yref_e_bar;        // [B][13] or null
    // read by the WGT instantiation only (qmpc_eval_adjoint_weights)
    const double* x;           // [B][N+1][13] the last solve's states
    const double* u;           // [B][N][4] the last solve's inputs
    const double* yref;        // [B][N][17] the reference that solve ran with
    const double* yref_e;      // [B][13]
    double* w_bar;             // [B][17] gradient w.r.t. w_diag, or null
    double* we_bar;            // [B][13] gradient w.r.t. we_diag, or null
};

// Reverse mode of the same solution map, now also w.r.t. the reference: K1 reads the reference only in the linear cost
// term (tile column 15, q = dt W_x (x_lin - xref)) and the solve only in rdel (from uref), so on the active set
// d<xb, x> + <ub, u> = <x0_bar, dx0> + <yref_bar, dyref> + <yref_e_bar, dyref_e> with, for the minimiser (dx, du) of the
// pinned LQR with linear costs -xb, -ub from dx_0 = 0:  yref_bar[k] = (Qd dx_k, Rd du_k), yref_e_bar = QNd dx_N and
// x0_bar = -p_0, the costate of x_0.  One warp per OCP: sens_factorise, backward_cotangent, forward_cotangent (skipped
// when no output it writes is wanted).  A vehicle whose active set is unknown gets NaN everywhere.
// WGT: also the gradients w.r.t. the cost weights.  The weights enter the QP only through its objective (Hessian dt W,
// tile column 15, rdel), never the linearisation, so with z the solution and (dx, du) the minimiser above,
// w_bar[i] = -dt sum_k (dx_k, du_k)_i (z_k - yref_k)_i and we_bar[i] = -dx_N,i (x_N - yref_e)_i (DESIGN.md §4).
// The fp64 factorisation spills at 16 resident warps as in qmpc_sens_kernel: the same register budget.
template <typename real, int WARPS, bool WGT = false>
__global__ void __launch_bounds__(WARPS * 32, SENS_MIN_WARPS / WARPS) qmpc_adjoint_kernel(AdjArgs<real> s)
{
    QMPC_DYN_SMEM(smem_raw);
    const IpmArgs<real>& a = s.b;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ocp = blockIdx.x * WARPS + warp;
    if (ocp >= a.B) return;
    const int N = a.N, E = 4 * N;
    const unsigned char* act = a.act + (size_t)ocp * E;
    const double* xb = s.x_bar ? s.x_bar + (size_t)ocp * (N + 1) * NX : nullptr;
    const double* ub = s.u_bar ? s.u_bar + (size_t)ocp * E : nullptr;
    double* x0b = s.x0_bar ? s.x0_bar + (size_t)ocp * NX : nullptr;
    double* yb = s.yref_bar ? s.yref_bar + (size_t)ocp * N * NY : nullptr;
    double* yeb = s.yref_e_bar ? s.yref_e_bar + (size_t)ocp * NX : nullptr;
    double* wb = (WGT && s.w_bar) ? s.w_bar + (size_t)ocp * NY : nullptr;
    double* web = (WGT && s.we_bar) ? s.we_bar + (size_t)ocp * NX : nullptr;
    int known = 1;
    for (int e = lane; e < E; e += 32) if (act[e] > 2) known = 0;
    if (!warp_min(known)) {
        const double qnan = nan("");
        if (x0b && lane < NX) x0b[lane] = qnan;
        if (yeb && lane < NX) yeb[lane] = qnan;
        if (yb) for (int i = lane; i < N * NY; i += 32) yb[i] = qnan;
        if constexpr (WGT) {
            if (wb && lane < NY) wb[lane] = qnan;
            if (web && lane < NX) web[lane] = qnan;
        }
        return;
    }
    WarpCtx<real> c{a};
    sens_factorise(c, smem_raw, warp, lane, ocp, act);
    c.backward_cotangent(xb, ub);
    if (x0b && lane < NX) x0b[lane] = -double(c.pv[lane]);
    if constexpr (WGT) {
        if (yb || yeb || wb || web)
            c.template forward_cotangent<true>(yb, yeb, s.x + (size_t)ocp * (N + 1) * NX, s.u + (size_t)ocp * E,
                                               s.yref + (size_t)ocp * N * NY, s.yref_e + (size_t)ocp * NX, wb, web);
    } else {
        if (yb || yeb) c.forward_cotangent(yb, yeb);
    }
}

// ------------------------------------------------------------------------------------------ forward-mode sensitivities

template <typename real>
struct JvpArgs {
    IpmArgs<real> b;           // as SensArgs::b
    int K;                     // tangent directions per vehicle, >= 1
    const double* dx0;         // [B][K][13] tangent of x0, or null (zero)
    const double* dyref;       // [B][K][N][17] tangent of the reference, or null
    const double* dyref_e;     // [B][K][13] or null
    const double* dw;          // [B][K][17] tangent of w_diag, or null
    const double* dwe;         // [B][K][13] tangent of we_diag, or null
    double* dx;                // [B][K][N+1][13] or null
    double* du;                // [B][K][N][4]
    const double* x;           // [B][N+1][13] the last solve's states
    const double* u;           // [B][N][4] the last solve's inputs
    const double* yref;        // [B][N][17] the reference that solve ran with
    const double* yref_e;      // [B][13]
};

// Forward mode of the solution map of qmpc_adjoint_kernel<.., true>: on the active set the solve ended on, the tangent
// (dx, du) for (dx0, dyref, dyref_e, dw, dwe) is the minimiser of the pinned LQR of the adjoint with the linear costs
// c_k = -(Qd, Rd) dyref_k + dt dw (z_k - yref_k), c_N = -QNd dyref_e + dwe (x_N - yref_e), from dx_0 = dx0 (DESIGN.md §4).
// One warp per OCP: sens_factorise once, then per direction backward_cotangent<true> (costs formed per stage, nothing
// stored) and forward_cotangent<false, true>; the K directions share the factorisation.  A vehicle whose active set is
// unknown gets NaN in every output of every direction.  The same register budget as qmpc_adjoint_kernel.
template <typename real, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, SENS_MIN_WARPS / WARPS) qmpc_jvp_kernel(JvpArgs<real> s)
{
    QMPC_DYN_SMEM(smem_raw);
    const IpmArgs<real>& a = s.b;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ocp = blockIdx.x * WARPS + warp;
    if (ocp >= a.B) return;
    const int N = a.N, E = 4 * N, K = s.K;
    const unsigned char* act = a.act + (size_t)ocp * E;
    double* dxo = s.dx ? s.dx + (size_t)ocp * K * (N + 1) * NX : nullptr;
    double* duo = s.du + (size_t)ocp * K * E;
    int known = 1;
    for (int e = lane; e < E; e += 32) if (act[e] > 2) known = 0;
    if (!warp_min(known)) {
        const double qnan = nan("");
        if (dxo) for (int i = lane; i < K * (N + 1) * NX; i += 32) dxo[i] = qnan;
        for (int i = lane; i < K * E; i += 32) duo[i] = qnan;
        return;
    }
    WarpCtx<real> c{a};
    sens_factorise(c, smem_raw, warp, lane, ocp, act);
    TanDir t;
    t.xs = s.x + (size_t)ocp * (N + 1) * NX; t.us = s.u + (size_t)ocp * E;
    t.yr = s.yref + (size_t)ocp * N * NY; t.yre = s.yref_e + (size_t)ocp * NX;
    for (int d = 0; d < K; ++d) {
        const size_t v = (size_t)ocp * K + d;          // (vehicle, direction)
        t.dyref = s.dyref ? s.dyref + v * N * NY : nullptr;
        t.dyref_e = s.dyref_e ? s.dyref_e + v * NX : nullptr;
        t.dw = s.dw ? s.dw + v * NY : nullptr;
        t.dwe = s.dwe ? s.dwe + v * NX : nullptr;
        c.template backward_cotangent<true>(nullptr, nullptr, &t);
        c.template forward_cotangent<false, true>(nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                                                  s.dx0 ? s.dx0 + v * NX : nullptr,
                                                  dxo ? dxo + (size_t)d * (N + 1) * NX : nullptr, duo + (size_t)d * E);
    }
}

}  // namespace qmpc
