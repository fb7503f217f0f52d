// host_params.h — host-side translation of qmpc_config into kernel argument blocks
// (shared by capi.cu and the test-only emulation harness).
#pragma once
#include <cmath>
#include "../../include/qmpc.h"
#include "mpc_kernels.cuh"

namespace qmpc {

typedef qmpc_config HostOcp;

template <typename real>
inline void fill_model(const qmpc_config& c, ModelParams<real>& mp)
{
    const double* q = c.quad;
    const double mass = q[0], T = q[1];
    const double* J = q + 2;
    mp.thrust_over_mass = real(T / mass);
    mp.T = real(T);
    for (int i = 0; i < 4; ++i) { mp.xf[i] = real(q[5 + i]); mp.yf[i] = real(q[9 + i]); mp.zt[i] = real(q[13 + i]); }
    for (int i = 0; i < 3; ++i) { mp.invJ[i] = real(1.0 / J[i]); mp.g[i] = real(q[17 + i]); }
    mp.Jc[0] = real(J[1] - J[2]); mp.Jc[1] = real(J[2] - J[0]); mp.Jc[2] = real(J[0] - J[1]);
    for (int d = 0; d < 3; ++d) {
        const double L = c.gp_theta[3 * d], sf = c.gp_theta[3 * d + 1];
        mp.sf2[d] = real(sf * sf);
        mp.iL2[d] = real(L != 0.0 ? 1.0 / (L * L) : 0.0);
    }
    mp.M = c.n_basis;
    for (int d = 0; d < 3; ++d) { mp.gx0[d] = 0; mp.gdx[d] = 0; mp.gidx[d] = 0; mp.gcc[d] = 0; }
}

// Equispaced basis points (the reference builds them with linspace, GPE.py:127-150) let K1 evaluate the M kernel values of an
// axis from three exps and a two-term recurrence; grid[d] = {first point, spacing} or spacing 0 when axis d is not equispaced
// to 1e-12 of its range.  X: host [3][M].
inline void gp_grid_detect(const double* X, int M, double grid[6])
{
    for (int d = 0; d < 3; ++d) {
        grid[2 * d] = 0; grid[2 * d + 1] = 0;
        if (!X || M < 2) continue;
        const double* x = X + (size_t)d * M;
        const double dx = (x[M - 1] - x[0]) / (M - 1);
        double span = std::fabs(x[M - 1] - x[0]), dev = 0;
        for (int i = 0; i < M; ++i) dev = std::fmax(dev, std::fabs(x[i] - (x[0] + i * dx)));
        if (dx > 0 && std::isfinite(dx) && dev <= 1e-12 * span) { grid[2 * d] = x[0]; grid[2 * d + 1] = dx; }
    }
}
template <typename real>
inline void fill_gp_grid(const double grid[6], ModelParams<real>& mp)
{
    for (int d = 0; d < 3; ++d) {
        const double dx = grid[2 * d + 1];
        mp.gx0[d] = real(grid[2 * d]); mp.gdx[d] = real(dx); mp.gidx[d] = real(dx > 0 ? 1.0 / dx : 0.0);
        mp.gcc[d] = real(std::exp(-dx * dx * double(mp.iL2[d])));
    }
}

inline double cfg_dt(const qmpc_config& c) { return c.t_horizon / c.n_nodes; }
// per-warp shared memory of the Riccati kernel (reals): working set, then (fp64 QMPC_RING builds) the tile ring and one
// 8-byte mbarrier per slot.  `full`: the IPM layout (13 vectors); otherwise the screening layout (6 vectors).
inline int ipm_ring_off(int N, bool full) { return (SM_VEC + (full ? SM_NVEC : 6) * 4 * N + (N + 1) * 13 + 9) & ~1; }
inline int ipm_smem_reals(int N, bool full, bool fp64)
{
    const int ring = fp64 ? QMPC_RING : 0;
    const int hist = fp64 ? HIST_REALS<double>() : HIST_REALS<float>();
    const int mbar = fp64 ? ring : 2 * ring;
    const int refine = fp64 ? 0 : 2 * ((N + 1) * 13 + 16 + 4 * N);  // fp32 handles: (N+1) x 13 + 16 + 4N doubles of refinement scratch
    return (ipm_ring_off(N, full) + hist + ring * WT + mbar + refine + 3) & ~3;
}
// fp32 handles: offset (in floats, 8-byte aligned) of the fp64 refinement scratch = right after the fingerprint history
inline int ipm_refine_off(int N, bool full) { return ipm_ring_off(N, full) + HIST_REALS<float>();
}

template <typename real, typename treal>
inline void fill_lin_args(const qmpc_config& c, LinArgs<real, treal>& a)
{
    a.B = c.batch; a.N = c.n_nodes; a.dt = real(cfg_dt(c));
    fill_model(c, a.mp);
    a.alpha_stride = 3 * c.n_basis;
    for (int i = 0; i < 13; ++i) a.Qd[i] = real(cfg_dt(c) * c.w_diag[i]);
}

template <typename real>
inline void fill_ipm_args(const qmpc_config& c, IpmArgs<real>& a)
{
    const double dt = cfg_dt(c);
    a.B = c.batch; a.N = c.n_nodes;
    for (int i = 0; i < 13; ++i) { a.Qd[i] = real(dt * c.w_diag[i]); a.QNd[i] = real(c.we_diag[i]); }
    for (int i = 0; i < 4; ++i) a.Rd[i] = real(dt * c.w_diag[13 + i]);
    a.dt = real(dt); a.lb = real(c.lbu); a.ub = real(c.ubu);
    const bool f64 = sizeof(real) == 8;
    a.mu_tol = real(c.ipm_mu_tol > 0 ? c.ipm_mu_tol : (f64 ? 1e-13 : 1e-6));
    a.max_iter = c.ipm_max_iter > 0 ? c.ipm_max_iter : 50;
    a.max_iter_failed = a.max_iter < 20 ? a.max_iter : 20;
    a.fail_streak = nullptr;
    a.mu_switch = real(c.ipm_mu_switch > 0 ? c.ipm_mu_switch : 1e-4);
    // initial multipliers of a cold IPM: clip(0.02 * mean|dJ/du(box centre)|, 0.1, 1e5).  The upper clip used to be 100: a vehicle
    // 30-80 m off its reference (gradients of 1e3-1e4, 75 of 80 inputs saturated) then spent 25-45 iterations growing the
    // multipliers, 8-15 now; ordinary problems are unaffected (profiles/r02_lam0_sweep.txt)
#ifndef QMPC_LAM0_SCALE
#define QMPC_LAM0_SCALE 0.02
#endif
    a.lam0_scale = real(QMPC_LAM0_SCALE); a.lam0_min = real(0.1); a.lam0_max = real(1e5);
#ifdef QMPC_EMU       // tuning hook of the test-only emulation build (scripts/replay_hard.py)
    if (getenv("EMU_LAM0_SCALE")) a.lam0_scale = real(atof(getenv("EMU_LAM0_SCALE")));
    if (getenv("EMU_LAM0_MAX")) a.lam0_max = real(atof(getenv("EMU_LAM0_MAX")));
#endif
    a.refine_gtol = real(f64 ? 1e-12 : 1e-5);
    a.resfac_final = real(f64 ? 1e-9 : 1e-3);
    a.max_refine = c.refine_max_rounds < 0 ? 0 : (c.refine_max_rounds == 0 ? (f64 ? 20 : 10) : c.refine_max_rounds);
    a.post_bail = f64 ? 0 : 1;
    a.warm_rounds = (c.warm_start_rounds < 0 || a.max_refine == 0) ? 0 : (c.warm_start_rounds == 0 ? 6 : c.warm_start_rounds);
    a.smem_per_warp = ipm_smem_reals(c.n_nodes, true, f64);
    a.ring_off = ipm_ring_off(c.n_nodes, true);
    a.refine_off = f64 ? 0 : ipm_refine_off(c.n_nodes, true);
    a.bail_round = c.bail_round > 0 ? c.bail_round : 2;
    a.bail_changed = c.bail_changed > 0 ? c.bail_changed : (1 << 20);
    a.final_rollout = c.final_rollout > 0 ? 1 : 0;
    a.dense_warm_rounds = 0;
    a.warm_rounds_busy = 0; a.bail_round_busy = a.bail_round; a.busy_threshold = 1 << 30; a.skip_screen_iters = 0; a.bail_to_ipm = 0;
    a.unsettled_prev = nullptr; a.unsettled_cur = nullptr;
    a.timeline = nullptr; a.hard_list = nullptr; a.hard_count = nullptr;
}

// 1 = Riccati kernel alone, 2 = Riccati screening launch + dense condensed launch (qmpc_config::solver_variant, 0 = auto)
inline int solver_variant(const qmpc_config& c, int dense_max_nodes)
{
    const bool dense_ok = c.precision != 32 && c.n_nodes <= dense_max_nodes;     // the condensed formulation is fp64-only
    if (c.solver_variant == 1 || !dense_ok) return 1;
    return 2;
}

// screening-mode arguments (variant 2): the screening launch tries `screen_rounds` warm-started rounds, the dense launch
// continues for `dense_warm_rounds`; with the warm start switched off (warm_start_rounds < 0) neither kernel looks at
// the remembered active set and every OCP takes the cold IPM of the dense kernel.
template <typename real>
inline void fill_screen_args(const qmpc_config& c, IpmArgs<real>& a)
{
    const int screen = c.screen_rounds > 0 ? c.screen_rounds : 3;
    const int dense_warm = c.dense_warm_rounds < 0 ? 0 : (c.dense_warm_rounds == 0 ? 8 : c.dense_warm_rounds);
    a.dense_warm_rounds = a.warm_rounds > 0 ? dense_warm : 0;
    if (a.warm_rounds > 0) {
        a.warm_rounds = screen;
        a.warm_rounds_busy = c.screen_rounds_busy < 0 ? 0 : (c.screen_rounds_busy == 0 ? 8 : c.screen_rounds_busy);
        a.bail_round_busy = a.bail_round > 3 ? a.bail_round : 3;
        const int pct = c.screen_busy_pct > 0 ? c.screen_busy_pct : 25;
        a.busy_threshold = (int)((long long)c.batch * pct / 100);
        a.skip_screen_iters = 12;
        a.bail_to_ipm = 0;       // measured (profiles/r02_policy_ab.txt): sending given-up OCPs straight to the dense IPM costs 3 %
    }
    a.smem_per_warp = ipm_smem_reals(c.n_nodes, false, sizeof(real) == 8);
    a.ring_off = ipm_ring_off(c.n_nodes, false);
    a.refine_off = 0;
}

// qmpc_eval_sens_x0 / qmpc_eval_adjoint: weights of the solve, per-warp shared memory of the screening layout; the caller
// sets the pointers
template <typename real>
inline void fill_sens_base(const qmpc_config& c, IpmArgs<real>& b)
{
    fill_ipm_args(c, b);
    b.smem_per_warp = ipm_smem_reals(c.n_nodes, false, sizeof(real) == 8);
    b.ring_off = ipm_ring_off(c.n_nodes, false);
    b.refine_off = 0;
}

template <typename real>
inline void fill_sens_args(const qmpc_config& c, int n_stages, SensArgs<real>& a)
{
    fill_sens_base(c, a.b);
    a.n_stages = n_stages;
}

}  // namespace qmpc
