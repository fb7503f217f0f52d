"""GPU parity tests: the CUDA path, called through the C-ABI (libqmpc.so) behind the reference's Python API,
against the CPU oracle and the committed golden fixtures.  Tolerances (BASELINE.json north_star / SURVEY §8d):
  fp64 solver: controls and predicted states within 1e-6 relative of the exact oracle, per step from identical
               (x0, yref, alpha, iterate);  RGP mean/covariance within 1e-9 relative (always fp64);
  distance to the acados logs is reported separately (<= 1e-5 abs on u0: HPIPM's own tolerance)."""
import os

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from conftest import rel_err
from helpers import make_gp, oracle_solve_batch, random_ocp_batch, u_rel, x_rel

pytestmark = pytest.mark.gpu

TOL_U64 = 1e-6
TOL_X64 = 1e-6
TOL_RGP = 1e-9


def _pkg():
    from mpc_quad_ros_b200.quad import Quadrotor3D
    from mpc_quad_ros_b200.quad_opt import quad_optimizer
    from mpc_quad_ros_b200.gp.GPE import GPEnsemble
    return Quadrotor3D, quad_optimizer, GPEnsemble


def _solve_batch(sc, B, N, gp, precision=64, quad_name="hummingbird", mu_tol=0.0, **policy):
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    quad = Quadrotor3D(drag=True, batch=B)
    quad = quad.set_hummingbird_params() if quad_name == "hummingbird" else quad.set_logged_pysim_params()
    gpe = None
    if gp is not None and policy.pop("basis_vectors", False):
        gpe = GPEnsemble.frombasisvectors([gp.X[d] for d in range(3)], [np.zeros(gp.M)] * 3, [None] * 3, [list(gp.theta[d]) for d in range(3)], batch=B)
    elif gp is not None:
        gpe = GPEnsemble.fromrange([(gp.X[d, 0], gp.X[d, -1]) for d in range(3)], [gp.M] * 3, theta=list(gp.theta[0]), batch=B)
    opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=gpe, precision=precision, ipm_mu_tol=mu_tol, **policy)
    opt.set_iterate(torch.as_tensor(sc["xit"]), torch.as_tensor(sc["uit"]))
    dev = opt.device
    import ctypes as C
    from mpc_quad_ros_b200 import _capi
    yref = torch.as_tensor(sc["yref"], device=dev).contiguous()
    yref_e = torch.as_tensor(sc["yref_e"], device=dev).contiguous()
    _capi.check(_capi.lib().qmpc_set_yref(opt._h, _capi.ptr(yref), _capi.ptr(yref_e), _capi.stream_ptr()))
    if gp is not None:
        opt.set_rgp_params(torch.as_tensor(sc["mu"]))
    x_opt, w_opt, t_cpu, cost = opt.run_optimization(torch.as_tensor(sc["x0"], device=dev))
    st, it = opt.solver_status()
    return x_opt.cpu().numpy(), w_opt.cpu().numpy(), cost.cpu().numpy(), st.cpu().numpy(), it.cpu().numpy()


@pytest.mark.parametrize("N,M,seed", [(20, 20, 140), (10, 0, 110), (50, 20, 170), (7, 50, 157), (20, 100, 220), (50, 20, 1070), (20, 50, 1070),
                                      (1, 0, 1), (2, 3, 2), (3, 20, 3), (21, 20, 21)])
def test_solve_fp64_vs_oracle(N, M, seed):
    """(50, 20, 1070) and (20, 50, 1070) are the cells of profiles/r01_sweep.md where an early exit of the post-IPM
    active-set rounds once left an IPM-accurate (3.5e-6) instead of an exact answer; N = 1, 2, 3 are horizons shorter than
    or equal to the tile ring / condensing chunk (TMA ring and mbarrier phases at their edges), N = 21 the largest horizon
    of the dense kernel"""
    B, dt = 48, 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp(M) if M else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=seed)
    x, u, cost, st, it = _solve_batch(sc, B, N, gp)
    xo, uo, co, ito = oracle_solve_batch(sc, quad, dt, N, gp)
    assert (st == 0).all(), st
    assert u_rel(u, uo) < TOL_U64, u_rel(u, uo)
    assert x_rel(x, xo) < TOL_X64, x_rel(x, xo)
    # the solver ends on an exact KKT point (active-set rounds), not on an IPM-accurate one: 1e-12 on the Riccati path,
    # <= 1e-8 through the condensed Hessian of the dense kernel
    assert u_rel(u, uo) < 1e-7 and x_rel(x, xo) < 1e-7, (u_rel(u, uo), x_rel(x, xo))
    assert np.abs(cost - co).max() < 1e-7 * max(1.0, np.abs(co).max())
    assert ((u > 0 - 1e-12) & (u < 1 + 1e-12)).all()
    assert np.abs(x[:, 0] - sc["x0"]).max() == 0.0
    nact = ((uo < 1e-9) | (uo > 1 - 1e-9)).sum()
    assert nact > 0 or N < 3                           # the batch does exercise active thrust limits
    print(f"N={N} M={M}: u_rel={u_rel(u, uo):.2e} x_rel={x_rel(x, xo):.2e} ipm iters mean={it.mean():.1f} (oracle {ito.mean():.1f})")


@pytest.mark.parametrize("layout", ["scattered", "narrow_kernel", "velocities_off_grid", "two_points"])
def test_gp_basis_point_layouts_vs_oracle(layout):
    """K1 evaluates an equispaced axis (linspace, GPE.fromrange) with three exps and a recurrence started at the basis point
    nearest to the velocity, any other layout with one exp per kernel value: scattered points take the general path; a
    length-scale far below the spacing, velocities outside the grid and a two-point grid stress the recurrence"""
    B, N, M, dt = 48, 20, 20, 1.0 / 20
    rng = np.random.default_rng(5)
    quad = orc.quad_hummingbird()
    if layout == "scattered":
        X = np.sort(rng.uniform(-10, 10, (3, M)), axis=1)
        gp = orc.GPSpec(X, np.array((3.0, 0.1, 0.01)))
    elif layout == "narrow_kernel":
        gp = orc.GPSpec(np.tile(np.linspace(-10, 10, M), (3, 1)), np.array((0.3, 0.5, 0.01)))
    elif layout == "velocities_off_grid":
        gp = orc.GPSpec(np.tile(np.linspace(-0.5, 0.5, M), (3, 1)), np.array((0.2, 0.3, 0.01)))
    else:
        M = 2
        gp = orc.GPSpec(np.tile(np.linspace(-3, 3, M), (3, 1)), np.array((3.0, 0.1, 0.01)))
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=31)
    x, u, cost, st, it = _solve_batch(sc, B, N, gp, basis_vectors=True)
    xo, uo, co, ito = oracle_solve_batch(sc, quad, dt, N, gp)
    assert (st == 0).all(), st
    assert u_rel(u, uo) < 1e-7 and x_rel(x, xo) < 1e-7, (layout, u_rel(u, uo), x_rel(x, xo))
    # the GP term does matter in these problems: the nominal model gives a different answer
    xn, un, _, _, _ = _solve_batch(sc, B, N, None)
    assert u_rel(un, uo) > 1e-5 or layout == "velocities_off_grid", u_rel(un, uo)
    print(f"{layout}: u_rel={u_rel(u, uo):.2e} x_rel={x_rel(x, xo):.2e}; nominal model differs by {u_rel(un, uo):.2e}")


def test_solve_full_baseline_batch_subset_vs_oracle():
    """BASELINE config 2 size (4096 vehicles, N=20, M=20): every vehicle converges; a random subset of 64 is compared
    with the oracle; the rest is covered by size-independent properties (bounds, x0 pin, determinism)."""
    B, N, M = 4096, 20, 20
    dt = 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp(M)
    base = random_ocp_batch(128, N, dt, quad, gp, seed=7)
    rep = B // 128
    sc = {k: (None if v is None else np.concatenate([v] * rep)) for k, v in base.items()}
    x, u, cost, st, it = _solve_batch(sc, B, N, gp)
    assert (st == 0).all()
    x2, u2, cost2, st2, it2 = _solve_batch(sc, B, N, gp)
    assert np.array_equal(u, u2) and np.array_equal(x, x2)          # deterministic
    assert np.array_equal(u[:128], u[128 * 5:128 * 6])               # replicated inputs -> identical outputs
    assert ((u >= 0) & (u <= 1)).all()
    idx = np.random.default_rng(0).choice(128, 64, replace=False)
    xo, uo, co, ito = oracle_solve_batch(base, quad, dt, N, gp, idx)
    assert u_rel(u[idx], uo) < TOL_U64 and x_rel(x[idx], xo) < TOL_X64


@pytest.mark.parametrize("name,use_gp,nmax", [("traj2_v10_a10_gp0", False, None), ("traj0_v10_a10_gp2", True, None),
                                              ("traj1_v15_a5_gp2", True, 46)])
def test_golden_log_replay_through_reference_api(golden, name, use_gp, nmax):
    """Replays the reference's shipped acados logs through quad_optimizer (single vehicle, numpy API)."""
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    g = golden(name)
    N, dt = 10, 0.1
    quad = Quadrotor3D(drag=True).set_logged_pysim_params()
    gpe, gp = None, None
    if use_gp:
        X, th = g["rgp_X"], g["rgp_theta"]
        gpe = GPEnsemble.fromrange([(X[d, 0], X[d, -1]) for d in range(3)], [X.shape[1]] * 3, theta=list(th[0]))
        gp = orc.GPSpec(X, th)
    opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=gpe)
    xit, uit = np.zeros((N + 1, 13)), np.zeros((N, 4))
    n = len(g["x_odom"]) if nmax is None else nmax
    e_log, e_orc, e_cost = [], [], []
    for i in range(min(n, len(g["x_ref"]) - N)):
        x_ref = g["x_ref"][i:i + N]
        yref, yref_N = opt.set_reference_trajectory(x_ref)
        assert yref.shape == (N, 17) and np.all(yref[:, 13:] == 0.16) and np.array_equal(yref_N, x_ref[-1])
        alpha = None
        if use_gp:
            p = np.zeros((3, gp.M)) if i == 0 else g["rgp_mu"][i - 1]
            opt.set_rgp_params(p)
            alpha = gp.alpha(p)
        x_opt, w_opt, t_cpu, cost = opt.run_optimization(g["x_odom"][i])
        yr, yre = orc.make_yref(x_ref)
        orc.rti_step(orc.quad_logged_pysim(), dt, N, g["x_odom"][i], yr, yre, xit, uit, gp=gp, alpha=alpha)
        e_log.append(np.abs(w_opt[0] - g["w_odom"][i]).max())
        e_orc.append(max(np.abs(w_opt - uit).max(), np.abs(x_opt - xit).max() / max(1.0, np.abs(xit).max())))
        e_cost.append(abs(cost - g["cost_solution"][i]) / abs(g["cost_solution"][i]))
        # keep both iterates identical so that every step is a per-step parity check (SURVEY §8c caveat)
        opt.set_iterate(xit[None], uit[None])
    e_log, e_orc = np.array(e_log), np.array(e_orc)
    print(f"{name}: vs acados log median {np.median(e_log):.1e} max {e_log.max():.1e}; vs oracle max {e_orc.max():.1e}; cost rel {max(e_cost):.1e}")
    assert e_orc.max() < TOL_U64
    assert np.median(e_log) < 5e-8 and e_log.max() < 1e-5
    assert max(e_cost) < 2e-5


def test_golden_log_free_running_replay(golden):
    """Same log, but the GPU solver carries its OWN iterate across all 289 steps (no injection): contractive log."""
    Quadrotor3D, quad_optimizer, _ = _pkg()
    g = golden("traj2_v10_a10_gp0")
    N = 10
    opt = quad_optimizer(Quadrotor3D(drag=True).set_logged_pysim_params(), t_horizon=1.0, n_nodes=N)
    errs = []
    for i in range(len(g["x_ref"]) - N):
        opt.set_reference_trajectory(g["x_ref"][i:i + N])
        x_opt, w_opt, _, cost = opt.run_optimization(g["x_odom"][i])
        errs.append(np.abs(w_opt[0] - g["w_odom"][i]).max())
    assert np.median(errs) < 5e-8 and max(errs) < 1e-5


@pytest.mark.parametrize("name,tol", [("traj0_v10_a10_gp2", TOL_RGP), ("traj1_v15_a5_gp2", TOL_RGP), ("traj0_v15_a5_gp2", TOL_RGP),
                                      ("traj2_v10_a10_gp2", 1e-7)])
def test_rgp_regress_golden_logs(golden, name, tol):
    """GPEnsemble.regress against the logged RGP state sequences (list-in / list-out reference API);
    the last log is the reference's own DIVERGING run (mu -> 1e12, SURVEY App. C-7), kept as an operand-order stress."""
    _, _, GPEnsemble = _pkg()
    g = golden(name)
    X, th = g["rgp_X"], g["rgp_theta"]
    gpe = GPEnsemble.fromrange([(X[d, 0], X[d, -1]) for d in range(3)], [X.shape[1]] * 3, theta=list(th[0]))
    assert gpe.type == "RGP" and np.allclose(gpe.gp[0].X, X[0])
    worst_mu = worst_C = 0.0
    for i in range(len(g["v_body"])):
        mu, Cm = gpe.regress([np.array([g["v_body"][i, d]]) for d in range(3)], [np.array([g["a_drag"][i, d]]) for d in range(3)])
        worst_mu = max(worst_mu, rel_err(np.stack(mu), g["rgp_mu"][i]))
        worst_C = max(worst_C, rel_err(np.stack(Cm), g["rgp_C"][i]))
    print(f"{name}: rgp rel err mu {worst_mu:.1e} C {worst_C:.1e}")
    assert worst_mu < tol and worst_C < tol
    assert np.array_equal(gpe.gp[1].mu_g_t, mu[1]) and gpe.gp[2].C_g_t.shape == (X.shape[1],) * 2


@pytest.mark.parametrize("tag", ["m20", "m50", "m7"])
def test_rgp_reference_code_fixture_batched(golden, tag):
    """RGP.regress / predict / predict_using_y outputs of the reference's own numpy code (M = 20, 50, 7), with the
    vehicles of a batch fed the same sequence at different offsets (ragged progress)."""
    _, _, GPEnsemble = _pkg()
    g = golden("reference_code")
    X, th = g[f"rgp_{tag}_X"], g[f"rgp_{tag}_theta"]
    M, T = X.shape[1], len(g[f"rgp_{tag}_xt"])
    B = 5
    gpe = GPEnsemble.fromrange([(X[d, 0], X[d, -1]) for d in range(3)], [M] * 3, theta=list(th[0]), batch=B)
    assert rel_err(gpe.K_x_inv, g[f"rgp_{tag}_Kx_inv"]) < 1e-9
    xt, yt = g[f"rgp_{tag}_xt"], g[f"rgp_{tag}_yt"]
    for t in range(T):
        # vehicle b is b samples behind; NaN = "no sample for this vehicle yet" (axis skipped by the kernel)
        xb = np.stack([xt[t - b] if t - b >= 0 else np.full(3, np.nan) for b in range(B)])
        yb = np.stack([yt[t - b] if t - b >= 0 else np.zeros(3) for b in range(B)])
        mu, Cm = gpe.regress(torch.as_tensor(xb), torch.as_tensor(yb))
    mu, Cm = mu.cpu().numpy(), Cm.cpu().numpy()
    for b in range(B):
        assert rel_err(mu[b], g[f"rgp_{tag}_mu"][T - 1 - b]) < TOL_RGP
        assert rel_err(Cm[b], g[f"rgp_{tag}_C"][T - 1 - b]) < TOL_RGP
    xs = g[f"rgp_{tag}_pred_x"]
    mean, std = gpe.predict(torch.as_tensor(np.broadcast_to(xs, (B, 3, len(xs))).copy()), std=True)
    assert rel_err(mean[0].cpu().numpy(), g[f"rgp_{tag}_pred_mean"]) < TOL_RGP
    var_ref = g[f"rgp_{tag}_pred_var"]
    assert np.abs(std[0].cpu().numpy() ** 2 - var_ref).max() < 1e-9 * max(1.0, np.abs(var_ref).max())
    y = g[f"rgp_{tag}_puy_y"]
    puy = gpe.predict_using_y(torch.as_tensor(np.broadcast_to(xs, (B, 3, len(xs))).copy()), torch.as_tensor(np.broadcast_to(y, (B, 3, M)).copy()))
    assert rel_err(puy[0].cpu().numpy(), g[f"rgp_{tag}_puy_mean"]) < TOL_RGP
    # alpha = K_x^-1 mu is what the OCP model consumes
    al = gpe.alpha_tensor().cpu().numpy()
    assert rel_err(al[0], np.einsum("dij,dj->di", g[f"rgp_{tag}_Kx_inv"], mu[0])) < 1e-9


def test_helpers_vs_golden(golden):
    from mpc_quad_ros_b200.utils import utils
    Quadrotor3D, quad_optimizer, _ = _pkg()
    g, gl = golden("reference_code"), golden("traj0_v10_a10_gp2")
    # compute_a_drag: reference list format for one vehicle, tensors for a batch
    vb, ad = utils.compute_a_drag(g["drag_x_now"][0], g["drag_x_pred"][0], float(g["drag_dt"]))
    assert isinstance(vb, list) and len(vb) == 3 and vb[0].shape == (1,)
    vbt, adt = utils.compute_a_drag(torch.as_tensor(g["drag_x_now"]).cuda(), torch.as_tensor(g["drag_x_pred"]).cuda(), float(g["drag_dt"]))
    assert np.abs(vbt.cpu().numpy() - g["drag_v_body"]).max() < 1e-13
    assert np.abs(adt.cpu().numpy() - g["drag_a_drag"]).max() < 1e-11
    assert abs(vb[1][0] - g["drag_v_body"][0, 1]) < 1e-13
    # get_reference_chunk incl. end padding and skip: bit exact
    for n, (idx, N, skip) in enumerate(g["chunk_cases"]):
        out = utils.get_reference_chunk(g["chunk_traj"], int(idx), int(N), int(skip))
        assert np.array_equal(out, g[f"chunk_{n}"]), (idx, N, skip)
    # discrete_dynamics (nominal RK4) against the logged one-step predictions
    quad = Quadrotor3D(drag=True).set_logged_pysim_params()
    opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=10)
    xp = opt.discrete_dynamics(torch.as_tensor(gl["x_odom"]).cuda(), torch.as_tensor(gl["w_odom"]).cuda(), 0.1)
    assert np.abs(xp.cpu().numpy() - gl["x_pred_odom"]).max() < 1e-13
    x1 = opt.discrete_dynamics(gl["x_odom"][3], gl["w_odom"][3], 0.1)
    assert x1.shape == (13,) and np.abs(x1 - gl["x_pred_odom"][3]).max() < 1e-13
    xb = opt.discrete_dynamics(gl["x_odom"][3], gl["w_odom"][3], 0.1, body_frame=True)
    assert np.abs(xb[7:10] - orc.compute_a_drag(x1, x1, 0.1)[0]).max() < 1e-13
    with pytest.raises(AssertionError):
        opt.discrete_dynamics(np.zeros(12), np.zeros(4), 0.1)
    with pytest.raises(ValueError):
        opt.run_optimization(None)
    # plant (Quadrotor3D.update over one control period) against the reference's own class
    for tag in ("hb", "log"):
        xs, us, xn = g[f"plant_{tag}_x"], g[f"plant_{tag}_u"], g[f"plant_{tag}_xnext"]
        q = Quadrotor3D(drag=True, batch=len(xs))
        q = q.set_hummingbird_params() if tag == "hb" else q.set_logged_pysim_params()
        q.set_state(xs)
        for _ in range(11):
            q.update(torch.as_tensor(us), 5e-3)
        assert np.abs(q.get_state(quaternion=True, stacked=True).cpu().numpy() - xn).max() < 1e-12


@pytest.mark.parametrize("use_gp", [True, False])
def test_closed_loop_vs_oracle(use_gp):
    """ClosedLoop (fused qmpc_step + plant + chunk on the GPU) against the oracle's closed loop, 32 vehicles x 12 steps,
    BASELINE shape N=20, M=20.  Both loops run freely (no injection): over 12 steps they stay within tolerance."""
    from mpc_quad_ros_b200.execute_trajectory import ClosedLoop
    from mpc_quad_ros_b200.trajectory import random_smooth_trajectories
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    B, N, M, steps = 32, 20, 20, 12
    dt = 1.0 / N
    quad = Quadrotor3D(drag=True, batch=B).set_hummingbird_params()
    gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [M] * 3, theta=[3.0, 0.1, 0.01], batch=B) if use_gp else None
    opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=gpe)
    traj = random_smooth_trajectories(B, steps + N + 3, dt)
    x0 = traj[:, 0, :].copy()
    x0[:, :3] += np.random.default_rng(3).uniform(-0.5, 0.5, (B, 3))
    loop = ClosedLoop(quad, opt, torch.as_tensor(traj), torch.as_tensor(x0))
    assert loop.n_sub == 11
    xs, us = loop.run(steps, record=True)
    ref = orc.ClosedLoop(orc.quad_hummingbird(), dt, N, traj, x0, gp=make_gp(M) if use_gp else None)
    r = ref.run(steps)
    assert r["bad"] == 0
    assert u_rel(us.cpu().numpy(), r["u0"]) < TOL_U64
    assert x_rel(xs.cpu().numpy(), r["x"]) < TOL_X64
    if use_gp:
        assert rel_err(gpe.mu_tensor().cpu().numpy(), ref.mu) < 1e-6      # closed-loop accumulation of 1e-9-level control differences
        assert rel_err(gpe.C_tensor().cpu().numpy(), ref.C) < 1e-6   # free-running loop: C sees the 1e-9-level state differences through Jt; per-step RGP parity (1e-9) is tested above


def test_simulate_trajectory_single_vehicle_reference_api():
    """The reference's loop, method by method, for ONE vehicle with numpy in/out (drop-in surface), RGP in the loop."""
    from mpc_quad_ros_b200.execute_trajectory import simulate_trajectory
    from mpc_quad_ros_b200.trajectory import sample_circle_trajectory_accelerating
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    N, steps = 10, 15
    quad = Quadrotor3D(payload=False, drag=True).set_logged_pysim_params()
    x0 = np.array([0.0, 0.0, 3.0] + [1.0, 0.0, 0.0, 0.0] + [0.0] * 6)
    quad.set_state(x0)
    gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [10] * 3, theta=[3.0, 0.1, 0.01])
    opt = quad_optimizer(quad, t_horizon=1, n_nodes=N, gpe=gpe)
    nominal = quad_optimizer(quad, t_horizon=1, n_nodes=N, gpe=None)
    traj, t = sample_circle_trajectory_accelerating(10, 10, 30, opt.optimization_dt)
    log = simulate_trajectory(quad, opt, nominal, x0, traj, max(t), steps, 5e-3)
    assert isinstance(log["w_odom"][0], np.ndarray) and log["w_odom"][0].shape == (4,)
    assert isinstance(log["rgp_mu_g_t"][0], list) and log["rgp_mu_g_t"][0][0].shape == (10,)
    ref = orc.ClosedLoop(orc.quad_logged_pysim(), 0.1, N, traj[None], x0[None], gp=make_gp(10))
    r = ref.run(steps)
    u = np.array(log["w_odom"])
    assert u_rel(u, r["u0"][:, 0]) < TOL_U64
    assert rel_err(np.stack(log["rgp_mu_g_t"][-1]), ref.mu[0]) < 1e-7


TOL_F32 = 1e-4      # north_star: controls and predicted trajectories within 1e-4 relative in the fp32 build


@pytest.mark.parametrize("N,M,seed,amps", [(20, 20, 11, (2.0,)), (20, 20, 140, (2.0, 8.0, 25.0)), (10, 0, 110, (2.0, 8.0, 25.0)),
                                           (50, 20, 170, (2.0, 8.0, 25.0)), (10, 50, 157, (2.0, 8.0)), (20, 100, 220, (2.0, 8.0, 25.0))])
def test_fp32_solver_within_1e4_of_oracle(N, M, seed, amps):
    """fp32 build (qmpc_config.precision = 32): the linearisation runs in fp64 and is rounded once into fp32 stage tiles, the
    Riccati / IPM / active-set solver runs in fp32 and its result takes one step of iterative refinement with an fp64
    residual (mpc_kernels.cuh refine_solution_fp64).  Tolerance of north_star for fp32: 1e-4 relative, also with the thrust
    limits active (amplitudes 8 and 25 saturate the inputs)."""
    B, dt = 48, 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp(M) if M else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=seed, amp_choices=amps)
    x, u, cost, st, it = _solve_batch(sc, B, N, gp, precision=32)
    xo, uo, co, ito = oracle_solve_batch(sc, quad, dt, N, gp)
    assert np.isfinite(u).all() and ((u >= 0) & (u <= 1)).all()
    print(f"fp32 N={N} M={M}: u_rel={u_rel(u, uo):.2e} x_rel={x_rel(x, xo):.2e} status={np.bincount(st)}")
    ok = st == 0
    assert ok.mean() >= 0.95
    assert u_rel(u[ok], uo[ok]) < TOL_F32 and x_rel(x[ok], xo[ok]) < TOL_F32


@pytest.mark.parametrize("M", [20, 50])
def test_shared_swarm_rgp_vs_sequential_oracle(M):
    """shared-swarm mode (BASELINE config 3): information-form accumulate + apply on the GPU equals the oracle's
    sequential single-sample regress over all vehicles (order independent), within the RGP tolerance."""
    from mpc_quad_ros_b200.swarm import SharedSwarmRGP
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    B, N = 96, 10
    gp = make_gp(M)
    gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [M] * 3, theta=[3.0, 0.1, 0.01], batch=1)
    quad = Quadrotor3D(drag=True, batch=B).set_hummingbird_params()
    opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=gpe)
    swarm = SharedSwarmRGP(gpe, opt)
    rng = np.random.default_rng(5)
    mu = np.zeros((3, M)); Cm = np.stack([orc.rgp_prior(gp.X[d], gp.theta[d])[0] for d in range(3)])
    for rnd in range(3):
        xt = rng.uniform(-9, 9, (B, 3)); yt = -0.3 * xt + 0.02 * rng.standard_normal((B, 3))
        swarm.update(torch.as_tensor(xt).cuda(), torch.as_tensor(yt).cuda())
        for v in range(B):
            for d in range(3):
                orc.rgp_regress(gp.X[d], gp.theta[d], gp.Kx_inv[d], mu[d], Cm[d], xt[v, d], yt[v, d])
        assert rel_err(gpe.mu_tensor()[0].cpu().numpy(), mu) < 1e-8
        assert rel_err(gpe.C_tensor()[0].cpu().numpy(), Cm) < 1e-8
    # the shared model feeds every vehicle's OCP (alpha broadcast): one fused step runs and matches per-vehicle alpha
    sc = random_ocp_batch(B, N, 1.0 / N, orc.quad_hummingbird(), gp, seed=9)
    alpha = gp.alpha(mu)
    x_ref = torch.as_tensor(sc["yref"][:, :, :13].copy()).cuda()
    xpp = torch.zeros((B, 13), dtype=torch.float64, device="cuda")
    u0 = torch.empty((B, 4), dtype=torch.float64, device="cuda")
    opt.set_iterate(torch.as_tensor(sc["xit"]), torch.as_tensor(sc["uit"]))
    opt.step(torch.as_tensor(sc["x0"]).cuda(), x_ref, xpp, True, u0)
    for b in range(0, B, 17):
        x, u = sc["xit"][b].copy(), sc["uit"][b].copy()
        yr, yre = orc.make_yref(sc["yref"][b][:, :13])
        orc.rti_step(orc.quad_hummingbird(), 1.0 / N, N, sc["x0"][b], yr, yre, x, u, gp=gp, alpha=alpha)
        assert np.abs(u0[b].cpu().numpy() - u[0]).max() < 1e-6
    swarm.update()        # residuals left by the fused step
    assert torch.isfinite(gpe.mu_tensor()).all()


def test_logger_schema_and_rgp_checkpoint(tmp_path):
    """log writer with the reference's pickle schema (SURVEY §8f-3) and RGP state checkpoint/restore"""
    from mpc_quad_ros_b200.Logger import Logger, load_log, load_rgp_state, save_rgp_state
    from mpc_quad_ros_b200.execute_trajectory import simulate_trajectory
    from mpc_quad_ros_b200.trajectory import sample_circle_trajectory_accelerating
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    quad = Quadrotor3D(drag=True).set_logged_pysim_params()
    x0 = np.array([0.0, 0.0, 3.0, 1.0, 0, 0, 0, 0, 0, 0, 0, 0, 0])
    quad.set_state(x0)
    gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [10] * 3, theta=[3.0, 0.1, 0.01])
    opt = quad_optimizer(quad, t_horizon=1, n_nodes=10, gpe=gpe)
    nominal = quad_optimizer(quad, t_horizon=1, n_nodes=10)
    traj, t = sample_circle_trajectory_accelerating(10, 10, 30, 0.1)
    logger = Logger(str(tmp_path / "run"))
    simulate_trajectory(quad, opt, nominal, x0, traj, max(t), 6, 5e-3, logger)
    d = load_log(logger.save_log())
    for k in ("x_odom", "x_pred_odom", "x_ref", "t_odom", "w_odom", "t_cpu", "cost_solution", "rgp_mu_g_t", "rgp_C_g_t", "v_body", "a_drag"):
        assert k in d and len(d[k]) == 6, k
    assert d["x_odom"][0].shape == (13,) and d["w_odom"][0].shape == (4,) and np.stack(d["rgp_C_g_t"][-1]).shape == (3, 10, 10)
    save_rgp_state(gpe, str(tmp_path / "rgp.npz"))
    mu = gpe.mu_tensor().clone()
    gpe.set_state(torch.zeros_like(mu), None)
    load_rgp_state(gpe, str(tmp_path / "rgp.npz"))
    assert torch.equal(gpe.mu_tensor(), mu)


def test_grouped_streams_equal_single_stream():
    """GroupedClosedLoop (vehicle groups on separate CUDA streams) against the single-stream loop.  Every OCP ends on the
    same exact minimiser whichever kernel solved it, but WHICH kernel (Riccati rounds or dense kernel) can depend on the
    handle's busy-step policy, i.e. on the other vehicles of the handle: equal to solver accuracy, not bit for bit."""
    from mpc_quad_ros_b200.execute_trajectory import ClosedLoop, GroupedClosedLoop
    from mpc_quad_ros_b200.trajectory import random_smooth_trajectories
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    B, N, M, steps = 64, 20, 20, 6
    traj = random_smooth_trajectories(B, steps + N + 3, 1.0 / N)
    x0 = traj[:, 0, :].copy()

    def make(first=0, count=B):
        quad = Quadrotor3D(drag=True, batch=count).set_hummingbird_params()
        gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [M] * 3, theta=[3.0, 0.1, 0.01], batch=count)
        opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=gpe)
        return ClosedLoop(quad, opt, torch.as_tensor(traj[first:first + count]), torch.as_tensor(x0[first:first + count]))

    single = make()
    for _ in range(steps):
        single.step()
    grouped = GroupedClosedLoop(make, B, 4)
    for _ in range(steps):
        grouped.step()
    torch.cuda.synchronize()
    xg = torch.cat([lp.x for lp in grouped.loops]); ug = torch.cat([lp.u0 for lp in grouped.loops])
    mug = torch.cat([lp.opt.gpe.mu_tensor() for lp in grouped.loops])
    assert (xg - single.x).abs().max().item() < 1e-8 and (ug - single.u0).abs().max().item() < 1e-8
    assert (mug - single.opt.gpe.mu_tensor()).abs().max().item() < 1e-8


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [1, 2])
def test_solver_kernel_variants_agree_with_oracle(variant):
    """qmpc_config.solver_variant selects the kernel mapping behind qmpc_solve (1 Riccati kernel alone, 2 = default for
    fp64 and N <= 21: Riccati screening + dense condensed kernel).  Both mappings land on the oracle's minimiser."""
    B, N, M = 67, 20, 20                      # odd batch: partial CTA paths
    dt = 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp(M)
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=7, amp_choices=(8.0, 2.0, 0.5))
    x, u, cost, st, it = _solve_batch(sc, B, N, gp, solver_variant=variant)
    xo, uo, co, ito = oracle_solve_batch(sc, quad, dt, N, gp)
    assert (st == 0).all(), st
    assert u_rel(u, uo) < TOL_U64 and x_rel(x, xo) < TOL_X64
    assert np.abs(cost - co).max() < 1e-7 * max(1.0, np.abs(co).max())


@pytest.mark.gpu
def test_failed_solve_reinitialises_iterate_on_reference():
    """A vehicle whose solve breaks down (here: a non-finite iterate) holds its previous control, and before the next solve
    its SQP iterate is re-initialised on the reference (aux_kernels.cuh reset_failed_kernel): the next solve is healthy
    again and equals a solve started from that reference iterate.  The other vehicles are untouched."""
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    import ctypes as C
    from mpc_quad_ros_b200 import _capi
    B, N = 8, 20
    dt = 1.0 / N
    quadp = orc.quad_hummingbird()
    sc = random_ocp_batch(B, N, dt, quadp, None, seed=11, amp_choices=(1.0,))
    quad = Quadrotor3D(drag=True, batch=B).set_hummingbird_params()
    opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=None)
    dev = opt.device
    xit, uit = sc["xit"].copy(), sc["uit"].copy()
    xit[3, 5, 2] = np.nan
    opt.set_iterate(torch.as_tensor(xit), torch.as_tensor(uit))
    yref = torch.as_tensor(sc["yref"], device=dev).contiguous()
    yref_e = torch.as_tensor(sc["yref_e"], device=dev).contiguous()
    _capi.check(_capi.lib().qmpc_set_yref(opt._h, _capi.ptr(yref), _capi.ptr(yref_e), _capi.stream_ptr()))
    x0 = torch.as_tensor(sc["x0"], device=dev)
    opt.run_optimization(x0)
    st, _ = opt.solver_status()
    assert st.cpu().numpy().tolist() == [0, 0, 0, 2, 0, 0, 0, 0]
    x1, u1 = (t.cpu().numpy() for t in opt.get_iterate())
    # second solve: vehicle 3 restarts from (reference states, reference inputs)
    opt.run_optimization(x0)
    st2, _ = opt.solver_status()
    assert (st2.cpu().numpy() == 0).all()
    x2, u2 = (t.cpu().numpy() for t in opt.get_iterate())
    xr, ur = x1.copy(), u1.copy()
    xr[3, :N] = sc["yref"][3, :, :13]; xr[3, N] = sc["yref_e"][3]; ur[3] = sc["yref"][3, :, 13:]
    sc2 = dict(sc); sc2["xit"], sc2["uit"] = xr, ur
    xo, uo, _, _ = oracle_solve_batch(sc2, quadp, dt, N, None)
    assert u_rel(u2, uo) < TOL_U64 and x_rel(x2, xo) < TOL_X64


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["m10", "m20", "m7"])
def test_rgp_learn_kernel_vs_reference_code(golden, tag):
    """qrgp_learn_kernel through the C-ABI (RGPLearner) against RGP.learn of the reference's numpy code: a batch of 5
    models fed the same 12 samples (every model must reproduce the fixture), plus the numpy-style batch-1 surface"""
    from mpc_quad_ros_b200.gp.RGP import RGPLearner
    g = golden("rgp_learn")
    X, theta = g[f"learn_{tag}_X"], g[f"learn_{tag}_theta"]
    B = 5
    lr = RGPLearner(X, theta=list(theta), batch=B)
    one = RGPLearner(X, np.zeros(X.shape[0]), theta=list(theta))
    for t, (xt, yt) in enumerate(zip(g[f"learn_{tag}_xt"], g[f"learn_{tag}_yt"])):
        mu_z, C_z = lr.learn(torch.full((B,), xt, dtype=torch.float64), torch.full((B,), yt, dtype=torch.float64))
        assert (lr.status() == 0).all()
        for b in (0, B - 1):
            assert rel_err(mu_z[b].cpu().numpy(), g[f"learn_{tag}_mu_z"][t]) < TOL_RGP
            assert rel_err(C_z[b].cpu().numpy(), g[f"learn_{tag}_C_z"][t]) < TOL_RGP
        mz1, Cz1 = one.learn(np.array([xt]), np.array([yt]))
        assert rel_err(mz1, g[f"learn_{tag}_mu_z"][t]) < TOL_RGP and rel_err(Cz1, g[f"learn_{tag}_C_z"][t]) < TOL_RGP
    for name, val in (("mu_g", lr.mu_g_t), ("C_g", lr.C_g_t), ("mu_eta", lr.mu_eta_t), ("C_eta", lr.C_eta_t), ("Kx_inv", lr.K_x_inv)):
        assert rel_err(val[B - 1].cpu().numpy(), g[f"learn_{tag}_{name}"][-1]) < TOL_RGP, name
    assert rel_err(np.array(one.get_theta()), g[f"learn_{tag}_mu_eta"][-1]) < TOL_RGP


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["m20", "m7"])
def test_rgp_predict_cov_and_gain_vs_reference_code(golden, tag):
    """RGP.predict(cov=True, return_Jt=True) (RGP.py:195-229): full posterior covariance and gain rows after 25 regress
    calls, against the reference's numpy code; also the var / std / return_Jt return conventions"""
    from mpc_quad_ros_b200.gp.RGP import RGP
    g = golden("rgp_predict_cov")
    X, theta = g[f"pc_{tag}_X"], list(g[f"pc_{tag}_theta"])
    r = RGP(X, np.zeros(X.shape[0]), theta=theta)
    for xt, yt in zip(g[f"pc_{tag}_xt"], g[f"pc_{tag}_yt"]):
        r.regress(np.array([xt]), np.array([yt]))
    xs = g[f"pc_{tag}_xs"]
    mean, C_p, Jt = r.predict(xs, cov=True, return_Jt=True)
    assert rel_err(mean, g[f"pc_{tag}_mean"]) < TOL_RGP and rel_err(Jt, g[f"pc_{tag}_Jt"]) < TOL_RGP
    assert rel_err(C_p, g[f"pc_{tag}_cov"]) < TOL_RGP
    m2, v2, J2 = r.predict(xs, var=True, return_Jt=True)
    assert np.allclose(v2, np.diag(C_p)) and np.array_equal(J2, Jt)
    m3, J3 = r.predict(xs, return_Jt=True)
    assert np.array_equal(m3, mean) and J3.shape == (xs.shape[0], X.shape[0])


# ------------------------------------------------------------------------------------------ round 2 additions

def test_device_reference_generators_match_host_sampling():
    """qmpc_reference_generate (SURVEY §8f-2) against the host-sampled trajectories cut with utils.get_reference_chunk:
    sinusoid sums (config 2), lemniscate (config 5) and the reference's accelerating circle incl. its '%.6f' rounding
    (config 1, TrajectoryGenerator.py:41-74), with end padding and skip"""
    from mpc_quad_ros_b200 import trajectory as T
    from mpc_quad_ros_b200.utils import utils
    B, N, dt = 7, 20, 0.05
    K = 90
    cases = [
        (T.KIND_SINUSOIDS, T.random_smooth_params(B, K, dt, seed=77), T.random_smooth_trajectories(B, K, dt, seed=77), 1e-12),
        (T.KIND_LEMNISCATE, T.lemniscate_params(B, v_peak=20.0, seed=5), T.lemniscate_trajectories(B, K, dt, v_peak=20.0, seed=5), 1e-12),
    ]
    circ, ts = T.sample_circle_trajectory_accelerating(10, 10, 30, dt)
    cases.append((T.KIND_CIRCLE, T.circle_params(10, 10, 30, dt, B=2), np.stack([circ, circ]), 0.0))
    for kind, par, traj, tol in cases:
        Bk, Kk = traj.shape[0], traj.shape[1]
        gen = T.DeviceReference(kind, par, Kk, dt)
        out = torch.empty((Bk, N, 13), dtype=torch.float64, device="cuda")
        for idx, skip in ((0, 1), (17, 1), (Kk - N - 1, 1), (Kk - 5, 1), (Kk - 1, 1), (3, 2), (Kk - 25, 2), (Kk - 2, 3)):
            gen.chunk(idx, N, out, skip=skip)
            got = out.cpu().numpy()
            for b in range(Bk):
                want = utils.get_reference_chunk(traj[b], idx, N, skip)
                err = np.abs(got[b] - want).max()
                assert err <= tol, (kind, idx, skip, b, err)


def test_closed_loop_with_device_reference_equals_sampled_reference():
    """ClosedLoop fed by DeviceReference (nothing but the state crosses the boundary) against the same loop fed by the
    host-sampled trajectory: references agree to 1e-12, so the closed loops stay together"""
    from mpc_quad_ros_b200 import trajectory as T
    from mpc_quad_ros_b200.execute_trajectory import ClosedLoop
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    B, N, M, steps = 24, 20, 20, 10
    dt = 1.0 / N
    K = steps + N + 3
    traj = T.random_smooth_trajectories(B, K, dt, seed=9)
    par = T.random_smooth_params(B, K, dt, seed=9)
    loops = []
    for src in (torch.as_tensor(traj), T.DeviceReference(T.KIND_SINUSOIDS, par, K, dt)):
        quad = Quadrotor3D(drag=True, batch=B).set_hummingbird_params()
        gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [M] * 3, theta=[3.0, 0.1, 0.01], batch=B)
        opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=gpe)
        loops.append(ClosedLoop(quad, opt, src, torch.as_tensor(traj[:, 0, :].copy())))
        loops[-1].run(steps)
    torch.cuda.synchronize()
    assert x_rel(loops[1].x.cpu().numpy(), loops[0].x.cpu().numpy()) < 1e-8
    assert u_rel(loops[1].u0.cpu().numpy(), loops[0].u0.cpu().numpy()) < 1e-8


def test_set_reference_state_constant_reference():
    """quad_optimizer.set_reference_state (quad_opt.py:271-292): constant target over the horizon, default hover inputs
    0.16 and default target [0,0,0,1,0,...]; the solve against it equals the oracle's"""
    Quadrotor3D, quad_optimizer, _ = _pkg()
    N, dt = 10, 0.1
    quadp = orc.quad_hummingbird()
    opt = quad_optimizer(Quadrotor3D(drag=True).set_hummingbird_params(), t_horizon=1.0, n_nodes=N)
    yref, yref_N = opt.set_reference_state()
    assert yref.shape == (N, 17) and np.array_equal(yref[:, :13], np.tile([0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0], (N, 1)))
    assert np.all(yref[:, 13:] == 0.16) and np.array_equal(yref_N, yref[-1, :13])
    x_target = np.array([1.0, -2.0, 3.0, 1.0, 0, 0, 0, 0, 0, 0, 0, 0, 0])
    u_target = np.array([0.2, 0.25, 0.3, 0.35])
    yref, yref_N = opt.set_reference_state(x_target, u_target)
    assert np.array_equal(yref, np.tile(np.concatenate([x_target, u_target]), (N, 1))) and np.array_equal(yref_N, x_target)
    x0 = np.array([0.5, -1.5, 2.5, 1.0, 0, 0, 0, 0.2, 0, -0.1, 0, 0, 0])
    x_opt, w_opt, _, cost = opt.run_optimization(x0)
    xit, uit = np.zeros((N + 1, 13)), np.zeros((N, 4))
    r = orc.rti_step(quadp, dt, N, x0, np.ascontiguousarray(yref), x_target.copy(), xit, uit)
    assert r["status"] == 0
    assert u_rel(w_opt, uit) < TOL_U64 and x_rel(x_opt, xit) < TOL_X64
    assert abs(cost - r["cost"]) < 1e-7 * max(1.0, abs(r["cost"]))


def test_cold_handle_runs_no_warm_rounds():
    """warm_start_rounds < 0 (ADVICE r1): every OCP of every solve takes the cold IPM, in the screening + dense mapping too
    (the dense kernel used to continue up to 8 warm rounds from the active set of its previous solve)"""
    B, N, M = 40, 20, 20
    dt = 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp(M)
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=4, amp_choices=(8.0, 2.0))
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    for variant in (1, 2):
        gpe = GPEnsemble.fromrange([(gp.X[d, 0], gp.X[d, -1]) for d in range(3)], [gp.M] * 3, theta=list(gp.theta[0]), batch=B)
        opt = quad_optimizer(Quadrotor3D(drag=True, batch=B).set_hummingbird_params(), t_horizon=1.0, n_nodes=N, gpe=gpe,
                             warm_start_rounds=-1, solver_variant=variant)
        opt.set_iterate(torch.as_tensor(sc["xit"]), torch.as_tensor(sc["uit"]))
        from mpc_quad_ros_b200 import _capi
        yref = torch.as_tensor(sc["yref"], device=opt.device).contiguous()
        yref_e = torch.as_tensor(sc["yref_e"], device=opt.device).contiguous()
        _capi.check(_capi.lib().qmpc_set_yref(opt._h, _capi.ptr(yref), _capi.ptr(yref_e), _capi.stream_ptr()))
        opt.set_rgp_params(torch.as_tensor(sc["mu"]))
        x0 = torch.as_tensor(sc["x0"], device=opt.device)
        for rep in range(3):        # the second and third solve have a remembered active set available: it must be ignored
            x_opt, w_opt, _, cost = opt.run_optimization(x0)
            st, it = opt.solver_status()
            assert (st == 0).all() and (it > 0).all(), (variant, rep, it.min().item())
        xo, uo, co, ito = oracle_solve_batch(sc, quad, dt, N, gp)
        # first solve of a fresh handle with the same data = the oracle's single RTI step
        opt.set_iterate(torch.as_tensor(sc["xit"]), torch.as_tensor(sc["uit"]))
        x_opt, w_opt, _, cost = opt.run_optimization(x0)
        assert u_rel(w_opt.cpu().numpy(), uo) < TOL_U64 and x_rel(x_opt.cpu().numpy(), xo) < TOL_X64


def test_fused_step_uses_rgp_means_only_after_first_regress():
    """reference: the solver parameters are zeros until the first regress pushes the means (quad_opt.py:101,402-404),
    also when the ensemble was built with non-zero means (frombasisvectors).  The fused qmpc_step and the method-by-method
    path agree on the very first solve (ADVICE r1)."""
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    B, N, M = 6, 10, 10
    dt = 1.0 / N
    quadp = orc.quad_hummingbird()
    gp = make_gp(M)
    sc = random_ocp_batch(B, N, dt, quadp, gp, seed=12, amp_choices=(2.0,))
    X = [gp.X[d] for d in range(3)]
    y = [0.4 * np.sin(0.3 * X[d]) for d in range(3)]                     # non-zero prior means
    Cs = [orc.rgp_prior(gp.X[d], gp.theta[d])[0] for d in range(3)]
    u_first = []
    for fused in (True, False):
        gpe = GPEnsemble.frombasisvectors(X, y, Cs, [list(gp.theta[d]) for d in range(3)], batch=B)
        opt = quad_optimizer(Quadrotor3D(drag=True, batch=B).set_hummingbird_params(), t_horizon=1.0, n_nodes=N, gpe=gpe)
        opt.set_iterate(torch.as_tensor(sc["xit"]), torch.as_tensor(sc["uit"]))
        x_ref = torch.as_tensor(sc["yref"][:, :, :13].copy(), device=opt.device)
        x0 = torch.as_tensor(sc["x0"], device=opt.device)
        if fused:
            xpp = torch.zeros((B, 13), dtype=torch.float64, device=opt.device)
            u0 = torch.empty((B, 4), dtype=torch.float64, device=opt.device)
            opt.step(x0, x_ref, xpp, True, u0)
            u_first.append(u0.cpu().numpy())
        else:
            opt.set_reference_trajectory(x_ref)
            _, w_opt, _, _ = opt.run_optimization(x0)
            u_first.append(w_opt[:, 0].cpu().numpy())
    # oracle: nominal model (alpha = 0) on the first solve
    xo, uo, _, _ = oracle_solve_batch(dict(sc, alpha=np.zeros_like(sc["alpha"])), quadp, dt, N, gp)
    assert np.abs(u_first[0] - u_first[1]).max() < 1e-9
    assert u_rel(u_first[0], uo[:, 0]) < TOL_U64


def _closed_loop_with_injection(workload, B, steps, seed, v_peak=20.0, M=20, N=20):
    """SURVEY §8d contract: B DISTINCT vehicles x `steps` closed-loop control steps.  Every step the GPU solve and the
    oracle start from the IDENTICAL (x0, reference, alpha, SQP iterate): after the comparison the oracle's iterate is
    injected into the GPU solver (qmpc_set_iterate), and the plant/RGP advance with the GPU's controls on both sides."""
    from mpc_quad_ros_b200 import trajectory as T
    from mpc_quad_ros_b200.utils import utils
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    dt = 1.0 / N
    K = steps + N + 2
    if workload == "lemniscate":
        traj = T.lemniscate_trajectories(B, K, dt, v_peak=v_peak, seed=seed, ramp=1.0)      # at full speed after 20 steps
    else:
        traj = T.random_smooth_trajectories(B, K, dt, seed=seed)
    quadp, gp = orc.quad_hummingbird(), make_gp(M)
    quad = Quadrotor3D(drag=True, batch=B).set_hummingbird_params()
    gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [M] * 3, theta=[3.0, 0.1, 0.01], batch=B)
    opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=gpe)
    dev = opt.device
    x = torch.as_tensor(traj[:, 0, :].copy(), device=dev)
    xpp = torch.zeros((B, 13), dtype=torch.float64, device=dev)
    u0 = torch.empty((B, 4), dtype=torch.float64, device=dev)
    traj_d = torch.as_tensor(traj, device=dev)
    xo, uo = np.zeros((B, N + 1, 13)), np.zeros((B, N, 4))          # the oracle's persistent iterate (zero start, like acados)
    mu_o = np.zeros((B, 3, M)); C_o = np.ascontiguousarray(np.broadcast_to(np.stack([orc.rgp_prior(gp.X[d], gp.theta[d])[0] for d in range(3)]), (B, 3, M, M)))
    worst_u = worst_x = worst_mu = worst_C = 0.0
    n_sat = n_tot = n_ipm = n_gpu_bad = 0
    plant = quad.plant_vector(); qv = quad.quad_vector()
    import ctypes as C
    from mpc_quad_ros_b200 import _capi
    for i in range(steps):
        chunk = utils.get_reference_chunk(traj_d, i, N)                       # [B,N,13] on the device
        x_now = x.clone()
        alpha = gpe.alpha_tensor().cpu().numpy() if i > 0 else np.zeros((B, 3, M))   # pushed after the first regress
        xit_before, uit_before = xo.copy(), uo.copy()
        act_before = opt.get_active_set().cpu().numpy()
        opt.step(x_now, chunk, xpp, first_step=(i == 0), u0_out=u0)
        xg, ug = (t.cpu().numpy() for t in opt.get_iterate())
        st, it = opt.solver_status()
        gpu_ok = (st == 0).cpu().numpy()
        n_gpu_bad += int((~gpu_ok).sum())
        assert gpu_ok.mean() > 0.99, (i, torch.bincount(st).tolist())       # a vehicle that tumbles may break down (status 2, contained)
        # oracle: the same step from the same iterate
        ch = chunk.cpu().numpy()
        yref = np.concatenate([ch, np.full((B, N, 4), 0.16)], axis=2)
        r = orc.rti_step_batch(quadp, dt, N, x_now.cpu().numpy(), yref, np.ascontiguousarray(ch[:, -1, :]), xo, uo, gp=gp, alpha=alpha)
        ok = (r["status"] == 0) & gpu_ok                                        # the oracle's own exactness flag (active set verified)
        assert ok.mean() > 0.97, (i, np.bincount(r["status"]))
        eu = np.abs(ug - uo).max(axis=(1, 2)); eu[~ok] = 0
        if eu.max() > worst_u and eu.max() > 1e-7 and os.environ.get("QMPC_DUMP_WORST"):
            b = int(eu.argmax())
            np.savez(os.environ["QMPC_DUMP_WORST"], step=i, b=b, x0=x_now[b].cpu().numpy(), chunk=ch[b], alpha=alpha[b], xit=xit_before[b], uit=uit_before[b],
                     act=act_before[b], u_gpu=ug[b], u_orc=uo[b], it=int(it[b]), rd=int(opt.solver_rounds()[b]), st_orc=int(r["status"][b]), it_orc=int(r["iters"][b]))
        worst_u = max(worst_u, u_rel(ug[ok], uo[ok])); worst_x = max(worst_x, x_rel(xg[ok], xo[ok]))
        n_sat += int(((uo[ok][:, 0] < 1e-9) | (uo[ok][:, 0] > 1 - 1e-9)).sum()); n_tot += int(ok.sum()) * 4
        n_ipm += int((it > 0).sum().item())
        # RGP: the oracle applies the same residual to its own state
        mu_g = gpe.mu_tensor().cpu().numpy()
        xp_prev = x_now.cpu().numpy() if i == 0 else xpp_prev_np
        for b in range(B):
            vb, ad = orc.compute_a_drag(x_now[b].cpu().numpy(), xp_prev[b], dt)
            for d in range(3):
                orc.rgp_regress(gp.X[d], gp.theta[d], gp.Kx_inv[d], mu_o[b, d], C_o[b, d], vb[d], ad[d])
        worst_mu = max(worst_mu, rel_err(mu_g, mu_o)); 
        if i % 10 == 9 or i == steps - 1:
            worst_C = max(worst_C, rel_err(gpe.C_tensor().cpu().numpy(), C_o))
        xpp_prev_np = xpp.cpu().numpy().copy()
        # injection: both sides continue from the oracle's iterate (vehicles the oracle gave up on keep the GPU's)
        xo[~ok], uo[~ok] = xg[~ok], ug[~ok]
        opt.set_iterate(torch.as_tensor(xo), torch.as_tensor(uo))
        gpe.set_state(torch.as_tensor(mu_o), None)           # keep the RGP means identical too (C compared, not injected)
        opt.set_rgp_params(torch.as_tensor(mu_o))
        _capi.check(_capi.lib().qmpc_plant_period(qv.ctypes.data_as(C.c_void_p), plant.ctypes.data_as(C.c_void_p), B, _capi.ptr(x),
                                                  _capi.ptr(u0), C.c_double(5e-3), 11, _capi.stream_ptr()))
    return dict(u=worst_u, x=worst_x, mu=worst_mu, C=worst_C, sat=n_sat / max(n_tot, 1), ipm_frac=n_ipm / (B * steps), gpu_bad=n_gpu_bad)


@pytest.mark.parametrize("workload,seed", [("random_smooth", 1234), ("lemniscate", 4321)])
def test_contract_size_parity_256_vehicles_50_steps_with_injection(workload, seed):
    """BASELINE configs[1] and configs[4] at the sample size SURVEY §8d asks for: 256 distinct vehicles x 50 closed-loop
    steps, per-step parity from identical (x0, reference, alpha, iterate); the lemniscate runs at v_peak 20 m/s with the
    thrust limits active.  fp64 tolerances: controls / predicted states 1e-6 rel, RGP 1e-9 rel."""
    r = _closed_loop_with_injection(workload, 256, 50, seed)
    print(f"{workload}: u_rel {r['u']:.2e} x_rel {r['x']:.2e} mu {r['mu']:.2e} C {r['C']:.2e}; saturated first inputs {100 * r['sat']:.1f} %, "
          f"solves through the IPM {100 * r['ipm_frac']:.1f} %, solves with status != 0: {r['gpu_bad']} of {256 * 50}")
    assert r["gpu_bad"] <= 5
    assert r["u"] < TOL_U64 and r["x"] < TOL_X64
    assert r["mu"] < TOL_RGP and r["C"] < TOL_RGP
    assert r["sat"] > (0.05 if workload == "lemniscate" else 0.01)          # the thrust limits are exercised


def test_free_running_4096_vehicles_100_steps_statistics_vs_oracle():
    """BASELINE configs[1] at full size, free-running (no injection, SURVEY §7 hard part 8): 4096 vehicles x 100 closed-loop
    steps on the GPU against the oracle's closed loop of the same vehicles.  RTI closed loops amplify differences on a few
    aggressive flights, so the comparison is statistical: the bulk of the vehicles must still agree tightly after 100
    steps, and the swarm-level statistics (tracking error, saturation, RGP means) must coincide."""
    from mpc_quad_ros_b200.execute_trajectory import ClosedLoop
    from mpc_quad_ros_b200.trajectory import random_smooth_trajectories
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    B, N, M, steps = 4096, 20, 20, 100
    dt = 1.0 / N
    traj = random_smooth_trajectories(B, steps + N + 2, dt, seed=1234)
    x0 = traj[:, 0, :].copy()
    quad = Quadrotor3D(drag=True, batch=B).set_hummingbird_params()
    gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [M] * 3, theta=[3.0, 0.1, 0.01], batch=B)
    opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=gpe)
    loop = ClosedLoop(quad, opt, torch.as_tensor(traj), torch.as_tensor(x0))
    xs, us = loop.run(steps, record=True)
    xs, us = xs.cpu().numpy(), us.cpu().numpy()
    ref = orc.ClosedLoop(orc.quad_hummingbird(), dt, N, traj, x0, gp=make_gp(M), reset_on_fail=True)
    r = ref.run(steps)
    # per-vehicle agreement at the last step
    e_x = np.abs(xs[-1] - r["x"][-1]).max(axis=1)
    e_u = np.abs(us - r["u0"]).max(axis=(0, 2))
    e_x[~np.isfinite(e_x)] = np.inf; e_u[~np.isfinite(e_u)] = np.inf      # a vehicle that crashed and blew up counts as a disagreement
    q = np.quantile(e_x, [0.5, 0.9, 0.99]); qu = np.quantile(e_u, [0.5, 0.9, 0.99])
    print(f"free-running 4096 x 100: |x-x_orc| at step 100 p50 {q[0]:.1e} p90 {q[1]:.1e} p99 {q[2]:.1e}; max_t |u0-u0_orc| p50 {qu[0]:.1e} p90 {qu[1]:.1e} p99 {qu[2]:.1e}")
    assert q[0] < 1e-8 and q[1] < 1e-6
    assert qu[0] < 1e-8 and qu[1] < 1e-6
    # swarm-level statistics
    track_g = np.linalg.norm(xs[:, :, :3] - traj[:, :steps, :3].transpose(1, 0, 2), axis=2)
    track_o = np.linalg.norm(r["x"][:, :, :3] - traj[:, :steps, :3].transpose(1, 0, 2), axis=2)
    # (the few per cent of flights that amplify 1e-10 differences move the median tracking error in the 5th digit)
    assert abs(np.nanmedian(track_g) - np.nanmedian(track_o)) < 1e-3 * np.nanmedian(track_o)
    sat_g = ((us < 1e-9) | (us > 1 - 1e-9)).mean(); sat_o = ((r["u0"] < 1e-9) | (r["u0"] > 1 - 1e-9)).mean()
    assert abs(sat_g - sat_o) < 2e-3, (sat_g, sat_o)
    mu_g = gpe.mu_tensor().cpu().numpy()
    good = e_x < 1e-6
    assert good.mean() > 0.9
    assert rel_err(mu_g[good], ref.mu[good]) < 1e-4        # 100 steps of accumulated 1e-6-level state differences


def test_step_with_odometry_dt_matches_method_by_method_path():
    """ROS-node variant of the loop (mpc_controller_node.py:278-315): reference cut with skip = control_freq_factor, the
    nominal prediction and the drag residual over ODOMETRY_DT instead of the OCP's dt.  The fused qmpc_step_dt equals the
    method-by-method sequence of the reference API."""
    from mpc_quad_ros_b200.utils import utils
    from mpc_quad_ros_b200.trajectory import random_smooth_trajectories
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    B, N, M = 12, 10, 10
    odo_dt, skip = 0.02, 5
    traj = random_smooth_trajectories(B, 200, 0.02, seed=3)                    # sampled at the odometry rate
    x_now = torch.as_tensor(traj[:, 3, :].copy()).cuda()
    x_now[:, :3] += 0.05
    x_prev_pred = torch.as_tensor(traj[:, 3, :].copy()).cuda()
    x_prev_pred[:, 7:10] += 0.3                                                # a non-zero drag residual
    outs = []
    for fused in (True, False):
        gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [M] * 3, theta=[3.0, 0.1, 0.01], batch=B)
        opt = quad_optimizer(Quadrotor3D(drag=True, batch=B).set_hummingbird_params(), t_horizon=1.0, n_nodes=N, gpe=gpe)
        nominal = quad_optimizer(Quadrotor3D(drag=True, batch=B).set_hummingbird_params(), t_horizon=1.0, n_nodes=N)
        x_ref = utils.get_reference_chunk(torch.as_tensor(traj).cuda(), 3, N, skip)
        xpp = x_prev_pred.clone()
        if fused:
            u0 = torch.empty((B, 4), dtype=torch.float64, device="cuda")
            opt.step(x_now, x_ref, xpp, False, u0, odometry_dt=odo_dt)
            x_pred = xpp
        else:
            opt.set_reference_trajectory(x_ref)
            _, w_opt, _, _ = opt.run_optimization(x_now)
            u0 = w_opt[:, 0].contiguous()
            x_pred = nominal.discrete_dynamics(x_now, u0, odo_dt)
            v_body, a_drag = utils.compute_a_drag(x_now, xpp, odo_dt)
            opt.regress_and_update_RGP_model(v_body, a_drag)
        outs.append((u0.cpu().numpy(), x_pred.cpu().numpy(), gpe.mu_tensor().cpu().numpy()))
    assert np.abs(outs[0][0] - outs[1][0]).max() < 1e-12
    assert np.abs(outs[0][1] - outs[1][1]).max() < 1e-12
    assert rel_err(outs[0][2], outs[1][2]) < 1e-12 and np.abs(outs[1][2]).max() > 0


def _nccl_shared_swarm_worker(rank, world, port, Bt, M, steps, out_path):
    import os
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{rank}"))
    from mpc_quad_ros_b200.execute_trajectory import ClosedLoop
    from mpc_quad_ros_b200.swarm import SharedSwarmRGP, shard_range
    from mpc_quad_ros_b200.trajectory import random_smooth_trajectories
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    N = 10
    dev = torch.device(f"cuda:{rank}")
    traj = random_smooth_trajectories(Bt, steps + N + 2, 1.0 / N, seed=50)
    first, count = shard_range(Bt, rank, world)
    quad = Quadrotor3D(drag=True, batch=count, device=dev).set_hummingbird_params()
    gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [M] * 3, theta=[3.0, 0.1, 0.01], batch=1, device=dev)
    opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=gpe)
    loop = ClosedLoop(quad, opt, torch.as_tensor(traj[first:first + count]), torch.as_tensor(traj[first:first + count, 0, :].copy()),
                      shared_swarm=SharedSwarmRGP(gpe, opt))
    xs, us = loop.run(steps, record=True)
    torch.cuda.synchronize()
    mu, Cm = gpe.mu_tensor()[0], gpe.C_tensor()[0]
    gathered = [torch.empty_like(mu) for _ in range(world)]
    dist.all_gather(gathered, mu)
    same = all(torch.equal(g, gathered[0]) for g in gathered)
    np.savez(out_path % rank, mu=mu.cpu().numpy(), C=Cm.cpu().numpy(), xs=xs.cpu().numpy(), us=us.cpu().numpy(), same=same, first=first, count=count)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_shared_swarm_two_ranks_nccl_vs_sequential_oracle(tmp_path):
    """BASELINE configs[2] over NCCL: two ranks, each with half of the vehicles, ONE shared RGP updated every control step
    by the overlapped accumulate -> all-reduce -> apply (SharedSwarmRGP.begin/end inside ClosedLoop).  The model is
    bit-identical on both ranks and equals the oracle's sequential single-sample regress over all vehicles of both ranks
    (order-free), fed with the residuals of the recorded states; the controls equal a single-rank run over all vehicles."""
    import torch.multiprocessing as mp
    Bt, M, steps, N = 48, 20, 5, 10
    out = str(tmp_path / "rank%d.npz")
    mp.spawn(_nccl_shared_swarm_worker, args=(2, 29611, Bt, M, steps, out), nprocs=2, join=True)
    r0, r1 = np.load(out % 0), np.load(out % 1)
    assert bool(r0["same"]) and bool(r1["same"])
    assert np.array_equal(r0["mu"], r1["mu"]) and np.array_equal(r0["C"], r1["C"])
    # oracle: sequential regress of every vehicle's residual, step by step
    gp = make_gp(M)
    dt = 1.0 / N
    xs = np.concatenate([r0["xs"], r1["xs"]], axis=1)                  # [steps, Bt, 13]
    us = np.concatenate([r0["us"], r1["us"]], axis=1)
    mu = np.zeros((3, M)); Cm = np.stack([orc.rgp_prior(gp.X[d], gp.theta[d])[0] for d in range(3)])
    quadp = orc.quad_hummingbird()
    for s in range(steps):
        for b in range(Bt):
            xprev = xs[s, b] if s == 0 else orc.rk4(quadp, xs[s - 1, b], us[s - 1, b], dt, None, None)
            vb, ad = orc.compute_a_drag(xs[s, b], xprev, dt)
            for d in range(3):
                orc.rgp_regress(gp.X[d], gp.theta[d], gp.Kx_inv[d], mu[d], Cm[d], vb[d], ad[d])
    assert rel_err(r0["mu"], mu) < 1e-8 and rel_err(r0["C"], Cm) < 1e-8
    # single rank over all vehicles: same controls (the shared model is the same to rounding of the summation order)
    from mpc_quad_ros_b200.execute_trajectory import ClosedLoop
    from mpc_quad_ros_b200.swarm import SharedSwarmRGP
    from mpc_quad_ros_b200.trajectory import random_smooth_trajectories
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    traj = random_smooth_trajectories(Bt, steps + N + 2, dt, seed=50)
    quad = Quadrotor3D(drag=True, batch=Bt).set_hummingbird_params()
    gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [M] * 3, theta=[3.0, 0.1, 0.01], batch=1)
    opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=gpe)
    loop = ClosedLoop(quad, opt, torch.as_tensor(traj), torch.as_tensor(traj[:, 0, :].copy()), shared_swarm=SharedSwarmRGP(gpe, opt))
    xs1, us1 = loop.run(steps, record=True)
    assert u_rel(us1.cpu().numpy(), us) < 1e-7 and x_rel(xs1.cpu().numpy(), xs) < 1e-7


def test_reference_semantics_without_reset_on_fail():
    """reset_on_fail = -1 restores the reference's behaviour (quad_opt.py:333 ignores the solver status): a vehicle whose
    solve broke down keeps whatever iterate it had, it is NOT re-initialised on the reference, and no fail streak is kept.
    The library default (reset on) is the documented deviation, tested in test_failed_solve_reinitialises_iterate_on_reference."""
    Quadrotor3D, quad_optimizer, GPEnsemble = _pkg()
    from mpc_quad_ros_b200 import _capi
    B, N = 6, 20
    dt = 1.0 / N
    sc = random_ocp_batch(B, N, dt, orc.quad_hummingbird(), None, seed=11, amp_choices=(1.0,))
    opt = quad_optimizer(Quadrotor3D(drag=True, batch=B).set_hummingbird_params(), t_horizon=1.0, n_nodes=N, reset_on_fail=-1)
    xit, uit = sc["xit"].copy(), sc["uit"].copy()
    xit[2, 5, 2] = np.nan
    opt.set_iterate(torch.as_tensor(xit), torch.as_tensor(uit))
    yref = torch.as_tensor(sc["yref"], device=opt.device).contiguous(); yref_e = torch.as_tensor(sc["yref_e"], device=opt.device).contiguous()
    _capi.check(_capi.lib().qmpc_set_yref(opt._h, _capi.ptr(yref), _capi.ptr(yref_e), _capi.stream_ptr()))
    x0 = torch.as_tensor(sc["x0"], device=opt.device)
    for rep in range(2):
        opt.run_optimization(x0)
        st, _ = opt.solver_status()
        assert st.cpu().numpy().tolist() == [0, 0, 2, 0, 0, 0]            # stays broken: nothing resets it
        x1, u1 = (t.cpu().numpy() for t in opt.get_iterate())
        assert np.isnan(x1[2, 5, 2])
        assert (opt.fail_streak().cpu().numpy() == 0).all()


@pytest.mark.parametrize("M", [64, 33, 100, 2])
def test_rgp_regress_kernel_dispatch_sizes(M):
    """qrgp_regress picks its kernel by the basis size: the TMA-staged one with 8 / 2 / 1 warps per CTA for even M <= 64
    (M = 20 / 50 are covered by the fixtures above, 64 is the one-warp-per-CTA case, 2 the smallest), the streaming one
    for odd or larger M; every branch against the C oracle's RGP.regress (itself pinned by the reference's numpy code)"""
    _, _, GPEnsemble = _pkg()
    B, T = 7, 12
    rng = np.random.default_rng(M)
    theta = [3.0, 0.1, 0.01]
    gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [M] * 3, theta=theta, batch=B)
    X = np.tile(np.linspace(-10, 10, M), (3, 1))
    pri = [orc.rgp_prior(X[d], np.array(theta)) for d in range(3)]
    mu = np.zeros((B, 3, M)); Cm = np.stack([np.stack([pri[d][0] for d in range(3)])] * B)
    for t in range(T):
        xt, yt = rng.uniform(-9, 9, (B, 3)), rng.standard_normal((B, 3))
        mg, Cg = gpe.regress(torch.as_tensor(xt), torch.as_tensor(yt))
        for b in range(B):
            for d in range(3):
                orc.rgp_regress(X[d], np.array(theta), pri[d][1], mu[b, d], Cm[b, d], xt[b, d], yt[b, d])     # in place
    assert rel_err(mg.cpu().numpy(), mu) < TOL_RGP and rel_err(Cg.cpu().numpy(), Cm) < TOL_RGP
    al = gpe.alpha_tensor().cpu().numpy()
    assert rel_err(al, np.einsum("dij,bdj->bdi", np.stack([p[1] for p in pri]), mu)) < 1e-8
