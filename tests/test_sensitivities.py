"""Sensitivities of the RTI step w.r.t. x0 (qmpc_eval_sens_x0, quad_optimizer.eval_sens; acados eval_param_sens "ex").

RTI linearises at the iterate, never at x0, so x0 -> (x, u) is the box-QP's solution map: piecewise affine, and on the
active set the solve ended on its Jacobian is the closed loop of the LQR with the active inputs pinned.  Three routes are
compared: central differences of the oracle's RTI step, 13 independent LQR solves with the oracle's routines
(tests/sens/rti_sens.c), and the kernel (one pinned factorisation + a 13-column forward sweep), emulated on the CPU
(tests/sens/emu_sens.cpp) and on the GPU."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as orc
from helpers import make_gp, random_ocp_batch
from emu import emu
from sens import sens_ref

TOL64 = 1e-9          # kernel vs oracle, fp64: two exact routes to the same linear map


def rel(a, ref):
    """max|a - ref| / max(1, max|ref|) (controls and states are O(1))"""
    return float(np.abs(a - ref).max() / max(1.0, np.abs(ref).max()))


def act_of(u, lb=0.0, ub=1.0):
    """active set implied by an exact solution: an input is pinned when it equals a bound"""
    u = u.reshape(u.shape[0], -1)
    return np.where(u == lb, 1, np.where(u == ub, 2, 0)).astype(np.uint8)


def oracle_solve(sc, b, quad, dt, N, gp, x0=None):
    x, u = sc["xit"][b].copy(), sc["uit"][b].copy()
    r = orc.rti_step(quad, dt, N, sc["x0"][b] if x0 is None else x0, sc["yref"][b], sc["yref_e"][b], x, u, gp=gp,
                     alpha=None if gp is None else sc["alpha"][b])
    assert r["status"] == 0, r
    return x, u


def oracle_sens(sc, b, quad, dt, N, gp, act, n_stages=None, states=True):
    return sens_ref.rti_sens(quad, dt, N, sc["xit"][b], sc["uit"][b], act, n_stages=n_stages, states=states, gp=gp,
                        alpha=None if gp is None else sc["alpha"][b])


# ------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("N,use_gp", [(20, True), (20, False), (7, True), (7, False)])
def test_oracle_sens_matches_central_differences(N, use_gp):
    B, dt, eps = 4, 1.0 / N, 1e-4
    quad = orc.quad_hummingbird()
    gp = make_gp() if use_gp else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=100 + N)
    kept = 0
    for b in range(B):
        x, u = oracle_solve(sc, b, quad, dt, N, gp)
        act = act_of(u[None])[0]
        sx, su = oracle_sens(sc, b, quad, dt, N, gp, act)
        assert np.abs(sx[0] - np.eye(13)).max() == 0.0
        assert (su.reshape(4 * N, 13)[act != 0] == 0).all()
        dx, du, same = np.empty_like(sx), np.empty_like(su), True
        for i in range(13):
            xs, us = [], []
            for s in (1, -1):
                x0 = sc["x0"][b].copy()
                x0[i] += s * eps
                xp, up = oracle_solve(sc, b, quad, dt, N, gp, x0=x0)
                same = same and np.array_equal(act_of(up[None])[0], act)
                xs.append(xp); us.append(up)
            dx[:, :, i] = (xs[0] - xs[1]) / (2 * eps)
            du[:, :, i] = (us[0] - us[1]).reshape(N, 4) / (2 * eps)
        if not same:
            continue
        kept += 1
        assert rel(sx, dx) < 1e-7 and rel(su, du) < 1e-7, (b, rel(sx, dx), rel(su, du))
    assert kept >= B // 2, kept
    print(f"N={N} gp={use_gp}: {kept}/{B} vehicles keep their active set under the perturbation")


def _emulated_case(N, use_gp, variant, B=3, seed=None):
    dt = 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp() if use_gp else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=N + 40 if seed is None else seed)
    cfg, keep = emu.make_config(B, N, 1.0, quad, orc.W_DIAG, orc.WE_DIAG, None if gp is None else gp.X,
                                None if gp is None else gp.theta)
    xe, ue = sc["xit"].copy(), sc["uit"].copy()
    r = emu.solve(cfg, sc["x0"], sc["yref"], sc["yref_e"], sc["alpha"], xe, ue, variant=variant)
    return sc, quad, dt, gp, cfg, keep, r


@pytest.mark.parametrize("variant", [1, 2], ids=["warp_per_ocp", "screen_plus_dense"])
@pytest.mark.parametrize("N,use_gp", [(20, True), (20, False), (7, True), (7, False), (1, True), (1, False)])
def test_emulated_sens_kernel_matches_oracle(N, use_gp, variant):
    sc, quad, dt, gp, cfg, keep, r = _emulated_case(N, use_gp, variant)
    B = cfg.batch
    assert (r["status"] == 0).all()
    sx, su = sens_ref.emu_sens(cfg, r, N)
    sx1, su1 = sens_ref.emu_sens(cfg, r, 1)
    _, su1n = sens_ref.emu_sens(cfg, r, 1, states=False)
    for b in range(B):
        _, uo = oracle_solve(sc, b, quad, dt, N, gp)
        act = act_of(uo[None])[0]
        assert np.array_equal(r["act"][b], act), b
        ox, ou = oracle_sens(sc, b, quad, dt, N, gp, act)
        assert rel(sx[b], ox) < TOL64 and rel(su[b], ou) < TOL64, (b, rel(sx[b], ox), rel(su[b], ou))
        assert (su[b].reshape(4 * N, 13)[act != 0] == 0).all()                 # pinned rows exactly 0
    assert np.array_equal(sx1, sx[:, :2]) and np.array_equal(su1, su[:, :1]) and np.array_equal(su1n, su1)
    assert np.array_equal(sx[:, 0], np.broadcast_to(np.eye(13), (B, 13, 13)))


def test_emulated_sens_kernel_without_tile_ring():
    """the A/B build flavour that reads the tiles in place with unpadded rows (QMPC_RING=0, QMPC_WR=16)"""
    N = 20
    dt = 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp()
    sc = random_ocp_batch(3, N, dt, quad, gp, seed=60)
    cfg, keep = emu.make_config(3, N, 1.0, quad, orc.W_DIAG, orc.WE_DIAG, gp.X, gp.theta)
    xe, ue = sc["xit"].copy(), sc["uit"].copy()
    r = emu.solve(cfg, sc["x0"], sc["yref"], sc["yref_e"], sc["alpha"], xe, ue, variant=1, flavour="noring")
    sx, su = sens_ref.emu_sens(cfg, r, N, flavour="noring")
    for b in range(3):
        ox, ou = oracle_sens(sc, b, quad, dt, N, gp, r["act"][b])
        assert rel(sx[b], ox) < TOL64 and rel(su[b], ou) < TOL64


def test_emulated_unknown_active_set_gives_nan():
    N, B = 20, 3
    dt = 1.0 / N
    quad = orc.quad_hummingbird()
    sc = random_ocp_batch(B, N, dt, quad, None, seed=77, amp_choices=(8.0,))
    cfg, keep = emu.make_config(B, N, 1.0, quad, orc.W_DIAG, orc.WE_DIAG, max_iter=1, warm_start_rounds=-1)
    xe, ue = sc["xit"].copy(), sc["uit"].copy()
    r = emu.solve(cfg, sc["x0"], sc["yref"], sc["yref_e"], None, xe, ue, variant=1)
    assert (r["status"] == 1).all() and (r["act"] == 255).all()
    sx, su = sens_ref.emu_sens(cfg, r, N)
    assert np.isnan(sx).all() and np.isnan(su).all()
    # one unknown entry makes one vehicle unknown; its neighbours are unaffected
    cfg2, keep2 = emu.make_config(B, N, 1.0, quad, orc.W_DIAG, orc.WE_DIAG)
    xe, ue = sc["xit"].copy(), sc["uit"].copy()
    r2 = emu.solve(cfg2, sc["x0"], sc["yref"], sc["yref_e"], None, xe, ue, variant=1)
    assert (r2["status"] == 0).all()
    r2["act"][1, 17] = 255
    sx, su = sens_ref.emu_sens(cfg2, r2, N)
    assert np.isnan(sx[1]).all() and np.isnan(su[1]).all()
    assert np.isfinite(sx[[0, 2]]).all() and np.isfinite(su[[0, 2]]).all()


# ------------------------------------------------------------------------------------------------------------- GPU

def _gpu_handle(sc, B, N, gp, precision=64, **policy):
    import torch
    from mpc_quad_ros_b200 import _capi
    from mpc_quad_ros_b200.gp.GPE import GPEnsemble
    from mpc_quad_ros_b200.quad import Quadrotor3D
    from mpc_quad_ros_b200.quad_opt import quad_optimizer
    quad = Quadrotor3D(drag=True, batch=B).set_hummingbird_params()
    gpe = None if gp is None else GPEnsemble.fromrange([(gp.X[d, 0], gp.X[d, -1]) for d in range(3)], [gp.M] * 3,
                                                         theta=list(gp.theta[0]), batch=B)
    opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=gpe, precision=precision, **policy)
    yref = torch.as_tensor(sc["yref"], device=opt.device).contiguous()
    yref_e = torch.as_tensor(sc["yref_e"], device=opt.device).contiguous()
    _capi.check(_capi.lib().qmpc_set_yref(opt._h, _capi.ptr(yref), _capi.ptr(yref_e), _capi.stream_ptr()))
    if gp is not None:
        opt.set_rgp_params(torch.as_tensor(sc["mu"]))
    return opt


def _gpu_solve(opt, xit, uit, x0, act=None):
    import torch
    opt.set_iterate(torch.as_tensor(xit), torch.as_tensor(uit))
    if act is not None:
        opt.set_active_set(act)
    x, u, _, _ = opt.run_optimization(torch.as_tensor(x0, device=opt.device))
    return x, u


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [1, 2], ids=["warp_per_ocp", "screen_plus_dense"])
@pytest.mark.parametrize("N,M,seed", [(20, 20, 140), (10, 0, 110), (50, 20, 170), (21, 20, 21), (1, 0, 1)])
def test_gpu_sens_vs_oracle(N, M, seed, variant):
    if variant == 2 and N > 21:
        pytest.skip("the screening + dense solver serves N <= 21")
    import torch
    B, dt = 48, 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp(M) if M else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=seed)      # the scenarios of test_gpu_parity's fp64 solve test
    opt = _gpu_handle(sc, B, N, gp, solver_variant=variant)
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"])
    sx, su = (t.cpu().numpy() for t in opt.eval_sens(N))
    sx1, su1 = (t.cpu().numpy() for t in opt.eval_sens(1))
    none, su1n = opt.eval_sens(1, states=False)
    act = opt.get_active_set().cpu().numpy()
    st = opt.solver_status()[0].cpu().numpy()
    assert none is None and np.array_equal(su1n.cpu().numpy(), su1)
    assert np.array_equal(sx1, sx[:, :2]) and np.array_equal(su1, su[:, :1])
    assert (st == 0).all()
    worst = 0.0
    for b in range(B):
        _, uo = oracle_solve(sc, b, quad, dt, N, gp)
        assert np.array_equal(act[b], act_of(uo[None])[0]), b
        ox, ou = oracle_sens(sc, b, quad, dt, N, gp, act[b])
        worst = max(worst, rel(sx[b], ox), rel(su[b], ou))
        assert (su[b].reshape(4 * N, 13)[act[b] != 0] == 0).all()
    print(f"N={N} M={M} variant {variant}: worst rel err vs the oracle {worst:.1e}")
    assert worst < TOL64, worst


@pytest.mark.gpu
@pytest.mark.parametrize("variant,tol", [(1, 1e-6), (2, 1e-4)], ids=["warp_per_ocp", "screen_plus_dense"])
def test_gpu_sens_vs_central_differences_of_the_library(variant, tol):
    """no oracle: 26 solves of the library itself from the same iterate and active set at x0 +- eps e_i"""
    import torch
    B, N, M, eps = 48, 20, 20, 1e-3
    dt = 1.0 / N
    gp = make_gp(M)
    sc = random_ocp_batch(B, N, dt, orc.quad_hummingbird(), gp, seed=900)
    opt = _gpu_handle(sc, B, N, gp, solver_variant=variant, reset_on_fail=-1)
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"])
    act0 = opt.get_active_set().clone()                  # injected before every solve below
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"], act=act0)
    sx, su = (t.cpu().numpy() for t in opt.eval_sens())
    acts = [opt.get_active_set().cpu().numpy()]
    dx, du = np.empty_like(sx), np.empty_like(su)
    for i in range(13):
        xs, us = [], []
        for s in (1, -1):
            x0 = sc["x0"].copy()
            x0[:, i] += s * eps
            x, u = _gpu_solve(opt, sc["xit"], sc["uit"], x0, act=act0)
            xs.append(x.cpu().numpy()); us.append(u.cpu().numpy()); acts.append(opt.get_active_set().cpu().numpy())
        dx[..., i] = (xs[0] - xs[1]) / (2 * eps)
        du[..., i] = ((us[0] - us[1]) / (2 * eps)).reshape(B, N, 4)
    keep = np.array([all(np.array_equal(a[b], acts[0][b]) for a in acts) and (acts[0][b] <= 2).all() for b in range(B)])
    print(f"variant {variant}: {keep.sum()}/{B} vehicles keep their active set in all 27 solves")
    assert keep.mean() >= 0.75
    ex, eu = rel(sx[keep], dx[keep]), rel(su[keep], du[keep])
    print(f"variant {variant}: rel err vs central differences: x {ex:.1e}, u {eu:.1e}")
    assert ex < tol and eu < tol


@pytest.mark.gpu
def test_gpu_sens_between_fused_steps_leaves_the_loop_unchanged():
    import torch
    from mpc_quad_ros_b200.execute_trajectory import ClosedLoop
    from mpc_quad_ros_b200.gp.GPE import GPEnsemble
    from mpc_quad_ros_b200.quad import Quadrotor3D
    from mpc_quad_ros_b200.quad_opt import quad_optimizer
    from mpc_quad_ros_b200.trajectory import random_smooth_trajectories
    B, N, M, steps = 256, 20, 20, 30
    traj = random_smooth_trajectories(B, steps + N + 2, 1.0 / N)

    def run(with_sens):
        quad = Quadrotor3D(drag=True, batch=B).set_hummingbird_params()
        gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [M] * 3, theta=[3.0, 0.1, 0.01], batch=B)
        opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=gpe)
        loop = ClosedLoop(quad, opt, torch.as_tensor(traj), torch.as_tensor(traj[:, 0, :].copy()))
        u0s, finite = [], True
        for _ in range(steps):
            loop.step()
            u0s.append(loop.u0.clone())
            if with_sens:
                sx, su = opt.eval_sens(N)
                ok = opt.solver_status()[0] == 0
                finite = finite and bool(torch.isfinite(sx[ok]).all() and torch.isfinite(su[ok]).all())
        x, u = opt.get_iterate()
        return torch.stack(u0s), x, u, gpe.mu_tensor(), gpe.C_tensor(), finite

    a, b = run(False), run(True)
    for ta, tb in zip(a[:5], b[:5]):
        assert torch.equal(ta, tb)
    assert b[5]


@pytest.mark.gpu
def test_gpu_sens_reference_api_batch_one():
    N, M, B = 20, 20, 4
    dt = 1.0 / N
    gp = make_gp(M)
    sc = random_ocp_batch(B, N, dt, orc.quad_hummingbird(), gp, seed=33)
    optb = _gpu_handle(sc, B, N, gp)
    _gpu_solve(optb, sc["xit"], sc["uit"], sc["x0"])
    sxb, sub = optb.eval_sens()
    one = {k: (None if v is None else v[:1]) for k, v in sc.items()}
    opt1 = _gpu_handle(one, 1, N, gp)
    opt1.set_iterate(sc["xit"][0], sc["uit"][0])
    opt1.run_optimization(sc["x0"][0])                  # numpy in: the reference API of one vehicle
    sx, su = opt1.eval_sens()
    assert isinstance(sx, np.ndarray) and sx.shape == (N + 1, 13, 13) and su.shape == (N, 4, 13)
    assert rel(sx, sxb[0].cpu().numpy()) < 1e-12 and rel(su, sub[0].cpu().numpy()) < 1e-12
    none, su5 = opt1.eval_sens(5, states=False)
    assert none is None and su5.shape == (5, 4, 13) and np.array_equal(su5, su[:5])


@pytest.mark.gpu
def test_gpu_sens_argument_errors_launch_nothing():
    import torch
    from mpc_quad_ros_b200 import _capi
    N, B = 10, 4
    sc = random_ocp_batch(B, N, 1.0 / N, orc.quad_hummingbird(), None, seed=3)
    opt = _gpu_handle(sc, B, N, None)
    lib = _capi.lib()
    su = torch.empty((B, N, 4, 13), dtype=torch.float64, device=opt.device)
    l0 = lib.qmpc_launch_count()
    with pytest.raises(_capi.QmpcError, match="no solve"):
        opt.eval_sens()
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"])
    torch.cuda.synchronize()
    l1 = lib.qmpc_launch_count()
    for n in (0, N + 1):
        with pytest.raises(_capi.QmpcError, match="n_stages"):
            opt.eval_sens(n)
    with pytest.raises(_capi.QmpcError, match="sens_u"):
        _capi.check(lib.qmpc_eval_sens_x0(opt._h, N, C.c_void_p(0), C.c_void_p(0), _capi.stream_ptr()))
    with pytest.raises(_capi.QmpcError, match="null handle"):
        _capi.check(lib.qmpc_eval_sens_x0(C.c_void_p(0), N, C.c_void_p(0), _capi.ptr(su), _capi.stream_ptr()))
    assert lib.qmpc_launch_count() == l1 and l1 > l0
    opt.eval_sens()
    assert lib.qmpc_launch_count() == l1 + 1
    # fp32 handles: the fp32 tiles and Riccati recursion measured up to 1.4e-3 off on the GPU (DESIGN section 4)
    opt32 = _gpu_handle(sc, B, N, None, precision=32)
    _gpu_solve(opt32, sc["xit"], sc["uit"], sc["x0"])
    torch.cuda.synchronize()
    l2 = lib.qmpc_launch_count()
    with pytest.raises(_capi.QmpcError, match="fp64"):
        opt32.eval_sens()
    assert lib.qmpc_launch_count() == l2
