"""Adjoint (reverse-mode) sensitivities of the RTI step w.r.t. x0 and the reference (qmpc_eval_adjoint,
quad_optimizer.eval_adjoint / differentiable_step).

K1 reads the reference only in the linear cost term and never reads x0, so (x0, yref, yref_e) -> (x, u) is the box-QP's
solution map: piecewise affine, and on the active set the solve ended on its reverse mode is one pinned LQR with the
cotangents as linear costs.  Routes compared: central differences of the oracle's RTI step, the oracle's LQR with an
explicit costate recursion (tests/sens/rti_adjoint.c), the transpose of the forward sensitivities (rti_sens / eval_sens),
and the kernel (one pinned factorisation, a backward and a forward vector sweep), emulated on the CPU
(tests/sens/emu_adjoint.cpp) and on the GPU."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as orc
from helpers import make_gp, random_ocp_batch
from emu import emu
from sens import adjoint_ref, sens_ref

TOL64 = 1e-9          # kernel vs oracle, fp64: two exact routes to the same linear map
NX, NU = 13, 4


def rel(a, ref):
    """max|a - ref| / max(1, max|ref|)"""
    return float(np.abs(a - ref).max() / max(1.0, np.abs(ref).max()))


def act_of(u, lb=0.0, ub=1.0):
    """active set implied by an exact solution: an input is pinned when it equals a bound"""
    u = u.reshape(u.shape[0], -1)
    return np.where(u == lb, 1, np.where(u == ub, 2, 0)).astype(np.uint8)


def cotangents(rng, B, N):
    return rng.standard_normal((B, N + 1, NX)), rng.standard_normal((B, N, NU))


def oracle_solve(sc, b, quad, dt, N, gp, x0=None, yref=None, yref_e=None):
    x, u = sc["xit"][b].copy(), sc["uit"][b].copy()
    r = orc.rti_step(quad, dt, N, sc["x0"][b] if x0 is None else x0, sc["yref"][b] if yref is None else yref,
                     sc["yref_e"][b] if yref_e is None else yref_e, x, u, gp=gp,
                     alpha=None if gp is None else sc["alpha"][b])
    assert r["status"] == 0, r
    return x, u


def oracle_adjoint(sc, b, quad, dt, N, gp, act, x_bar=None, u_bar=None):
    return adjoint_ref.rti_adjoint(quad, dt, N, sc["xit"][b], sc["uit"][b], act, x_bar=x_bar, u_bar=u_bar, gp=gp,
                                alpha=None if gp is None else sc["alpha"][b])


def transpose_of_sens(sx, su, xb, ub):
    """sum_k sens_x[k]^T x_bar[k] + sens_u[k]^T u_bar[k] (leading dimensions broadcast)"""
    return np.einsum("...kij,...ki->...j", sx, xb) + np.einsum("...kij,...ki->...j", su, ub)


# ------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("N,use_gp", [(20, True), (20, False), (7, True), (7, False)])
def test_oracle_adjoint_matches_central_differences(N, use_gp):
    B, dt, eps = 4, 1.0 / N, 1e-4
    quad = orc.quad_hummingbird()
    gp = make_gp() if use_gp else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=300 + N)
    rng = np.random.default_rng(N)
    xbs, ubs = cotangents(rng, B, N)
    kept = 0
    for b in range(B):
        x, u = oracle_solve(sc, b, quad, dt, N, gp)
        act = act_of(u[None])[0]
        x0b, yb, yeb = oracle_adjoint(sc, b, quad, dt, N, gp, act, xbs[b], ubs[b])
        assert (yb[0, :NX] == 0).all() and (yb[:, NX:].reshape(-1)[act != 0] == 0).all()
        # directions: x0 alone, the stage reference alone, the terminal reference alone, all three at once
        dirs = []
        for part in range(4):
            d0 = rng.standard_normal(NX) if part in (0, 3) else np.zeros(NX)
            dy = rng.standard_normal((N, NX + NU)) if part in (1, 3) else np.zeros((N, NX + NU))
            de = rng.standard_normal(NX) if part in (2, 3) else np.zeros(NX)
            dirs.append((d0, dy, de))
        same, errs = True, []
        for d0, dy, de in dirs:
            vals = []
            for s in (1, -1):
                xp, up = oracle_solve(sc, b, quad, dt, N, gp, x0=sc["x0"][b] + s * eps * d0,
                                      yref=sc["yref"][b] + s * eps * dy, yref_e=sc["yref_e"][b] + s * eps * de)
                same = same and np.array_equal(act_of(up[None])[0], act)
                vals.append(np.vdot(xbs[b], xp) + np.vdot(ubs[b], up))
            fd = (vals[0] - vals[1]) / (2 * eps)
            ad = np.vdot(x0b, d0) + np.vdot(yb, dy) + np.vdot(yeb, de)
            errs.append(abs(fd - ad) / max(1.0, abs(ad)))
        if not same:
            continue
        kept += 1
        assert max(errs) < 1e-7, (b, errs)
    assert kept >= B // 2, kept
    print(f"N={N} gp={use_gp}: {kept}/{B} vehicles keep their active set under the perturbation")


@pytest.mark.parametrize("N,use_gp", [(20, True), (7, False), (1, True)])
def test_oracle_adjoint_x0_is_the_transpose_of_the_forward_sensitivities(N, use_gp):
    B, dt = 4, 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp() if use_gp else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=400 + N)
    xbs, ubs = cotangents(np.random.default_rng(7), B, N)
    for b in range(B):
        _, u = oracle_solve(sc, b, quad, dt, N, gp)
        act = act_of(u[None])[0]
        x0b, _, _ = oracle_adjoint(sc, b, quad, dt, N, gp, act, xbs[b], ubs[b])
        sx, su = sens_ref.rti_sens(quad, dt, N, sc["xit"][b], sc["uit"][b], act, gp=gp,
                                   alpha=None if gp is None else sc["alpha"][b])
        assert rel(x0b, transpose_of_sens(sx, su, xbs[b], ubs[b])) < 1e-12


def _emulated_case(N, use_gp, variant, B=3, seed=None, flavour=""):
    dt = 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp() if use_gp else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=N + 40 if seed is None else seed)
    cfg, keep = emu.make_config(B, N, 1.0, quad, orc.W_DIAG, orc.WE_DIAG, None if gp is None else gp.X,
                                None if gp is None else gp.theta)
    xe, ue = sc["xit"].copy(), sc["uit"].copy()
    r = emu.solve(cfg, sc["x0"], sc["yref"], sc["yref_e"], sc["alpha"], xe, ue, variant=variant, flavour=flavour)
    return sc, quad, dt, gp, cfg, keep, r


@pytest.mark.parametrize("variant", [1, 2], ids=["warp_per_ocp", "screen_plus_dense"])
@pytest.mark.parametrize("N,use_gp", [(20, True), (20, False), (7, True), (7, False), (1, True), (1, False)])
def test_emulated_adjoint_kernel_matches_oracle(N, use_gp, variant):
    sc, quad, dt, gp, cfg, keep, r = _emulated_case(N, use_gp, variant)
    B = cfg.batch
    assert (r["status"] == 0).all()
    xbs, ubs = cotangents(np.random.default_rng(N + variant), B, N)
    x0b, yb, yeb = adjoint_ref.emu_adjoint(cfg, r, xbs, ubs)
    for b in range(B):
        _, uo = oracle_solve(sc, b, quad, dt, N, gp)
        act = act_of(uo[None])[0]
        assert np.array_equal(r["act"][b], act), b
        ox0, oy, oye = oracle_adjoint(sc, b, quad, dt, N, gp, act, xbs[b], ubs[b])
        errs = rel(x0b[b], ox0), rel(yb[b], oy), rel(yeb[b], oye)
        assert max(errs) < TOL64, (b, errs)
        assert (yb[b, :, NX:].reshape(-1)[act != 0] == 0).all()                 # pinned inputs exactly 0
    assert (yb[:, 0, :NX] == 0).all()                                             # x_0 is pinned at x0: exactly 0
    # a NULL cotangent is zero, unrequested outputs change nothing, the map is linear in the cotangents
    x0x, yx, yex = adjoint_ref.emu_adjoint(cfg, r, xbs, None)
    x0u, yu, yeu = adjoint_ref.emu_adjoint(cfg, r, None, ubs)
    assert rel(x0x + x0u, x0b) < 1e-12 and rel(yx + yu, yb) < 1e-12 and rel(yex + yeu, yeb) < 1e-12
    for b in range(B):
        ox0, oy, oye = oracle_adjoint(sc, b, quad, dt, N, gp, r["act"][b], x_bar=xbs[b])
        assert max(rel(x0x[b], ox0), rel(yx[b], oy), rel(yex[b], oye)) < TOL64
    only_x0, none1, none2 = adjoint_ref.emu_adjoint(cfg, r, xbs, ubs, outputs=(True, False, False))
    assert none1 is None and none2 is None and np.array_equal(only_x0, x0b)
    n0, only_y, n2 = adjoint_ref.emu_adjoint(cfg, r, xbs, ubs, outputs=(False, True, False))
    assert np.array_equal(only_y, yb)
    # cotangents on pinned inputs have no effect
    ub2 = ubs.copy().reshape(B, -1)
    ub2[r["act"] != 0] += 5.0
    x0p, yp, yep = adjoint_ref.emu_adjoint(cfg, r, xbs, ub2.reshape(B, N, NU))
    assert np.array_equal(x0p, x0b) and np.array_equal(yp, yb) and np.array_equal(yep, yeb)


def test_emulated_adjoint_kernel_without_tile_ring():
    """the A/B build flavour that reads the tiles in place with unpadded rows (QMPC_RING=0, QMPC_WR=16)"""
    N = 20
    sc, quad, dt, gp, cfg, keep, r = _emulated_case(N, True, 1, seed=60, flavour="noring")
    xbs, ubs = cotangents(np.random.default_rng(60), 3, N)
    x0b, yb, yeb = adjoint_ref.emu_adjoint(cfg, r, xbs, ubs, flavour="noring")
    for b in range(3):
        ox0, oy, oye = oracle_adjoint(sc, b, quad, dt, N, gp, r["act"][b], xbs[b], ubs[b])
        assert max(rel(x0b[b], ox0), rel(yb[b], oy), rel(yeb[b], oye)) < TOL64


def test_emulated_adjoint_unknown_active_set_gives_nan():
    N, B = 20, 3
    dt = 1.0 / N
    quad = orc.quad_hummingbird()
    sc = random_ocp_batch(B, N, dt, quad, None, seed=77, amp_choices=(8.0,))
    xbs, ubs = cotangents(np.random.default_rng(77), B, N)
    cfg, keep = emu.make_config(B, N, 1.0, quad, orc.W_DIAG, orc.WE_DIAG)
    xe, ue = sc["xit"].copy(), sc["uit"].copy()
    r = emu.solve(cfg, sc["x0"], sc["yref"], sc["yref_e"], None, xe, ue, variant=1)
    assert (r["status"] == 0).all()
    ref = adjoint_ref.emu_adjoint(cfg, r, xbs, ubs)
    r["act"][1, 17] = 255               # one unknown entry makes one vehicle unknown; its neighbours are unaffected
    out = adjoint_ref.emu_adjoint(cfg, r, xbs, ubs)
    for o, o_ref in zip(out, ref):
        assert np.isnan(o[1]).all()
        assert np.array_equal(o[[0, 2]], o_ref[[0, 2]])


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
def test_gpu_adjoint_vs_oracle_and_eval_sens(N, M, seed, variant):
    if variant == 2 and N > 21:
        pytest.skip("the screening + dense solver serves N <= 21")
    B, dt = 48, 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp(M) if M else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=seed)      # the scenarios of test_gpu_sens_vs_oracle
    opt = _gpu_handle(sc, B, N, gp, solver_variant=variant)
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"])
    xbs, ubs = cotangents(np.random.default_rng(seed), B, N)
    x0b, yb, yeb = (t.cpu().numpy() for t in opt.eval_adjoint(xbs, ubs))
    sx, su = (t.cpu().numpy() for t in opt.eval_sens(N))
    act = opt.get_active_set().cpu().numpy()
    assert (opt.solver_status()[0].cpu().numpy() == 0).all()
    worst = worst_t = 0.0
    for b in range(B):
        _, uo = oracle_solve(sc, b, quad, dt, N, gp)
        assert np.array_equal(act[b], act_of(uo[None])[0]), b
        ox0, oy, oye = oracle_adjoint(sc, b, quad, dt, N, gp, act[b], xbs[b], ubs[b])
        worst = max(worst, rel(x0b[b], ox0), rel(yb[b], oy), rel(yeb[b], oye))
        worst_t = max(worst_t, rel(x0b[b], transpose_of_sens(sx[b], su[b], xbs[b], ubs[b])))
        assert (yb[b, :, NX:].reshape(-1)[act[b] != 0] == 0).all()
    assert (yb[:, 0, :NX] == 0).all()
    print(f"N={N} M={M} variant {variant}: worst rel err vs the oracle {worst:.1e}, vs eval_sens transposed {worst_t:.1e}")
    assert worst < TOL64 and worst_t < TOL64, (worst, worst_t)


@pytest.mark.gpu
@pytest.mark.parametrize("variant,tol", [(1, 1e-6), (2, 1e-4)], ids=["warp_per_ocp", "screen_plus_dense"])
def test_gpu_adjoint_vs_central_differences_of_the_library(variant, tol):
    """no oracle: solves of the library itself from the same iterate and active set at reference +- eps * direction"""
    import torch
    B, N, M, eps = 48, 20, 20, 1e-3
    dt = 1.0 / N
    gp = make_gp(M)
    sc = random_ocp_batch(B, N, dt, orc.quad_hummingbird(), gp, seed=900)
    opt = _gpu_handle(sc, B, N, gp, solver_variant=variant, reset_on_fail=-1)
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"])
    act0 = opt.get_active_set().clone()                  # injected before every solve below
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"], act=act0)
    rng = np.random.default_rng(901)
    xbs, ubs = cotangents(rng, B, N)
    x0b, yb, yeb = (t.cpu().numpy() for t in opt.eval_adjoint(xbs, ubs))
    acts = [opt.get_active_set().cpu().numpy()]
    from mpc_quad_ros_b200 import _capi
    fds, ads = [], []
    for part in range(3):                                # the stage reference, the terminal reference, x0 with both
        dy = rng.standard_normal((B, N, NX + NU)) if part in (0, 2) else np.zeros((B, N, NX + NU))
        de = rng.standard_normal((B, NX)) if part in (1, 2) else np.zeros((B, NX))
        d0 = rng.standard_normal((B, NX)) if part == 2 else np.zeros((B, NX))
        vals = []
        for s in (1, -1):
            yref = torch.as_tensor(sc["yref"] + s * eps * dy, device=opt.device).contiguous()
            yref_e = torch.as_tensor(sc["yref_e"] + s * eps * de, device=opt.device).contiguous()
            _capi.check(_capi.lib().qmpc_set_yref(opt._h, _capi.ptr(yref), _capi.ptr(yref_e), _capi.stream_ptr()))
            x, u = _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"] + s * eps * d0, act=act0)
            acts.append(opt.get_active_set().cpu().numpy())
            vals.append((xbs * x.cpu().numpy()).sum(axis=(1, 2)) + (ubs * u.cpu().numpy()).sum(axis=(1, 2)))
        fds.append((vals[0] - vals[1]) / (2 * eps))
        ads.append((x0b * d0).sum(1) + (yb * dy).sum(axis=(1, 2)) + (yeb * de).sum(1))
    keep = np.array([all(np.array_equal(a[b], acts[0][b]) for a in acts) and (acts[0][b] <= 2).all() for b in range(B)])
    print(f"variant {variant}: {keep.sum()}/{B} vehicles keep their active set in all 7 solves")
    assert keep.mean() >= 0.75
    fd, ad = np.array(fds)[:, keep], np.array(ads)[:, keep]
    err = float((np.abs(fd - ad) / np.maximum(1.0, np.abs(ad))).max())
    print(f"variant {variant}: rel err vs central differences {err:.1e}")
    assert err < tol


def _stable_vehicles(opt, sc, N, act0, xit, uit, x_ref, u_ref, eps, n_dirs=6):
    """vehicles whose active set survives +-eps in random directions of (x0, x_ref, u_ref) and in each direction's
    coordinate-wise worst case (every coordinate at once, sign of the direction)"""
    import torch
    rng = np.random.default_rng(5)
    x0 = torch.as_tensor(sc["x0"], device=opt.device)
    ok = np.ones(opt.batch, dtype=bool)
    for i in range(n_dirs):
        d = [torch.as_tensor(rng.standard_normal(t.shape), device=opt.device) for t in (x0, x_ref, u_ref)]
        if i % 2:
            d = [torch.sign(t) for t in d]
        for s in (1, -1):
            opt.set_active_set(act0)
            opt.differentiable_step(x0 + s * eps * d[0], x_ref + s * eps * d[1], u_ref + s * eps * d[2],
                                    iterate=(xit, uit))
            ok &= (opt.get_active_set() == act0).all(1).cpu().numpy()
    return ok


@pytest.mark.gpu
def test_gpu_differentiable_step_gradcheck():
    import torch
    Bc, B, N, M, eps = 8, 4, 10, 20, 1e-6
    dt = 1.0 / N
    gp = make_gp(M)
    sc = random_ocp_batch(Bc, N, dt, orc.quad_hummingbird(), gp, seed=1000)
    dev = torch.device("cuda:0")
    x_ref = torch.as_tensor(sc["yref"][..., :NX], device=dev).contiguous()
    u_ref = torch.as_tensor(sc["yref"][..., NX:], device=dev).contiguous()
    xit, uit = torch.as_tensor(sc["xit"], device=dev), torch.as_tensor(sc["uit"], device=dev)
    opt = _gpu_handle(sc, Bc, N, gp, solver_variant=1, reset_on_fail=-1)
    opt.differentiable_step(torch.as_tensor(sc["x0"], device=dev), x_ref, u_ref, iterate=(xit, uit))
    act0 = opt.get_active_set().clone()
    assert (opt.solver_status()[0] == 0).all() and (act0 <= 2).all()
    stable = _stable_vehicles(opt, sc, N, act0, xit, uit, x_ref, u_ref, eps)
    idx = np.flatnonzero(stable)[:B]
    assert len(idx) == B, stable
    sub = {k: (None if v is None else v[idx]) for k, v in sc.items()}
    # gradcheck solves again for every perturbed input before it runs the backward of its first call: that first call
    # gets a handle of its own, so that its backward still finds the tiles it was taken from
    opts = [_gpu_handle(sub, B, N, gp, solver_variant=1, reset_on_fail=-1) for _ in range(2)]
    it = (xit[idx].contiguous(), uit[idx].contiguous())
    act = act0[idx].contiguous()
    calls = [0]

    def f(x0, xr, ur):
        o = opts[min(calls[0], 1)]
        calls[0] += 1
        o.set_active_set(act)
        return o.differentiable_step(x0, xr, ur, iterate=it)

    inputs = tuple(t.detach().clone().requires_grad_(True) for t in
                   (torch.as_tensor(sub["x0"], device=dev), x_ref[idx].contiguous(), u_ref[idx].contiguous()))
    # check_undefined_grad runs the forward three more times before it runs their three backwards, which a handle that
    # keeps only its last solve's tiles refuses by design; test_gpu_differentiable_step_backward_refuses_stale_tiles
    # covers zero and undefined output gradients
    assert torch.autograd.gradcheck(f, inputs, eps=eps, atol=1e-6, rtol=1e-4, check_undefined_grad=False)
    assert all((o.get_active_set() == act).all() for o in opts)


@pytest.mark.gpu
def test_gpu_differentiable_step_backward_refuses_stale_tiles():
    import torch
    N, B = 10, 4
    sc = random_ocp_batch(B, N, 1.0 / N, orc.quad_hummingbird(), None, seed=3)
    opt = _gpu_handle(sc, B, N, None)
    dev = opt.device
    x0 = torch.as_tensor(sc["x0"], device=dev).requires_grad_(True)
    x_ref = torch.as_tensor(sc["yref"][..., :NX], device=dev).requires_grad_(True)
    it = (torch.as_tensor(sc["xit"], device=dev), torch.as_tensor(sc["uit"], device=dev))
    x, u = opt.differentiable_step(x0, x_ref, iterate=it)
    g = torch.autograd.grad((x,), (x0, x_ref), (torch.zeros_like(x),), retain_graph=True, allow_unused=True)   # u_bar undefined
    assert all(t is None or (t == 0).all() for t in g)
    g = torch.autograd.grad((u,), (x0, x_ref), (torch.ones_like(u),), retain_graph=True, allow_unused=True)    # x_bar undefined
    assert all(t is not None and torch.isfinite(t).all() for t in g)
    (x.sum() + u.sum()).backward()
    assert x0.grad is not None and x_ref.grad is not None
    x, u = opt.differentiable_step(x0, x_ref, iterate=it)
    opt.differentiable_step(x0.detach(), x_ref.detach(), iterate=it)
    with pytest.raises(RuntimeError, match="solved again or had its active set changed"):
        u.sum().backward()
    x, u = opt.differentiable_step(x0, x_ref, iterate=it)
    opt.set_active_set(opt.get_active_set())
    with pytest.raises(RuntimeError, match="solved again or had its active set changed"):
        x.sum().backward()
    with pytest.raises(ValueError, match="iterate"):
        opt.differentiable_step(x0, x_ref, iterate=(it[0].clone().requires_grad_(True), it[1]))


@pytest.mark.gpu
def test_gpu_sens_epoch():
    import torch
    from mpc_quad_ros_b200.execute_trajectory import ClosedLoop
    from mpc_quad_ros_b200.quad import Quadrotor3D
    from mpc_quad_ros_b200.quad_opt import quad_optimizer
    from mpc_quad_ros_b200.trajectory import random_smooth_trajectories
    B, N = 8, 10
    traj = random_smooth_trajectories(B, 20 + N, 1.0 / N)
    quad = Quadrotor3D(drag=True, batch=B).set_hummingbird_params()
    opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N)
    loop = ClosedLoop(quad, opt, torch.as_tensor(traj), torch.as_tensor(traj[:, 0, :].copy()))
    e = [opt.sens_epoch()]
    loop.step()                                            # fused step (qmpc_closed_loop_step / qmpc_step)
    e.append(opt.sens_epoch())
    x0 = loop.x.clone()
    opt.run_optimization(x0)                               # qmpc_solve
    e.append(opt.sens_epoch())
    xbs, ubs = cotangents(np.random.default_rng(0), B, N)
    opt.eval_sens()
    opt.eval_adjoint(xbs, ubs)
    e.append(opt.sens_epoch())
    opt.set_active_set(opt.get_active_set())
    e.append(opt.sens_epoch())
    opt.reset_warm_start()
    e.append(opt.sens_epoch())
    assert e[1] != e[0] and e[2] != e[1] and e[3] == e[2] and e[4] != e[3] and e[5] != e[4], e


@pytest.mark.gpu
def test_gpu_adjoint_between_fused_steps_leaves_the_loop_unchanged():
    import torch
    from mpc_quad_ros_b200.execute_trajectory import ClosedLoop
    from mpc_quad_ros_b200.gp.GPE import GPEnsemble
    from mpc_quad_ros_b200.quad import Quadrotor3D
    from mpc_quad_ros_b200.quad_opt import quad_optimizer
    from mpc_quad_ros_b200.trajectory import random_smooth_trajectories
    B, N, M, steps = 256, 20, 20, 30
    traj = random_smooth_trajectories(B, steps + N + 2, 1.0 / N)
    xbs, ubs = (torch.as_tensor(t, device="cuda:0") for t in cotangents(np.random.default_rng(1), B, N))

    def run(with_adjoint):
        quad = Quadrotor3D(drag=True, batch=B).set_hummingbird_params()
        gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [M] * 3, theta=[3.0, 0.1, 0.01], batch=B)
        opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=gpe)
        loop = ClosedLoop(quad, opt, torch.as_tensor(traj), torch.as_tensor(traj[:, 0, :].copy()))
        u0s, finite = [], True
        for _ in range(steps):
            loop.step()
            u0s.append(loop.u0.clone())
            if with_adjoint:
                out = opt.eval_adjoint(xbs, ubs)
                ok = opt.solver_status()[0] == 0
                finite = finite and all(bool(torch.isfinite(t[ok]).all()) for t in out)
        x, u = opt.get_iterate()
        return torch.stack(u0s), x, u, gpe.mu_tensor(), gpe.C_tensor(), finite

    a, b = run(False), run(True)
    for ta, tb in zip(a[:5], b[:5]):
        assert torch.equal(ta, tb)
    assert b[5]


@pytest.mark.gpu
def test_gpu_adjoint_reference_api_batch_one():
    N, M, B = 20, 20, 4
    dt = 1.0 / N
    gp = make_gp(M)
    sc = random_ocp_batch(B, N, dt, orc.quad_hummingbird(), gp, seed=33)
    xbs, ubs = cotangents(np.random.default_rng(33), B, N)
    optb = _gpu_handle(sc, B, N, gp)
    _gpu_solve(optb, sc["xit"], sc["uit"], sc["x0"])
    refb = [t[0].cpu().numpy() for t in optb.eval_adjoint(xbs, ubs)]
    one = {k: (None if v is None else v[:1]) for k, v in sc.items()}
    opt1 = _gpu_handle(one, 1, N, gp)
    opt1.set_iterate(sc["xit"][0], sc["uit"][0])
    opt1.run_optimization(sc["x0"][0])                  # numpy in: the reference API of one vehicle
    out = opt1.eval_adjoint(xbs[0], ubs[0])
    assert all(isinstance(t, np.ndarray) for t in out)
    assert [t.shape for t in out] == [(13,), (N, 17), (13,)]
    for t, r in zip(out, refb):
        assert rel(t, r) < 1e-12
    x0u, _, _ = opt1.eval_adjoint(u_bar=ubs[0])
    x0x, _, _ = opt1.eval_adjoint(x_bar=xbs[0])
    assert rel(x0u + x0x, out[0]) < 1e-12


@pytest.mark.gpu
def test_gpu_adjoint_argument_errors_launch_nothing():
    import torch
    from mpc_quad_ros_b200 import _capi
    N, B = 10, 4
    sc = random_ocp_batch(B, N, 1.0 / N, orc.quad_hummingbird(), None, seed=3)
    opt = _gpu_handle(sc, B, N, None)
    lib = _capi.lib()
    xb = torch.zeros((B, N + 1, 13), dtype=torch.float64, device=opt.device)
    x0b = torch.empty((B, 13), dtype=torch.float64, device=opt.device)
    s = _capi.stream_ptr()
    null = C.c_void_p(0)
    l0 = lib.qmpc_launch_count()
    with pytest.raises(_capi.QmpcError, match="no solve"):
        opt.eval_adjoint(xb)
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"])
    torch.cuda.synchronize()
    l1 = lib.qmpc_launch_count()
    with pytest.raises(_capi.QmpcError, match="both NULL"):
        _capi.check(lib.qmpc_eval_adjoint(opt._h, null, null, _capi.ptr(x0b), null, null, s))
    with pytest.raises(_capi.QmpcError, match="all NULL"):
        _capi.check(lib.qmpc_eval_adjoint(opt._h, _capi.ptr(xb), null, null, null, null, s))
    with pytest.raises(_capi.QmpcError, match="null handle"):
        _capi.check(lib.qmpc_eval_adjoint(null, _capi.ptr(xb), null, _capi.ptr(x0b), null, null, s))
    with pytest.raises(_capi.QmpcError, match="null argument"):
        _capi.check(lib.qmpc_get_sens_epoch(opt._h, null))
    assert lib.qmpc_launch_count() == l1 and l1 > l0
    _capi.check(lib.qmpc_eval_adjoint(opt._h, _capi.ptr(xb), null, _capi.ptr(x0b), null, null, s))
    assert lib.qmpc_launch_count() == l1 + 1
    opt32 = _gpu_handle(sc, B, N, None, precision=32)
    _gpu_solve(opt32, sc["xit"], sc["uit"], sc["x0"])
    torch.cuda.synchronize()
    l2 = lib.qmpc_launch_count()
    with pytest.raises(_capi.QmpcError, match="fp64"):
        opt32.eval_adjoint(xb)
    assert lib.qmpc_launch_count() == l2
