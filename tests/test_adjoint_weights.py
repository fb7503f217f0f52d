"""Gradients of the RTI step w.r.t. the cost weights (qmpc_eval_adjoint_weights, quad_optimizer.eval_adjoint(weights=True)
and differentiable_step(w_diag=, we_diag=)), and the weights settable between solves (qmpc_set_weights).

The linearisation does not read the weights: they enter only the QP's objective, so on the active set the solve ended on
the solution z = (x, u) is a smooth function of them.  With (xh, uh) the minimiser the adjoint already builds (the pinned
LQR with linear costs -x_bar, -u_bar from xh_0 = 0):
    w_bar[i] = -dt sum_k (xh_k, uh_k)_i (z_k - yref_k)_i,   we_bar[i] = -xh_N,i (x_N - yref_e)_i.
Scaling every weight by one factor leaves z unchanged, so sum_i w_i w_bar_i + sum_i we_i we_bar_i = 0 for every vehicle.
Routes compared: central differences of the oracle's RTI step and of the library's own solves, the formula on the
oracle's LQR (tests/sens/rti_adjoint_weights.c), and the kernel, emulated on the CPU
(tests/sens/emu_adjoint_weights.cpp) and on the GPU."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as orc
from helpers import make_gp, random_ocp_batch
from emu import emu
from sens import adjoint_ref, adjoint_weights_ref

TOL64 = 1e-9          # kernel vs oracle, fp64: two exact routes to the same linear map (as tests/test_adjoint.py)
NX, NU, NY = 13, 4, 17


def rel(a, ref):
    """max|a - ref| / max(1, max|ref|)"""
    return float(np.abs(a - ref).max() / max(1.0, np.abs(ref).max()))


def act_of(u, lb=0.0, ub=1.0):
    u = u.reshape(u.shape[0], -1)
    return np.where(u == lb, 1, np.where(u == ub, 2, 0)).astype(np.uint8)


def cotangents(rng, B, N):
    return rng.standard_normal((B, N + 1, NX)), rng.standard_normal((B, N, NU))


def scale_residual(wb, web, Wd=orc.W_DIAG, Wed=orc.WE_DIAG):
    """|sum w w_bar + sum we we_bar| / sum of the magnitudes of its terms, per vehicle (0 for the exact minimiser)"""
    t = np.concatenate([np.asarray(Wd) * wb, np.asarray(Wed) * web], axis=-1)
    return np.abs(t.sum(-1)) / np.maximum(np.abs(t).sum(-1), 1e-300)


def oracle_solve(sc, b, quad, dt, N, gp, Wd=orc.W_DIAG, Wed=orc.WE_DIAG):
    x, u = sc["xit"][b].copy(), sc["uit"][b].copy()
    r = orc.rti_step(quad, dt, N, sc["x0"][b], sc["yref"][b], sc["yref_e"][b], x, u, gp=gp,
                     alpha=None if gp is None else sc["alpha"][b], Wd=Wd, Wed=Wed)
    assert r["status"] == 0, r
    return x, u


def reference(sc, b, quad, dt, N, gp, act, x, u, x_bar, u_bar):
    return adjoint_weights_ref.rti_adjoint_weights(quad, dt, N, sc["xit"][b], sc["uit"][b], act, x, u, sc["yref"][b],
                                           sc["yref_e"][b], x_bar=x_bar, u_bar=u_bar, gp=gp,
                                           alpha=None if gp is None else sc["alpha"][b])


# ------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("N,use_gp", [(20, True), (20, False), (7, True), (7, False)])
def test_reference_matches_central_differences_and_the_scale_identity(N, use_gp):
    B, dt, eps = 6, 1.0 / N, 1e-5
    quad = orc.quad_hummingbird()
    gp = make_gp(20) if use_gp else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=140 + N)
    rng = np.random.default_rng(140 + N)
    xbs, ubs = cotangents(rng, B, N)
    kept, worst, worst_scale = 0, 0.0, 0.0
    for b in range(B):
        x, u = oracle_solve(sc, b, quad, dt, N, gp)
        act = act_of(u[None])[0]
        wb, web = reference(sc, b, quad, dt, N, gp, act, x, u, xbs[b], ubs[b])
        worst_scale = max(worst_scale, float(scale_residual(wb, web)))
        same, errs = True, []
        for _ in range(3):             # relative directions: the weights span 0.05 .. 10
            dw, dwe = orc.W_DIAG * rng.standard_normal(NY), orc.WE_DIAG * rng.standard_normal(NX)
            vals = []
            for s in (1, -1):
                xp, up = oracle_solve(sc, b, quad, dt, N, gp, Wd=orc.W_DIAG + s * eps * dw, Wed=orc.WE_DIAG + s * eps * dwe)
                same = same and np.array_equal(act_of(up[None])[0], act)
                vals.append(np.vdot(xbs[b], xp) + np.vdot(ubs[b], up))
            fd = (vals[0] - vals[1]) / (2 * eps)
            ad = np.vdot(wb, dw) + np.vdot(web, dwe)
            errs.append(abs(fd - ad) / max(1.0, abs(ad)))
        if same:
            kept += 1
            worst = max(worst, max(errs))
    print(f"N={N} gp={use_gp}: {kept}/{B} vehicles keep their active set; worst rel err vs central differences "
          f"{worst:.1e}, scale identity {worst_scale:.1e}")
    assert kept >= B // 2, kept
    # central differences at eps = 1e-5 carry a truncation error ~ eps^2 and a rounding error ~ 1e-16 / eps relative:
    # at most 4.0e-8 measured on these cases, so 1e-6 leaves room and still fails any wrong term (those are O(1))
    assert worst < 1e-6, worst
    assert worst_scale < 1e-12, worst_scale


def _emulated_case(N, use_gp, variant, B=3, seed=None, flavour=""):
    dt = 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp() if use_gp else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=N + 40 if seed is None else seed)
    cfg, keep = emu.make_config(B, N, 1.0, quad, orc.W_DIAG, orc.WE_DIAG, None if gp is None else gp.X,
                                None if gp is None else gp.theta)
    xe, ue = sc["xit"].copy(), sc["uit"].copy()
    r = emu.solve(cfg, sc["x0"], sc["yref"], sc["yref_e"], sc["alpha"], xe, ue, variant=variant, flavour=flavour)
    return sc, quad, dt, gp, cfg, keep, r, xe, ue


def _check_emulated(sc, quad, dt, gp, cfg, r, xe, ue, xbs, ubs, flavour=""):
    B, N = cfg.batch, cfg.n_nodes
    out = adjoint_weights_ref.emu_adjoint_weights(cfg, r, xe, ue, sc["yref"], sc["yref_e"], xbs, ubs, flavour=flavour)
    # the first three outputs are those of qmpc_eval_adjoint, bit for bit
    for o, o_ref in zip(out[:3], adjoint_ref.emu_adjoint(cfg, r, xbs, ubs, flavour=flavour)):
        assert np.array_equal(o, o_ref)
    wb, web = out[3], out[4]
    for b in range(B):
        owb, oweb = reference(sc, b, quad, dt, N, gp, r["act"][b], xe[b], ue[b], xbs[b], ubs[b])
        assert max(rel(wb[b], owb), rel(web[b], oweb)) < TOL64, (b, rel(wb[b], owb), rel(web[b], oweb))
    assert (scale_residual(wb, web) < 1e-9).all(), scale_residual(wb, web)
    return out


@pytest.mark.parametrize("variant", [1, 2], ids=["warp_per_ocp", "screen_plus_dense"])
@pytest.mark.parametrize("N,use_gp", [(20, True), (20, False), (7, True), (7, False), (1, True), (1, False)])
def test_emulated_kernel_matches_reference(N, use_gp, variant):
    sc, quad, dt, gp, cfg, keep, r, xe, ue = _emulated_case(N, use_gp, variant)
    B = cfg.batch
    assert (r["status"] == 0).all()
    for b in range(B):                                  # the emulated solve ends on the oracle's solution
        xo, uo = oracle_solve(sc, b, quad, dt, N, gp)
        assert np.array_equal(r["act"][b], act_of(uo[None])[0]) and rel(ue[b], uo) < 1e-8
    xbs, ubs = cotangents(np.random.default_rng(N + variant), B, N)
    x0b, yb, yeb, wb, web = _check_emulated(sc, quad, dt, gp, cfg, r, xe, ue, xbs, ubs)
    # any output may be NULL, the weight outputs alone included; each output is the same whatever else is asked for
    ysl = (sc["yref"], sc["yref_e"])
    for mask in [(False, False, False, True, True), (False, False, False, True, False), (False, False, False, False, True),
                 (True, False, False, False, True), (False, True, True, False, False)]:
        part = adjoint_weights_ref.emu_adjoint_weights(cfg, r, xe, ue, *ysl, xbs, ubs, outputs=mask)
        for want, o, full in zip(mask, part, (x0b, yb, yeb, wb, web)):
            assert (o is None) if not want else np.array_equal(o, full)
    # a NULL cotangent is zero: the map is linear in the cotangents
    _, _, _, wx, wex = adjoint_weights_ref.emu_adjoint_weights(cfg, r, xe, ue, *ysl, xbs, None)
    _, _, _, wu, weu = adjoint_weights_ref.emu_adjoint_weights(cfg, r, xe, ue, *ysl, None, ubs)
    assert rel(wx + wu, wb) < 1e-12 and rel(wex + weu, web) < 1e-12


def test_emulated_kernel_without_tile_ring():
    """the A/B build flavour that reads the tiles in place with unpadded rows (QMPC_RING=0, QMPC_WR=16)"""
    N = 20
    sc, quad, dt, gp, cfg, keep, r, xe, ue = _emulated_case(N, True, 1, seed=60, flavour="noring")
    xbs, ubs = cotangents(np.random.default_rng(60), 3, N)
    _check_emulated(sc, quad, dt, gp, cfg, r, xe, ue, xbs, ubs, flavour="noring")


def test_emulated_unknown_active_set_gives_nan():
    N, B = 20, 3
    dt = 1.0 / N
    quad = orc.quad_hummingbird()
    sc = random_ocp_batch(B, N, dt, quad, None, seed=77, amp_choices=(8.0,))
    xbs, ubs = cotangents(np.random.default_rng(77), B, N)
    cfg, keep = emu.make_config(B, N, 1.0, quad, orc.W_DIAG, orc.WE_DIAG)
    xe, ue = sc["xit"].copy(), sc["uit"].copy()
    r = emu.solve(cfg, sc["x0"], sc["yref"], sc["yref_e"], None, xe, ue, variant=1)
    assert (r["status"] == 0).all()
    ref = adjoint_weights_ref.emu_adjoint_weights(cfg, r, xe, ue, sc["yref"], sc["yref_e"], xbs, ubs)
    r["act"][1, 17] = 255               # one unknown entry makes one vehicle unknown; its neighbours are unaffected
    out = adjoint_weights_ref.emu_adjoint_weights(cfg, r, xe, ue, sc["yref"], sc["yref_e"], xbs, ubs)
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
def test_gpu_adjoint_weights_vs_reference(N, M, seed, variant):
    import torch
    if variant == 2 and N > 21:
        pytest.skip("the screening + dense solver serves N <= 21")
    B, dt = 48, 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp(M) if M else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=seed)      # the scenarios of test_gpu_adjoint_vs_oracle_and_eval_sens
    opt = _gpu_handle(sc, B, N, gp, solver_variant=variant)
    x, u = (t.cpu().numpy() for t in _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"]))
    xbs, ubs = cotangents(np.random.default_rng(seed), B, N)
    out = opt.eval_adjoint(xbs, ubs, weights=True)
    for o, o_ref in zip(out[:3], opt.eval_adjoint(xbs, ubs)):
        assert torch.equal(o, o_ref)
    wb, web = (t.cpu().numpy() for t in out[3:])
    act = opt.get_active_set().cpu().numpy()
    assert (opt.solver_status()[0].cpu().numpy() == 0).all()
    worst = 0.0
    for b in range(B):
        owb, oweb = reference(sc, b, quad, dt, N, gp, act[b], x[b], u[b], xbs[b], ubs[b])
        worst = max(worst, rel(wb[b], owb), rel(web[b], oweb))
    scale = float(scale_residual(wb, web).max())
    print(f"N={N} M={M} variant {variant}: worst rel err vs the reference {worst:.1e}, scale identity {scale:.1e}")
    assert worst < TOL64, worst
    assert scale < 1e-9, scale            # exact for the exact minimiser; the solve is exact to ~1e-12 relative


@pytest.mark.gpu
@pytest.mark.parametrize("variant,tol", [(1, 1e-6), (2, 1e-4)], ids=["warp_per_ocp", "screen_plus_dense"])
def test_gpu_adjoint_weights_vs_central_differences_of_the_library(variant, tol):
    """no oracle: solves of the library itself from the same iterate and active set at weights w +- eps * d"""
    import torch
    from mpc_quad_ros_b200.quad_opt import Q_DIAGONAL, R_COST
    B, N, M, eps = 48, 20, 20, 1e-4
    dt = 1.0 / N
    gp = make_gp(M)
    sc = random_ocp_batch(B, N, dt, orc.quad_hummingbird(), gp, seed=900)
    opt = _gpu_handle(sc, B, N, gp, solver_variant=variant, reset_on_fail=-1)
    w0, we0 = np.concatenate([Q_DIAGONAL, R_COST]), Q_DIAGONAL.copy()
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"])
    act0 = opt.get_active_set().clone()                  # injected before every solve below
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"], act=act0)
    rng = np.random.default_rng(901)
    xbs, ubs = cotangents(rng, B, N)
    wb, web = (t.cpu().numpy() for t in opt.eval_adjoint(xbs, ubs, weights=True)[3:])
    acts = [opt.get_active_set().cpu().numpy()]
    fds, ads = [], []
    for part in range(3):                                # stage weights, terminal weights, both
        dw = w0 * rng.standard_normal(NY) if part in (0, 2) else np.zeros(NY)
        dwe = we0 * rng.standard_normal(NX) if part in (1, 2) else np.zeros(NX)
        vals = []
        for s in (1, -1):
            opt.set_weights(w0 + s * eps * dw, we0 + s * eps * dwe)
            x, u = _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"], act=act0)
            acts.append(opt.get_active_set().cpu().numpy())
            vals.append((xbs * x.cpu().numpy()).sum(axis=(1, 2)) + (ubs * u.cpu().numpy()).sum(axis=(1, 2)))
        fds.append((vals[0] - vals[1]) / (2 * eps))
        ads.append(wb @ dw + web @ dwe)
    keep = np.array([all(np.array_equal(a[b], acts[0][b]) for a in acts) and (acts[0][b] <= 2).all() for b in range(B)])
    print(f"variant {variant}: {keep.sum()}/{B} vehicles keep their active set in all 7 solves")
    assert keep.mean() >= 0.75
    fd, ad = np.array(fds)[:, keep], np.array(ads)[:, keep]
    err = float((np.abs(fd - ad) / np.maximum(1.0, np.abs(ad))).max())
    print(f"variant {variant}: rel err vs central differences {err:.1e}")
    assert err < tol


def _outputs(opt):
    import torch
    x, u = opt.get_iterate()
    cost = torch.empty((opt.batch,), dtype=torch.float64, device=opt.device)
    from mpc_quad_ros_b200 import _capi
    _capi.check(_capi.lib().qmpc_get_cost(opt._h, _capi.ptr(cost), _capi.stream_ptr()))
    st, it = opt.solver_status()
    return [x, u, cost, st, it, opt.get_active_set()]


def _run_sequence(opt, sc, traj):
    """three qmpc_solve calls from the persistent iterate, then five fused closed-loop steps (qmpc_step)"""
    import torch
    from mpc_quad_ros_b200.execute_trajectory import ClosedLoop
    outs = []
    opt.set_iterate(torch.as_tensor(sc["xit"]), torch.as_tensor(sc["uit"]))
    for i in range(3):
        opt.run_optimization(torch.as_tensor(sc["x0"] * (1 + 0.01 * i), device=opt.device))
        outs += _outputs(opt)
    loop = ClosedLoop(opt.quad, opt, torch.as_tensor(traj), torch.as_tensor(traj[:, 0, :].copy()))
    for _ in range(5):
        loop.step()
        outs += _outputs(opt) + [loop.u0.clone()]
    return outs


@pytest.mark.gpu
@pytest.mark.parametrize("precision,variant", [(64, 1), (64, 2), (32, 1)], ids=["fp64_warp_per_ocp",
                                                                                 "fp64_screen_plus_dense", "fp32"])
def test_gpu_set_weights_equals_creating_with_them(precision, variant, monkeypatch):
    import torch
    from mpc_quad_ros_b200 import quad_opt
    from mpc_quad_ros_b200.trajectory import random_smooth_trajectories
    B, N = 64, 20
    sc = random_ocp_batch(B, N, 1.0 / N, orc.quad_hummingbird(), None, seed=7)
    traj = random_smooth_trajectories(B, 10 + N, 1.0 / N)
    q1, r1 = quad_opt.Q_DIAGONAL.copy(), quad_opt.R_COST.copy()
    q2, r2 = q1 * np.linspace(0.5, 3.0, NX), r1 * np.array([2.0, 0.5, 1.5, 3.0])
    make = lambda: _gpu_handle(sc, B, N, None, precision=precision, solver_variant=variant)
    a = make()                                                    # created with W1, set to W2
    a.set_weights(np.concatenate([q2, r2]), q2)
    e = make()                                                    # created with W1, set to W2 and back to W1
    e.set_weights(np.concatenate([q2, r2]), q2)
    e.set_weights(np.concatenate([q1, r1]), q1)
    f = make()                                                    # created with W1, never changed
    monkeypatch.setattr(quad_opt, "Q_DIAGONAL", q2)               # quad_optimizer builds W and W_e from these
    monkeypatch.setattr(quad_opt, "R_COST", r2)
    b = make()                                                    # created with W2
    assert np.array_equal(np.diag(a.W), np.diag(b.W)) and np.array_equal(np.diag(a.W_e), np.diag(b.W_e))
    ra, rb, re_, rf = (_run_sequence(o, sc, traj) for o in (a, b, e, f))
    same = lambda x, y: torch.equal(x, y) or bool(((x == y) | (x.isnan() & y.isnan())).all())
    assert all(same(x, y) for x, y in zip(ra, rb))
    assert all(same(x, y) for x, y in zip(re_, rf))
    assert not all(same(x, y) for x, y in zip(ra, rf))             # the weights did change the solutions


@pytest.mark.gpu
def test_gpu_set_weights_after_a_solve_leaves_its_sensitivities():
    import torch
    N, M, B = 20, 20, 32
    gp = make_gp(M)
    sc = random_ocp_batch(B, N, 1.0 / N, orc.quad_hummingbird(), gp, seed=44)
    opt = _gpu_handle(sc, B, N, gp)
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"])
    xbs, ubs = cotangents(np.random.default_rng(44), B, N)
    calls = lambda: list(opt.eval_sens()) + list(opt.eval_adjoint(xbs, ubs)) + list(opt.eval_adjoint(xbs, ubs, weights=True))
    before, e0 = calls(), opt.sens_epoch()
    opt.set_weights(np.diag(opt.W) * 2.5, np.diag(opt.W_e) * 0.3)
    after = calls()
    assert opt.sens_epoch() == e0
    for x, y in zip(before, after):
        assert torch.equal(x, y)


def _stable_vehicles(opt, sc, act0, xit, uit, x_ref, w, we, eps, n_dirs=6):
    """vehicles whose active set survives +-eps in random directions of (x0, x_ref, w, we), and in each direction's
    coordinate-wise worst case"""
    import torch
    rng = np.random.default_rng(5)
    x0 = torch.as_tensor(sc["x0"], device=opt.device)
    ok = np.ones(opt.batch, dtype=bool)
    for i in range(n_dirs):
        d = [torch.as_tensor(rng.standard_normal(t.shape), device=opt.device) for t in (x0, x_ref, w, we)]
        if i % 2:
            d = [torch.sign(t) for t in d]
        for s in (1, -1):
            opt.set_active_set(act0)
            opt.differentiable_step(x0 + s * eps * d[0], x_ref + s * eps * d[1], iterate=(xit, uit),
                                    w_diag=w + s * eps * d[2], we_diag=we + s * eps * d[3])
            ok &= (opt.get_active_set() == act0).all(1).cpu().numpy()
    return ok


@pytest.mark.gpu
def test_gpu_differentiable_step_gradcheck_weights():
    import torch
    from mpc_quad_ros_b200.quad_opt import Q_DIAGONAL, R_COST
    Bc, B, N, M, eps = 8, 4, 10, 20, 1e-6
    dt = 1.0 / N
    gp = make_gp(M)
    sc = random_ocp_batch(Bc, N, dt, orc.quad_hummingbird(), gp, seed=1000)
    dev = torch.device("cuda:0")
    x_ref = torch.as_tensor(sc["yref"][..., :NX], device=dev).contiguous()
    xit, uit = torch.as_tensor(sc["xit"], device=dev), torch.as_tensor(sc["uit"], device=dev)
    w = torch.as_tensor(np.concatenate([Q_DIAGONAL, R_COST]), device=dev)
    we = torch.as_tensor(Q_DIAGONAL, device=dev)
    opt = _gpu_handle(sc, Bc, N, gp, solver_variant=1, reset_on_fail=-1)
    opt.differentiable_step(torch.as_tensor(sc["x0"], device=dev), x_ref, iterate=(xit, uit))
    act0 = opt.get_active_set().clone()
    assert (opt.solver_status()[0] == 0).all() and (act0 <= 2).all()
    stable = _stable_vehicles(opt, sc, act0, xit, uit, x_ref, w, we, eps)
    idx = np.flatnonzero(stable)[:B]
    assert len(idx) == B, stable
    sub = {k: (None if v is None else v[idx]) for k, v in sc.items()}
    # the first call gets a handle of its own, so that its backward still finds its tiles (as in test_adjoint.py)
    opts = [_gpu_handle(sub, B, N, gp, solver_variant=1, reset_on_fail=-1) for _ in range(2)]
    it = (xit[idx].contiguous(), uit[idx].contiguous())
    act = act0[idx].contiguous()
    calls = [0]

    def f(x0, xr, wd, wed):
        o = opts[min(calls[0], 1)]
        calls[0] += 1
        o.set_active_set(act)
        return o.differentiable_step(x0, xr, iterate=it, w_diag=wd, we_diag=wed)

    inputs = tuple(t.detach().clone().requires_grad_(True) for t in
                   (torch.as_tensor(sub["x0"], device=dev), x_ref[idx].contiguous(), w, we))
    assert torch.autograd.gradcheck(f, inputs, eps=eps, atol=1e-6, rtol=1e-4, check_undefined_grad=False)
    assert all((o.get_active_set() == act).all() for o in opts)


@pytest.mark.gpu
def test_gpu_imitation_of_the_expert_weights():
    """learn the Q/R weights from an expert's controls by gradient descent on log-weights through the controller"""
    import torch
    from mpc_quad_ros_b200.quad_opt import Q_DIAGONAL, R_COST
    B, N, M = 64, 20, 20
    gp = make_gp(M)
    sc = random_ocp_batch(B, N, 1.0 / N, orc.quad_hummingbird(), gp, seed=2024)
    dev = torch.device("cuda:0")
    opt = _gpu_handle(sc, B, N, gp, solver_variant=1, reset_on_fail=-1)
    x0 = torch.as_tensor(sc["x0"], device=dev)
    x_ref = torch.as_tensor(sc["yref"][..., :NX], device=dev).contiguous()
    it = (torch.as_tensor(sc["xit"], device=dev), torch.as_tensor(sc["uit"], device=dev))
    w_star = torch.as_tensor(np.concatenate([Q_DIAGONAL, R_COST, Q_DIAGONAL]), device=dev)
    with torch.no_grad():
        _, u_star = opt.differentiable_step(x0, x_ref, iterate=it, w_diag=w_star[:NY], we_diag=w_star[NY:])
    log_w = torch.log(w_star).clone()
    log_w[[0, 4, 13, 15, 17]] += np.log(3.0)            # a few stage, input and terminal weights x3
    log_w.requires_grad_(True)
    adam = torch.optim.Adam([log_w], lr=0.05)
    losses = []
    for _ in range(40):
        adam.zero_grad()
        w = torch.exp(log_w)
        _, u = opt.differentiable_step(x0, x_ref, iterate=it, w_diag=w[:NY], we_diag=w[NY:])
        ok = opt.solver_status()[0] == 0
        loss = ((u - u_star)[ok] ** 2).mean()
        loss.backward()
        adam.step()
        losses.append(float(loss.detach()))
    print(f"imitation loss {losses[0]:.3e} -> {losses[-1]:.3e} (min {min(losses):.3e}) in {len(losses)} steps")
    assert np.isfinite(losses).all()
    # measured on a B200 (1000 W power limit): 1.80e-2 -> 2.66e-4 in 40 steps
    assert losses[-1] < 0.1 * losses[0], losses


@pytest.mark.gpu
def test_gpu_refusals_launch_nothing():
    import torch
    from mpc_quad_ros_b200 import _capi
    N, B = 10, 4
    sc = random_ocp_batch(B, N, 1.0 / N, orc.quad_hummingbird(), None, seed=3)
    opt = _gpu_handle(sc, B, N, None, solver_variant=1)
    lib = _capi.lib()
    s, null = _capi.stream_ptr(), C.c_void_p(0)
    xb = torch.zeros((B, N + 1, NX), dtype=torch.float64, device=opt.device)
    wb = torch.empty((B, NY), dtype=torch.float64, device=opt.device)
    hp = lambda a: null if a is None else a.ctypes.data_as(C.c_void_p)          # a: float64 arrays kept alive by the caller
    w_ok, we_ok = np.diag(opt.W).copy(), np.diag(opt.W_e).copy()
    torch.cuda.synchronize()
    l0 = lib.qmpc_launch_count()
    with pytest.raises(_capi.QmpcError, match="no solve"):
        _capi.check(lib.qmpc_eval_adjoint_weights(opt._h, _capi.ptr(xb), null, null, null, null, _capi.ptr(wb), null, s))
    assert lib.qmpc_launch_count() == l0
    opt.reset_warm_start()             # both solves below start from the same iterate and the same (unknown) active set
    x_first, u_first = (t.clone() for t in _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"]))
    torch.cuda.synchronize()
    l1 = lib.qmpc_launch_count()
    bad = []
    for i, v in [(0, np.nan), (3, -1e-3), (8, np.inf), (13, 0.0), (16, -0.1)]:
        w = w_ok.copy()
        w[i] = v
        bad.append((w, None))
    for i, v in [(0, np.nan), (12, -1.0)]:
        we = we_ok.copy()
        we[i] = v
        bad.append((None, we))
    bad.append((w_ok * 2, np.where(np.arange(NX) == 5, -1.0, we_ok)))          # one bad array refuses both
    for w, we in bad:
        with pytest.raises(_capi.QmpcError, match="w_diag|we_diag"):
            _capi.check(lib.qmpc_set_weights(opt._h, hp(w), hp(we)))
    with pytest.raises(_capi.QmpcError, match="both NULL"):
        _capi.check(lib.qmpc_set_weights(opt._h, null, null))
    with pytest.raises(_capi.QmpcError, match="null handle"):
        _capi.check(lib.qmpc_set_weights(null, hp(w_ok), null))
    with pytest.raises(_capi.QmpcError, match="null handle"):
        _capi.check(lib.qmpc_eval_adjoint_weights(null, _capi.ptr(xb), null, null, null, null, _capi.ptr(wb), null, s))
    with pytest.raises(_capi.QmpcError, match="both NULL"):
        _capi.check(lib.qmpc_eval_adjoint_weights(opt._h, null, null, null, null, null, _capi.ptr(wb), null, s))
    with pytest.raises(_capi.QmpcError, match="all NULL"):
        _capi.check(lib.qmpc_eval_adjoint_weights(opt._h, _capi.ptr(xb), null, null, null, null, null, null, s))
    assert lib.qmpc_launch_count() == l1
    # the refused calls changed nothing: the same solve again gives the same bits
    opt.reset_warm_start()
    x, u = _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"])
    assert torch.equal(x, x_first) and torch.equal(u, u_first)
    torch.cuda.synchronize()
    l2 = lib.qmpc_launch_count()
    _capi.check(lib.qmpc_eval_adjoint_weights(opt._h, _capi.ptr(xb), null, null, null, null, _capi.ptr(wb), null, s))
    assert lib.qmpc_launch_count() == l2 + 1
    opt32 = _gpu_handle(sc, B, N, None, precision=32)
    opt32.set_weights(w_ok * 2, we_ok * 2)                         # fp32 handles take new weights
    _gpu_solve(opt32, sc["xit"], sc["uit"], sc["x0"])
    torch.cuda.synchronize()
    l3 = lib.qmpc_launch_count()
    with pytest.raises(_capi.QmpcError, match="fp64"):
        opt32.eval_adjoint(xb, weights=True)
    assert lib.qmpc_launch_count() == l3
