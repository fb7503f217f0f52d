"""Forward mode of the RTI step w.r.t. x0, the reference and the cost weights (qmpc_eval_jvp, quad_optimizer.eval_jvp)
and forward-mode autograd through differentiable_step (_RTIStep.jvp).

The linearisation does not read x0, the reference or the weights, so on the active set the solve ended on the step is
linear in their tangents: (dx, du) is the minimiser of the pinned LQR of the adjoint with dx_0 = dx0 and the linear
costs c_k = -dt W dyref_k + dt dw (z_k - yref_k), c_N = -W_e dyref_e + dwe (x_N - yref_e).  Routes compared: central
differences of the oracle's RTI step and of the library's own solves, that LQR on the oracle's routines
(tests/sens/rti_jvp.c), the kernel emulated on the CPU (tests/sens/emu_jvp.cpp) and on the GPU; and three identities:
the dot product with the adjoint, the x0 columns of eval_sens and the scale invariance of the minimiser."""
import numpy as np
import pytest

from oracle import oracle as orc
from helpers import make_gp, random_ocp_batch
from emu import emu
from sens import adjoint_ref, adjoint_weights_ref, jvp_ref, sens_ref

TOL64 = 1e-9          # kernel vs oracle, fp64: two exact routes to the same linear map (as tests/test_adjoint.py)
NX, NU, NY = 13, 4, 17
NAMES = ("dx0", "dyref", "dyref_e", "dw", "dwe")


def rel(a, ref):
    """max|a - ref| / max(1, max|ref|)"""
    return float(np.abs(a - ref).max() / max(1.0, np.abs(ref).max()))


def act_of(u, lb=0.0, ub=1.0):
    u = u.reshape(u.shape[0], -1)
    return np.where(u == lb, 1, np.where(u == ub, 2, 0)).astype(np.uint8)


def tangents(rng, lead, N, parts=NAMES):
    """random tangents with a leading shape `lead`; the weight directions relative to the weights (they span 0.05 .. 10)"""
    full = dict(dx0=rng.standard_normal(lead + (NX,)), dyref=rng.standard_normal(lead + (N, NY)),
                dyref_e=rng.standard_normal(lead + (NX,)), dw=orc.W_DIAG * rng.standard_normal(lead + (NY,)),
                dwe=orc.WE_DIAG * rng.standard_normal(lead + (NX,)))
    return {k: (full[k] if k in parts else None) for k in NAMES}


def oracle_solve(sc, b, quad, dt, N, gp, x0=None, yref=None, yref_e=None, Wd=orc.W_DIAG, Wed=orc.WE_DIAG):
    x, u = sc["xit"][b].copy(), sc["uit"][b].copy()
    r = orc.rti_step(quad, dt, N, sc["x0"][b] if x0 is None else x0, sc["yref"][b] if yref is None else yref,
                     sc["yref_e"][b] if yref_e is None else yref_e, x, u, gp=gp,
                     alpha=None if gp is None else sc["alpha"][b], Wd=Wd, Wed=Wed)
    assert r["status"] == 0, r
    return x, u


def reference(sc, b, quad, dt, N, gp, act, x, u, t):
    return jvp_ref.rti_jvp(quad, dt, N, sc["xit"][b], sc["uit"][b], act, x, u, sc["yref"][b], sc["yref_e"][b],
                           gp=gp, alpha=None if gp is None else sc["alpha"][b], **t)


def adjoint_side(sc, b, quad, dt, N, gp, act, x, u, xb, ub, t):
    """<x0_bar, dx0> + <yref_bar, dyref> + ... from the two adjoint references, and the sum of the magnitudes of its terms"""
    alpha = None if gp is None else sc["alpha"][b]
    bars = adjoint_ref.rti_adjoint(quad, dt, N, sc["xit"][b], sc["uit"][b], act, xb, ub, gp=gp, alpha=alpha)
    bars += adjoint_weights_ref.rti_adjoint_weights(quad, dt, N, sc["xit"][b], sc["uit"][b], act, x, u, sc["yref"][b],
                                                    sc["yref_e"][b], xb, ub, gp=gp, alpha=alpha)
    terms = [np.vdot(bar, t[n]) for bar, n in zip(bars, NAMES) if t[n] is not None]
    return float(np.sum(terms)), float(np.sum(np.abs(terms)))


# ------------------------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("N,use_gp", [(20, True), (20, False), (7, True), (7, False)])
def test_reference_matches_central_differences(N, use_gp):
    B, dt, eps = 6, 1.0 / N, 1e-5
    quad = orc.quad_hummingbird()
    gp = make_gp(20) if use_gp else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=240 + N)
    rng = np.random.default_rng(240 + N)
    kept, worst = 0, 0.0
    for b in range(B):
        x, u = oracle_solve(sc, b, quad, dt, N, gp)
        act = act_of(u[None])[0]
        same, errs = True, []
        for parts in [(n,) for n in NAMES] + [NAMES]:          # each tangent alone, then all together
            t = tangents(rng, (), N, parts)
            dx, du = reference(sc, b, quad, dt, N, gp, act, x, u, t)
            fd = []
            for s in (1, -1):
                at = lambda base, n: base if t[n] is None else base + s * eps * t[n]
                xp, up = oracle_solve(sc, b, quad, dt, N, gp, x0=at(sc["x0"][b], "dx0"), yref=at(sc["yref"][b], "dyref"),
                                      yref_e=at(sc["yref_e"][b], "dyref_e"), Wd=at(orc.W_DIAG, "dw"),
                                      Wed=at(orc.WE_DIAG, "dwe"))
                same = same and np.array_equal(act_of(up[None])[0], act)
                fd.append((xp, up))
            fdx, fdu = ((p - m) / (2 * eps) for p, m in zip(*fd))
            errs.append(max(rel(dx, fdx), rel(du, fdu)))
        if same:
            kept += 1
            worst = max(worst, max(errs))
    print(f"N={N} gp={use_gp}: {kept}/{B} vehicles keep their active set; worst rel err vs central differences {worst:.1e}")
    assert kept >= B // 2, kept
    # eps = 1e-5: truncation ~ eps^2 and rounding ~ 1e-16 / eps relative, as in tests/test_adjoint_weights.py; a wrong
    # term is O(1)
    assert worst < 1e-6, worst


@pytest.mark.parametrize("N,use_gp", [(20, True), (7, False)])
def test_reference_identities(N, use_gp):
    """the dot product with the adjoint references, the x0 columns of rti_sens and the scale invariance"""
    B, dt = 6, 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp(20) if use_gp else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=340 + N)
    rng = np.random.default_rng(340 + N)
    w_dot = w_col = w_scale = 0.0
    for b in range(B):
        x, u = oracle_solve(sc, b, quad, dt, N, gp)
        act = act_of(u[None])[0]
        t = tangents(rng, (), N)
        dx, du = reference(sc, b, quad, dt, N, gp, act, x, u, t)
        xb, ub = rng.standard_normal((N + 1, NX)), rng.standard_normal((N, NU))
        rhs, mag = adjoint_side(sc, b, quad, dt, N, gp, act, x, u, xb, ub, t)
        lhs = np.vdot(xb, dx) + np.vdot(ub, du)
        w_dot = max(w_dot, abs(lhs - rhs) / (mag + abs(lhs)))
        sx, su = sens_ref.rti_sens(quad, dt, N, sc["xit"][b], sc["uit"][b], act, gp=gp,
                                   alpha=None if gp is None else sc["alpha"][b])
        for i in range(NX):
            dxi, dui = reference(sc, b, quad, dt, N, gp, act, x, u, dict(dx0=np.eye(NX)[i]))
            w_col = max(w_col, rel(dxi, sx[:, :, i]), rel(dui, su[:, :, i]))
        # scaling every weight leaves the minimiser unchanged: the stage and the terminal halves cancel
        xs, us = reference(sc, b, quad, dt, N, gp, act, x, u, dict(dw=orc.W_DIAG))
        xe, ue = reference(sc, b, quad, dt, N, gp, act, x, u, dict(dwe=orc.WE_DIAG))
        scale = max(np.abs(xs).max(), np.abs(us).max())
        w_scale = max(w_scale, max(np.abs(xs + xe).max(), np.abs(us + ue).max()) / scale)
    print(f"N={N} gp={use_gp}: dot product {w_dot:.1e}, x0 columns {w_col:.1e}, scale identity {w_scale:.1e}")
    assert w_dot < 1e-12 and w_col < 1e-12, (w_dot, w_col)
    assert w_scale < 1e-10, w_scale        # exact for the exact minimiser; the oracle's solve is exact to ~1e-13


def _emulated_case(N, use_gp, variant, B=3, seed=None, flavour=""):
    dt = 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp() if use_gp else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=N + 50 if seed is None else seed)
    cfg, keep = emu.make_config(B, N, 1.0, quad, orc.W_DIAG, orc.WE_DIAG, None if gp is None else gp.X,
                                None if gp is None else gp.theta)
    xe, ue = sc["xit"].copy(), sc["uit"].copy()
    r = emu.solve(cfg, sc["x0"], sc["yref"], sc["yref_e"], sc["alpha"], xe, ue, variant=variant, flavour=flavour)
    return sc, quad, dt, gp, cfg, keep, r, xe, ue


def _emu(cfg, r, sc, xe, ue, t, K, **kw):
    return jvp_ref.emu_jvp(cfg, r, xe, ue, sc["yref"], sc["yref_e"], n_dir=K, **t, **kw)


def _check_emulated(sc, quad, dt, gp, cfg, r, xe, ue, t, K, flavour=""):
    B, N = cfg.batch, cfg.n_nodes
    dx, du = _emu(cfg, r, sc, xe, ue, t, K, flavour=flavour)
    worst = 0.0
    for b in range(B):
        for d in range(K):
            tb = {n: (None if v is None else v[b, d]) for n, v in t.items()}
            odx, odu = reference(sc, b, quad, dt, N, gp, r["act"][b], xe[b], ue[b], tb)
            worst = max(worst, rel(dx[b, d], odx), rel(du[b, d], odu))
    assert worst < TOL64, worst
    return dx, du


@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("variant", [1, 2], ids=["warp_per_ocp", "screen_plus_dense"])
@pytest.mark.parametrize("N,use_gp", [(20, True), (20, False), (7, True), (7, False), (1, True), (1, False)])
def test_emulated_kernel_matches_reference(N, use_gp, variant, K):
    sc, quad, dt, gp, cfg, keep, r, xe, ue = _emulated_case(N, use_gp, variant)
    B = cfg.batch
    assert (r["status"] == 0).all()
    for b in range(B):                                  # the emulated solve ends on the oracle's solution
        xo, uo = oracle_solve(sc, b, quad, dt, N, gp)
        assert np.array_equal(r["act"][b], act_of(uo[None])[0]) and rel(ue[b], uo) < 1e-8
    rng = np.random.default_rng(N + 10 * variant + K)
    t = tangents(rng, (B, K), N)
    dx, du = _check_emulated(sc, quad, dt, gp, cfg, r, xe, ue, t, K)
    # every direction of a K-direction call is the one-direction call on it, bit for bit; dx NULL leaves du alone
    for d in range(K):
        one = _emu(cfg, r, sc, xe, ue, {n: (None if v is None else v[:, d]) for n, v in t.items()}, 1)
        assert np.array_equal(one[0][:, 0], dx[:, d]) and np.array_equal(one[1][:, 0], du[:, d])
    assert np.array_equal(_emu(cfg, r, sc, xe, ue, t, K, states=False)[1], du)
    # a NULL tangent is zero: the map is linear in the tangents
    sx, su = np.zeros_like(dx), np.zeros_like(du)
    for n in NAMES:
        px, pu = _emu(cfg, r, sc, xe, ue, {m: (t[m] if m == n else None) for m in NAMES}, K)
        sx, su = sx + px, su + pu
    assert rel(sx, dx) < 1e-12 and rel(su, du) < 1e-12


def test_emulated_kernel_without_tile_ring():
    """the A/B build flavour that reads the tiles in place with unpadded rows (QMPC_RING=0, QMPC_WR=16)"""
    N, K = 20, 3
    sc, quad, dt, gp, cfg, keep, r, xe, ue = _emulated_case(N, True, 1, seed=61, flavour="noring")
    t = tangents(np.random.default_rng(61), (3, K), N)
    _check_emulated(sc, quad, dt, gp, cfg, r, xe, ue, t, K, flavour="noring")


def test_emulated_unknown_active_set_gives_nan():
    N, B, K = 20, 3, 2
    dt = 1.0 / N
    quad = orc.quad_hummingbird()
    sc = random_ocp_batch(B, N, dt, quad, None, seed=78, amp_choices=(8.0,))
    cfg, keep = emu.make_config(B, N, 1.0, quad, orc.W_DIAG, orc.WE_DIAG)
    xe, ue = sc["xit"].copy(), sc["uit"].copy()
    r = emu.solve(cfg, sc["x0"], sc["yref"], sc["yref_e"], None, xe, ue, variant=1)
    assert (r["status"] == 0).all()
    t = tangents(np.random.default_rng(78), (B, K), N)
    ref = _emu(cfg, r, sc, xe, ue, t, K)
    r["act"][1, 17] = 255               # one unknown entry makes one vehicle unknown; its neighbours are unaffected
    out = _emu(cfg, r, sc, xe, ue, t, K)
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
    _set_yref(opt, sc["yref"], sc["yref_e"])
    if gp is not None:
        opt.set_rgp_params(torch.as_tensor(sc["mu"]))
    return opt


def _set_yref(opt, yref, yref_e):
    import torch
    from mpc_quad_ros_b200 import _capi
    y = torch.as_tensor(yref, device=opt.device).contiguous()
    ye = torch.as_tensor(yref_e, device=opt.device).contiguous()
    _capi.check(_capi.lib().qmpc_set_yref(opt._h, _capi.ptr(y), _capi.ptr(ye), _capi.stream_ptr()))


def _gpu_solve(opt, xit, uit, x0, act=None):
    import torch
    opt.set_iterate(torch.as_tensor(xit), torch.as_tensor(uit))
    if act is not None:
        opt.set_active_set(act)
    x, u, _, _ = opt.run_optimization(torch.as_tensor(x0, device=opt.device))
    return x, u


def _gpu_vs_reference(opt, sc, quad, dt, N, gp, t, K):
    """eval_jvp with K directions against rti_jvp per vehicle and direction, for the vehicles whose solve succeeded;
    returns the worst relative error"""
    x, u = (a.cpu().numpy() for a in opt.get_iterate())
    act = opt.get_active_set().cpu().numpy()
    dx, du = (a.cpu().numpy() for a in opt.eval_jvp(**t))
    worst = 0.0
    for b in np.flatnonzero(opt.solver_status()[0].cpu().numpy() == 0):
        for d in range(K):
            tb = {n: (None if v is None else v[b, d]) for n, v in t.items()}
            odx, odu = reference(sc, b, quad, dt, N, gp, act[b], x[b], u[b], tb)
            worst = max(worst, rel(dx[b, d], odx), rel(du[b, d], odu))
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [1, 2], ids=["warp_per_ocp", "screen_plus_dense"])
@pytest.mark.parametrize("N,M,seed", [(20, 20, 140), (10, 0, 110), (50, 20, 170), (21, 20, 21), (1, 0, 1)])
def test_gpu_jvp_vs_reference(N, M, seed, variant):
    if variant == 2 and N > 21:
        pytest.skip("the screening + dense solver serves N <= 21")
    B, K, dt = 48, 2, 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp(M) if M else None
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=seed)      # the scenarios of the eval_sens / eval_adjoint tests
    opt = _gpu_handle(sc, B, N, gp, solver_variant=variant)
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"])
    assert (opt.solver_status()[0].cpu().numpy() == 0).all()
    worst = _gpu_vs_reference(opt, sc, quad, dt, N, gp, tangents(np.random.default_rng(seed), (B, K), N), K)
    print(f"N={N} M={M} variant {variant}: worst rel err vs the reference {worst:.1e}")
    assert worst < TOL64, worst


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [1, 2], ids=["warp_per_ocp", "screen_plus_dense"])
def test_gpu_identities(variant):
    """the dot product with qmpc_eval_adjoint_weights, the x0 unit directions against qmpc_eval_sens_x0, scale invariance"""
    import torch
    B, N, M = 64, 20, 20
    gp = make_gp(M)
    sc = random_ocp_batch(B, N, 1.0 / N, orc.quad_hummingbird(), gp, seed=31)
    opt = _gpu_handle(sc, B, N, gp, solver_variant=variant)
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"])
    assert (opt.solver_status()[0] == 0).all()
    rng = np.random.default_rng(31)
    K = 3
    t = tangents(rng, (B, K), N)
    dx, du = (a.cpu().numpy() for a in opt.eval_jvp(**t))
    xb, ub = rng.standard_normal((B, N + 1, NX)), rng.standard_normal((B, N, NU))
    bars = [a.cpu().numpy() for a in opt.eval_adjoint(xb, ub, weights=True)]
    lhs = np.einsum("bkij,bij->bk", dx, xb) + np.einsum("bkij,bij->bk", du, ub)
    terms = np.stack([(bar.reshape(B, 1, -1) * t[n].reshape(B, K, -1)).sum(-1) for bar, n in zip(bars, NAMES)])
    w_dot = float((np.abs(lhs - terms.sum(0)) / (np.abs(terms).sum(0) + np.abs(lhs))).max())
    sx, su = (a.cpu().numpy() for a in opt.eval_sens())
    cx, cu = (a.cpu().numpy() for a in opt.eval_jvp(dx0=np.tile(np.eye(NX), (B, 1, 1))))
    w_col = max(rel(cx, np.moveaxis(sx, -1, 1)), rel(cu, np.moveaxis(su, -1, 1)))
    w = torch.as_tensor(np.diag(opt.W).copy())
    we = torch.as_tensor(np.diag(opt.W_e).copy())
    xs, us = (a.cpu().numpy() for a in opt.eval_jvp(dw=w))                   # [17]: shared by every vehicle
    xe, ue = (a.cpu().numpy() for a in opt.eval_jvp(dwe=we))
    both = [a.cpu().numpy() for a in opt.eval_jvp(dw=w, dwe=we)]
    scale = np.maximum(np.abs(xs).max(axis=(1, 2)), np.abs(us).max(axis=(1, 2)))
    w_scale = float((np.maximum(np.abs(both[0]).max(axis=(1, 2)), np.abs(both[1]).max(axis=(1, 2))) / scale).max())
    assert rel(both[0], xs + xe) < 1e-12 and rel(both[1], us + ue) < 1e-12
    print(f"variant {variant}: dot product {w_dot:.1e}, x0 columns {w_col:.1e}, scale identity {w_scale:.1e}")
    assert w_dot < 1e-11, w_dot
    assert w_col < 1e-12, w_col             # the same factorisation and the same forward algebra as qmpc_sens_kernel
    assert w_scale < 1e-8, w_scale          # exact for the exact minimiser; the solve is exact to ~1e-12 relative


@pytest.mark.gpu
@pytest.mark.parametrize("variant,tol", [(1, 1e-6), (2, 1e-4)], ids=["warp_per_ocp", "screen_plus_dense"])
def test_gpu_jvp_vs_central_differences_of_the_library(variant, tol):
    """no oracle: solves of the library itself from the same iterate and active set at reference / weights +- eps * d"""
    import torch
    B, N, M, eps = 48, 20, 20, 1e-4
    gp = make_gp(M)
    sc = random_ocp_batch(B, N, 1.0 / N, orc.quad_hummingbird(), gp, seed=910)
    opt = _gpu_handle(sc, B, N, gp, solver_variant=variant, reset_on_fail=-1)
    w0, we0 = np.diag(opt.W).copy(), np.diag(opt.W_e).copy()
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"])
    act0 = opt.get_active_set().clone()                  # injected before every solve below
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"], act=act0)
    rng = np.random.default_rng(911)
    dirs = [tangents(rng, (B,), N, p) for p in (("dyref", "dyref_e"), ("dw", "dwe"), ("dyref", "dyref_e", "dw", "dwe"))]
    for t in dirs:                                       # one weight direction for the whole batch: the handle shares them
        for n in ("dw", "dwe"):
            if t[n] is not None:
                t[n] = t[n][0]
    ads = [[a.cpu().numpy() for a in opt.eval_jvp(**t)] for t in dirs]
    acts, errs = [act0.cpu().numpy()], []
    for t, ad in zip(dirs, ads):
        sol = []
        for s in (1, -1):
            at = lambda base, n: base if t[n] is None else base + s * eps * t[n]
            _set_yref(opt, at(sc["yref"], "dyref"), at(sc["yref_e"], "dyref_e"))
            opt.set_weights(at(w0, "dw"), at(we0, "dwe"))
            x, u = _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"], act=act0)
            acts.append(opt.get_active_set().cpu().numpy())
            sol.append((x.cpu().numpy(), u.cpu().numpy()))
        fd = [(p - m) / (2 * eps) for p, m in zip(*sol)]
        errs.append([np.abs(f - a).max(axis=(1, 2)) / np.maximum(1.0, np.abs(a).max(axis=(1, 2))) for f, a in zip(fd, ad)])
    keep = np.array([all(np.array_equal(a[b], acts[0][b]) for a in acts) and (acts[0][b] <= 2).all() for b in range(B)])
    print(f"variant {variant}: {keep.sum()}/{B} vehicles keep their active set in all 7 solves")
    assert keep.mean() >= 0.75
    err = float(np.max([e[keep] for part in errs for e in part]))
    print(f"variant {variant}: rel err vs central differences {err:.1e}")
    assert err < tol


def _stable_subset(sc, B, N, gp, dev, w, we, eps, n_dirs=6):
    """a handle's solve of the scenario, and the vehicles whose active set survives +-eps in random directions of
    (x0, x_ref, u_ref, w, we) and in each direction's coordinate-wise worst case"""
    import torch
    opt = _gpu_handle(sc, B, N, gp, solver_variant=1, reset_on_fail=-1)
    x0 = torch.as_tensor(sc["x0"], device=dev)
    xr = torch.as_tensor(sc["yref"][..., :NX], device=dev).contiguous()
    ur = torch.as_tensor(sc["yref"][..., NX:], device=dev).contiguous()
    it = (torch.as_tensor(sc["xit"], device=dev), torch.as_tensor(sc["uit"], device=dev))
    opt.differentiable_step(x0, xr, ur, iterate=it)
    act0 = opt.get_active_set().clone()
    assert (opt.solver_status()[0] == 0).all() and (act0 <= 2).all()
    rng = np.random.default_rng(6)
    ok = np.ones(B, dtype=bool)
    for i in range(n_dirs):
        d = [torch.as_tensor(rng.standard_normal(t.shape), device=dev) for t in (x0, xr, ur, w, we)]
        if i % 2:
            d = [torch.sign(t) for t in d]
        for s in (1, -1):
            opt.set_active_set(act0)
            opt.differentiable_step(x0 + s * eps * d[0], xr + s * eps * d[1], ur + s * eps * d[2], iterate=it,
                                    w_diag=w + s * eps * d[3], we_diag=we + s * eps * d[4])
            ok &= (opt.get_active_set() == act0).all(1).cpu().numpy()
    return x0, xr, ur, it, act0, ok


@pytest.mark.gpu
def test_gpu_differentiable_step_gradcheck_forward_ad():
    import torch
    from mpc_quad_ros_b200.quad_opt import Q_DIAGONAL, R_COST
    Bc, B, N, M, eps = 8, 4, 10, 20, 1e-6
    gp = make_gp(M)
    sc = random_ocp_batch(Bc, N, 1.0 / N, orc.quad_hummingbird(), gp, seed=1000)   # as the backward gradcheck
    dev = torch.device("cuda:0")
    w = torch.as_tensor(np.concatenate([Q_DIAGONAL, R_COST]), device=dev)
    we = torch.as_tensor(Q_DIAGONAL, device=dev)
    x0, xr, ur, it, act0, stable = _stable_subset(sc, Bc, N, gp, dev, w, we, eps)
    idx = np.flatnonzero(stable)[:B]
    assert len(idx) == B, stable
    sub = {k: (None if v is None else v[idx]) for k, v in sc.items()}
    opts = [_gpu_handle(sub, B, N, gp, solver_variant=1, reset_on_fail=-1) for _ in range(2)]
    its = (it[0][idx].contiguous(), it[1][idx].contiguous())
    act = act0[idx].contiguous()
    calls = [0]

    def f(x0_, xr_, ur_, wd, wed):
        o = opts[min(calls[0], 1)]
        calls[0] += 1
        o.set_active_set(act)
        return o.differentiable_step(x0_, xr_, ur_, iterate=its, w_diag=wd, we_diag=wed)

    inputs = tuple(t.detach().clone().requires_grad_(True) for t in
                   (x0[idx].contiguous(), xr[idx].contiguous(), ur[idx].contiguous(), w, we))
    # the backward w.r.t. these inputs has gradchecks of its own (tests/test_adjoint*.py)
    assert torch.autograd.gradcheck(f, inputs, eps=eps, atol=1e-6, rtol=1e-4, check_undefined_grad=False,
                                    check_forward_ad=True, check_backward_ad=False)
    assert all((o.get_active_set() == act).all() for o in opts)


@pytest.mark.gpu
def test_gpu_func_jvp_and_dual_tensors_equal_eval_jvp():
    import torch
    import torch.autograd.forward_ad as fwAD
    B, N, M = 16, 20, 20
    gp = make_gp(M)
    sc = random_ocp_batch(B, N, 1.0 / N, orc.quad_hummingbird(), gp, seed=12)
    dev = torch.device("cuda:0")
    opt = _gpu_handle(sc, B, N, gp, solver_variant=1)
    prim = [torch.as_tensor(a, device=dev).contiguous() for a in
            (sc["x0"], sc["yref"][..., :NX], sc["yref"][..., NX:], np.diag(opt.W), np.diag(opt.W_e))]
    it = (torch.as_tensor(sc["xit"], device=dev), torch.as_tensor(sc["uit"], device=dev))
    rng = np.random.default_rng(12)
    tan = [torch.as_tensor(rng.standard_normal(p.shape), device=dev) for p in prim]
    tan[3], tan[4] = tan[3] * prim[3], tan[4] * prim[4]
    step = lambda *p: opt.differentiable_step(p[0], p[1], p[2], iterate=it, w_diag=p[3], we_diag=p[4])
    (x, u), (jx, ju) = torch.func.jvp(step, tuple(prim), tuple(tan))
    # the same solve (from the same cold start), then eval_jvp with the mapping written out: yref_e = x_ref[:, N-1]
    opt.reset_warm_start()
    step(*prim)
    assert torch.equal(opt.get_iterate()[0], x)
    dyref = torch.cat([tan[1], tan[2]], dim=2)
    ex, eu = opt.eval_jvp(dx0=tan[0], dyref=dyref, dyref_e=tan[1][:, N - 1], dw=tan[3], dwe=tan[4])
    assert torch.equal(jx, ex) and torch.equal(ju, eu)
    opt.reset_warm_start()
    with fwAD.dual_level():
        dual = [fwAD.make_dual(p, t) for p, t in zip(prim, tan)]
        ox, ou = step(*dual)
        fx, fu = fwAD.unpack_dual(ox).tangent, fwAD.unpack_dual(ou).tangent
    assert torch.equal(fx, ex) and torch.equal(fu, eu)
    # a tangent of x0 alone, u_ref None (the hover input, a constant): the x0 columns of eval_sens
    with fwAD.dual_level():
        ox, ou = opt.differentiable_step(fwAD.make_dual(prim[0], tan[0]), prim[1], iterate=it)
        fx = fwAD.unpack_dual(ox).tangent
    sx, _ = opt.eval_sens()
    assert rel(fx.cpu().numpy(), torch.einsum("bkij,bj->bki", sx, tan[0]).cpu().numpy()) < 1e-12


@pytest.mark.gpu
def test_gpu_iterate_tangent_is_refused():
    import torch
    import torch.autograd.forward_ad as fwAD
    B, N = 4, 10
    sc = random_ocp_batch(B, N, 1.0 / N, orc.quad_hummingbird(), None, seed=13)
    dev = torch.device("cuda:0")
    opt = _gpu_handle(sc, B, N, None)
    x0 = torch.as_tensor(sc["x0"], device=dev)
    xr = torch.as_tensor(sc["yref"][..., :NX], device=dev).contiguous()
    xit, uit = torch.as_tensor(sc["xit"], device=dev), torch.as_tensor(sc["uit"], device=dev)
    with fwAD.dual_level():
        with pytest.raises(ValueError, match="iterate"):
            opt.differentiable_step(x0, xr, iterate=(fwAD.make_dual(xit, torch.ones_like(xit)), uit))
    with pytest.raises(ValueError, match="iterate"):
        torch.func.jvp(lambda u_: opt.differentiable_step(x0, xr, iterate=(xit, u_))[1], (uit,), (torch.ones_like(uit),))


@pytest.mark.gpu
def test_gpu_jvp_has_no_side_effects():
    """a fused closed loop with an eval_jvp after every step is bit-identical to one without; the epoch stays"""
    import torch
    from mpc_quad_ros_b200.execute_trajectory import ClosedLoop
    from mpc_quad_ros_b200.trajectory import random_smooth_trajectories
    B, N, M, steps = 64, 20, 20, 8
    gp = make_gp(M)
    sc = random_ocp_batch(B, N, 1.0 / N, orc.quad_hummingbird(), gp, seed=14)
    traj = random_smooth_trajectories(B, steps + N + 2, 1.0 / N, seed=14)
    rng = np.random.default_rng(14)
    t = tangents(rng, (B, 3), N)
    runs = []
    for with_jvp in (False, True):
        opt = _gpu_handle(sc, B, N, gp)
        loop = ClosedLoop(opt.quad, opt, torch.as_tensor(traj), torch.as_tensor(traj[:, 0, :].copy()))
        outs = []
        for _ in range(steps):
            loop.step()
            if with_jvp:
                e0 = opt.sens_epoch()
                opt.eval_jvp(**t)
                assert opt.sens_epoch() == e0
            outs += [loop.u0.clone(), *opt.get_iterate(), opt.get_active_set(), *opt.solver_status()]
        runs.append(outs)
    same = lambda x, y: torch.equal(x, y) or bool(((x == y) | (x.isnan() & y.isnan())).all())
    assert all(same(a, b) for a, b in zip(*runs))


@pytest.mark.gpu
def test_gpu_argument_errors_launch_nothing():
    import torch
    from mpc_quad_ros_b200 import _capi
    N, B = 10, 4
    sc = random_ocp_batch(B, N, 1.0 / N, orc.quad_hummingbird(), None, seed=15)
    opt = _gpu_handle(sc, B, N, None, solver_variant=1)
    lib = _capi.lib()
    s, null = _capi.stream_ptr(), None
    dx0 = torch.zeros((B, 1, NX), dtype=torch.float64, device=opt.device)
    du = torch.empty((B, 1, N, NU), dtype=torch.float64, device=opt.device)
    P = _capi.ptr
    torch.cuda.synchronize()
    l0 = lib.qmpc_launch_count()
    with pytest.raises(_capi.QmpcError, match="no solve"):
        _capi.check(lib.qmpc_eval_jvp(opt._h, 1, P(dx0), null, null, null, null, null, P(du), s))
    assert lib.qmpc_launch_count() == l0
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"])
    torch.cuda.synchronize()
    l1 = lib.qmpc_launch_count()
    with pytest.raises(_capi.QmpcError, match="null handle"):
        _capi.check(lib.qmpc_eval_jvp(null, 1, P(dx0), null, null, null, null, null, P(du), s))
    for k in (0, -3):
        with pytest.raises(_capi.QmpcError, match="n_dir"):
            _capi.check(lib.qmpc_eval_jvp(opt._h, k, P(dx0), null, null, null, null, null, P(du), s))
    with pytest.raises(_capi.QmpcError, match="all NULL"):
        _capi.check(lib.qmpc_eval_jvp(opt._h, 1, null, null, null, null, null, null, P(du), s))
    with pytest.raises(_capi.QmpcError, match="du is NULL"):
        _capi.check(lib.qmpc_eval_jvp(opt._h, 1, P(dx0), null, null, null, null, null, null, s))
    with pytest.raises(_capi.QmpcError, match="all NULL"):
        opt.eval_jvp()
    with pytest.raises(ValueError, match="directions"):
        opt.eval_jvp(dx0=np.zeros((B, 2, NX)), dw=np.zeros((B, 3, NY)))
    assert lib.qmpc_launch_count() == l1
    _capi.check(lib.qmpc_eval_jvp(opt._h, 1, P(dx0), null, null, null, null, null, P(du), s))
    assert lib.qmpc_launch_count() == l1 + 1
    opt32 = _gpu_handle(sc, B, N, None, precision=32)
    _gpu_solve(opt32, sc["xit"], sc["uit"], sc["x0"])
    torch.cuda.synchronize()
    l2 = lib.qmpc_launch_count()
    with pytest.raises(_capi.QmpcError, match="fp64"):
        opt32.eval_jvp(dx0=dx0)
    assert lib.qmpc_launch_count() == l2


@pytest.mark.gpu
@pytest.mark.parametrize("N,K", [(1, 30), (256, 30), (256, 1)])
def test_gpu_size_envelope(N, K):
    """the shortest and the longest horizon the C-ABI accepts, up to 30 directions"""
    B, M, dt = 5, 20, 1.0 / N
    quad = orc.quad_hummingbird()
    gp = make_gp(M)
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=N + K)
    opt = _gpu_handle(sc, B, N, gp)
    _gpu_solve(opt, sc["xit"], sc["uit"], sc["x0"])
    assert (opt.solver_status()[0].cpu().numpy() == 0).sum() >= B - 1
    worst = _gpu_vs_reference(opt, sc, quad, dt, N, gp, tangents(np.random.default_rng(N + K), (B, K), N), K)
    print(f"N={N} K={K}: worst rel err vs the reference {worst:.1e}")
    assert worst < TOL64, worst
