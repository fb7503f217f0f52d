"""The solver and its derivatives over the whole size range qmpc_create accepts (n_nodes 1..256, n_basis 0..128).

The other suites stop at N = 50 and M = 100.  The sizes here are where the kernels change shape: the per-CTA shared
memory of the Riccati kernel (ipm_smem_reals, host_params.h) grows with N and first goes over 48 KB at N = 82 for fp64
handles, at N = 120 for fp32 handles (they also carry the fp64 refinement scratch) and at N = 143 for the screening
layout that qmpc_sens_kernel and qmpc_adjoint_kernel use; at N = 256 an fp64 solve takes 140 KB per CTA and the TMA tile
ring cycles its mbarrier phases over 256 stages.  n_basis = 128 is the largest GP the linearisation accepts.

Every case is compared with the exact CPU oracle (oracle/qmpc_oracle.c) and, for the derivatives, with the references of
tests/sens.  The lane emulation of tests/emu runs a subset of the same cases on the CPU."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as orc
from helpers import make_gp, oracle_solve_batch, random_ocp_batch, u_rel, x_rel
from emu import emu
from sens import adjoint_ref, sens_ref

TOL_EXACT = 1e-7      # the solver ends on an exact KKT point: the Riccati path's bound in test_solve_fp64_vs_oracle
TOL_F32 = 1e-4        # fp32 handles: north_star tolerance of test_fp32_solver_within_1e4_of_oracle
TOL_SENS = 1e-9       # kernel vs reference, fp64: two exact routes to the same linear map (test_gpu_sens_vs_oracle)
NX, NU = 13, 4
QMPC_ERR_ARG = -1
FP32_MAX_NODES = 64   # QMPC_FP32_MAX_NODES (include/qmpc.h)

HORIZONS = [64, 81, 82, 119, 120, 128, 200, 256]


def rel(a, ref):
    """max|a - ref| / max(1, max|ref|)"""
    return float(np.abs(a - ref).max() / max(1.0, np.abs(ref).max()))


def act_of(u, lb=0.0, ub=1.0):
    """active set implied by an exact solution: an input is pinned when it equals a bound"""
    u = u.reshape(u.shape[0], -1)
    return np.where(u == lb, 1, np.where(u == ub, 2, 0)).astype(np.uint8)


def n_active(uo):
    return int(((uo < 1e-9) | (uo > 1 - 1e-9)).sum())


def scenario(B, N, M, t_horizon, seed, scattered=False, dup=None):
    """random_ocp_batch at dt = t_horizon / N; dup = (src, dst) copies vehicle src over vehicle dst"""
    dt = t_horizon / N
    quad = orc.quad_hummingbird()
    gp = None
    if M and scattered:
        X = np.sort(np.random.default_rng(M + N).uniform(-10, 10, (3, M)), axis=1)
        gp = orc.GPSpec(X, np.array((3.0, 0.1, 0.01)))
    elif M:
        gp = make_gp(M)
    sc = random_ocp_batch(B, N, dt, quad, gp, seed=seed)
    if dup is not None:
        for k, v in sc.items():
            if v is not None:
                v[dup[1]] = v[dup[0]]
    return sc, quad, dt, gp


# ------------------------------------------------------------------------------------------------------------- GPU

def _handle(sc, B, N, gp, t_horizon, precision=64, **policy):
    """quad_optimizer with the scenario's reference, alpha and iterate loaded.  alpha goes in as it is (qmpc_set_alpha),
    so that the handle and the oracle use the same GP weights and only the solver is compared."""
    import torch
    from mpc_quad_ros_b200 import _capi
    from mpc_quad_ros_b200.gp.GPE import GPEnsemble
    from mpc_quad_ros_b200.quad import Quadrotor3D
    from mpc_quad_ros_b200.quad_opt import quad_optimizer
    quad = Quadrotor3D(drag=True, batch=B).set_hummingbird_params()
    gpe = None
    if gp is not None:
        gpe = GPEnsemble.frombasisvectors([gp.X[d] for d in range(3)], [np.zeros(gp.M)] * 3, [None] * 3,
                                          [list(gp.theta[d]) for d in range(3)], batch=B)
    opt = quad_optimizer(quad, t_horizon=t_horizon, n_nodes=N, gpe=gpe, precision=precision, **policy)
    dev = opt.device
    s = _capi.stream_ptr()
    yref = torch.as_tensor(sc["yref"], device=dev).contiguous()
    yref_e = torch.as_tensor(sc["yref_e"], device=dev).contiguous()
    _capi.check(_capi.lib().qmpc_set_yref(opt._h, _capi.ptr(yref), _capi.ptr(yref_e), s))
    if gp is not None:
        alpha = torch.as_tensor(sc["alpha"], device=dev).contiguous()
        _capi.check(_capi.lib().qmpc_set_alpha(opt._h, _capi.ptr(alpha), s))
    opt.set_iterate(torch.as_tensor(sc["xit"]), torch.as_tensor(sc["uit"]))
    return opt


def _solve(sc, B, N, gp, t_horizon, precision=64, **policy):
    import torch
    opt = _handle(sc, B, N, gp, t_horizon, precision, **policy)
    x, u, _, cost = opt.run_optimization(torch.as_tensor(sc["x0"], device=opt.device))
    st, it = opt.solver_status()
    return opt, x.cpu().numpy(), u.cpu().numpy(), cost.cpu().numpy(), st.cpu().numpy(), it.cpu().numpy()


def _long_cases(horizons=HORIZONS):
    for N in horizons:
        for M in (0, 20):
            for th in ("1s", "10ms"):
                yield pytest.param(N, M, th, id=f"N{N}-M{M}-dt_{th}")


def _t_horizon(N, th):
    return 1.0 if th == "1s" else 0.01 * N


@pytest.mark.gpu
@pytest.mark.parametrize("N,M,th", list(_long_cases()))
def test_long_horizon_fp64_vs_oracle(N, M, th):
    """B = 37 is not a multiple of the 32 nodes of a linearisation block; vehicle 5 is repeated as vehicle 36, which sits
    in another CTA; two fresh handles solving the same batch must agree bit for bit"""
    B, t_horizon = 37, _t_horizon(N, th)
    sc, quad, dt, gp = scenario(B, N, M, t_horizon, seed=1000 + N + M, dup=(5, 36))
    _, x, u, cost, st, it = _solve(sc, B, N, gp, t_horizon)
    xo, uo, co, ito = oracle_solve_batch(sc, quad, dt, N, gp)
    assert (st == 0).all(), st
    eu, ex = u_rel(u, uo), x_rel(x, xo)
    print(f"fp64 N={N} M={M} dt={dt:.4f}: u_rel={eu:.2e} x_rel={ex:.2e} cost {np.abs(cost - co).max():.1e} "
          f"active inputs {n_active(uo)}")
    assert ((u >= 0) & (u <= 1)).all()
    assert np.abs(x[:, 0] - sc["x0"]).max() == 0.0
    assert n_active(uo) > 0                                   # the batch does exercise active thrust limits
    assert np.array_equal(u[5], u[36]) and np.array_equal(x[5], x[36]) and cost[5] == cost[36]
    _, x2, u2, cost2, st2, _ = _solve(sc, B, N, gp, t_horizon)
    assert np.array_equal(u, u2) and np.array_equal(x, x2) and np.array_equal(cost, cost2) and np.array_equal(st, st2)
    assert eu < TOL_EXACT and ex < TOL_EXACT, (eu, ex)
    assert np.abs(cost - co).max() < TOL_EXACT * max(1.0, np.abs(co).max())


@pytest.mark.gpu
@pytest.mark.parametrize("N,M,th", list(_long_cases([N for N in HORIZONS if N <= FP32_MAX_NODES])))
def test_long_horizon_fp32_vs_oracle(N, M, th):
    """the longest horizon an fp32 handle accepts; longer ones are refused (test_create_refuses_sizes_outside_the_envelope)"""
    B, t_horizon = 37, _t_horizon(N, th)
    sc, quad, dt, gp = scenario(B, N, M, t_horizon, seed=1000 + N + M, dup=(5, 36))
    _, x, u, cost, st, it = _solve(sc, B, N, gp, t_horizon, precision=32)
    xo, uo, co, ito = oracle_solve_batch(sc, quad, dt, N, gp)
    ok = st == 0
    eu, ex = u_rel(u[ok], uo[ok]), x_rel(x[ok], xo[ok])
    print(f"fp32 N={N} M={M} dt={dt:.4f}: u_rel={eu:.2e} x_rel={ex:.2e} status={np.bincount(st)}")
    assert np.isfinite(u).all() and ((u >= 0) & (u <= 1)).all()
    assert ok.mean() >= 0.95, np.bincount(st)
    assert eu < TOL_F32 and ex < TOL_F32, (eu, ex)
    assert np.array_equal(u[5], u[36]) and np.array_equal(x[5], x[36])
    _, x2, u2, _, st2, _ = _solve(sc, B, N, gp, t_horizon, precision=32)
    assert np.array_equal(u, u2) and np.array_equal(x, x2) and np.array_equal(st, st2)


def _cotangents(rng, B, N):
    return rng.standard_normal((B, N + 1, NX)), rng.standard_normal((B, N, NU))


def _transpose_of_sens(sx, su, xb, ub):
    return np.einsum("kij,ki->j", sx, xb) + np.einsum("kij,ki->j", su, ub)


@pytest.mark.gpu
@pytest.mark.parametrize("N,M,t_horizon", [(128, 20, 1.0), (128, 0, 1.28), (143, 20, 1.43), (143, 0, 1.0),
                                           (256, 20, 1.0), (256, 0, 2.56)])
def test_long_horizon_sens_and_adjoint_vs_oracle(N, M, t_horizon):
    """qmpc_eval_sens_x0 with n_stages = N and 1, and qmpc_eval_adjoint with every cotangent, against the references of
    tests/sens and against each other.  B = 12: sens_x at N = 256 is 347 KB per vehicle."""
    B = 12
    sc, quad, dt, gp = scenario(B, N, M, t_horizon, seed=2000 + N + M)
    opt, x, u, _, st, _ = _solve(sc, B, N, gp, t_horizon)
    assert (st == 0).all(), st
    sx, su = (t.cpu().numpy() for t in opt.eval_sens(N))
    sx1, su1 = (t.cpu().numpy() for t in opt.eval_sens(1))
    xbs, ubs = _cotangents(np.random.default_rng(N + M), B, N)
    x0b, yb, yeb = (t.cpu().numpy() for t in opt.eval_adjoint(xbs, ubs))
    act = opt.get_active_set().cpu().numpy()
    assert np.array_equal(sx1, sx[:, :2]) and np.array_equal(su1, su[:, :1])
    worst_s = worst_a = worst_t = 0.0
    for b in range(B):
        xo, uo, _, _ = oracle_solve_batch(sc, quad, dt, N, gp, idx=[b])
        assert np.array_equal(act[b], act_of(uo)[0]), b
        kw = dict(gp=gp, alpha=None if gp is None else sc["alpha"][b])
        ox, ou = sens_ref.rti_sens(quad, dt, N, sc["xit"][b], sc["uit"][b], act[b], **kw)
        ox1, ou1 = sens_ref.rti_sens(quad, dt, N, sc["xit"][b], sc["uit"][b], act[b], n_stages=1, **kw)
        worst_s = max(worst_s, rel(sx[b], ox), rel(su[b], ou), rel(sx1[b], ox1), rel(su1[b], ou1))
        assert (su[b].reshape(4 * N, 13)[act[b] != 0] == 0).all()
        ax0, ay, aye = adjoint_ref.rti_adjoint(quad, dt, N, sc["xit"][b], sc["uit"][b], act[b], x_bar=xbs[b],
                                               u_bar=ubs[b], **kw)
        worst_a = max(worst_a, rel(x0b[b], ax0), rel(yb[b], ay), rel(yeb[b], aye))
        worst_t = max(worst_t, rel(x0b[b], _transpose_of_sens(sx[b], su[b], xbs[b], ubs[b])))
        assert (yb[b, :, NX:].reshape(-1)[act[b] != 0] == 0).all()
    assert (yb[:, 0, :NX] == 0).all()
    assert np.array_equal(sx[:, 0], np.broadcast_to(np.eye(13), (B, 13, 13)))
    print(f"N={N} M={M} dt={dt:.4f}: sens {worst_s:.1e}, adjoint {worst_a:.1e}, adjoint vs eval_sens^T {worst_t:.1e}, "
          f"active inputs {int((act != 0).sum())}")
    assert worst_s < TOL_SENS and worst_a < TOL_SENS and worst_t < TOL_SENS, (worst_s, worst_a, worst_t)
    # one cotangent at a time: linear in the cotangents, and each half against the reference
    x0x, yx, yex = (t.cpu().numpy() for t in opt.eval_adjoint(x_bar=xbs))
    x0u, yu, yeu = (t.cpu().numpy() for t in opt.eval_adjoint(u_bar=ubs))
    assert rel(x0x + x0u, x0b) < 1e-12 and rel(yx + yu, yb) < 1e-12 and rel(yex + yeu, yeb) < 1e-12
    for b in (0, B - 1):
        kw = dict(gp=gp, alpha=None if gp is None else sc["alpha"][b])
        ref = adjoint_ref.rti_adjoint(quad, dt, N, sc["xit"][b], sc["uit"][b], act[b], u_bar=ubs[b], **kw)
        assert max(rel(x0u[b], ref[0]), rel(yu[b], ref[1]), rel(yeu[b], ref[2])) < TOL_SENS


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["equispaced", "scattered"])
@pytest.mark.parametrize("N", [20, 64])
def test_largest_gp_basis_vs_oracle(N, layout):
    """n_basis = 128 in the linearisation: an equispaced grid takes the recurrence of three exps, scattered points the
    general path (K1 in mpc_kernels.cuh).  N = 20 runs the screening + dense mapping, N = 64 the Riccati kernel alone."""
    B, t_horizon = 37, 1.0
    sc, quad, dt, gp = scenario(B, N, 128, t_horizon, seed=3000 + N, scattered=layout == "scattered")
    _, x, u, cost, st, _ = _solve(sc, B, N, gp, t_horizon)
    xo, uo, co, _ = oracle_solve_batch(sc, quad, dt, N, gp)
    assert (st == 0).all(), st
    eu, ex = u_rel(u, uo), x_rel(x, xo)
    assert eu < TOL_EXACT and ex < TOL_EXACT, (eu, ex)
    assert np.abs(cost - co).max() < TOL_EXACT * max(1.0, np.abs(co).max())
    # the GP term does matter in these problems: the nominal model gives a different answer
    _, xn, un, _, _, _ = _solve(sc, B, N, None, t_horizon)
    print(f"M=128 {layout} N={N}: u_rel={eu:.2e} x_rel={ex:.2e}; nominal model differs by {u_rel(un, uo):.2e}")
    assert u_rel(un, uo) > 1e-5, u_rel(un, uo)


def _config(N, M, precision=64):
    """a valid qmpc_config (hummingbird, reference weights) with n_nodes = N, n_basis = M"""
    from mpc_quad_ros_b200._capi import QmpcConfig
    from mpc_quad_ros_b200.quad_opt import Q_DIAGONAL, R_COST
    c = QmpcConfig()
    c.batch, c.n_nodes, c.n_basis, c.precision, c.t_horizon = 4, N, M, precision, 1.0
    c.quad[:] = list(orc.quad_hummingbird())
    c.w_diag[:] = list(np.concatenate((Q_DIAGONAL, R_COST)))
    c.we_diag[:] = list(Q_DIAGONAL)
    c.lbu, c.ubu = 0.0, 1.0
    X = np.ascontiguousarray(np.tile(np.linspace(-10, 10, max(M, 1)), (3, 1)))
    c.gp_theta[:] = [3.0, 0.1, 0.01] * 3
    c.gp_X = X.ctypes.data_as(C.POINTER(C.c_double))
    return c, X


@pytest.mark.parametrize("N,M,precision,what", [(257, 20, 64, "n_nodes"), (0, 20, 64, "n_nodes"), (256, 129, 64, "n_basis"),
                                                (20, -1, 64, "n_basis")] +
                         [(N, M, 32, "fp32") for N in HORIZONS + [FP32_MAX_NODES + 1] if N > FP32_MAX_NODES for M in (0, 20)])
def test_create_refuses_sizes_outside_the_envelope(N, M, precision, what):
    """qmpc_create checks its sizes before it touches the device: QMPC_ERR_ARG, no handle, nothing launched.  fp32 handles
    stop at QMPC_FP32_MAX_NODES: past it their controls end up to 2.5e-2 off the exact minimiser (include/qmpc.h)"""
    from mpc_quad_ros_b200 import _capi
    lib = _capi.lib()
    cfg, keep = _config(N, M, precision)
    h = C.c_void_p()
    l0 = lib.qmpc_launch_count()
    assert lib.qmpc_create(C.byref(cfg), C.byref(h)) == QMPC_ERR_ARG
    assert not h.value and lib.qmpc_launch_count() == l0
    assert what in lib.qmpc_last_error().decode()


@pytest.mark.parametrize("M", [65, 0])
def test_learner_create_refuses_basis_outside_its_tile(M):
    """the RGP* learner keeps its (M+4)^2 joint covariance and an M x 2M tableau in shared memory: n_basis <= 64"""
    from mpc_quad_ros_b200 import _capi
    lib = _capi.lib()
    X = np.linspace(-10, 10, max(M, 1))
    th = np.array([3.0, 0.1, 0.01])
    h = C.c_void_p()
    l0 = lib.qmpc_launch_count()
    rc = lib.qrgpl_create(5, M, X.ctypes.data_as(C.c_void_p), th.ctypes.data_as(C.c_void_p), 0, C.byref(h))
    assert rc == QMPC_ERR_ARG and not h.value and lib.qmpc_launch_count() == l0
    assert "n_basis" in lib.qmpc_last_error().decode()


# ------------------------------------------------------------------------------------------------------------- CPU
# The same kernels under the lane emulation of tests/emu (B = 2; an emulated solve at these sizes takes seconds).

def _emulated(N, M, t_horizon, seed, f32=False, flavour=""):
    B = 2
    sc, quad, dt, gp = scenario(B, N, M, t_horizon, seed=seed)
    cfg, keep = emu.make_config(B, N, t_horizon, quad, orc.W_DIAG, orc.WE_DIAG, None if gp is None else gp.X,
                                None if gp is None else gp.theta)
    xe, ue = sc["xit"].copy(), sc["uit"].copy()
    r = emu.solve(cfg, sc["x0"], sc["yref"], sc["yref_e"], sc["alpha"], xe, ue, f32=f32, variant=1, flavour=flavour)
    xo, uo, co, _ = oracle_solve_batch(sc, quad, dt, N, gp)
    return sc, quad, dt, gp, cfg, keep, r, xe, ue, xo, uo


@pytest.mark.parametrize("N,M,t_horizon,f32,flavour", [
    pytest.param(82, 20, 1.0, False, "", id="fp64-N82-M20"),
    pytest.param(128, 20, 1.28, False, "", id="fp64-N128-M20"),
    pytest.param(64, 0, 1.0, True, "", id="fp32-N64-M0"),
    pytest.param(128, 20, 1.0, False, "noring", id="noring-N128-M20")])
def test_emulated_long_horizon_vs_oracle(N, M, t_horizon, f32, flavour):
    sc, quad, dt, gp, cfg, keep, r, xe, ue, xo, uo = _emulated(N, M, t_horizon, 4000 + N + M, f32, flavour)
    assert (r["status"] == 0).all(), r["status"]
    eu, ex = u_rel(ue, uo), x_rel(xe, xo)
    print(f"emulated {'fp32' if f32 else 'fp64'} {flavour} N={N} M={M}: u_rel={eu:.2e} x_rel={ex:.2e} "
          f"active inputs {n_active(uo)}")
    tol = TOL_F32 if f32 else TOL_EXACT
    assert eu < tol and ex < tol, (eu, ex)
    assert np.abs(xe[:, 0] - sc["x0"]).max() == 0.0 and ((ue >= 0) & (ue <= 1)).all()
    assert n_active(uo) > 0
    if not f32:
        assert np.array_equal(r["act"], act_of(uo))


def test_emulated_rounds_retried_from_the_converged_ipm_point():
    """N = 256, dt = 1/256: vehicles 16 and 19 of test_long_horizon_fp64_vs_oracle[N256-M0-dt_1s].  Their active-set rounds
    do not settle within the two attempts during the IPM (40 rounds); the IPM point at ipm_mu_tol was then returned with
    status 0 although its controls were 3.4e-4 and 4.4e-5 off the minimiser.  The rounds now run once more from that
    point and settle, so both vehicles end on the exact minimiser; a point that still does not settle is flagged MAXITER."""
    N, t_horizon = 256, 1.0
    sc, quad, dt, gp = scenario(37, N, 0, t_horizon, seed=1000 + N, dup=(5, 36))
    sub = {k: (None if v is None else np.ascontiguousarray(v[[16, 19]])) for k, v in sc.items()}
    cfg, keep = emu.make_config(2, N, t_horizon, quad, orc.W_DIAG, orc.WE_DIAG)
    xe, ue = sub["xit"].copy(), sub["uit"].copy()
    r = emu.solve(cfg, sub["x0"], sub["yref"], sub["yref_e"], None, xe, ue, variant=1)
    xo, uo, co, _ = oracle_solve_batch(sub, quad, dt, N, None)
    print(f"emulated N={N}: status {r['status']}, rounds {r['rounds']}, u_rel {u_rel(ue, uo):.2e}")
    assert (r["rounds"] > 40).all()                       # the case still needs the retry
    assert (r["status"] == 0).all(), r["status"]
    assert u_rel(ue, uo) < TOL_EXACT and x_rel(xe, xo) < TOL_EXACT, (u_rel(ue, uo), x_rel(xe, xo))
    assert np.array_equal(r["act"], act_of(uo))


def test_emulated_sens_and_adjoint_at_screening_smem_boundary():
    """N = 143: the first horizon whose screening layout (the one of the sensitivity kernels) needs more than 48 KB"""
    N, M = 143, 20
    sc, quad, dt, gp, cfg, keep, r, xe, ue, xo, uo = _emulated(N, M, 1.0, 4143)
    assert (r["status"] == 0).all()
    sx, su = sens_ref.emu_sens(cfg, r, N)
    sx1, su1 = sens_ref.emu_sens(cfg, r, 1)
    xbs, ubs = _cotangents(np.random.default_rng(143), 2, N)
    x0b, yb, yeb = adjoint_ref.emu_adjoint(cfg, r, xbs, ubs)
    worst_s = worst_a = 0.0
    for b in range(2):
        act = r["act"][b]
        assert np.array_equal(act, act_of(uo[b:b + 1])[0])
        kw = dict(gp=gp, alpha=sc["alpha"][b])
        ox, ou = sens_ref.rti_sens(quad, dt, N, sc["xit"][b], sc["uit"][b], act, **kw)
        worst_s = max(worst_s, rel(sx[b], ox), rel(su[b], ou))
        ax0, ay, aye = adjoint_ref.rti_adjoint(quad, dt, N, sc["xit"][b], sc["uit"][b], act, x_bar=xbs[b], u_bar=ubs[b],
                                               **kw)
        worst_a = max(worst_a, rel(x0b[b], ax0), rel(yb[b], ay), rel(yeb[b], aye),
                      rel(x0b[b], _transpose_of_sens(sx[b], su[b], xbs[b], ubs[b])))
    print(f"emulated N={N} M={M}: sens {worst_s:.1e}, adjoint {worst_a:.1e}, active inputs {int((r['act'] != 0).sum())}")
    assert worst_s < TOL_SENS and worst_a < TOL_SENS, (worst_s, worst_a)
    assert np.array_equal(sx1, sx[:, :2]) and np.array_equal(su1, su[:, :1])
