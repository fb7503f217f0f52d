"""The RGP kernels (rgp_kernels.cuh) at every basis size where their launch changes shape.

regress_launch (capi.cu) runs the TMA-staged update with 8 warps per CTA for even M <= 24, 2 warps for even M <= 52 and
1 warp for even M <= 64, and the streaming kernel for odd M and for M > 64, whose lanes stride the basis RGP_MAXT = 4
times (M in 97..128 reaches the fourth stride).  predict, predict_cov and predict_using_y loop over the query points
inside one warp.  The RGP* learner keeps its state in shared memory up to M = 64; the shared-swarm accumulate picks
1..8 warps from its 200 KB tile and the shared apply takes M <= 118.

The reference here restates the formulas of RGP.py (regress :303-330, predict :195-229, predict_using_y :264-300) in
np.longdouble and is given the K_x^-1 the handle holds, so that what is measured is the kernels' own rounding."""
import numpy as np
import pytest

from oracle import oracle as orc
from conftest import rel_err

# Tolerance: with theta = (L, sigma_f, sigma_n) = (3, 0.1, 0.01) on [-10, 10], cond(K_x) <= 4.4e3 for M <= 128 (and
# |K_x^-1| <= 1e4).  A kernel's fp64 dot products of length M then lose at most about M * cond * 2^-53 ~ 1e-10 relative;
# TOL_RGP = 1e-9, the suite's RGP tolerance, leaves a factor of ten for the accumulation over 20 regress steps.
THETA = (3.0, 0.1, 0.01)
TOL_RGP = 1e-9
LD = np.longdouble
QMPC_ERR_ARG = -1

# The shared swarm is compared with a different computation, not with its own formulas in long double: one
# information-form update (C <- (C^-1 + sum j^T j / r)^-1 by Gauss-Jordan on I + C Lambda) against the oracle's B x 3
# sequential fp64 rank-1 updates.  Both carry their own rounding, the sequential one over up to 30 000 updates, so the
# bound is the suite's shared-swarm bound (test_shared_swarm_rgp_vs_sequential_oracle), 1e-8.  Measured on a B200 at a
# 1000 W power limit: <= 2.8e-12 at M <= 118 with B = 96, 4.5e-11 at B = 10007.
TOL_SHARED = 1e-8

M_DISPATCH = [1, 2, 24, 26, 31, 32, 33, 52, 54, 63, 64, 65, 96, 97, 127, 128]


# --------------------------------------------------------------------------------------- long double reference

def _k(a, b, theta):
    """RBF kernel sigma_f^2 exp(-1/2 (a-b)^2 / L^2) on the outer grid of a [..., p] and b [..., q] -> [..., p, q]"""
    L, sf = LD(theta[0]), LD(theta[1])
    e = np.asarray(a, dtype=LD)[..., :, None] - np.asarray(b, dtype=LD)[..., None, :]
    return sf * sf * np.exp(LD(-0.5) * e * (LD(1) / (L * L)) * e)


class RefRGP:
    """RGP.py's formulas for one 1-D model in long double: X [M], K_x^-1 [M, M] as the handle holds it, the state
    (mu = 0, C = K_x) starting from the handle's fp64 K_x"""

    def __init__(self, X, theta, Kx, Kx_inv):
        self.X, self.theta = np.asarray(X, dtype=LD), tuple(float(t) for t in theta)
        self.Ki = np.asarray(Kx_inv, dtype=LD)
        self.mu = np.zeros(self.X.shape[0], dtype=LD)
        self.C = np.asarray(Kx, dtype=LD).copy()

    def gain(self, xs):
        """Jt = k(xs, X) K_x^-1 [m, M]"""
        return _k(np.atleast_1d(xs), self.X, self.theta) @ self.Ki

    def regress(self, xt, yt):
        """single-sample RGP.regress (:303-330); a non-finite sample leaves the model as it is"""
        if not (np.isfinite(xt) and np.isfinite(yt)):
            return
        J = self.gain(xt)[0]
        b = _k([xt], [xt], self.theta)[0, 0] - J @ _k(self.X, [xt], self.theta)[:, 0]
        w = J @ self.C                       # Jt C
        cj = self.C @ J                      # C Jt^T
        s = b + w @ J + LD(self.theta[2]) ** 2
        g = cj / s
        self.mu = self.mu + g * (LD(yt) - J @ self.mu)
        self.C = self.C - np.outer(g, w)

    def predict(self, xs, y=None):
        """posterior mean and variance at xs (:195-210); with y: predict_using_y (:264-300), mean only"""
        J = self.gain(xs)
        mean = J @ (self.mu if y is None else np.asarray(y, dtype=LD))
        var = np.diag(self.cov(xs, J))
        return mean, var

    def cov(self, xs, J=None):
        """full posterior covariance K(xs,xs) - Jt K(X,xs) + Jt C Jt^T (predict(cov=True), :212-229)"""
        J = self.gain(xs) if J is None else J
        return _k(xs, xs, self.theta) - J @ _k(self.X, xs, self.theta) + J @ self.C @ J.T


def _grid(M):
    return np.linspace(-10.0, 10.0, M) if M > 1 else np.array([0.5])


@pytest.mark.parametrize("M", [1, 2, 33, 128])
def test_long_double_reference_matches_the_oracle(M):
    """the reference against the C oracle's rgp_regress / rgp_predict (fp64), same K_x^-1, 20 samples"""
    from mpc_quad_ros_b200.gp.RGP import prior
    X = _grid(M)
    Kx, Ki = prior(X, THETA)
    ref = RefRGP(X, THETA, Kx, Ki)
    mu, Cm = np.zeros(M), Kx.copy()
    rng = np.random.default_rng(M)
    th = np.array(THETA)
    for t in range(20):
        xt, yt = rng.uniform(-9, 9), rng.standard_normal()
        orc.rgp_regress(X, th, Ki, mu, Cm, xt, yt)
        ref.regress(xt, yt)
    xs = np.concatenate([rng.uniform(-11, 11, 32), [X[0], 12.0]])
    mean, var = orc.rgp_predict(X, th, Ki, mu, Cm, xs)
    rmean, rvar = ref.predict(xs)
    errs = (rel_err(mu, ref.mu.astype(np.float64)), rel_err(Cm, ref.C.astype(np.float64)),
            rel_err(mean, rmean.astype(np.float64)), np.abs(var - rvar.astype(np.float64)).max() / THETA[1] ** 2)
    print(f"M={M}: oracle vs long double: mu {errs[0]:.1e} C {errs[1]:.1e} mean {errs[2]:.1e} var {errs[3]:.1e}")
    assert max(errs) < 1e-10, errs


# ------------------------------------------------------------------------------------------------------------- GPU

def _ensemble(M, B):
    from mpc_quad_ros_b200.gp.GPE import GPEnsemble
    X = _grid(M)
    gpe = GPEnsemble.frombasisvectors([X] * 3, [np.zeros(M)] * 3, [None] * 3, [list(THETA)] * 3, batch=B)
    refs = [[RefRGP(X, THETA, gpe.K_x[d], gpe.K_x_inv[d]) for d in range(3)] for _ in range(B)]
    return gpe, refs


def _ref_state(refs):
    mu = np.array([[r.mu for r in rb] for rb in refs], dtype=LD)
    Cm = np.array([[r.C for r in rb] for rb in refs], dtype=LD)
    return mu, Cm


@pytest.mark.gpu
@pytest.mark.parametrize("M", M_DISPATCH)
def test_rgp_kernels_at_dispatch_boundaries(M):
    """B = 7 (21 models: a partly empty CTA in every warp count), 20 regress steps with NaN samples on some
    (vehicle, axis) pairs, then predict / predict_cov / predict_using_y at m = 1 and m = 33 query points"""
    import torch
    B, T = 7, 20
    gpe, refs = _ensemble(M, B)
    rng = np.random.default_rng(100 + M)
    worst = dict(mu=0.0, C=0.0, alpha=0.0)
    for t in range(T):
        xt, yt = rng.uniform(-9, 9, (B, 3)), rng.standard_normal((B, 3))
        skip = rng.uniform(size=(B, 3)) < 0.2
        skip[t % B, t % 3] = True
        xt[skip & (rng.uniform(size=(B, 3)) < 0.5)] = np.nan
        yt[skip & ~np.isnan(xt)] = np.nan
        mu0, C0 = gpe.mu_tensor().cpu().numpy(), gpe.C_tensor().cpu().numpy()
        mg, Cg = (a.cpu().numpy() for a in gpe.regress(torch.as_tensor(xt), torch.as_tensor(yt)))
        for b in range(B):
            for d in range(3):
                refs[b][d].regress(xt[b, d], yt[b, d])
        # a non-finite sample leaves its model untouched, bit for bit
        assert np.array_equal(mg[skip], mu0[skip]) and np.array_equal(Cg[skip], C0[skip]), t
        assert not np.array_equal(mg[~skip], mu0[~skip])
        mu_r, C_r = _ref_state(refs)
        worst["mu"] = max(worst["mu"], rel_err(mg, mu_r.astype(np.float64)))
        worst["C"] = max(worst["C"], rel_err(Cg, C_r.astype(np.float64)))
        # alpha = K_x^-1 mu, of the kernel's own mu (the product's rounding only)
        al = gpe.alpha_tensor().cpu().numpy()
        al_r = np.einsum("dij,bdj->bdi", np.asarray(gpe.K_x_inv, dtype=LD), mg.astype(LD)).astype(np.float64)
        worst["alpha"] = max(worst["alpha"], rel_err(al, al_r))
    for m in (1, 33):
        xs = rng.uniform(-11, 11, (B, 3, m))
        y = rng.standard_normal((B, 3, M))
        mean, var = (a.cpu().numpy() for a in gpe.predict_tensor(torch.as_tensor(xs).cuda(), want_var=True))
        Jt, cov = (a.cpu().numpy() for a in gpe.predict_cov_tensor(torch.as_tensor(xs).cuda()))
        puy = gpe.predict_using_y(torch.as_tensor(xs), torch.as_tensor(y)).cpu().numpy()
        r_mean, r_var, r_J, r_cov, r_puy = (np.empty(a.shape, dtype=LD) for a in (mean, var, Jt, cov, puy))
        for b in range(B):
            for d in range(3):
                r = refs[b][d]
                r_mean[b, d], r_var[b, d] = r.predict(xs[b, d])
                r_J[b, d] = r.gain(xs[b, d])
                r_cov[b, d] = r.cov(xs[b, d])
                r_puy[b, d] = r.predict(xs[b, d], y=y[b, d])[0]
        f = lambda a: a.astype(np.float64)
        # variances are differences of O(sigma_f^2) terms: measured against the prior variance sigma_f^2
        e = dict(mean=rel_err(mean, f(r_mean)), var=rel_err(var, f(r_var), floor=THETA[1] ** 2),
                 Jt=rel_err(Jt, f(r_J)), cov=rel_err(cov, f(r_cov), floor=THETA[1] ** 2), puy=rel_err(puy, f(r_puy)))
        for k, v in e.items():
            worst[k] = max(worst.get(k, 0.0), v)
        assert np.abs(cov - cov.transpose(0, 1, 3, 2)).max() < TOL_RGP * THETA[1] ** 2
        assert np.abs(np.diagonal(cov, axis1=2, axis2=3) - var).max() < TOL_RGP * THETA[1] ** 2
    print(f"M={M}: " + " ".join(f"{k} {v:.1e}" for k, v in worst.items()))
    assert max(worst.values()) < TOL_RGP, worst


@pytest.mark.gpu
@pytest.mark.parametrize("M", [1, 2, 33, 64])
def test_rgp_learner_vs_oracle(M):
    """qrgpl_learn (one CTA per model, state in shared memory up to M = 64) against the oracle's RGP.learn: 5 models,
    each fed its own 10 samples, every return value and the full state after the last one"""
    import torch
    from mpc_quad_ros_b200.gp.RGP import RGPLearner
    n, T = 5, 10
    X = _grid(M)
    lr = RGPLearner(X, theta=list(THETA), batch=n)
    # the oracle starts from the learner's own initial state (its K_x^-1 comes from the host-side Gauss-Jordan)
    st = [lr._state(k).cpu().numpy() for k in ("mu_g", "C_g", "mu_eta", "C_eta", "Kx_inv")]
    mu_g, C_g, mu_eta, C_eta, Kx_inv = (np.ascontiguousarray(a) for a in st)
    assert (mu_g == 0).all() and np.array_equal(mu_eta, np.tile(THETA, (n, 1)))
    C_g_eta = np.zeros((M, 3))
    rng = np.random.default_rng(200 + M)
    worst = 0.0
    for t in range(T):
        xt = rng.uniform(-9, 9, n)
        yt = 0.3 * np.sin(0.4 * xt) + 0.01 * rng.standard_normal(n)
        mu_z, C_z = (a.cpu().numpy() for a in lr.learn(torch.as_tensor(xt), torch.as_tensor(yt)))
        assert (lr.status().cpu().numpy() == 0).all(), t
        for b in range(n):
            oz, oC = orc.rgp_learn(X, mu_g[b], C_g[b], mu_eta[b], C_eta[b], C_g_eta, Kx_inv[b], xt[b], yt[b])
            worst = max(worst, rel_err(mu_z[b], oz), rel_err(C_z[b], oC))
    fin = [lr._state(k).cpu().numpy() for k in ("mu_g", "C_g", "mu_eta", "C_eta", "Kx_inv")]
    es = [rel_err(a, o) for a, o in zip(fin, (mu_g, C_g, mu_eta, C_eta, Kx_inv))]
    print(f"M={M}: learn mu_z / C_z {worst:.1e}; state mu_g {es[0]:.1e} C_g {es[1]:.1e} mu_eta {es[2]:.1e} "
          f"C_eta {es[3]:.1e} Kx_inv {es[4]:.1e}")
    assert worst < TOL_RGP and max(es) < TOL_RGP, (worst, es)


def _shared_model(M):
    from mpc_quad_ros_b200.gp.GPE import GPEnsemble
    import torch
    X = _grid(M)
    gpe = GPEnsemble.frombasisvectors([X] * 3, [np.zeros(M)] * 3, [None] * 3, [list(THETA)] * 3, batch=1)
    info = torch.zeros((3, M * M + M), dtype=torch.float64, device="cuda:0")
    return gpe, X, info


def _shared_update(gpe, info, xt, yt):
    import torch
    from mpc_quad_ros_b200 import _capi
    lib, s = _capi.lib(), _capi.stream_ptr()
    xt, yt = torch.as_tensor(xt, device="cuda:0").contiguous(), torch.as_tensor(yt, device="cuda:0").contiguous()
    _capi.check(lib.qrgp_shared_accumulate(gpe._h, xt.shape[0], _capi.ptr(xt), _capi.ptr(yt), _capi.ptr(info), s))
    return lib.qrgp_shared_apply(gpe._h, _capi.ptr(info), s)


def _sequential(X, Kx_inv, mu, Cm, xt, yt):
    th = np.array(THETA)
    for v in range(xt.shape[0]):
        for d in range(3):
            if np.isfinite(xt[v, d]) and np.isfinite(yt[v, d]):
                orc.rgp_regress(X, th, Kx_inv[d], mu[d], Cm[d], xt[v, d], yt[v, d])


@pytest.mark.gpu
@pytest.mark.parametrize("M,B,rounds", [(64, 96, 3), (100, 96, 3), (118, 96, 3), (20, 10007, 1)])
def test_shared_swarm_vs_sequential_oracle(M, B, rounds):
    """one information-form update over B vehicles equals the oracle's sequential single-sample regress over all of
    them.  M = 64 / 100 / 118 run the accumulate with 5 / 2 / 1 warps per CTA, 118 is the largest apply tile;
    B = 10007 at M = 20 is more vehicles than the 148 CTAs x 8 warps x 8 of the strided vehicle loop cover in one pass"""
    gpe, X, info = _shared_model(M)
    rng = np.random.default_rng(300 + M)
    mu = np.zeros((3, M))
    Cm = np.ascontiguousarray(gpe.K_x.copy())
    for _ in range(rounds):
        xt = rng.uniform(-9, 9, (B, 3))
        yt = -0.3 * xt + 0.02 * rng.standard_normal((B, 3))
        xt[3, 1] = np.nan                                       # a non-finite residual is left out, not summed
        assert _shared_update(gpe, info, xt, yt) == 0
        _sequential(X, gpe.K_x_inv, mu, Cm, xt, yt)
        e_mu, e_C = rel_err(gpe.mu_tensor()[0].cpu().numpy(), mu), rel_err(gpe.C_tensor()[0].cpu().numpy(), Cm)
        print(f"shared M={M} B={B}: mu {e_mu:.1e} C {e_C:.1e}")
        assert e_mu < TOL_SHARED and e_C < TOL_SHARED, (e_mu, e_C)
    al = gpe.alpha_tensor()[0].cpu().numpy()
    assert rel_err(al, np.einsum("dij,dj->di", np.asarray(gpe.K_x_inv, dtype=LD), gpe.mu_tensor()[0].cpu().numpy().astype(LD)).astype(np.float64)) < TOL_RGP


@pytest.mark.gpu
def test_shared_apply_refuses_basis_beyond_its_tile():
    """M = 119 needs M (2M + 1) doubles = 222 KB for the apply tile: QMPC_ERR_ARG, nothing launched, model unchanged"""
    import torch
    from mpc_quad_ros_b200 import _capi
    M = 119
    gpe, X, info = _shared_model(M)
    lib = _capi.lib()
    rng = np.random.default_rng(119)
    xt = torch.as_tensor(rng.uniform(-9, 9, (32, 3)), device="cuda:0")
    yt = torch.as_tensor(rng.standard_normal((32, 3)), device="cuda:0")
    _capi.check(lib.qrgp_shared_accumulate(gpe._h, 32, _capi.ptr(xt), _capi.ptr(yt), _capi.ptr(info), _capi.stream_ptr()))
    torch.cuda.synchronize()
    assert torch.isfinite(info).all() and (info != 0).any()
    mu0, C0 = gpe.mu_tensor(), gpe.C_tensor()
    l0 = lib.qmpc_launch_count()
    assert lib.qrgp_shared_apply(gpe._h, _capi.ptr(info), _capi.stream_ptr()) == QMPC_ERR_ARG
    assert "shared apply tile" in lib.qmpc_last_error().decode()
    assert lib.qmpc_launch_count() == l0
    assert torch.equal(gpe.mu_tensor(), mu0) and torch.equal(gpe.C_tensor(), C0)
