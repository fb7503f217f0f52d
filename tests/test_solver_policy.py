"""The solver's status-0 contract under every policy knob, non-default input boxes and any warm-start state.

include/qmpc.h promises that QMPC_STATUS_OK means the exact active set was verified (refine_max_rounds < 0: the IPM
reached ipm_mu_tol), that the policy fields of qmpc_config steer the path a solve takes but not its answer, and that
the remembered active sets (qmpc_set_active_set) never change the answer either.  Every case here runs two consecutive
solves, a cold one and a second one from the first's iterate and active set with a perturbed x0 (the warm-start rounds
and the hand-over to the dense kernel run there), and checks every vehicle of both against the exact CPU oracle.

A vehicle is EXACT when its status is 0, every flag is 0, 1 or 2, the inputs flagged 1 / 2 equal lbu / ubu bit for bit
and the inputs flagged 0 lie strictly inside the box, its flags equal the oracle's active set (read off the oracle's
polished u by exact equality with a bound) and its u and x are within TOL_RICCATI / TOL_DENSE of the oracle.  The
bit-exact bound test is what tells an unverified IPM point from the minimiser: the IPM clips its inputs into the box
but does not put them on it.  A vehicle may instead report status MAXITER with all flags 255; status 0 on anything that
is not exact fails.

The emulated half (tests/emu, B = 8) runs on the CPU; the -m gpu half runs the same table at B = 256 on the device,
plus the launch geometry of the dense work queue, the busy step and a default-settings sweep over 4096 vehicles."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as orc
from helpers import make_gp, random_ocp_batch, u_rel, x_rel
from emu import emu

N, T_HORIZON = 20, 1.0
DT = T_HORIZON / N
NX, NU = 13, 4
STATUS_OK, STATUS_MAXITER, STATUS_NAN = 0, 1, 2
QMPC_ERR_ARG = -1
# the Riccati path (solver_variant 1) ends on a KKT point of the exact active set solved by the same Riccati recursion
# as the oracle: 2e-13 was the worst seen; 1e-9 leaves room for conditioning and is still 20x below the error of the
# unverified IPM points this file guards against (2e-10 .. 2e-8 at refine_max_rounds = 1)
TOL_RICCATI = 1e-9
# the dense path (solver_variant 2) solves the condensed QP with a Cholesky of H = R + G'QG, whose condition number
# costs digits against the Riccati recursion: 4e-11 worst emulated at B = 8, 5.3e-8 on a verified active set in 512
# aggressive-reference vehicles on a B200; 1e-7 as test_gpu_parity.py allows the dense kernel on the GPU.  An IPM point
# handed back as status 0 is caught by the bit-exact bound test whatever this tolerance is.
TOL_DENSE = 1e-7
# refine_max_rounds < 0: status 0 only promises the IPM reached ipm_mu_tol = 1e-13; at N = 20 that point was up to
# 3e-6 off the minimiser in 256 vehicles (complementarity over multipliers of order dt)
TOL_IPM = 1e-5
# two runs of the Riccati path that end on the same active set differ only in the rounding of the final pinned sweep
# (0 in most knob cases); final_rollout = 1 re-rolls the states through the dynamics instead of taking the sweep's,
# another summation order: 1.8e-11 in x on a B200
TOL_SAME_PATH = 1e-10
# the same problem on the dense path from a different start (warm set vs cold IPM) ends on the same active set; the
# final condensed solve's rounding is then the only difference, bounded by the dense tolerance
TOL_SAME_DENSE = TOL_DENSE
TOL_SWEEP = 1e-6
X0_KICK = 0.02                  # x0 perturbation of the second solve (metres, rad-ish, m/s): a few active inputs change


def tol_of(variant):
    return TOL_RICCATI if variant == 1 else TOL_DENSE


def act_of(u, lb, ub):
    """the active set of an exact solution: an input is pinned when it equals a bound"""
    u = u.reshape(u.shape[0], -1)
    return np.where(u == lb, 1, np.where(u == ub, 2, 0)).astype(np.uint8)


def scenario(B, seed, lb=0.0, ub=1.0, amp_choices=(2.0, 8.0, 25.0), n_nodes=N):
    """random_ocp_batch at dt = T_HORIZON / n_nodes with the GP; the iterate's inputs clipped into the box"""
    quad, gp = orc.quad_hummingbird(), make_gp(20)
    sc = random_ocp_batch(B, n_nodes, T_HORIZON / n_nodes, quad, gp, seed=seed, amp_choices=amp_choices)
    sc["uit"] = np.clip(sc["uit"], lb, ub)
    return sc, quad, gp


def n_of(sc):
    return sc["uit"].shape[1]


def oracle(sc, quad, gp, x0, xit, uit, lb, ub):
    """the exact RTI step from the given pre-solve iterate (copied).  returns (x, u, ok): ok marks the vehicles whose
    active set the oracle verified.  On a few percent of the warm second solves its polish rejects the active set
    (status 1: its IPM point, which can be far from the minimiser; rarely status 2, out of iterations); those
    vehicles have no exact reference."""
    x, u = np.ascontiguousarray(xit).copy(), np.ascontiguousarray(uit).copy()
    n = n_of(sc)
    r = orc.rti_step_batch(quad, T_HORIZON / n, n, np.ascontiguousarray(x0), sc["yref"], sc["yref_e"], x, u, gp=gp,
                           alpha=sc["alpha"], lbu=lb, ubu=ub)
    ok = r["status"] == 0
    assert ok.mean() >= 0.95, np.bincount(r["status"])
    return x, u, ok


def check(r, xo, uo, ok, lb, ub, tol, ipm_only=False):
    """the contract for every vehicle of a solve r (dict x, u, status, act) against the oracle's xo, uo; where the
    oracle has no verified active set (not ok) there is no exact reference: only the flags and bounds are checked.
    returns (failures [(vehicle, reasons)], MAXITER vehicles, worst error of the vehicles that passed)"""
    B = r["u"].shape[0]
    u, act, st = r["u"].reshape(B, -1), r["act"].reshape(B, -1), r["status"]
    oact = act_of(uo, lb, ub)
    fails, n_max, worst = [], 0, 0.0
    for b in range(B):
        e = max(u_rel(r["u"][b], uo[b]), x_rel(r["x"][b], xo[b]))
        tol_b = tol if ok[b] else np.inf
        if ipm_only:
            why = ([f"status {st[b]}"] if st[b] != STATUS_OK else []) + ([f"{e:.1e} off"] if not e < tol else [])
        elif st[b] == STATUS_MAXITER and (act[b] == 255).all():
            n_max += 1
            continue
        else:
            why = []
            if st[b] != STATUS_OK:
                why.append(f"status {st[b]}")
            if not np.isin(act[b], (0, 1, 2)).all():
                why.append("flags outside {0, 1, 2}")
            elif not ((u[b][act[b] == 1] == lb).all() and (u[b][act[b] == 2] == ub).all()):
                why.append("a pinned input is not on its bound")
            free = u[b][act[b] == 0]
            if not ((free > lb) & (free < ub)).all():
                why.append("a free input is not strictly inside the box")
            if ok[b] and not np.array_equal(act[b], oact[b]):
                why.append(f"flags differ from the oracle's active set in {int((act[b] != oact[b]).sum())} inputs")
            if not e < tol_b:
                why.append(f"{e:.1e} off the oracle")
        if why:
            fails.append((b, why))
        elif ok[b]:
            worst = max(worst, e)
    return fails, n_max, worst


# ------------------------------------------------------------------------------------------------------ backends
# Both run the product kernels: tests/emu under the lane emulation, _Gpu through the C-ABI.  A backend keeps the
# iterate and the remembered active sets between solves, as a handle does.

class _Emu:
    name = "emulated"

    def __init__(self, cfg, keep, sc):
        self.cfg, self.keep, self.sc = cfg, keep, sc
        self.x, self.u = sc["xit"].copy(), sc["uit"].copy()
        self.act = np.full((cfg.batch, 4 * cfg.n_nodes), 255, dtype=np.uint8)

    def iterate(self):
        """the iterate the next solve starts from"""
        return self.x.copy(), self.u.copy()

    def set_act(self, act):
        self.act = np.ascontiguousarray(act, dtype=np.uint8).copy()

    def reset_warm_start(self):
        self.act[:] = 255

    def set_iterate(self, x, u):
        self.x, self.u = x.copy(), u.copy()

    def solve(self, x0):
        sc = self.sc
        r = emu.solve(self.cfg, x0, sc["yref"], sc["yref_e"], sc["alpha"], self.x, self.u, act=self.act)
        return dict(x=self.x.copy(), u=self.u.copy(), status=r["status"].copy(), act=self.act.copy(),
                    rounds=r["rounds"].copy(), hard=r["hard"])


class _Gpu:
    """a handle created from a QmpcConfig (any lbu / ubu, which quad_optimizer fixes at [0, 1])"""
    name = "gpu"

    def __init__(self, cfg, keep, sc):
        import torch
        from mpc_quad_ros_b200 import _capi
        self.torch, self.capi, self.L = torch, _capi, _capi.lib()
        self.B, self.N, self.sc, self.dev = cfg.batch, cfg.n_nodes, sc, torch.device("cuda:0")
        self.h = C.c_void_p()
        _capi.check(self.L.qmpc_create(C.byref(cfg), C.byref(self.h)))
        self.s = _capi.stream_ptr()
        self.status = np.zeros(self.B, dtype=np.int32)         # a fresh handle's status: nothing to reset
        yref, yref_e, alpha = self._t(sc["yref"]), self._t(sc["yref_e"]), self._t(sc["alpha"])
        _capi.check(self.L.qmpc_set_yref(self.h, _capi.ptr(yref), _capi.ptr(yref_e), self.s))
        _capi.check(self.L.qmpc_set_alpha(self.h, _capi.ptr(alpha), self.s))
        self.set_iterate(sc["xit"], sc["uit"])

    def __del__(self):
        if getattr(self, "h", None):
            self.L.qmpc_destroy(self.h)

    def _t(self, a, dtype=None):
        """a device copy of a; the caller keeps it alive until the call that reads it has been queued (a tensor freed
        earlier may hand its memory to the next upload before the library's copy from it has run)"""
        return self.torch.as_tensor(np.ascontiguousarray(a), device=self.dev, dtype=dtype).contiguous()

    def _get(self, fn, shape, dtype):
        out = self.torch.empty(shape, dtype=dtype, device=self.dev)
        self.capi.check(fn(self.h, self.capi.ptr(out), self.s))
        return out.cpu().numpy()

    def iterate(self):
        """the iterate the next solve starts from: a vehicle whose last solve failed restarts from the reference
        (reset_on_fail, on by default: reset_failed_kernel)"""
        B, N = self.B, self.N
        x = self.torch.empty((B, N + 1, NX), dtype=self.torch.float64, device=self.dev)
        u = self.torch.empty((B, N, NU), dtype=self.torch.float64, device=self.dev)
        self.capi.check(self.L.qmpc_get_iterate(self.h, self.capi.ptr(x), self.capi.ptr(u), self.s))
        x, u = x.cpu().numpy(), u.cpu().numpy()
        for b in np.flatnonzero(self.status != STATUS_OK):
            x[b, :N], x[b, N], u[b] = self.sc["yref"][b, :, :NX], self.sc["yref_e"][b], self.sc["yref"][b, :, NX:]
        return x, u

    def set_act(self, act):
        a = self._t(act, self.torch.uint8)
        self.capi.check(self.L.qmpc_set_active_set(self.h, self.capi.ptr(a), self.s))

    def reset_warm_start(self):
        self.capi.check(self.L.qmpc_reset_warm_start(self.h, self.s))

    def set_iterate(self, x, u):
        xt, ut = self._t(x), self._t(u)
        self.capi.check(self.L.qmpc_set_iterate(self.h, self.capi.ptr(xt), self.capi.ptr(ut), self.s))

    def solve(self, x0):
        torch, L, N = self.torch, self.L, self.N
        x0 = self._t(x0)
        self.capi.check(L.qmpc_set_x0(self.h, self.capi.ptr(x0), self.s))
        self.capi.check(L.qmpc_solve(self.h, self.s))
        i32 = torch.int32
        st = self.torch.empty(self.B, dtype=i32, device=self.dev)
        self.capi.check(L.qmpc_get_status(self.h, self.capi.ptr(st), None, self.s))
        hard = C.c_int()
        self.capi.check(L.qmpc_get_hard_count(self.h, C.byref(hard), self.s))
        r = dict(x=self._get(L.qmpc_get_x, (self.B, N + 1, NX), torch.float64),
                 u=self._get(L.qmpc_get_u, (self.B, N, NU), torch.float64), status=st.cpu().numpy(),
                 act=self._get(L.qmpc_get_active_set, (self.B, 4 * N), torch.uint8),
                 rounds=self._get(L.qmpc_get_refine_rounds, (self.B,), i32), hard=hard.value)
        self.status = r["status"].copy()
        return r


def make(backend, sc, quad, gp, lb=0.0, ub=1.0, variant=1, **policy):
    cfg, keep = emu.make_config(sc["x0"].shape[0], n_of(sc), T_HORIZON, quad, orc.W_DIAG, orc.WE_DIAG, gp.X, gp.theta,
                                lbu=lb, ubu=ub, solver_variant=variant, **policy)
    return backend(cfg, keep, sc)


def kicked_x0(sc, k):
    """x0 of the k-th solve of a case (k = 0: the scenario's)"""
    if k == 0:
        return sc["x0"]
    return sc["x0"] + X0_KICK * np.random.default_rng(100 + k).standard_normal(sc["x0"].shape)


def run(h, sc, quad, gp, lb, ub, n_solves=2):
    """n_solves consecutive solves on backend h, each with the oracle's answer from the same pre-solve iterate.
    returns [(r, xo, uo, ok)]"""
    out = []
    for k in range(n_solves):
        x0 = kicked_x0(sc, k)
        xit, uit = h.iterate()
        xo, uo, ok = oracle(sc, quad, gp, x0, xit, uit, lb, ub)
        out.append((h.solve(x0), xo, uo, ok))
    return out


def assert_contract(res, lb, ub, tol, what, ipm_only=False):
    """every solve of a case honours the contract; returns (worst error, MAXITER vehicles)"""
    worst, n_max = 0.0, 0
    for k, (r, xo, uo, ok) in enumerate(res):
        fails, nm, w = check(r, xo, uo, ok, lb, ub, tol, ipm_only)
        assert not fails, f"{what}, solve {k}: {fails}"
        worst, n_max = max(worst, w), n_max + nm
    return worst, n_max


def diff(ra, rb, ok):
    """distance of two answers over the vehicles the oracle verified"""
    return max(float(np.abs(ra["u"][ok] - rb["u"][ok]).max()), x_rel(ra["x"][ok], rb["x"][ok]))


# ------------------------------------------------------------------------------------------------------- the table

B_EMU, B_GPU = 8, 256
SEED = 5
BACKENDS = [pytest.param(_Emu, id="emu"), pytest.param(_Gpu, id="gpu", marks=pytest.mark.gpu)]
_DEFAULTS = {}


def batch_of(backend):
    return B_EMU if backend is _Emu else B_GPU


def defaults(backend, variant):
    """the two solves of the scenario under the library defaults (shared by the knob cases)"""
    key = (backend, variant)
    if key not in _DEFAULTS:
        sc, quad, gp = scenario(batch_of(backend), SEED)
        res = run(make(backend, sc, quad, gp, variant=variant), sc, quad, gp, 0.0, 1.0)
        assert_contract(res, 0.0, 1.0, tol_of(variant), f"defaults, variant {variant}")
        _DEFAULTS[key] = res
    return _DEFAULTS[key]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("variant", [1, 2])
@pytest.mark.parametrize("rounds", [1, 2, 3, 20, -1])
def test_status_zero_means_exact(backend, variant, rounds):
    """refine_max_rounds in {1, 2, 3, 20}: status 0 only on the verified active set; the few rounds of 1 and 2 leave
    vehicles whose hand-over from the IPM does not settle twice, which must get a third attempt or report MAXITER.
    refine_max_rounds = -1: the pure IPM, status 0 means it reached ipm_mu_tol"""
    sc, quad, gp = scenario(batch_of(backend), SEED)
    res = run(make(backend, sc, quad, gp, variant=variant, refine_max_rounds=rounds), sc, quad, gp, 0.0, 1.0)
    tol = TOL_IPM if rounds < 0 else tol_of(variant)
    worst, n_max = assert_contract(res, 0.0, 1.0, tol, f"refine_max_rounds={rounds}", ipm_only=rounds < 0)
    print(f"{backend.name} variant {variant} refine_max_rounds={rounds}: worst {worst:.1e}, MAXITER {n_max}")


@pytest.mark.parametrize("rounds,bad", [(1, [0, 2, 5, 6]), (2, [5])])
def test_emulated_dense_kernel_third_attempt(rounds, bad):
    """random_ocp_batch(8, 20, seed 5, amplitudes 8 / 25 / 2) at refine_max_rounds = 1 and 2.  The dense kernel used to
    stop after its second failed hand-over from the IPM and return the IPM point at mu_tol with status 0: vehicles
    0, 2, 5, 6 came back 2e-10 .. 2e-8 off the minimiser (5 alone at 2 rounds), their flags already equal to the
    oracle's active set but their pinned inputs not on the bound.  It now makes a third attempt from that point, as
    qmpc_ipm_kernel does; on this batch every vehicle settles on the exact minimiser."""
    sc, quad, gp = scenario(8, SEED, amp_choices=(8.0, 25.0, 2.0))
    h = make(_Emu, sc, quad, gp, variant=2, refine_max_rounds=rounds)
    xo, uo, ok = oracle(sc, quad, gp, sc["x0"], sc["xit"], sc["uit"], 0.0, 1.0)
    assert ok.all()
    r = h.solve(sc["x0"])
    fails, n_max, worst = check(r, xo, uo, ok, 0.0, 1.0, TOL_DENSE)
    print(f"refine_max_rounds={rounds}: status {r['status']}, rounds {r['rounds']}, worst {worst:.1e}")
    assert not fails and n_max == 0, fails
    assert (r["rounds"][bad] >= 3).all(), r["rounds"]       # the third attempt ran for the vehicles that need it


KNOBS = [("bail_changed", 1), ("bail_changed", 3), ("bail_round", 1), ("bail_round", 5), ("final_rollout", 1),
         ("warm_start_rounds", 1), ("warm_start_rounds", 30), ("ipm_mu_switch", 1e-9), ("ipm_mu_switch", 1e-2),
         ("ipm_mu_switch", 1.0)]
DENSE_KNOBS = [("screen_rounds", 1), ("screen_rounds", 20), ("dense_warm_rounds", -1), ("dense_warm_rounds", 1),
               ("dense_warm_rounds", 30)]       # fields of the screening + dense mapping only


def _knob_cases():
    for k, v in KNOBS:
        for variant in (1, 2):
            yield pytest.param(k, v, variant, id=f"{k}={v}-v{variant}")
    for k, v in DENSE_KNOBS:
        yield pytest.param(k, v, 2, id=f"{k}={v}-v2")


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("knob,value,variant", list(_knob_cases()))
def test_policy_knob_keeps_the_answer(backend, knob, value, variant):
    """each policy field alone on top of the defaults: exact, and the answer of the defaults.  The Riccati path ends
    on the same pinned sweep (TOL_SAME_PATH); the dense path is compared with the Riccati path's default answer
    (TOL_SAME_DENSE)"""
    sc, quad, gp = scenario(batch_of(backend), SEED)
    res = run(make(backend, sc, quad, gp, variant=variant, **{knob: value}), sc, quad, gp, 0.0, 1.0)
    worst, n_max = assert_contract(res, 0.0, 1.0, tol_of(variant), f"{knob}={value}")
    assert n_max == 0
    ref = defaults(backend, 1)
    d = max(diff(r, rr, ok & okr) for (r, _, _, ok), (rr, _, _, okr) in zip(res, ref))
    print(f"{backend.name} {knob}={value} variant {variant}: worst vs oracle {worst:.1e}, vs defaults {d:.1e}")
    assert d < (TOL_SAME_PATH if variant == 1 else TOL_SAME_DENSE), d


BOXES = [(0.1, 0.6), (-0.5, 0.5), (0.25, 0.35), (0.0, 2.0)]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("variant", [1, 2])
@pytest.mark.parametrize("lb,ub", BOXES)
def test_input_box(backend, variant, lb, ub):
    """lbu / ubu other than [0, 1]: (0.25, 0.35) pins about 96 % of the inputs and excludes the 0.16 hover input a
    failed vehicle restarts from; (-0.5, 0.5) puts the box centre, where the IPM starts, at 0"""
    sc, quad, gp = scenario(batch_of(backend), SEED, lb, ub)
    res = run(make(backend, sc, quad, gp, lb, ub, variant=variant), sc, quad, gp, lb, ub)
    worst, n_max = assert_contract(res, lb, ub, tol_of(variant), f"box ({lb}, {ub})")
    pinned = np.mean([(r["act"] != 0).mean() for r, *_ in res])
    print(f"{backend.name} variant {variant} box ({lb}, {ub}): worst {worst:.1e}, MAXITER {n_max}, pinned {pinned:.0%}")
    assert pinned > 0


@pytest.mark.parametrize("lb,ub", [(0.5, 0.5), (1.0, 0.0), (np.nan, 1.0), (0.0, np.nan), (-np.inf, 1.0),
                                   (0.0, np.inf), (-np.inf, np.inf)])
def test_create_refuses_input_box(lb, ub):
    """ubu <= lbu, NaN and infinite bounds: QMPC_ERR_ARG, no handle, nothing launched (the IPM starts from the box
    centre, which is NaN or infinite then)"""
    from mpc_quad_ros_b200 import _capi
    L = _capi.lib()
    sc, quad, gp = scenario(2, 0)
    cfg, keep = emu.make_config(2, N, T_HORIZON, quad, orc.W_DIAG, orc.WE_DIAG, gp.X, gp.theta, lbu=lb, ubu=ub)
    h = C.c_void_p()
    l0 = L.qmpc_launch_count()
    assert L.qmpc_create(C.byref(cfg), C.byref(h)) == QMPC_ERR_ARG
    assert not h.value and L.qmpc_launch_count() == l0
    assert "bounds" in L.qmpc_last_error().decode()


def _adversarial(kind, right):
    rng = np.random.default_rng(7)
    if kind == "all_lower":
        return np.ones_like(right)
    if kind == "all_upper":
        return np.full_like(right, 2)
    if kind == "random":
        return rng.integers(0, 3, right.shape).astype(np.uint8)
    if kind == "random_unknown":
        a = rng.integers(0, 3, right.shape).astype(np.uint8)
        a[rng.uniform(size=right.shape) < 0.3] = 255
        return a
    assert kind == "complement"         # every flag wrong: free <-> pinned at the other bound's side
    return np.where(right == 0, np.where(rng.uniform(size=right.shape) < 0.5, 1, 2), 0).astype(np.uint8)


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("variant", [1, 2])
def test_adversarial_warm_start_keeps_the_answer(backend, variant):
    """qmpc_set_active_set before the second solve with a wrong set (all at lbu, all at ubu, random, random with 30 %
    unknown, the complement of the right set): the same u, x and flags as that solve after qmpc_reset_warm_start,
    and exact.  Each second solve runs on a fresh handle given the first solve's iterate."""
    sc, quad, gp = scenario(batch_of(backend), SEED)
    h = make(backend, sc, quad, gp, variant=variant)
    first = run(h, sc, quad, gp, 0.0, 1.0, n_solves=1)
    assert_contract(first, 0.0, 1.0, tol_of(variant), "first solve")
    right = first[0][0]["act"]
    x1, u1 = h.iterate()
    x0 = kicked_x0(sc, 1)
    xo, uo, ok = oracle(sc, quad, gp, x0, x1, u1, 0.0, 1.0)

    def second(act):
        h2 = make(backend, sc, quad, gp, variant=variant)
        h2.set_iterate(x1, u1)
        if act is None:
            h2.set_act(right)
            h2.reset_warm_start()
        else:
            h2.set_act(act)
        r = h2.solve(x0)
        assert_contract([(r, xo, uo, ok)], 0.0, 1.0, tol_of(variant), "reset" if act is None else kind)
        return r

    reset = second(None)
    tol_same = TOL_SAME_PATH if variant == 1 else TOL_SAME_DENSE
    worst = 0.0
    for kind in ("all_lower", "all_upper", "random", "random_unknown", "complement"):
        r = second(_adversarial(kind, right))
        d = diff(r, reset, ok)
        worst = max(worst, d)
        assert d < tol_same, (kind, d)
        assert np.array_equal(r["act"][ok], reset["act"][ok]) and np.array_equal(r["status"], reset["status"]), kind
    print(f"{backend.name} variant {variant}: adversarial warm starts vs reset {worst:.1e}")


# --------------------------------------------------------------------------------------------------------- GPU only

@pytest.mark.gpu
def test_adjoint_at_a_non_default_box():
    """qmpc_eval_adjoint after a solve in the box (0.1, 0.6): the adjoint kernels read the flags, not the bounds, so
    this checks that the flags of a non-default box reach them (reference: tests/sens/adjoint_ref.py)"""
    from sens import adjoint_ref
    lb, ub = 0.1, 0.6
    B = 16
    sc, quad, gp = scenario(B, 11, lb, ub)
    h = make(_Gpu, sc, quad, gp, lb, ub)
    xit, uit = h.iterate()
    res = run(h, sc, quad, gp, lb, ub, n_solves=1)
    assert_contract(res, lb, ub, TOL_DENSE, "adjoint box")
    act = res[0][0]["act"]
    rng = np.random.default_rng(3)
    xb, ub_ = rng.standard_normal((B, N + 1, NX)), rng.standard_normal((B, N, NU))
    x0b, yb, yeb = (h.torch.empty(s, dtype=h.torch.float64, device=h.dev) for s in ((B, NX), (B, N, NX + NU), (B, NX)))
    p = h.capi.ptr
    xbt, ubt = h._t(xb), h._t(ub_)
    h.capi.check(h.L.qmpc_eval_adjoint(h.h, p(xbt), p(ubt), p(x0b), p(yb), p(yeb), h.s))
    x0b, yb, yeb = x0b.cpu().numpy(), yb.cpu().numpy(), yeb.cpu().numpy()
    worst = 0.0
    for b in range(B):
        ref = adjoint_ref.rti_adjoint(quad, DT, N, xit[b], uit[b], act[b], x_bar=xb[b], u_bar=ub_[b], gp=gp,
                                      alpha=sc["alpha"][b])
        for a, r in zip((x0b[b], yb[b], yeb[b]), ref):
            worst = max(worst, float(np.abs(a - r).max() / max(1.0, np.abs(r).max())))
    print(f"adjoint at box ({lb}, {ub}): {worst:.1e}, pinned inputs {int((act != 0).sum())}")
    assert worst < 1e-9, worst          # two exact routes to the same linear map (TOL_SENS of test_size_envelope.py)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 5, 33, 129])
def test_dense_work_queue_geometry(B):
    """dense_grid in {1, 2, 7, 4096} persistent CTAs, B = 1 and 5 fewer items than CTAs: with the warm start off every
    vehicle goes through the queue; the answer is bit-identical to the default grid and exact"""
    sc, quad, gp = scenario(B, 20 + B)
    base = run(make(_Gpu, sc, quad, gp, variant=2, warm_start_rounds=-1), sc, quad, gp, 0.0, 1.0)
    assert_contract(base, 0.0, 1.0, TOL_DENSE, f"B={B} default grid")
    for grid in (1, 2, 7, 4096):
        res = run(make(_Gpu, sc, quad, gp, variant=2, warm_start_rounds=-1, dense_grid=grid), sc, quad, gp, 0.0, 1.0)
        for (r, *_), (rb, *_) in zip(res, base):
            for k in ("x", "u", "status", "act", "rounds"):
                assert np.array_equal(r[k], rb[k]), (B, grid, k)


@pytest.mark.gpu
@pytest.mark.parametrize("busy_rounds", [-1, 4, 12])
def test_busy_step(busy_rounds):
    """screen_rounds_busy with screen_busy_pct 1 (every step after the cold start is busy) and 100 (never), over three
    solves; the first is a start-up transient that leaves every vehicle unsettled.  Exact either way; the busy path
    must really have run (another hand-over count), and with screen_rounds_busy = -1 (no busy limit) nothing changes"""
    B = 512
    sc, quad, gp = scenario(B, 31, amp_choices=(8.0, 25.0))
    runs = {}
    for pct in (1, 100):
        h = make(_Gpu, sc, quad, gp, variant=2, screen_rounds_busy=busy_rounds, screen_busy_pct=pct)
        runs[pct] = run(h, sc, quad, gp, 0.0, 1.0, n_solves=3)
        worst, n_max = assert_contract(runs[pct], 0.0, 1.0, TOL_DENSE, f"busy {busy_rounds} pct {pct}")
        print(f"screen_rounds_busy={busy_rounds} pct={pct}: worst {worst:.1e}, MAXITER {n_max}, hand-overs "
              f"{[r['hard'] for r, *_ in runs[pct]]}, max rounds {[int(r['rounds'].max()) for r, *_ in runs[pct]]}")
    if busy_rounds < 0:
        for (a, *_), (b, *_) in zip(runs[1], runs[100]):
            assert all(np.array_equal(a[k], b[k]) for k in ("x", "u", "status", "act", "rounds")) and a["hard"] == b["hard"]
    else:       # the busy limit changed the hand-overs or the rounds of the solves after the cold one
        assert any(a["hard"] != b["hard"] or not np.array_equal(a["rounds"], b["rounds"])
                   for (a, *_), (b, *_) in zip(runs[1][1:], runs[100][1:]))


@pytest.mark.gpu
@pytest.mark.parametrize("n_nodes", [20, 21])
def test_default_settings_sweep(n_nodes):
    """4096 vehicles under the library defaults (screening + dense kernel), a cold and a warm solve: no status-0
    vehicle that is not exact.  The distance bound is TOL_SWEEP: over 4096 vehicles at N = 21 the condensed Cholesky
    left a verified active set 2.0e-7 off on a B200"""
    B = 4096
    sc, quad, gp = scenario(B, 4000 + n_nodes, amp_choices=(8.0, 25.0), n_nodes=n_nodes)
    res = run(make(_Gpu, sc, quad, gp, variant=0), sc, quad, gp, 0.0, 1.0)
    n_max, n_nan, worst, bad = 0, 0, 0.0, []
    for k, (r, xo, uo, ok) in enumerate(res):
        fails, nm, w = check(r, xo, uo, ok, 0.0, 1.0, TOL_SWEEP)
        bad += [(k, f) for f in fails if r["status"][f[0]] == STATUS_OK]
        n_nan += int((r["status"] == STATUS_NAN).sum())
        n_max, worst = n_max + nm, max(worst, w)
    print(f"default settings N={n_nodes}, B={B}: status-0 not exact {len(bad)}, MAXITER {n_max}, NaN {n_nan}, worst {worst:.1e}")
    assert not bad, bad[:10]
