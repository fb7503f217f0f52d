"""quad_optimizer — the reference's controller API (reference src/quad_opt.py:35-406) over libqmpc.so.

Same method names, argument meaning and return values as the reference for one vehicle (numpy in / numpy out);
with batch > 1 the same methods take and return CUDA tensors with a leading vehicle dimension.
acados/CasADi are replaced by two CUDA kernels (RK4 + sensitivities, Riccati IPM); nothing here computes on the CPU.
"""
import ctypes as C
import time

import numpy as np
import torch

from . import _capi
from ._capi import QmpcConfig

# LINEAR_LS weights of the reference OCP (quad_opt.py:122-130)
_Q_COST = np.array([10, 10, 10] + [0.1, 0.1, 0.1] + [0.05, 0.05, 0.05] + [0.05, 0.05, 0.05], dtype=np.float64)
Q_DIAGONAL = np.concatenate((_Q_COST[:3], np.mean(_Q_COST[3:6])[np.newaxis], _Q_COST[3:]))
R_COST = np.array([0.1, 0.1, 0.1, 0.1])


class quad_optimizer:
    def __init__(self, quad, t_horizon=1, n_nodes=100, gpe=None, batch=None, device=None, precision=64,
                 ipm_mu_tol=0.0, ipm_max_iter=50, ipm_mu_switch=0.0, refine_max_rounds=0, warm_start_rounds=0,
                 solver_variant=0, reset_on_fail=0, screen_rounds=0, dense_warm_rounds=0, bail_round=0, bail_changed=0,
                 final_rollout=0, dense_grid=0, screen_rounds_busy=0, screen_busy_pct=0):
        """The arguments after `gpe` have no counterpart in the reference (one vehicle, acados defaults): batch/device/
        precision select the GPU path, the rest is the per-handle solver policy of include/qmpc.h (0 = library default;
        reset_on_fail=-1 keeps whatever a failed solve left, which is what the reference does, quad_opt.py:333)."""
        self.n_nodes, self.t_horizon, self.gpe = n_nodes, t_horizon, gpe
        self.optimization_dt = self.t_horizon / self.n_nodes
        self.terminal_cost = 1
        self.quad = quad
        self.batch = batch if batch is not None else getattr(quad, "batch", 1)
        self.device = torch.device(device if device is not None else getattr(quad, "device", "cuda:0"))
        if gpe is not None:
            if gpe.type != "RGP":
                raise ValueError("Unknown GPE type")     # quad_opt.py:232 ('GP' ensembles are the offline mode)
            assert gpe.batch in (self.batch, 1), "gpe.batch must equal the solver batch (or 1 for a shared model)"
        self.nx, self.nu = 13, 4
        self.np = 0 if gpe is None else gpe.M          # quirk kept: acados_model.p is M x 3 (SURVEY App. C-1)
        self.ny = self.nx + self.nu
        self.W = np.diag(np.concatenate((Q_DIAGONAL, R_COST)))
        self.W_e = np.diag(Q_DIAGONAL) * self.terminal_cost

        cfg = QmpcConfig()
        cfg.batch, cfg.n_nodes, cfg.n_basis = self.batch, n_nodes, (0 if gpe is None else gpe.M)
        cfg.precision, cfg.device = precision, (self.device.index or 0)
        cfg.ipm_max_iter, cfg.ipm_mu_tol, cfg.t_horizon = ipm_max_iter, ipm_mu_tol, float(t_horizon)
        cfg.ipm_mu_switch, cfg.refine_max_rounds = ipm_mu_switch, refine_max_rounds   # 0 -> library defaults
        cfg.warm_start_rounds = warm_start_rounds                                     # 0 -> 6 rounds, <0 -> cold IPM every step
        cfg.solver_variant, cfg.reset_on_fail, cfg.screen_rounds = solver_variant, reset_on_fail, screen_rounds
        cfg.dense_warm_rounds, cfg.bail_round, cfg.bail_changed = dense_warm_rounds, bail_round, bail_changed
        cfg.final_rollout, cfg.dense_grid = final_rollout, dense_grid
        cfg.screen_rounds_busy, cfg.screen_busy_pct = screen_rounds_busy, screen_busy_pct
        cfg.quad[:] = list(quad.quad_vector())
        cfg.w_diag[:] = list(np.diag(self.W))
        cfg.we_diag[:] = list(np.diag(self.W_e))
        cfg.lbu, cfg.ubu = 0.0, 1.0                    # quad_opt.py:142-143
        self._gpX = None
        if gpe is not None:
            self._gpX = np.ascontiguousarray(gpe.X, dtype=np.float64)
            cfg.gp_theta[:] = list(gpe.theta.ravel())
            cfg.gp_X = self._gpX.ctypes.data_as(C.POINTER(C.c_double))
        self._cfg = cfg
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            _capi.check(_capi.lib().qmpc_create(C.byref(cfg), C.byref(self._h)))
        self._Kx_inv = None if gpe is None else torch.as_tensor(gpe.K_x_inv, device=self.device).contiguous()
        self.yref = self.yref_N = None
        self._numpy_io = self.batch == 1      # eval_sens answers like the last run_optimization (numpy for one vehicle)

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _capi.lib().qmpc_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # ---- plumbing -----------------------------------------------------------------------------------------------
    def _dev(self, a, shape):
        t = a if torch.is_tensor(a) else torch.as_tensor(np.asarray(a, dtype=np.float64))
        return t.to(self.device, torch.float64).reshape(shape).contiguous()

    def _s(self):
        return _capi.stream_ptr()

    def _single(self, *inputs):
        return self.batch == 1 and not any(torch.is_tensor(a) for a in inputs if a is not None)

    # ---- reference API --------------------------------------------------------------------------------------------
    def set_quad_state(self, x):
        """quad_opt.py:265-269: only forwards to the quad object"""
        self.quad.set_state(x)

    def set_reference_state(self, x_target=None, u_target=None):
        """quad_opt.py:271-292: constant reference over the horizon. returns (yref [N,17], yref_N [13])"""
        if u_target is None:
            u_target = np.ones((self.nu,)) * 0.16
        if x_target is None:
            x_target = np.array([0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0])
        single = self._single(x_target, u_target)
        xt = self._dev(x_target, (-1, 1, 13)).expand(self.batch, self.n_nodes, 13).contiguous()
        ut = self._dev(u_target, (-1, 1, 4)).expand(self.batch, self.n_nodes, 4).contiguous()
        return self._set_ref(xt, ut, single)

    def set_reference_trajectory(self, x_trajectory, u_trajectory=None):
        """quad_opt.py:295-317: x_trajectory [N,13] (or [B,N,13]), u_trajectory [N,4] or None (0.16 hover)."""
        single = self._single(x_trajectory, u_trajectory)
        xt = self._dev(x_trajectory, (self.batch, self.n_nodes, 13))
        ut = None if u_trajectory is None else self._dev(u_trajectory, (self.batch, self.n_nodes, 4))
        return self._set_ref(xt, ut, single)

    def _set_ref(self, xt, ut, single):
        _capi.check(_capi.lib().qmpc_set_reference(self._h, _capi.ptr(xt), _capi.ptr(ut), self._s()))
        u_part = ut if ut is not None else torch.full((self.batch, self.n_nodes, 4), 0.16, dtype=torch.float64, device=self.device)
        self.yref = torch.cat([xt, u_part], dim=2)
        self.yref_N = xt[:, -1, :].clone()
        if single:
            self.yref, self.yref_N = self.yref[0].cpu().numpy(), self.yref_N[0].cpu().numpy()
        return self.yref, self.yref_N

    def run_optimization(self, x_init):
        """quad_opt.py:321-350: pin x0, ONE SQP-RTI iteration, read back the whole trajectory.
        returns (x_opt [N+1,13], w_opt [N,4], t_cpu, cost); batched: tensors with a leading B and cost [B]."""
        if x_init is None:
            raise ValueError("x_init has to be set before running the optimization")
        single = self._single(x_init)
        self._numpy_io = single
        x0 = self._dev(x_init, (self.batch, 13))
        lib = _capi.lib()
        t0 = time.perf_counter()
        _capi.check(lib.qmpc_set_x0(self._h, _capi.ptr(x0), self._s()))
        _capi.check(lib.qmpc_solve(self._h, self._s()))
        x_opt = torch.empty((self.batch, self.n_nodes + 1, 13), dtype=torch.float64, device=self.device)
        w_opt = torch.empty((self.batch, self.n_nodes, 4), dtype=torch.float64, device=self.device)
        cost = torch.empty((self.batch,), dtype=torch.float64, device=self.device)
        _capi.check(lib.qmpc_get_x(self._h, _capi.ptr(x_opt), self._s()))
        _capi.check(lib.qmpc_get_u(self._h, _capi.ptr(w_opt), self._s()))
        _capi.check(lib.qmpc_get_cost(self._h, _capi.ptr(cost), self._s()))
        if single:
            out = x_opt[0].cpu().numpy(), w_opt[0].cpu().numpy()
            c = float(cost[0].item())
            return out[0], out[1], time.perf_counter() - t0, c
        return x_opt, w_opt, time.perf_counter() - t0, cost

    def eval_sens(self, n_stages=None, states=True):
        """acados eval_param_sens(field="ex") + get(k, "sens_u" / "sens_x"): derivatives of the last solve's u[k], x[k]
        w.r.t. x0 at the active set that solve ended on (qmpc_eval_sens_x0), for every x0 component at once.
        n_stages (default N): stages covered, 1 gives the feedback gain sens_u[0] = du0/dx0 and sens_x[1] only.
        returns (sens_x [n+1,13,13] or None when states=False, sens_u [n,4,13]), column = x0 component; batched: CUDA
        tensors with a leading B.  NaN for vehicles whose active set is unknown (a failed solve).  Valid until the next
        solve: the derivatives are taken from that solve's linearisation.  fp64 handles only (QmpcError otherwise)."""
        n = self.n_nodes if n_stages is None else int(n_stages)
        sx = torch.empty((self.batch, max(n, 0) + 1, 13, 13), dtype=torch.float64, device=self.device) if states else None
        su = torch.empty((self.batch, max(n, 0), 4, 13), dtype=torch.float64, device=self.device)
        _capi.check(_capi.lib().qmpc_eval_sens_x0(self._h, n, _capi.ptr(sx), _capi.ptr(su), self._s()))
        if self._numpy_io:
            return (None if sx is None else sx[0].cpu().numpy()), su[0].cpu().numpy()
        return sx, su

    def eval_adjoint(self, x_bar=None, u_bar=None):
        """Reverse mode of the last solve (qmpc_eval_adjoint): for cotangents x_bar [N+1,13] and u_bar [N,4] of its x_opt,
        w_opt (None = zero; batched: a leading B), the gradients of <x_bar, x_opt> + <u_bar, w_opt> w.r.t. x0, yref and
        yref_N at the active set that solve ended on.  returns (x0_bar [13], yref_bar [N,17], yref_N_bar [13]); batched:
        CUDA tensors with a leading B.  NaN for vehicles whose active set is unknown.  Valid until the next solve;
        fp64 handles only (QmpcError otherwise)."""
        x0b, yb, yeb = self._adjoint(x_bar, u_bar)
        if self._numpy_io:
            return x0b[0].cpu().numpy(), yb[0].cpu().numpy(), yeb[0].cpu().numpy()
        return x0b, yb, yeb

    def _adjoint(self, x_bar, u_bar):
        B, N = self.batch, self.n_nodes
        xb = None if x_bar is None else self._dev(x_bar, (B, N + 1, 13))
        ub = None if u_bar is None else self._dev(u_bar, (B, N, 4))
        x0b = torch.empty((B, 13), dtype=torch.float64, device=self.device)
        yb = torch.empty((B, N, 17), dtype=torch.float64, device=self.device)
        yeb = torch.empty((B, 13), dtype=torch.float64, device=self.device)
        _capi.check(_capi.lib().qmpc_eval_adjoint(self._h, _capi.ptr(xb), _capi.ptr(ub), _capi.ptr(x0b), _capi.ptr(yb),
                                                  _capi.ptr(yeb), self._s()))
        return x0b, yb, yeb

    def sens_epoch(self):
        """qmpc_get_sens_epoch: changes with every solve (also the fused steps) and every set / reset of the active set"""
        e = C.c_longlong()
        _capi.check(_capi.lib().qmpc_get_sens_epoch(self._h, C.byref(e)))
        return e.value

    def differentiable_step(self, x0, x_ref, u_ref=None, iterate=None):
        """set_reference_trajectory(x_ref, u_ref), optionally set_iterate(*iterate), run_optimization(x0) as a function
        torch.autograd can differentiate w.r.t. x0 [B,13], x_ref [B,N,13] and u_ref [B,N,4] (tensors; no leading B for
        batch 1 is accepted too).  returns (x_opt [B,N+1,13], u_opt [B,N,4]).  The backward is eval_adjoint: exact on
        the active set of this solve; the iterate is the linearisation point and counts as a constant.  The backward
        must run before the handle solves again or has its active set changed (RuntimeError otherwise).  With
        reset_on_fail on, a vehicle whose previous solve failed is linearised at a point built from the reference: its
        gradient is the one at that fixed linearisation."""
        if iterate is not None and any(torch.is_tensor(t) and t.requires_grad for t in iterate):
            raise ValueError("differentiable_step: the iterate is the linearisation point and is not differentiated; "
                             "pass it detached")
        return _RTIStep.apply(self, x0, x_ref, u_ref, iterate)

    def solver_status(self):
        """per-vehicle (status, iters) of the last solve; the reference discards acados' status (quad_opt.py:333)"""
        st = torch.empty((self.batch,), dtype=torch.int32, device=self.device)
        it = torch.empty_like(st)
        _capi.check(_capi.lib().qmpc_get_status(self._h, _capi.ptr(st), _capi.ptr(it), self._s()))
        return st, it

    def fail_streak(self):
        """consecutive failed solves per vehicle (0 = the last solve was fine), [B] int32"""
        r = torch.empty((self.batch,), dtype=torch.int32, device=self.device)
        _capi.check(_capi.lib().qmpc_get_fail_streak(self._h, _capi.ptr(r), self._s()))
        return r

    def solver_rounds(self):
        """active-set refinement rounds of the last solve (warm-start rounds + rounds after the IPM), [B] int32"""
        r = torch.empty((self.batch,), dtype=torch.int32, device=self.device)
        _capi.check(_capi.lib().qmpc_get_refine_rounds(self._h, _capi.ptr(r), self._s()))
        return r

    def get_active_set(self):
        """remembered active sets [B, 4N] uint8 (0 free, 1 lower, 2 upper, 255 unknown)"""
        a = torch.empty((self.batch, 4 * self.n_nodes), dtype=torch.uint8, device=self.device)
        _capi.check(_capi.lib().qmpc_get_active_set(self._h, _capi.ptr(a), self._s()))
        return a

    def set_active_set(self, act):
        a = act.to(self.device, torch.uint8).reshape(self.batch, 4 * self.n_nodes).contiguous()
        _capi.check(_capi.lib().qmpc_set_active_set(self._h, _capi.ptr(a), self._s()))

    def reset_warm_start(self):
        _capi.check(_capi.lib().qmpc_reset_warm_start(self._h, self._s()))

    def get_iterate(self):
        x = torch.empty((self.batch, self.n_nodes + 1, 13), dtype=torch.float64, device=self.device)
        u = torch.empty((self.batch, self.n_nodes, 4), dtype=torch.float64, device=self.device)
        _capi.check(_capi.lib().qmpc_get_iterate(self._h, _capi.ptr(x), _capi.ptr(u), self._s()))
        return x, u

    def set_iterate(self, x, u):
        x, u = self._dev(x, (self.batch, self.n_nodes + 1, 13)), self._dev(u, (self.batch, self.n_nodes, 4))
        _capi.check(_capi.lib().qmpc_set_iterate(self._h, _capi.ptr(x), _capi.ptr(u), self._s()))

    def set_rgp_params(self, mu):
        """solver.set(ii,'p',rgp_params) for all stages (quad_opt.py:402-404); mu [B,3,M] (or (3M,) for batch 1)"""
        assert self.gpe is not None, "RGP model has to be initialized before calling this method"
        mu = self._dev(mu, (self.batch, 3, self.gpe.M))
        _capi.check(_capi.lib().qmpc_set_params(self._h, _capi.ptr(mu), _capi.ptr(self._Kx_inv), self._s()))

    def discrete_dynamics(self, x, u, dt, body_frame=False):
        """quad_opt.py:353-377: fixed-step RK4 of the NOMINAL model (the reference calls it without p)."""
        single = self._single(x, u)
        if single:
            assert np.asarray(x).shape == (self.nx,), f"x has to be of shape ({self.nx},)"
            assert np.asarray(u).shape == (self.nu,), f"u has to be of shape ({self.nu},)"
        xt, ut = self._dev(x, (-1, 13)), self._dev(u, (-1, 4))
        out = torch.empty_like(xt)
        q = self.quad.quad_vector()
        _capi.check(_capi.lib().qmpc_predict_nominal(q.ctypes.data_as(C.c_void_p), xt.shape[0], _capi.ptr(xt), _capi.ptr(ut),
                                                     C.c_double(dt), int(bool(body_frame)), _capi.ptr(out), self._s()))
        return out[0].cpu().numpy() if single else out

    def regress_and_update_RGP_model(self, v_body, a_drag):
        """quad_opt.py:380-406: gpe.regress, then push concatenate(mu_g_t) as the solver parameters of every stage."""
        if not torch.is_tensor(v_body):
            assert len(v_body) == 3, "v_body has to be a list of length 3"
            assert len(a_drag) == 3, "a_drag has to be a list of length 3"
        assert self.gpe is not None, "RGP model has to be initialized before calling this method"
        assert self.gpe.type == "RGP", "Only RGP models are supported for online regression"
        mu_g_t, C_g_t = self.gpe.regress(v_body, a_drag)
        alpha = self.gpe.alpha_tensor()       # K_x^-1 mu, computed by the regress kernel's epilogue
        if self.gpe.batch == 1 and self.batch > 1:
            alpha = alpha.expand(self.batch, 3, self.gpe.M).contiguous()
        _capi.check(_capi.lib().qmpc_set_alpha(self._h, _capi.ptr(alpha), self._s()))
        return mu_g_t, C_g_t

    # ---- fused closed-loop step (execute_trajectory.py:196-277 in one call, all on the GPU) ------------------------------
    def step(self, x_now, x_ref, x_pred_prev, first_step, u0_out=None, rgp=True, odometry_dt=None):
        """reference chunk -> solve -> u0 -> nominal prediction -> residual -> RGP regress -> alpha for the next solve.
        x_now [B,13], x_ref [B,N,13], x_pred_prev [B,13] (updated in place), u0_out [B,4] (optional) CUDA tensors.
        rgp=False: solve and prediction only (the RGP update of this step is run elsewhere, swarm.SharedSwarmRGP.begin)."""
        g = self.gpe._h if (self.gpe is not None and rgp) else C.c_void_p(0)
        # odometry_dt: the ROS node predicts and differences over the odometry period (mpc_controller_node.py:298,315)
        _capi.check(_capi.lib().qmpc_step_dt(self._h, g, _capi.ptr(x_now), _capi.ptr(x_ref), _capi.ptr(x_pred_prev),
                                             int(bool(first_step)), _capi.ptr(u0_out),
                                             C.c_double(0.0 if odometry_dt is None else float(odometry_dt)), self._s()))


class _RTIStep(torch.autograd.Function):
    """quad_optimizer.differentiable_step: forward = one RTI solve, backward = qmpc_eval_adjoint on that solve's tiles"""

    @staticmethod
    def forward(ctx, opt, x0, x_ref, u_ref, iterate):
        B, N = opt.batch, opt.n_nodes
        opt.set_reference_trajectory(x_ref.detach().to(opt.device, torch.float64).reshape(B, N, 13),
                                     None if u_ref is None else u_ref.detach().to(opt.device, torch.float64).reshape(B, N, 4))
        if iterate is not None:
            opt.set_iterate(*iterate)
        x, u, _, _ = opt.run_optimization(x0.detach().to(opt.device, torch.float64).reshape(B, 13))
        ctx.opt, ctx.epoch = opt, opt.sens_epoch()
        ctx.like = [None if t is None else (t.shape, t.device, t.dtype) for t in (x0, x_ref, u_ref)]
        ctx.set_materialize_grads(False)
        lead = x0.shape[:-1]
        return x.reshape(*lead, N + 1, 13), u.reshape(*lead, N, 4)

    @staticmethod
    def backward(ctx, x_bar, u_bar):
        opt = ctx.opt
        if x_bar is None and u_bar is None:
            return None, None, None, None, None
        if opt.sens_epoch() != ctx.epoch:
            raise RuntimeError("differentiable_step: the handle has solved again or had its active set changed since "
                               "this step's forward; the stage tiles and active set its backward needs are gone")
        x0b, yb, yeb = opt._adjoint(x_bar, u_bar)
        N = opt.n_nodes
        x_ref_bar = yb[..., :13].clone()
        x_ref_bar[:, N - 1] += yeb                     # yref_e = x_ref[:, N-1] (set_reference_kernel)
        like = lambda g, i: g.reshape(ctx.like[i][0]).to(ctx.like[i][1], ctx.like[i][2]) if ctx.needs_input_grad[i + 1] else None
        return None, like(x0b, 0), like(x_ref_bar, 1), like(yb[..., 13:], 2), None
