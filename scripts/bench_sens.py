"""Cost of qmpc_eval_sens_x0 (derivatives of the RTI step w.r.t. x0) and of qmpc_eval_adjoint (its reverse mode, w.r.t. x0
and the reference) beside the solve they differentiate.

Workload: bench.py's random_smooth closed loop, B = 4096, N = 20, M = 20, fp64; 40 fused closed-loop steps first (the
last 20 with qmpc_timing_* on, for the solve time), then 200 timed calls of each case with CUDA events around every call:
  gain    n_stages = 1 without states (K0 = du0/dx0 and nothing else)
  full    n_stages = N with states
  adjoint       qmpc_eval_adjoint with u_bar on stage 0 only (x_bar NULL), all three outputs
  adjoint_full  qmpc_eval_adjoint with every cotangent (x_bar and u_bar), all three outputs
Prints one JSON line and writes it to --out.  Needs a GPU.

    python scripts/bench_sens.py --out bench_outputs/sens.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--nodes", type=int, default=20)
    ap.add_argument("--basis", type=int, default=20)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--calls", type=int, default=200)
    a = ap.parse_args()

    import torch
    assert torch.cuda.is_available(), "bench_sens.py needs a GPU"
    from mpc_quad_ros_b200 import _capi
    from mpc_quad_ros_b200.execute_trajectory import ClosedLoop
    from mpc_quad_ros_b200.gp.GPE import GPEnsemble
    from mpc_quad_ros_b200.quad import Quadrotor3D
    from mpc_quad_ros_b200.quad_opt import quad_optimizer
    from mpc_quad_ros_b200.trajectory import random_smooth_trajectories
    lib = _capi.lib()
    B, N, M = a.batch, a.nodes, a.basis
    dev = torch.device("cuda:0")

    traj = random_smooth_trajectories(B, a.steps + N + 2, 1.0 / N, seed=1234)     # bench.py's workload, rank 0
    quad = Quadrotor3D(drag=True, batch=B, device=dev).set_hummingbird_params()
    gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [M] * 3, theta=[3.0, 0.1, 0.01], batch=B, device=dev) if M else None
    opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=gpe)
    loop = ClosedLoop(quad, opt, torch.as_tensor(traj), torch.as_tensor(traj[:, 0, :].copy()))
    half = a.steps // 2
    for _ in range(half):
        loop.step()
    torch.cuda.synchronize()
    _capi.check(lib.qmpc_timing_enable(opt._h, 1))
    for _ in range(a.steps - half):
        loop.step()
    ms_lin, ms_ipm, cnt = C.c_double(), C.c_double(), C.c_int()
    _capi.check(lib.qmpc_timing_read(opt._h, C.byref(ms_lin), C.byref(ms_ipm), C.byref(cnt)))
    _capi.check(lib.qmpc_timing_enable(opt._h, 0))
    solve_ms = (ms_lin.value + ms_ipm.value) / max(cnt.value, 1)

    sx = torch.empty((B, N + 1, 13, 13), dtype=torch.float64, device=dev)
    su = torch.empty((B, N, 4, 13), dtype=torch.float64, device=dev)
    s = _capi.stream_ptr()
    cases = {"gain": (1, None), "full": (N, sx)}
    out = {"workload": f"random_smooth closed loop, B={B}, N={N}, M={M}, fp64, after {a.steps} fused steps",
           "timing": f"CUDA events around each of {a.calls} calls (after 10 untimed), per case",
           "card": card(), "solve_ms_per_step": solve_ms,
           "solve_note": f"qmpc_timing_* over the last {cnt.value} solves of the loop (linearize + solver kernels)"}
    for name, (n, sxp) in cases.items():
        for _ in range(10):
            _capi.check(lib.qmpc_eval_sens_x0(opt._h, n, _capi.ptr(sxp), _capi.ptr(su), s))
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.calls)]
        for e0, e1 in ev:
            e0.record()
            _capi.check(lib.qmpc_eval_sens_x0(opt._h, n, _capi.ptr(sxp), _capi.ptr(su), s))
            e1.record()
        torch.cuda.synchronize()
        t = np.array([e0.elapsed_time(e1) for e0, e1 in ev])
        st = opt.solver_status()[0]
        ok = st == 0
        sun = su.view(-1)[:B * n * 4 * 13].view(B, n, 4, 13)          # the call packs [B][n][4][13]
        finite = bool(torch.isfinite(sun[ok]).all()) and (sxp is None or bool(torch.isfinite(sx[ok]).all()))
        out[name] = {"n_stages": n, "states": sxp is not None, "median_ms": float(np.median(t)),
                     "p99_ms": float(np.percentile(t, 99)), "min_ms": float(t.min()),
                     "vehicles_status_ok": int(ok.sum().item()), "finite_for_status_ok": finite}

    g = torch.Generator(device=dev).manual_seed(5)
    xb = torch.randn((B, N + 1, 13), dtype=torch.float64, device=dev, generator=g)
    ub = torch.randn((B, N, 4), dtype=torch.float64, device=dev, generator=g)
    ub0 = torch.zeros_like(ub)
    ub0[:, 0] = ub[:, 0]
    x0b = torch.empty((B, 13), dtype=torch.float64, device=dev)
    yb = torch.empty((B, N, 17), dtype=torch.float64, device=dev)
    yeb = torch.empty((B, 13), dtype=torch.float64, device=dev)
    adj = {"adjoint": (None, ub0), "adjoint_full": (xb, ub)}
    for name, (xbp, ubp) in adj.items():
        call = lambda: _capi.check(lib.qmpc_eval_adjoint(opt._h, _capi.ptr(xbp), _capi.ptr(ubp), _capi.ptr(x0b),
                                                         _capi.ptr(yb), _capi.ptr(yeb), s))
        for _ in range(10):
            call()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.calls)]
        for e0, e1 in ev:
            e0.record()
            call()
            e1.record()
        torch.cuda.synchronize()
        t = np.array([e0.elapsed_time(e1) for e0, e1 in ev])
        ok = opt.solver_status()[0] == 0
        finite = all(bool(torch.isfinite(o[ok]).all()) for o in (x0b, yb, yeb))
        out[name] = {"x_bar": xbp is not None, "u_bar": "stage 0" if name == "adjoint" else "all",
                     "median_ms": float(np.median(t)), "p99_ms": float(np.percentile(t, 99)), "min_ms": float(t.min()),
                     "vehicles_status_ok": int(ok.sum().item()), "finite_for_status_ok": finite}
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
