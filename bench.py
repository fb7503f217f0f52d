#!/usr/bin/env python
"""bench.py — closed-loop RTI-MPC + RGP control steps/sec on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one closed-loop control step of EVERY vehicle on this rank: reference chunk -> RTI solve (RK4+sens,
Riccati IPM) -> u0 -> nominal prediction -> drag residual -> RGP regress x3 -> alpha, plus the plant period that
closes the loop; everything resident on the GPU.  Workload = BASELINE configs[1]: 4096 independent quads per GPU,
N=20, per-vehicle RGP (3 axes x 20 basis points), random-smooth references (SURVEY.md §8d).  Vehicles shard over
ranks with no data-path collective (weak scaling).

Legs of one run (all in the same JSON line; every key says which leg it belongs to):
  value            8 vehicle groups on 8 streams, `--steps` timed steps after `--warmup` (the driver's window)
  roofline         the same steps again on ONE stream with CUDA events around the solver launches (kernel durations)
  latency_ms       one stream, >= 200 steps after the warm-up: p50 / p99 / max of the batched step (CUDA events per step)
  e2e              host buffers in/out every step through quad_optimizer.step (pinned memory), references generated on the GPU
  lemniscate_leg   N = 1 only: BASELINE configs[4], 16384 vehicles, v_peak 20 m/s (thrust limits active), >= 200 steps, p99
  shared_rgp_leg   N > 1 only: BASELINE configs[2], 65536 vehicles over the ranks, ONE shared RGP, all-reduce every step
  cpu_baseline     N = 1 only: the C oracle on the host cores (+ the numpy RGP restatement on 1 core)

The library is not built here: run __graft_entry__.build() first.  bench.py writes nothing into the source tree.
"""
import argparse
import atexit
import ctypes as C
import gc
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: no __pycache__ next to the package
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # one hardware queue per vehicle-group stream

METRIC = "closed_loop_rti_mpc_rgp_control_steps_per_sec"
UNIT = "control_steps/s"
# dram__bytes_read.sum + dram__bytes_write.sum of the two solver launches of one control step (screening + dense) in the
# committed ncu --set full capture of the default shape (profiles/r02_solver_summary.txt); a profile constant
PROFILE_TRAFFIC_BYTES = 345.0e6      # step 60: 268.3 + 55.7 (screening) + 21.0 + 0.0 (dense) MB


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=4096, help="vehicles per GPU")
    ap.add_argument("--nodes", type=int, default=20)
    ap.add_argument("--basis", type=int, default=20)
    ap.add_argument("--precision", type=int, default=64, choices=[64, 32])
    ap.add_argument("--workload", default="random_smooth", choices=["random_smooth", "lemniscate"])
    ap.add_argument("--cpu-sample-vehicles", type=int, default=0, help="0 = auto (about 15 s of CPU work)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cold", action="store_true", help="disable the active-set warm start (cold IPM every step)")
    ap.add_argument("--groups", type=int, default=8, help="independent vehicle groups per GPU, one CUDA stream each (value leg)")
    ap.add_argument("--shared-rgp", action="store_true", help="BASELINE config 3: ONE RGP shared by all vehicles on all ranks (NCCL all-reduce per step)")
    ap.add_argument("--v-peak", type=float, default=15.0, help="lemniscate peak speed (m/s)")
    ap.add_argument("--warm-rounds", type=int, default=0, help="active-set rounds tried from the previous active set (0 = library default)")
    ap.add_argument("--mu-switch", type=float, default=0.0, help="IPM -> refinement hand-over complementarity (0 = library default)")
    ap.add_argument("--solver-opts", default="", help="qmpc_config solver-policy fields for A/B runs, e.g. screen_rounds=6,bail_round=3")
    ap.add_argument("--latency-steps", type=int, default=200, help="steps of the dedicated latency leg (p99 needs >= 200)")
    ap.add_argument("--no-extra-legs", action="store_true", help="skip the lemniscate (N=1) / shared-RGP (N>1) legs")
    ap.add_argument("--lemniscate-batch", type=int, default=16384)
    ap.add_argument("--swarm-total", type=int, default=65536, help="vehicles of the shared-RGP leg, over all ranks")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what their last step computed to DIR/<name>.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    a.policy = {kv.split("=")[0]: int(kv.split("=")[1]) for kv in a.solver_opts.split(",") if kv}
    return a


def workload_config(a, n_gpus):
    rgp = (f"ONE shared RGP 3x{a.basis} (information-form all-reduce per step, BASELINE configs[2])" if a.shared_rgp
           else f"per-vehicle RGP 3x{a.basis} basis points (BASELINE configs[1])")
    return {"workload": f"{a.batch} independent quads per GPU, N={a.nodes}, {rgp}, "
                        f"{a.workload} references, hummingbird model, closed loop with plant",
            "vehicles_per_gpu": a.batch, "n_nodes": a.nodes, "n_basis": a.basis, "t_horizon": 1.0,
            "references": a.workload,
            "sharding": (f"vehicles x{n_gpus} ranks; shared RGP: information-form all-reduce (NCCL) of [3][M*M+M] fp64 per control step"
                         if a.shared_rgp else f"vehicles x{n_gpus} ranks, no collective"),
            "reset_on_fail": a.policy.get("reset_on_fail", 0) >= 0,
            "groups_per_gpu": a.groups,
            "l2": "per-step working set (stage tiles 136 MB + factors 47 MB + RGP covariances 39 MB at the default "
                  "shape) exceeds the 126 MB L2; no explicit flush"}


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, arrays, B):
    """Writes the arrays a caller of the timed closed loop holds after its last step (rank 0's vehicles, in order) as
    out_dir/<name>.npy (float64): u0 [B,4] the control applied, x [B,13] the plant state after the control period,
    x_pred [B,13] the nominal one-period prediction, x_opt [B,N+1,13] / w_opt [B,N,4] the solver iterate, and with an
    RGP rgp_mu [*,3,M] / rgp_C [*,3,M,M] (one model per vehicle, or one shared).  Above DUMP_BYTES in all, the
    per-vehicle arrays keep a fixed seeded sample of vehicles whose indices go to vehicle_index.npy."""
    per_vehicle = {k for k, v in arrays.items() if v.shape[0] == B}
    vehicle_bytes = sum(arrays[k][0].size for k in per_vehicle) * 8
    shared_bytes = sum(v.size for k, v in arrays.items() if k not in per_vehicle) * 8
    keep = max(1, min(B, (DUMP_BYTES - shared_bytes) // (vehicle_bytes + 8)))     # + 8: its entry in vehicle_index
    idx = None if keep == B else np.sort(np.random.default_rng(0).choice(B, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        if idx is not None and k in per_vehicle:
            v = v[idx]
        np.save(os.path.join(out_dir, k + ".npy"), np.ascontiguousarray(v, dtype=np.float64))
    if idx is not None:
        np.save(os.path.join(out_dir, "vehicle_index.npy"), idx.astype(np.float64))


def make_trajectories(a, first_vehicle, count, K):
    from mpc_quad_ros_b200.trajectory import lemniscate_trajectories, random_smooth_trajectories
    dt = 1.0 / a.nodes
    # per-vehicle Philox stream (seed 1234 + global vehicle index): a rank generates only its own vehicles
    if a.workload == "lemniscate":
        return lemniscate_trajectories(count, K, dt, v_peak=a.v_peak, seed=1234 + first_vehicle)
    return random_smooth_trajectories(count, K, dt, seed=1234 + first_vehicle)


def make_refgen_params(a, first_vehicle, count, K):
    """generator parameters of the same references (trajectory.DeviceReference): (kind, params [count,32])"""
    from mpc_quad_ros_b200 import trajectory as T
    dt = 1.0 / a.nodes
    if a.workload == "lemniscate":
        return T.KIND_LEMNISCATE, T.lemniscate_params(count, v_peak=a.v_peak, seed=1234 + first_vehicle)
    return T.KIND_SINUSOIDS, T.random_smooth_params(count, K, dt, seed=1234 + first_vehicle)


# ------------------------------------------------------------------------------------------------ CPU legs

def host_threads():
    """all host threads this process may use (torchrun exports OMP_NUM_THREADS=1; the CPU legs override it)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_closed_loop(a, traj, x0, steps, nthreads):
    """the oracle's closed loop (oracle/qmpc_oracle.c, OpenMP over vehicles) on a bounded sample; returns steps/s"""
    from oracle import oracle as orc
    dt = 1.0 / a.nodes
    gp = orc.GPSpec(np.tile(np.linspace(-10, 10, a.basis), (3, 1)), np.array([3.0, 0.1, 0.01])) if a.basis else None
    loop = orc.ClosedLoop(orc.quad_hummingbird(), dt, a.nodes, traj, x0, gp=gp, nthreads=nthreads, mu_tol=1e-6)
    t0 = time.perf_counter()
    r = loop.run(steps, log=True)
    el = time.perf_counter() - t0
    return traj.shape[0] * steps / el, el, float(r["iters"].mean())


def reference_arm(a):
    """--impl reference: the reference's CPU path (C oracle port of acados RTI + numpy RGP, all host threads)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    nthreads = host_threads()
    # bounded sample of the same workload: first vehicles of the same trajectories, `steps` control steps
    Bs = a.cpu_sample_vehicles or min(a.batch, 64 * nthreads)
    K = a.warmup + a.steps + a.nodes + 2
    traj = make_trajectories(a, 0, Bs, K)
    x0 = traj[:, 0, :].copy()
    dt = 1.0 / a.nodes
    gp = orc.GPSpec(np.tile(np.linspace(-10, 10, a.basis), (3, 1)), np.array([3.0, 0.1, 0.01])) if a.basis else None
    loop = orc.ClosedLoop(orc.quad_hummingbird(), dt, a.nodes, traj, x0, gp=gp, nthreads=nthreads, mu_tol=1e-6)
    loop.run(a.warmup, log=False)
    t0 = time.perf_counter()
    loop.run(a.steps, log=False)
    el = time.perf_counter() - t0
    if a.dump_outputs:
        out = {"u0": loop.uit[:, 0], "x": loop.x, "x_pred": loop.xpred_prev, "x_opt": loop.xit, "w_opt": loop.uit}
        if gp is not None:
            out.update(rgp_mu=loop.mu, rgp_C=loop.C)
        dump_outputs(a.dump_outputs, out, Bs)
    val = Bs * a.steps / el
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": 1e3 * el / a.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(a, a.gpus),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": nthreads, "kind": "port",
                             "sample": f"{Bs} vehicles x {a.steps} steps of the same workload (C oracle, OpenMP over vehicles, "
                                       f"cold IPM to 1e-6 + exact active-set refinement)"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ clocks

class ClockSampler:
    """nvidia-smi in loop mode, started BEFORE the warm-up steps (the process takes ~0.1 s to deliver its first line, the
    driver's timed window is 40 ms long) and sampling every 10 ms; `mark()` brackets the timed region on the host clock.
    stop() reports the samples that fall inside the marks, or - if the window was too short to catch one - those taken
    under load since the warm-up began, and says which in `window`."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.marks = []
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "10",
                                       "-i", str(index)], stdout=self.f, stderr=subprocess.DEVNULL)
            atexit.register(self.p.kill)          # never outlives bench.py, also when a leg raises before stop()
        except Exception:
            self.p = None

    def mark(self):
        import datetime
        self.marks.append(datetime.datetime.now())

    def stop(self):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        rows = []
        for ln in self.f.read().splitlines():
            c = [t.strip() for t in ln.split(",")]
            if len(c) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f")
                rows.append((ts, float(c[1]), float(c[2]), [v.lower().startswith("active") for v in c[5:9]]))
            except ValueError:
                continue
        inside = [r for r in rows if len(self.marks) >= 2 and self.marks[0] <= r[0] <= self.marks[1]]
        use, window = (inside, "timed region") if inside else (rows, "warm-up + timed region (no sample fell inside the timed region)")
        if use:
            reasons = {name for r in use for name, on in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3]) if on}
            out = {"sm_mhz": float(np.median([r[1] for r in use])), "sm_max_mhz": float(max(r[2] for r in use)), "reasons": sorted(reasons),
                   "samples": len(use), "window": window}
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


# ------------------------------------------------------------------------------------------------ extra legs

def lemniscate_leg(a, dev, make_loop_generic):
    """BASELINE configs[4]: high-speed lemniscate (thrust limits active, many IPM iterations), 16384 quads on one GPU,
    references generated on the GPU; steps/s over the leg and the p50/p99/max latency of the batched step (one stream)"""
    import torch
    from mpc_quad_ros_b200 import trajectory as T
    Bl, N = a.lemniscate_batch, a.nodes
    steps, warm = max(a.latency_steps, 200), 20
    K = warm + steps + N + 2
    par = T.lemniscate_params(Bl, v_peak=20.0, seed=1234)
    x0 = T.lemniscate_trajectories(Bl, 1, 1.0 / N, v_peak=20.0, seed=1234)[:, 0, :]
    loop = make_loop_generic(Bl, None, x0, (T.KIND_LEMNISCATE, par, K))
    for _ in range(warm):
        loop.step()
    torch.cuda.synchronize()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    evs[0].record()
    for s in range(steps):
        loop.step()
        evs[s + 1].record()
    torch.cuda.synchronize()
    lat = np.array([evs[s].elapsed_time(evs[s + 1]) for s in range(steps)])
    st, it = loop.opt.solver_status()
    sat = float(((loop.u0 <= 1e-9) | (loop.u0 >= 1 - 1e-9)).double().mean().item())
    return {"workload": f"{Bl} quads, lemniscate a=10 m, v_peak 20 m/s, N={N}, per-vehicle RGP 3x{a.basis} (BASELINE configs[4])",
            "leg": f"one stream, {steps} timed steps after {warm} warm-up steps, references generated on the GPU",
            "value": Bl * steps / (lat.sum() * 1e-3), "unit": UNIT, "ms_per_step": float(lat.mean()),
            "latency_ms": {"p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99)), "max": float(lat.max())},
            "saturated_u0_frac_last_step": sat, "status_not_ok_last_step": int((st != 0).sum().item()),
            "ipm_iters_mean_last_step": float(it.double().mean().item())}


def shared_rgp_leg(a, dev, rank, world, make_loop_generic, barrier):
    """BASELINE configs[2]: 65536-quad swarm sharded over the ranks with ONE shared RGP; every control step all-reduces
    the information-form block [3][M*M+M] (NCCL), overlapped with the step's solve (swarm.SharedSwarmRGP.begin/end)"""
    import torch
    import torch.distributed as dist
    from mpc_quad_ros_b200 import trajectory as T
    from mpc_quad_ros_b200.swarm import shard_range
    N, M = a.nodes, a.basis
    first, count = shard_range(a.swarm_total, rank, world)
    steps, warm = max(a.steps, 20), max(a.warmup, 3)
    K = warm + steps + N + 2
    par = T.random_smooth_params(count, K, 1.0 / N, seed=1234 + first)
    x0 = np.zeros((count, 13)); x0[:, 3] = 1.0; x0[:, 2] = 3.0
    amp, ph = par[:, 0:9].reshape(count, 3, 3), par[:, 18:27].reshape(count, 3, 3)
    f = par[:, 9:18].reshape(count, 3, 3)
    x0[:, 7:10] = (amp * 2 * np.pi * f * np.cos(ph)).sum(2) * par[:, 27:28]           # reference velocity at t = 0
    loop = make_loop_generic(count, None, x0, (T.KIND_SINUSOIDS, par, K), shared=True)
    loop.shared_swarm.time_allreduce = True
    for _ in range(warm):
        loop.step()
    barrier()
    loop.shared_swarm.allreduce_ms.clear()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loop.step()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ar = [x.elapsed_time(y) for x, y in loop.shared_swarm.allreduce_ms]
    ar_t = torch.tensor([float(np.mean(ar)) if ar else 0.0], dtype=torch.float64, device=dev)
    dist.all_reduce(ar_t, op=dist.ReduceOp.MAX)
    mu = loop.opt.gpe.mu_tensor()
    mu_max = mu.clone(); mu_min = mu.clone()
    dist.all_reduce(mu_max, op=dist.ReduceOp.MAX); dist.all_reduce(mu_min, op=dist.ReduceOp.MIN)
    st, _ = loop.opt.solver_status()
    bad = torch.tensor([int((st != 0).sum().item())], dtype=torch.int64, device=dev)
    dist.all_reduce(bad)
    return {"workload": f"{a.swarm_total} quads over {world} ranks ({count} per rank), N={N}, ONE shared RGP 3x{M} (BASELINE configs[2]), "
                        "random_smooth references generated on the GPU",
            "leg": f"one stream + side stream per rank, {steps} timed steps after {warm} warm-up steps, max over ranks",
            "value": a.swarm_total * steps / (float(t.item()) * 1e-3), "unit": UNIT, "ms_per_step": float(t.item()) / steps,
            "allreduce_us_per_step": 1e3 * float(ar_t.item()), "allreduce_bytes": 3 * (M * M + M) * 8,
            "allreduce_note": "CUDA events around dist.all_reduce on the side stream (includes waiting for the slowest rank's "
                              "accumulate); the exchange overlaps the solve of the same step",
            "model_identical_on_all_ranks": bool(torch.equal(mu_max, mu_min)),
            "status_not_ok_last_step": int(bad.item())}


# ------------------------------------------------------------------------------------------------ B200 arm

def flops_per_step(N, M, n_ipm):
    """ALGORITHMIC flops per vehicle-step (SURVEY.md §8d): N*(22116+108M) + n_ipm*12067*N + 24M^2+45M + 2000"""
    return N * (22116 + 108 * M) + n_ipm * 12067 * N + 24 * M * M + 45 * M + 2000


def b200_arm(a):
    import torch
    import torch.distributed as dist
    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
        dist.barrier()
    assert torch.cuda.is_available(), "bench.py --impl b200 needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    from mpc_quad_ros_b200 import _capi
    from mpc_quad_ros_b200.execute_trajectory import ClosedLoop, GroupedClosedLoop
    from mpc_quad_ros_b200.gp.GPE import GPEnsemble
    from mpc_quad_ros_b200.quad import Quadrotor3D
    from mpc_quad_ros_b200.quad_opt import quad_optimizer
    from mpc_quad_ros_b200.swarm import SharedSwarmRGP
    lib = _capi.lib()

    B, N, M = a.batch, a.nodes, a.basis
    K = a.warmup + a.steps + N + 2
    traj_np = make_trajectories(a, rank * B, B, K)
    x0_np = traj_np[:, 0, :].copy()

    par_kind, par_np = make_refgen_params(a, rank * B, B, K)

    def make_loop_generic(count, traj, x0, refgen_spec=None, shared=False, policy=None):
        """closed loop over `count` vehicles; refgen_spec = (kind, params, K): references generated on the GPU"""
        from mpc_quad_ros_b200.trajectory import DeviceReference
        quad = Quadrotor3D(drag=True, batch=count, device=dev).set_hummingbird_params()
        gpe = GPEnsemble.fromrange([(-10, 10)] * 3, [M] * 3, theta=[3.0, 0.1, 0.01], batch=(1 if shared else count), device=dev) if M else None
        opt = quad_optimizer(quad, t_horizon=1.0, n_nodes=N, gpe=gpe, precision=a.precision,
                             warm_start_rounds=(-1 if a.cold else a.warm_rounds), ipm_mu_switch=a.mu_switch,
                             **(a.policy if policy is None else policy))
        swarm = SharedSwarmRGP(gpe, opt) if (shared and M) else None
        src = torch.as_tensor(traj) if refgen_spec is None else DeviceReference(refgen_spec[0], refgen_spec[1], refgen_spec[2], 1.0 / N, device=dev)
        return ClosedLoop(quad, opt, src, torch.as_tensor(x0), shared_swarm=swarm)

    def make_loop(first=0, count=None, refgen=False):
        count = B if count is None else count
        spec = (par_kind, par_np[first:first + count], K) if refgen else None
        return make_loop_generic(count, traj_np[first:first + count], x0_np[first:first + count], spec, shared=a.shared_rgp)

    def barrier():
        # handles of finished legs are released here, never inside a timed region (their destructors call cudaFree,
        # which synchronises the device); the collector stays off while a region is timed
        gc.collect()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    gc.disable()

    # ---------------- value: everything resident, K timed steps
    if B % max(a.groups, 1) != 0:
        a.groups = 1
    grouped = a.groups > 1 and not a.shared_rgp
    loop = GroupedClosedLoop(make_loop, B, a.groups) if grouped else make_loop()
    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(a.warmup):
        loop.step()
    barrier()
    if sampler:
        sampler.mark()
    l0 = lib.qmpc_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    if grouped:
        loop.fork()
    for _ in range(a.steps):
        loop.step()
    if grouped:
        loop.join()
    e1.record()
    barrier()
    if sampler:
        sampler.mark()
    ms = e0.elapsed_time(e1)
    launches = lib.qmpc_launch_count() - l0
    clocks = sampler.stop() if sampler else None
    opts = [lp.opt for lp in loop.loops] if grouped else [loop.opt]
    st = torch.cat([o.solver_status()[0] for o in opts]); it = torch.cat([o.solver_status()[1] for o in opts])
    n_ipm_last = float(it.double().mean().item())
    bad = int((st != 0).sum().item())
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * B * a.steps / (ms_max * 1e-3)
    if a.dump_outputs and rank == 0:
        lps = loop.loops if grouped else [loop]
        host = lambda ts: torch.cat(ts).cpu().numpy()
        its = [lp.opt.get_iterate() for lp in lps]
        out = {"u0": host([lp.u0 for lp in lps]), "x": host([lp.x for lp in lps]), "x_pred": host([lp.x_pred_prev for lp in lps]),
               "x_opt": host([i[0] for i in its]), "w_opt": host([i[1] for i in its])}
        if M:
            gpes = [lp.opt.gpe for lp in lps]
            out.update(rgp_mu=host([g.mu_tensor() for g in gpes]), rgp_C=host([g.C_tensor() for g in gpes]))
        dump_outputs(a.dump_outputs, out, B)

    # ---------------- roofline leg: same steps again on ONE stream with cudaEvents around the solve kernels
    loop2 = make_loop()
    for _ in range(a.warmup):
        loop2.step()
    gc.collect()
    torch.cuda.synchronize()
    _capi.check(lib.qmpc_timing_enable(loop2.opt._h, 1))
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record()
    for s in range(a.steps):
        loop2.step()
    r1.record()
    torch.cuda.synchronize()
    ms_single = r0.elapsed_time(r1) / a.steps
    ms_lin, ms_ipm, cnt = C.c_double(), C.c_double(), C.c_int()
    _capi.check(lib.qmpc_timing_read(loop2.opt._h, C.byref(ms_lin), C.byref(ms_ipm), C.byref(cnt)))
    ms_dense = C.c_double()
    _capi.check(lib.qmpc_timing_read_dense(loop2.opt._h, C.byref(ms_dense)))
    _capi.check(lib.qmpc_timing_enable(loop2.opt._h, 0))
    del loop2

    # ---------------- latency leg: one stream, >= 200 steps after the warm-up, CUDA events around every batched step
    # (SURVEY 8d: p99 from inputs-ready to u0-ready; p99 over 20 samples would be the maximum)
    n_lat = max(a.latency_steps, 1)
    K_lat = a.warmup + n_lat + N + 2                    # its own, longer references (same generator and seeds)
    kind_l, par_l = make_refgen_params(a, rank * B, B, K_lat)
    x0_l = make_trajectories(a, rank * B, B, 1)[:, 0, :] if a.workload == "lemniscate" else x0_np
    loopL = make_loop_generic(B, None, x0_l, (kind_l, par_l, K_lat), shared=a.shared_rgp)
    for _ in range(a.warmup):
        loopL.step()
    gc.collect()
    torch.cuda.synchronize()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_lat + 1)]
    evs[0].record()
    for s in range(n_lat):
        loopL.step()
        evs[s + 1].record()
    torch.cuda.synchronize()
    lat = np.array([evs[s].elapsed_time(evs[s + 1]) for s in range(n_lat)])
    del loopL, evs

    # mean IPM iterations over a few sampled steps of a third short pass (host reads are outside any timed region)
    loop3 = make_loop()
    n_ipm, n_rounds, n_warm_ok = [], [], []
    for s in range(a.warmup + min(a.steps, 20)):
        loop3.step()
        if s >= a.warmup:
            it3 = loop3.opt.solver_status()[1].double()
            n_ipm.append(float(it3.mean().item()))
            n_rounds.append(float(loop3.opt.solver_rounds().double().mean().item()))
            n_warm_ok.append(float((it3 == 0).double().mean().item()))
    del loop3
    n_ipm_mean = float(np.mean(n_ipm)) if n_ipm else n_ipm_last
    n_rounds_mean = float(np.mean(n_rounds)) if n_rounds else 0.0
    n_fact = n_ipm_mean + n_rounds_mean          # Riccati factorisations per vehicle-step
    peak = C.c_double()
    _capi.check(lib.qmpc_fma_peak(a.precision, C.byref(peak), _capi.stream_ptr()))
    ipm_ms = ms_ipm.value / max(cnt.value, 1)
    ipm_flops = B * n_fact * 12067 * N                # algorithmic flops of the solver launches per step (SURVEY §8d F_ipm per factorisation)
    achieved = ipm_flops / (ipm_ms * 1e-3) / 1e12 if ipm_ms > 0 else 0.0
    # DRAM traffic of the solver launches: constant of the committed ncu --set full capture of this exact shape
    # (profiles/r02_solver_summary.txt: screening launch + dense launch), NOT measured in this run; other shapes: null
    traffic = PROFILE_TRAFFIC_BYTES if (B, N, M, a.precision, a.workload, a.cold) == (4096, 20, 20, 64, "random_smooth", False) else None
    roofline = {"kernel": "qmpc_ipm_kernel (warm-started Riccati screening) + qmpc_dense_kernel (condensed IPM/active-set for the rest)"
                          if a.precision == 64 and N <= 21 else "qmpc_ipm_kernel",
                "leg": "roofline: single-stream replay of the timed steps, cudaEvents around the launches on their own stream",
                "bound": "fp%d_fma" % a.precision, "achieved": achieved, "peak": peak.value,
                "unit": "TFLOP/s", "frac": achieved / peak.value if peak.value else None, "traffic": traffic,
                "traffic_source": "profile constant (ncu --set full, profiles/r02_solver_summary.txt), not measured in this run",
                "peak_source": "measured in this run by qmpc_fma_peak (register-resident FMA microbenchmark); "
                               "MEASURED_PEAKS.json has no FMA figure",
                "ms_per_launch": ipm_ms, "ms_dense_per_launch": ms_dense.value / max(cnt.value, 1),
                "ms_linearize_per_launch": ms_lin.value / max(cnt.value, 1),
                "ms_per_step_single_stream": ms_single,
                "share_of_step": ipm_ms / ms_single if ms_single > 0 else None,   # within this single-stream leg
                "n_ipm_mean": n_ipm_mean, "n_refine_rounds_mean": n_rounds_mean, "n_factorisations_mean": n_fact,
                "warm_start_success_frac": float(np.mean(n_warm_ok)) if n_warm_ok else None,
                "algorithmic_flops_per_vehicle_step": flops_per_step(N, M, n_fact),
                "whole_step_tflops": value / world * flops_per_step(N, M, n_fact) / 1e12,
                "whole_step_frac": (value / world * flops_per_step(N, M, n_fact) / 1e12) / peak.value if peak.value else None}

    # ---------------- secondary roofline: the linearisation kernel (K1), the one FMA-throughput-bound kernel of the step
    lin_ms = ms_lin.value / max(cnt.value, 1)
    lin_flops = B * N * (22116 + 108 * M)
    lin_ach = lin_flops / (lin_ms * 1e-3) / 1e12 if lin_ms > 0 else 0.0
    roofline_lin = {"kernel": "qmpc_linearize_kernel", "leg": "roofline", "bound": "fp%d_fma" % a.precision, "achieved": lin_ach, "peak": peak.value,
                    "unit": "TFLOP/s", "frac": lin_ach / peak.value if peak.value else None, "traffic": None,
                    "ms_per_launch": lin_ms, "note": "algorithmic flops N*(22116+108M) per vehicle (SURVEY 8d), i.e. dense Jacobians and one exp per kernel value; the "
                                                      "kernel itself evaluates the primal + GP once per node (3 exps per equispaced axis) and 14 tangent "
                                                      "columns on cached Jacobian blocks: 51M warp instructions per launch at 4096x20 (round-2 start: 258M)"}

    # ---------------- secondary roofline: the HBM-bound RGP update (K3), timed alone with CUDA events
    roofline_rgp = None
    if M and not a.shared_rgp:
        gtest = GPEnsemble.fromrange([(-10, 10)] * 3, [M] * 3, theta=[3.0, 0.1, 0.01], batch=B, device=dev)
        xt = torch.rand((B, 3), dtype=torch.float64, device=dev) * 16 - 8
        yt = -0.3 * xt
        for _ in range(3):
            _capi.check(lib.qrgp_regress(gtest._h, _capi.ptr(xt), _capi.ptr(yt), _capi.stream_ptr()))
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20
        g0.record()
        for _ in range(reps):
            _capi.check(lib.qrgp_regress(gtest._h, _capi.ptr(xt), _capi.ptr(yt), _capi.stream_ptr()))
        g1.record()
        torch.cuda.synchronize()
        rgp_ms = g0.elapsed_time(g1) / reps
        rgp_bytes = B * 3 * 16 * M * M                 # C read + written once per (vehicle, axis): 16 M^2 bytes
        hbm_peak = None
        try:
            hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        except Exception:
            pass
        peak_gbs = hbm_peak if hbm_peak else 6650.0
        ach = rgp_bytes / (rgp_ms * 1e-3) / 1e9
        roofline_rgp = {"kernel": "qrgp_regress_tma_kernel", "leg": "stand-alone launches", "bound": "hbm", "achieved": ach, "peak": peak_gbs, "unit": "GB/s",
                        "frac": ach / peak_gbs, "traffic": None, "ms_per_launch": rgp_ms,
                        "peak_source": "MEASURED_PEAKS.json hbm_gbs" if hbm_peak else "fallback 6650 GB/s (B200_PROFILING.md)",
                        "note": "covariances of 4096 vehicles (39 MB) fit the 126 MB L2 when launched back to back"}
        del gtest

    # ---------------- e2e: host state in, host control out, every step, through the Python API (pinned memory).
    # The references are generated on the GPU (trajectory.DeviceReference): only x_now [B,13] goes up, u0 [B,4] comes down.
    e2e = None
    if not a.no_e2e:
        rec = make_loop()
        xs, us = rec.run(a.warmup + a.steps, record=True)          # states a closed loop really visits
        torch.cuda.synchronize()
        xs_host = xs.cpu().pin_memory()
        del rec, xs, us
        # G independent vehicle groups, one stream each: a group's copies overlap the other groups' kernels
        G = 1 if a.shared_rgp else a.groups
        per = B // G
        streams = [torch.cuda.Stream() for _ in range(G)]
        grp = []
        for gi in range(G):
            with torch.cuda.stream(streams[gi]):
                grp.append(dict(lp=make_loop(gi * per, per, refgen=True), lo=gi * per, hi=(gi + 1) * per,
                                x=torch.empty((per, 13), dtype=torch.float64, device=dev)))
        torch.cuda.synchronize()
        u_host = torch.empty((B, 4), dtype=torch.float64).pin_memory()

        done = [None] * G      # per group: event recorded after the D2H copy of its previous step

        def e2e_step(i):
            # every group is its own closed loop: the host waits for THAT group's u0 of the previous step, then feeds
            # its next state (pinned host -> device), runs the control step and reads u0 back
            for gi, (st_, g) in enumerate(zip(streams, grp)):
                if done[gi] is not None:
                    done[gi].synchronize()
                with torch.cuda.stream(st_):
                    g["x"].copy_(xs_host[i, g["lo"]:g["hi"]], non_blocking=True)
                    u0 = g["lp"].control(g["x"], i)
                    u_host[g["lo"]:g["hi"]].copy_(u0, non_blocking=True)
                    done[gi] = torch.cuda.Event()
                    done[gi].record(st_)

        def e2e_drain():
            for ev in done:
                if ev is not None:
                    ev.synchronize()

        for i in range(a.warmup):
            e2e_step(i)
        e2e_drain()
        barrier()
        t0 = time.perf_counter()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for i in range(a.warmup, a.warmup + a.steps):
            e2e_step(i)
        e2e_drain()                                                 # every u0 of the last step is on the host
        wall = (time.perf_counter() - t0) * 1e3                     # host clock: ends when the host holds the last control
        g1.record()
        barrier()
        te = torch.tensor([max(g0.elapsed_time(g1), wall)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = {"value": world * B * a.steps / (float(te.item()) * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": B * 13 * 8, "d2h_bytes_per_step": B * 4 * 8,
               "ms_per_step": float(te.item()) / a.steps,
               "note": "per step: pinned-host x_now [B,13] -> device, reference chunk generated on the GPU, quad_optimizer.step, "
                       "u0 [B,4] -> pinned host; each vehicle group (own stream) waits for its own u0 before its next step; "
                       "states replayed from a recorded closed loop"}
        del grp

    # ---------------- extra legs: the other BASELINE configs in front of the driver
    lem_leg = swarm_leg = None
    if not a.no_extra_legs and world == 1 and not a.shared_rgp and a.workload == "random_smooth":
        lem_leg = lemniscate_leg(a, dev, make_loop_generic)
    if not a.no_extra_legs and world > 1 and M:
        swarm_leg = shared_rgp_leg(a, dev, rank, world, make_loop_generic, barrier)

    # ---------------- CPU baseline beside it (rank 0, N=1 only): bounded sample of the same workload
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        nthreads = host_threads()
        Bc = min(B, 4 * nthreads)
        v, el, _ = cpu_closed_loop(a, traj_np[:Bc], x0_np[:Bc], 5, nthreads)          # calibrate
        steps_cpu = a.warmup + a.steps                                               # same control steps as the GPU run
        Bs = a.cpu_sample_vehicles or int(max(nthreads, min(B, 15.0 * v / steps_cpu)))  # about 15 s of CPU work
        v, el, it_cpu = cpu_closed_loop(a, traj_np[:Bs], x0_np[:Bs], steps_cpu, nthreads)
        cpu = {"value": v, "unit": UNIT, "cores": nthreads, "kind": "port",
               "sample": f"first {Bs} vehicles x {steps_cpu} steps of the same workload, {el:.1f} s, C oracle with OpenMP over vehicles "
                         f"(exact QP: cold IPM to 1e-6 + active-set refinement, mean {it_cpu:.1f} IPM iterations)"}
        if M:
            # SURVEY 8d-ii: the reference's numpy RGP as shipped (Python-level loops), 1 core: oracle/rgp_numpy.py
            from oracle.rgp_numpy import time_three_axis_updates
            sec = time_three_axis_updates(M, 200)
            cpu["numpy_rgp_1core"] = {"ms_per_vehicle_step": 1e3 * sec, "vehicle_steps_per_s": 1.0 / sec, "cores": 1, "kind": "port",
                                      "sample": f"200 three-axis RGP.regress updates at M={M} (numpy restatement of reference src/gp/RGP.py:303-330 "
                                                "with its per-entry kernel calls)"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": ms_max / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f%d" % a.precision, "data": "synthetic", "config": workload_config(a, world),
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "roofline_linearize": roofline_lin, "roofline_rgp": roofline_rgp, "cpu_baseline": cpu,
                "latency_ms": {"leg": f"latency: one stream, {n_lat} steps after {a.warmup} warm-up steps", "steps": n_lat,
                               "p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99)), "max": float(lat.max())},
                "lemniscate_leg": lem_leg, "shared_rgp_leg": swarm_leg,
                "solver": {"status_not_ok_last_step": bad, "ipm_iters_mean": n_ipm_mean, "refine_rounds_mean": n_rounds_mean,
                           "warm_start": (not a.cold)}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        reference_arm(args)
    else:
        b200_arm(args)
