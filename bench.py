#!/usr/bin/env python
"""Benchmark of the per-timestep hot path: full-timestep Mcell-updates/s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--scaling strong|weak]
                    [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the example loop body (reference ``examples/3d_examples/*``):
``dt = compute_stable_timestep()``, ``interactor()``, ``interactor.time_step(dt)``,
``flow_sim.time_step(dt)``, on synthetic fields.  Default workload: ``fsi_512_f32``, the north-star
target (512^3 float32, flow_type "navier_stokes_with_forcing" with a virtual-boundary-forcing sphere:
forcing update + rotational-form update + diffusion + penalise + unbounded FFT Poisson + curl +
immersed-boundary interpolation / spreading), strong-scaled over z-slabs for N > 1
(BASELINE.json configs[4]).  One JSON line is printed by rank 0.

The K timed steps always start from the synthetic initial condition, whatever number of warm-up steps
it took to bring the clocks up, so that the same arguments compute the same steps.  ``--dump-outputs
DIR`` (one process) writes what the last timed step handed its caller as ``DIR/<name>.npy``: see
``dump_outputs``.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

# stdout carries ONE JSON line: while the benchmark runs, file descriptor 1 points at stderr so that
# anything the libraries print (NCCL's version banner, ...) stays out of it; emit() restores it
_STDOUT_FD = None


def capture_stdout():
    """Called by main() only (importing this module must not touch the descriptors)."""
    global _STDOUT_FD
    if _STDOUT_FD is None:
        sys.stdout.flush()
        _STDOUT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    if _STDOUT_FD is not None:
        os.dup2(_STDOUT_FD, 1)
    print(json.dumps(line), flush=True)
    if _STDOUT_FD is not None:
        os.dup2(2, 1)


ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "full_timestep_Mcell_updates_per_s"
UNIT = "Mcell-updates/s"
FALLBACK_HBM_GBS = 6650.0
DEFAULT_WORKLOAD = "fsi_512_f32"
# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel, per workload, written
# by `tools/ncu_summary.py --traffic-json` from the `ncu --set full` captures kept under profiles/
NCU_TRAFFIC_JSON = os.path.join(ROOT, "profiles", "ncu_traffic.json")

WORKLOADS = {
    # name: (grid (z,y,x), flow_type, immersed body, real_t)
    # north-star target / BASELINE configs[4]: full FSI step at 512^3 float32 (sphere, D = 0.4, ~1.3e5 points)
    "fsi_512_f32": ((512, 512, 512), "navier_stokes_with_forcing", "sphere", "f32"),
    "fsi_256_f32": ((256, 256, 256), "navier_stokes_with_forcing", "sphere", "f32"),
    # BASELINE configs[1]
    "vortex_ring_256_f32": ((256, 256, 256), "navier_stokes", None, "f32"),
    "vortex_ring_128_f32": ((128, 128, 128), "navier_stokes", None, "f32"),
    "vortex_ring_512_f32": ((512, 512, 512), "navier_stokes", None, "f32"),
    "vortex_ring_256_f64": ((256, 256, 256), "navier_stokes", None, "f64"),
    "vortex_ring_128_f64": ((128, 128, 128), "navier_stokes", None, "f64"),
    # BASELINE configs[2]
    "sphere_vbf_512x256x256_f32": ((256, 256, 512), "navier_stokes_with_forcing", "sphere", "f32"),
    # BASELINE configs[3]: rod in cross-flow; x_range 1.8, Laplacian filter order 1 (multiplicative),
    # synthetic rod surface grid (160 rings x 64 points + caps ~ 10 k points), 3 velocity
    # interpolations (rod sub-steps) + 1 full interaction per flow step (SURVEY 8(d))
    "rod_fsi_512x256x256_f32": ((256, 256, 512), "navier_stokes_with_forcing", "rod", "f32"),
    "rod_fsi_128x64x64_f32": ((64, 64, 128), "navier_stokes_with_forcing", "rod", "f32"),
}


def rod_surface_points(x_range, y_range, z_range, n_elem=160, n_ring=64):
    """Straight rod of length 1 along x, diameter y_range / 5, centred in the box."""
    length, radius = 1.0, y_range / 10.0
    x0 = 0.5 * (x_range - length)
    xs = x0 + (np.arange(n_elem) + 0.5) * length / n_elem
    th = 2 * np.pi * np.arange(n_ring) / n_ring
    ring = np.stack([np.zeros(n_ring), radius * np.cos(th), radius * np.sin(th)])
    pts = [np.stack([np.full(n_ring, x), 0.5 * y_range + ring[1], 0.5 * z_range + ring[2]]) for x in xs]
    for xc in (x0, x0 + length):  # caps: concentric rings
        for frac in (0.25, 0.5, 0.75):
            m = max(int(n_ring * frac), 4)
            t2 = 2 * np.pi * np.arange(m) / m
            pts.append(np.stack([np.full(m, xc), 0.5 * y_range + frac * radius * np.cos(t2),
                                 0.5 * z_range + frac * radius * np.sin(t2)]))
    return np.concatenate(pts, axis=1)


def vortex_ring(x, y, z, real_t):
    """Gaussian-core vortex ring (SURVEY 8(d) config 2): R=0.125, a=0.2R, centre
    (0.5,0.5,0.35), axis +z, Gamma=1.  x,y,z: broadcastable coordinate arrays."""
    R, gamma = 0.125, 1.0
    a = 0.2 * R
    rho = np.sqrt((x - 0.5) ** 2 + (y - 0.5) ** 2)
    w_theta = gamma / (np.pi * a * a) * np.exp(-((rho - R) ** 2 + (z - 0.35) ** 2) / (a * a))
    rho = np.maximum(rho, 1e-12)
    wx = -w_theta * (y - 0.5) / rho
    wy = w_theta * (x - 0.5) / rho
    return np.stack([wx + 0 * z, wy + 0 * z, 0 * wx + 0 * z]).astype(real_t)


def sphere_points(centre, diameter, spacing):
    """latitude rings with (about) `spacing` between neighbours"""
    r = diameter / 2
    n_lat = max(int(np.pi * r / spacing), 2)
    pts = []
    for i in range(n_lat + 1):
        th = np.pi * i / n_lat
        n_lon = max(int(2 * np.pi * r * np.sin(th) / spacing), 1)
        ph = 2 * np.pi * np.arange(n_lon) / n_lon
        pts.append(np.stack([centre[0] + r * np.sin(th) * np.cos(ph), centre[1] + r * np.sin(th) * np.sin(ph),
                             np.full(n_lon, centre[2] + r * np.cos(th))]))
    return np.ascontiguousarray(np.concatenate(pts, axis=1))


def workload_setup(name, grid):
    """Everything both arms (GPU product, CPU oracle) need to build the same problem."""
    _, flow_type, body, prec = WORKLOADS[name]
    nz, ny, nx = grid
    real_t = np.float32 if prec == "f32" else np.float64
    x_range = 1.8 if body == "rod" else 1.0
    y_range, z_range = x_range * ny / nx, x_range * nz / nx
    dx = x_range / nx
    w = dict(name=name, grid=tuple(grid), flow_type=flow_type, body=body, real_t=real_t, prec=prec, x_range=x_range,
             y_range=y_range, z_range=z_range, dx=dx, nu=1.0 / 1000.0, sim_kw={}, points=None, lag_vel=None,
             u_inf=[1.0, 0.0, 0.0] if body else [0.0, 0.0, 0.0], substeps=0)
    if body == "rod":
        w["sim_kw"] = dict(filter_vorticity=True, filter_setting_dict={"order": 1, "type": "multiplicative"})
        w["points"] = rod_surface_points(x_range, y_range, z_range)
        w["lag_vel"] = 0.01 * np.random.default_rng(1234).standard_normal(w["points"].shape)
        w["k"], w["c"] = -2e5, -1e2  # flow_past_rod_case.py:24-25
        w["substeps"] = 3
    elif body == "sphere":
        diameter = 0.4 * min(nz, ny) / nx * x_range
        w["points"] = sphere_points((0.25 * x_range, 0.5 * y_range, 0.5 * z_range), diameter, dx)
        w["lag_vel"] = np.zeros_like(w["points"])
        w["k"], w["c"] = -6e5 / 4, -3.5e2 / 4  # flow_past_sphere_case.py
    return w


def initial_vorticity(w, local_x, local_y, local_z):
    """the ring, every axis scaled to the unit cube so that it sits inside non-cubic boxes too"""
    x = np.asarray(local_x)[None, None, :].astype(np.float64) / w["x_range"]
    y = np.asarray(local_y)[None, :, None].astype(np.float64) / w["y_range"]
    z = np.asarray(local_z)[:, None, None].astype(np.float64) / w["z_range"]
    return vortex_ring(x, y, z, w["real_t"])


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic(name):
    try:
        return float(json.load(open(NCU_TRAFFIC_JSON))[name]["dram_bytes_per_launch"])
    except Exception:
        return None


class ClockSampler:
    def __init__(self, device_index):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(device_index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        self.first = 0

    def mark(self):
        """Samples taken from now on belong to the timed region."""
        try:
            self.first = sum(1 for _ in open(self.path))
        except OSError:
            self.first = 0

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = open(self.path).read().splitlines()
        timed = lines[self.first:]
        # a short timed region may see no 20 ms sample of its own: fall back to the last samples of
        # the (>= 1 s, same workload) warm-up that precedes it
        for line in (timed if len(timed) >= 2 else lines[-10:]):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons)}
        try:
            os.remove(self.path)
        except OSError:
            pass
        return out


# ------------------------------------------------------------------ CPU arm (oracle/)
# Host-memory need of the oracle at the workload's grid: ~16 padded fields + the doubled-domain FFT
# buffers (real, two spectra, result, Green's function and its spectrum) ~ 64 reals per cell.
def cpu_oracle_worker(name, grid, steps, warmup):
    """Runs in its own process (see run_cpu_oracle): the reference's CPU path restated (oracle/: numpy
    stencils, scipy.fft on all host cores, vectorised numpy gather / scatter for the Lagrangian
    kernels) on the SAME workload as the GPU arm: same grid, flow type, body, step sequence."""
    from oracle import ib as ib_oracle
    from oracle.simulator import FlowSimulatorOracle3D

    w = workload_setup(name, grid)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    t_setup = time.perf_counter()
    sim = FlowSimulatorOracle3D(w["grid"], w["x_range"], w["nu"], flow_type=w["flow_type"], real_t=w["real_t"],
                                with_free_stream_flow=bool(w["body"]), fft_workers=cores, **w["sim_kw"])
    sim.vorticity_field[...] = initial_vorticity(w, sim.local_x, sim.local_y, sim.local_z)
    u_inf = w["u_inf"]
    sim.compute_flow_velocity(u_inf)
    vbf = None
    if w["body"]:
        area = w["dx"] ** 2
        vbf = ib_oracle.VirtualBoundaryForcingOracle(w["k"] * area, w["c"] * area, 3, sim.dx, w["real_t"], np.float64,
                                                     sim.gs, fast=True)
    pts, vel = w["points"], w["lag_vel"]

    def one_step():
        dt = sim.compute_stable_timestep(dt_prefac=0.5)
        if vbf is not None:
            for _ in range(w["substeps"]):
                vbf.compute_interaction_force_on_lag_grid(sim.velocity_field, pts, vel)
            vbf.compute_interaction_force_on_eul_and_lag_grid(sim.eul_grid_forcing_field, sim.velocity_field, pts, vel)
            vbf.time_step(dt)
        sim.time_step(dt, u_inf)

    for _ in range(warmup):
        one_step()
    setup_s = time.perf_counter() - t_setup
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    cells = float(np.prod(grid))
    print(json.dumps({"value": cells / dt / 1e6, "ms_per_step": dt * 1e3, "cores": cores, "steps": steps,
                      "warmup": warmup, "setup_s": setup_s, "grid": list(grid),
                      "lagrangian_points": 0 if pts is None else int(pts.shape[1])}), flush=True)


def run_cpu_oracle(name, grid, steps, warmup, timeout_s=1500):
    """The CPU oracle in a child process with a clean threading environment: torchrun exports
    OMP_NUM_THREADS=1, which (read at library load) cut scipy.fft's worker pool and made this arm 2.4x
    slower under `torch.distributed.run` than stand-alone in round 1."""
    env = {k: v for k, v in os.environ.items()
           if k not in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS", "RANK", "WORLD_SIZE",
                        "LOCAL_RANK")}
    env["CUDA_VISIBLE_DEVICES"] = ""
    cmd = [sys.executable, os.path.abspath(__file__), "--cpu-worker", name, "--cpu-grid",
           ",".join(str(int(g)) for g in grid), "--steps", str(steps), "--warmup", str(warmup)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s, env=env)
    if r.returncode != 0:
        raise RuntimeError(f"cpu oracle worker failed ({r.returncode}): {r.stderr[-2000:]}")
    return json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][-1])


def cpu_arm_steps(cells, steps, warmup):
    """The CPU arm runs a BOUNDED number of steps of the same workload (a 512^3 step is tens of seconds
    on the host): at most ~90 s of stepping, never more than asked for."""
    est = cells / 2.5e6  # seconds per step at ~2.5 Mcell-updates/s (8 cores; faster on the box)
    k = int(max(1, min(steps, 90.0 // max(est, 1e-9))))
    w = int(min(warmup, 1 if est < 10 else 0))
    return k, w


def cpu_sample_text(res, name):
    return (f"oracle/ (numpy + scipy.fft restatement of the reference CPU path; the reference itself needs "
            f"mpi4py/sopht/pystencils, absent from the image) on the SAME workload {name}: grid "
            f"{'x'.join(str(g) for g in res['grid'])}, {res['lagrangian_points']} Lagrangian points, "
            f"{res['steps']} timed step(s) after {res['warmup']} warm-up, scipy.fft workers = {res['cores']}, "
            f"numpy stencils single-threaded (as the reference's serial-per-rank pystencils loops)")


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.workload or DEFAULT_WORKLOAD
    grid, flow_type, body, prec = WORKLOADS[name]
    cells = float(np.prod(grid))
    k, wu = cpu_arm_steps(cells, args.steps, args.warmup)
    res = run_cpu_oracle(name, grid, k, wu)
    sample = cpu_sample_text(res, name)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": prec, "data": "synthetic",
        "config": {"workload": name, "grid_zyx": list(grid), "flow_type": flow_type,
                   "lagrangian_points": res["lagrangian_points"], "cpu_steps_run": res["steps"],
                   "cpu_warmup_run": res["warmup"], "kind": "port (oracle/), not the reference binary"},
        "cpu_baseline": {"value": res["value"], "unit": UNIT, "cores": res["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ----------------------------------------------------------------------- own arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", type=str, default=None)
    ap.add_argument("--impl", type=str, default="b200")
    ap.add_argument("--scaling", type=str, default="strong", choices=["weak", "strong"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fused", action="store_true")
    ap.add_argument("--poisson-backend", type=str, default="auto")
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (one process only)")
    ap.add_argument("--cpu-worker", type=str, default=None, help=argparse.SUPPRESS)
    ap.add_argument("--cpu-grid", type=str, default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path, not of --impl reference")
    if args.cpu_worker:
        cpu_oracle_worker(args.cpu_worker, tuple(int(v) for v in args.cpu_grid.split(",")), args.steps, args.warmup)
        return
    capture_stdout()
    if args.impl == "reference":
        reference_arm(args)
        return

    import torch
    import torch.distributed as dist

    from sopht_mpi_b200 import _lib
    from sopht_mpi_b200.simulator import (PrescribedForcingGrid, RigidBodyFlowInteractionMPI,
                                          UnboundedFlowSimulator3D)
    from sopht_mpi_b200.utils.comm import init_process_group_if_needed

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    _lib.load()
    init_process_group_if_needed()
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs needs a single process (each rank only holds its own slab)")
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)

    name = args.workload or DEFAULT_WORKLOAD
    grid = list(WORKLOADS[name][0])
    if os.environ.get("SB200_BENCH_GRID"):  # developer aid (e.g. the per-rank slab of a larger job on fewer GPUs)
        grid = [int(v) for v in os.environ["SB200_BENCH_GRID"].split(",")]
    if args.scaling == "weak" and world > 1:
        # fixed cells per GPU: the box doubles along z, then y, then x; the decomposition stays z-slabs
        f, axis = world, 0
        while f > 1:
            grid[axis % 3] *= 2
            f //= 2
            axis += 1
    w = workload_setup(name, grid)
    real_t, flow_type, u_inf = w["real_t"], w["flow_type"], w["u_inf"]
    w_bytes = 4 if real_t == np.float32 else 8
    sim = UnboundedFlowSimulator3D(
        grid_size=tuple(grid), x_range=w["x_range"], kinematic_viscosity=w["nu"], flow_type=flow_type,
        real_t=real_t, with_free_stream_flow=bool(w["body"]), use_fused_kernels=not args.no_fused,
        poisson_backend=args.poisson_backend, rank_distribution=(0, 1, 1), **w["sim_kw"])
    gs = sim.ghost_size
    w0 = initial_vorticity(w, sim.local_x, sim.local_y, sim.local_z)
    host_w = torch.from_numpy(w0).pin_memory()
    sim.vorticity_field[...] = host_w.to(device)
    sim.compute_flow_velocity(free_stream_velocity=u_inf)

    interactor, n_lag, substeps = None, 0, w["substeps"]
    if w["body"]:
        pts = w["points"]
        n_lag = pts.shape[1]

        class _Body:
            pass

        interactor = RigidBodyFlowInteractionMPI(
            mpi_construct=sim.mpi_construct,
            mpi_ghost_exchange_communicator=sim.mpi_ghost_exchange_communicator,
            rigid_body=_Body(), eul_grid_forcing_field=sim.eul_grid_forcing_field,
            eul_grid_velocity_field=sim.velocity_field, virtual_boundary_stiffness_coeff=w["k"],
            virtual_boundary_damping_coeff=w["c"], dx=sim.dx, grid_dim=3,
            forcing_grid_cls=lambda grid_dim, rigid_body: PrescribedForcingGrid(
                grid_dim, pts, velocity_field=w["lag_vel"], max_lag_grid_dx=w["dx"], static=True))

    cells = float(np.prod(grid))

    def one_step():
        dt = sim.compute_stable_timestep(dt_prefac=0.5)
        if interactor is not None:
            for _ in range(substeps):  # rod sub-steps: flow forces on the body only
                interactor.compute_flow_forces_and_torques()
            interactor()
            interactor.time_step(dt)
        sim.time_step(dt=dt, free_stream_velocity=u_inf)
        return dt

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # W warm-up steps, extended (never shortened) until the GPU has been busy for about a second: three
    # steps of a few ms do not bring the SM clock up from idle.  The number of extra steps is decided on
    # rank 0 and broadcast (the steps contain collectives).
    n_warm = max(args.warmup, 3)
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    t_warm = time.perf_counter()
    for _ in range(n_warm):
        one_step()
    barrier()
    per_step = max((time.perf_counter() - t_warm) / n_warm, 1e-5)
    extra = torch.tensor([max(0, min(400, int(1.0 / per_step)) - n_warm)], dtype=torch.int64, device=device)
    if world > 1:
        dist.broadcast(extra, src=0)
    for _ in range(int(extra.item())):
        one_step()
    n_warm += int(extra.item())
    # back to the initial condition: how many warm-up steps ran depends on the speed of the build and
    # of the GPU, what the timed steps compute must not
    sim.vorticity_field[...] = host_w.to(device)
    sim.compute_flow_velocity(free_stream_velocity=u_inf)
    if interactor is not None:
        interactor.global_lag_grid_position_mismatch_field = 0.0
    barrier()
    if sampler:
        sampler.mark()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        dt_last = one_step()
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    t = torch.tensor([ms_total], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = t.item() / args.steps
    clocks = sampler.stop() if sampler else {}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, sim, interactor, dt_last)

    if os.environ.get("SB200_TRACE"):
        # developer aid: kernel-level timeline (CUPTI through torch.profiler) of three more steps, one
        # chrome trace per rank; read with tools/trace_summary.py
        from torch.profiler import ProfilerActivity, profile

        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                one_step()
            barrier()
        prof.export_chrome_trace(f"{os.environ['SB200_TRACE']}_rank{rank}.json")

    # ---- per-stage device times (untimed extra pass) -> roofline of the dominant stage
    stage_ms = {}

    def timed(label, fn, reps=5):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        stage_ms[label] = a.elapsed_time(b) / reps

    dt_fix = sim.compute_stable_timestep(dt_prefac=0.5)
    solver = sim.unbounded_poisson_solver
    timed("poisson_vector_solve", lambda: solver.vector_field_solve(
        solution_vector_field=sim.stream_func_field, rhs_vector_field=sim.vorticity_field))
    timed("flow_step", lambda: sim.time_step(dt=dt_fix, free_stream_velocity=u_inf))
    if interactor is not None:
        timed("interaction", lambda: interactor())
    local_cells = cells / world
    peak, peak_src = hbm_peak()
    # ---- roofline of the dominant kernel: the fused z pass of the Poisson solve (forward FFT x Green's
    # spectrum x inverse FFT, in place).  Its launches are timed live with CUDA events recorded by the
    # library on the solve's stream (sb200_poisson_set_profiling), averaged over `steps` solves.
    # ALGORITHMIC bytes per launch: read 4 W + write 4 W per cell and component (DESIGN.md section 4).
    roofline = None
    if solver.backend == "fft":
        solver.set_profiling(True)
        acc = {}
        reps = max(args.steps, 5)
        for _ in range(reps):
            solver.vector_field_solve(solution_vector_field=sim.stream_func_field,
                                      rhs_vector_field=sim.vorticity_field)
            for k, v in solver.last_stage_ms().items():
                acc[k] = acc.get(k, 0.0) + v / reps
        solver.set_profiling(False)
        stage_ms.update({"poisson_" + k: v for k, v in acc.items()})
        zk = "z_fused_forward_green_inverse"
        if zk not in acc:  # z-slabs: the y and z passes are timed together (20 W per cell and component)
            zk = "y_forward_z_fused_y_inverse"
        z_bytes = (8 if zk.startswith("z_") else 20) * w_bytes * 3 * local_cells
        achieved = z_bytes / (acc[zk] * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": "fused z pass of the Poisson vector solve (forward FFT x Green x "
                    "inverse FFT, in place): sb_fft_zconvw_kernel (float, 2nz = 512 / 1024; one line per warp, "
                    "bulk-copy tiles), sb_fft_strided_kernel <MODE 1> otherwise",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": ncu_traffic(name) if world == 1 else None,
                    "peak_source": peak_src,
                    "launch_ms": acc[zk], "algorithmic_bytes_per_launch": z_bytes,
                    "algorithmic_bytes_per_cell": z_bytes / local_cells,
                    "share_of_step": acc[zk] / (ms_step if world == 1 else stage_ms["flow_step"]),
                    "per_gpu": world > 1,
                    "note": "bound by FP32 issue, not by HBM: two 2nz-point transforms per line = ~7 FP32 "
                            "lane-operations per byte (FMA pipe 66 % busy, DRAM 1.19 x algorithmic); see "
                            "DESIGN.md 'Fused z pass' and profiles/r02_ncu_zconvw_512.txt"}
    nvlink = None
    if world > 1 and "poisson_all_to_all_z_to_kx" in stage_ms:
        # each all-to-all moves the x-pass output (nx/2 + 1 complex bins per row = 2 W per cell) of this
        # GPU's planes, minus the block that stays local
        kxl = ((grid[2] + 1 + world - 1) // world + 3) // 4 * 4
        a2a_bytes = 2 * w_bytes * 3 * (grid[0] / world) * grid[1] * kxl * (world - 1)
        nvlink = {"all_to_all_bytes_out_per_gpu": a2a_bytes,
                  "GBps_out_per_gpu": [a2a_bytes / (stage_ms[k] * 1e-3) / 1e9
                                       for k in ("poisson_all_to_all_z_to_kx", "poisson_all_to_all_kx_to_z")],
                  "peak_GBps_per_direction": 900.0,
                  "exchange": getattr(solver, "exchange_mode", None)}
    poisson_bytes = 86 * w_bytes * local_cells
    poisson_gbs = poisson_bytes / (stage_ms["poisson_vector_solve"] * 1e-3) / 1e9
    w_per_cell = 107 if flow_type == "navier_stokes_with_forcing" else 101
    if w["sim_kw"].get("filter_vorticity"):
        w_per_cell += 3 * 3 * w["sim_kw"]["filter_setting_dict"]["order"] * 2  # SURVEY 8(d)
    step_bytes = w_per_cell * w_bytes * local_cells
    step_gbs = step_bytes / (ms_step * 1e-3) / 1e9

    # ---- end to end through the public API with HOST buffers, every step:
    #   in : the body's Lagrangian kinematics (positions + velocities of the forcing grid, host numpy ->
    #        pinned staging -> device) -- what the reference's interactor receives from the body solver;
    #   out: the Lagrangian forces (device -> host numpy, what compute_flow_forces_and_torques hands
    #        back), dt (compute_stable_timestep) and the max-vorticity diagnostic.
    # Workloads without a body have no per-step host input: there the whole vorticity field is uploaded and
    # vorticity + velocity are read back every step (the round-1 definition), which is also reported for
    # the body workloads as `full_field_io_value`.
    e2e_steps = max(3, min(args.steps, 10))

    def measure(step_fn):
        step_fn(0)
        barrier()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            step_fn(i + 1)
        barrier()
        s = torch.tensor([(time.perf_counter() - t0) / e2e_steps], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(s, op=dist.ReduceOp.MAX)
        return cells / s.item() / 1e6

    field_bytes = host_w.numel() * host_w.element_size()
    host_out_w = torch.empty_like(host_w).pin_memory()
    host_out_u = torch.empty_like(host_w).pin_memory()

    def e2e_fields(i):
        sim.vorticity_field.tensor.copy_(host_w, non_blocking=True)
        one_step()
        host_out_w.copy_(sim.vorticity_field.tensor, non_blocking=True)
        host_out_u.copy_(sim.velocity_field.tensor, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    if interactor is not None:
        fg = interactor.forcing_grid
        pos_a = np.array(fg.position_field)
        pos_b = pos_a + 1e-9  # a second host array: the body "moved", every step uploads fresh kinematics
        sink = np.zeros(3)

        def e2e_api(i):
            fg.position_field[...] = pos_a if i % 2 else pos_b
            getattr(fg, "mark_moved", lambda: None)()  # (ranks other than the master hold an empty grid)
            one_step()
            sink[...] = np.asarray(interactor.global_lag_grid_forcing_field).sum(axis=1)  # host read of the forces
            sink[0] += sim.get_max_vorticity()

        lag_bytes = fg.position_field.nbytes
        e2e = {"value": measure(e2e_api), "unit": UNIT, "h2d_bytes_per_step": 2 * lag_bytes,
               "d2h_bytes_per_step": lag_bytes * (substeps + 1) + 16,
               "what": "public API, host buffers: the body moves every step, so its Lagrangian positions + "
                       "velocities (host numpy) are staged and uploaded every step; Lagrangian forces (every "
                       "interaction), dt and max vorticity are read back on the host",
               "full_field_io_value": measure(e2e_fields),
               "full_field_io_bytes_per_step": {"h2d": field_bytes, "d2h": 2 * field_bytes}}
        fg.position_field[...] = pos_a
        getattr(fg, "mark_moved", lambda: None)()
    else:
        e2e = {"value": measure(e2e_fields), "unit": UNIT, "h2d_bytes_per_step": field_bytes,
               "d2h_bytes_per_step": 2 * field_bytes,
               "what": "operator API with host buffers: vorticity H2D from pinned memory, step, "
                       "vorticity+velocity D2H, every step"}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        k, wu = cpu_arm_steps(cells, 1 if cells > 3e7 else 3, 1)
        try:
            res = run_cpu_oracle(name, grid, k, wu)
            cpu_baseline = {"value": res["value"], "unit": UNIT, "cores": res["cores"], "kind": "port",
                            "ms_per_step": res["ms_per_step"], "sample": cpu_sample_text(res, name)}
        except Exception as exc:  # the baseline is a reported number, never a reason to lose the line
            cpu_baseline = {"value": None, "unit": UNIT, "cores": None, "kind": "port",
                            "sample": f"failed: {type(exc).__name__}: {str(exc)[-300:]}"}

    # every rank runs the counted step (it contains collectives)
    launches_per_step = count_launches(sim, interactor, u_inf, substeps)
    if rank == 0:
        line = {
            "metric": METRIC, "value": cells / (ms_step * 1e-3) / 1e6, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": n_warm, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": w["prec"],
            "data": "synthetic",
            "config": {"workload": name, "grid_zyx": grid, "flow_type": flow_type, "lagrangian_points": n_lag,
                       "ghost_size": gs, "parallelism": f"z-slabs x{world}",
                       "poisson_backend": sim.unbounded_poisson_solver.backend,
                       "l2": "working set (>= 1.2 GB of fields per step) is far larger than the 126 MB L2",
                       "requested_warmup": args.warmup,
                       "step_algorithmic_W_per_cell": w_per_cell,
                       "step_algorithmic_GBps": step_gbs, "step_hbm_frac_of_measured": step_gbs / peak,
                       "step_hbm_frac_of_nominal_8TBps": step_gbs / 8000.0,
                       "poisson_algorithmic_GBps": poisson_gbs, "poisson_hbm_frac_of_measured": poisson_gbs / peak,
                       "stage_ms": stage_ms, "nvlink": nvlink},
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": launches_per_step * args.steps,
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
        }
        emit(line)
    if world > 1:
        # release the CUDA-IPC mappings of the other ranks' exchange buffers before any rank exits
        import gc

        solver.close()
        halo = getattr(sim.mpi_construct, "_peer_halo", None)
        if halo is not None:
            halo.close()
        del solver, sim, interactor
        gc.collect()
        torch.cuda.ipc_collect()
        dist.barrier()
        dist.destroy_process_group()


DUMP_MAX_BYTES = 60 << 20  # with the .npy headers, under 64 MB in decimal units too
DUMP_SEED = 0


def dump_outputs(out_dir, sim, interactor, dt):
    """What the last step handed its caller, as ``out_dir/<name>.npy`` (at most DUMP_MAX_BYTES in all):
    ``dt`` (float64), the vorticity, velocity and stream-function fields as (3, n) arrays in the workload's
    precision over the same n interior cells, and for workloads with a body the Lagrangian forcing and
    position mismatch of every forcing point.  The cells are all interior cells when they fit, otherwise
    a sample drawn with DUMP_SEED (sorted flat interior indices, z-major), so every run with the same
    arguments writes the same cells."""
    os.makedirs(out_dir, exist_ok=True)
    out = {"dt": np.array([float(dt)], dtype=np.float64)}
    if interactor is not None:
        out["lag_grid_forcing_field"] = np.array(interactor.global_lag_grid_forcing_field)
        out["lag_grid_position_mismatch_field"] = np.array(interactor.global_lag_grid_position_mismatch_field)
    fields = ("vorticity_field", "velocity_field", "stream_func_field")
    gs = sim.ghost_size
    padded = tuple(int(v) for v in sim.local_grid_size_with_ghost)
    interior = tuple(v - 2 * gs for v in padded)
    n_interior = int(np.prod(interior))
    per_cell = len(fields) * 3 * np.dtype(sim.real_t).itemsize
    n = (DUMP_MAX_BYTES - sum(a.nbytes for a in out.values())) // per_cell
    if n >= n_interior:
        cells = np.arange(n_interior)
    else:
        cells = np.unique(np.random.default_rng(DUMP_SEED).integers(0, n_interior, size=n))
    zyx = np.unravel_index(cells, interior)
    flat = np.ravel_multi_index(tuple(c + gs for c in zyx), padded)
    import torch

    index = torch.from_numpy(flat).to(sim.vorticity_field.tensor.device)
    for name in fields:
        t = getattr(sim, name).tensor
        out[name] = t.reshape(t.shape[0], -1).index_select(1, index).cpu().numpy()
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_MAX_BYTES and all(a.dtype in (np.float32, np.float64) for a in out.values()), total
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def count_launches(sim, interactor, u_inf, substeps=0):
    """kernels of libsophtb200 launched by one step (counted by wrapping the ctypes calls)."""
    from sopht_mpi_b200 import _lib

    lib = _lib.load()
    counts = {"n": 0}
    per_call = {"sb200_diffusion_timestep": 6, "sb200_laplacian_filter": 12, "sb200_penalise_field_boundary": 2,
                "sb200_poisson_solve": 5, "sb200_poisson_slab_spectral": 3, "sb200_velocity_from_stream_function": 2,
                "sb200_max_abs_sum": 2}
    originals = {}
    for fname in _lib.PROTOTYPES:
        fn = getattr(lib, fname)
        originals[fname] = fn

        def wrap(*a, _fn=fn, _name=fname):
            counts["n"] += per_call.get(_name, 1)
            return _fn(*a)

        setattr(lib, fname, wrap)
    try:
        dt = sim.compute_stable_timestep(dt_prefac=0.5)
        if interactor is not None:
            for _ in range(substeps):
                interactor.compute_flow_forces_and_torques()
            interactor()
            interactor.time_step(dt)
        sim.time_step(dt=dt, free_stream_velocity=u_inf)
    finally:
        for fname, fn in originals.items():
            setattr(lib, fname, fn)
    return counts["n"]


if __name__ == "__main__":
    main()
