"""Replicated vs z-slab Poisson solve of grids that are not powers of two (the cuFFT backend), over a ladder of
grids.  Writes one JSON file.

    # P ranks as P virtual handles on ONE GPU: the work each GPU does per vector solve on either path, without
    # the exchanges (the replicated path's all-gather, the slab path's two all-to-alls per component).  This
    # bounds the crossover from one side only; the exchange times need the torchrun mode on P GPUs.
    python tools/bench_slab_cufft.py --virtual 2,3,4,6,8 --out profiles/r03_slab_cufft_ladder.json

    # P processes on P GPUs: both paths end to end through UnboundedPoissonSolverMPI3D (vector solve, stage
    # times from the slab profiling marks) and the navier_stokes_with_forcing step at 768 x 384 x 384
    torchrun --nproc-per-node P tools/bench_slab_cufft.py --out profiles/r03_slab_cufft_nP.json

The replicated path is measured through its own code: the size floor of the slab selection is raised above
every grid for the replicated solver of each pair."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from sopht_mpi_b200 import _lib  # noqa: E402
from sopht_mpi_b200.utils.device import dptr  # noqa: E402

GS = 2
# (6P, 20, 36) at P = 8 up to the sphere shape 1.5x refined and 384^3; nz a multiple of 24 (2, 3, 4, 6, 8 slabs)
LADDER = [(48, 20, 36), (48, 48, 60), (48, 72, 80), (96, 96, 120), (192, 120, 150), (192, 192, 240),
          (384, 192, 192), (384, 384, 384), (768, 384, 384)]


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.TimeoutExpired):
        out = []
    return {"query": q, "gpus": out, "torch_name": torch.cuda.get_device_name(0)}


def timed(fn, reps, warmup=2):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def virtual_ladder(ranks, reps):
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    rows = []
    for n in LADDER:
        nz, ny, nx = n
        cells = nz * ny * nx
        rhs = torch.rand((3,) + tuple(v + 2 * GS for v in n), device=dev)
        sol = torch.zeros_like(rhs)
        h = ctypes.c_void_p()
        _lib.check(lib, lib.sb200_poisson_create(ctypes.byref(h), 3, _lib.F32, nz, ny, nx, GS, 1.0, 0, 1, 0, None))
        whole_ms = timed(lambda: _lib.check(lib, lib.sb200_poisson_solve(h, dptr(sol), dptr(rhs), 3, None)), reps)
        whole_ws = int(lib.sb200_poisson_workspace_bytes(h))
        lib.sb200_poisson_destroy(h)
        row = {"grid": list(n), "cells": cells, "single_rank_vector_solve_ms": whole_ms,
               "single_rank_workspace_bytes": whole_ws, "slabs": []}
        for P in ranks:
            if nz % P or nz // P < 2 * GS:
                continue
            nzl = nz // P
            stage = {"forward": 0.0, "spectral": 0.0, "backward": 0.0}
            ws, xbytes = 0, 0
            for r in range(P):  # the slowest rank of each stage bounds the step
                hr = ctypes.c_void_p()
                _lib.check(lib, lib.sb200_poisson_create(ctypes.byref(hr), 3, _lib.F32, nz, ny, nx, GS, 1.0, r, P, 0,
                                                         None))
                xbytes = int(lib.sb200_poisson_slab_buffer_bytes(hr, 1))
                send = torch.zeros(xbytes // 4, device=dev)
                recv = torch.rand(xbytes // 4, device=dev)
                loc = rhs[:, r * nzl:r * nzl + nzl + 2 * GS].contiguous()
                out = torch.zeros_like(loc)
                vol = loc[0].numel() * 4

                def comp(t, c):
                    return ctypes.c_void_p(t.data_ptr() + c * vol)

                fns = {
                    "forward": lambda: [_lib.check(lib, lib.sb200_poisson_slab_forward(hr, comp(loc, c), 1, dptr(send),
                                                                                       None)) for c in range(3)],
                    "spectral": lambda: [_lib.check(lib, lib.sb200_poisson_slab_spectral(hr, dptr(recv), 1, None))
                                         for c in range(3)],
                    "backward": lambda: [_lib.check(lib, lib.sb200_poisson_slab_backward(hr, comp(out, c), 1,
                                                                                         dptr(send), None))
                                         for c in range(3)],
                }
                for k, fn in fns.items():
                    stage[k] = max(stage[k], timed(fn, reps))
                ws = max(ws, int(lib.sb200_poisson_workspace_bytes(hr)))
                lib.sb200_poisson_destroy(hr)
                del send, recv, loc, out
            row["slabs"].append({
                "ranks": P, "stage_ms_max_over_ranks": stage, "local_ms": sum(stage.values()),
                "workspace_bytes_per_rank": ws, "exchange_bytes_per_component": xbytes,
                "exchange_bytes_per_vector_solve": 6 * xbytes,
                "replicated_all_gather_bytes_per_vector_solve": 3 * cells * 4,
                "exchange_ms": "not measured (one GPU)"})
            print(json.dumps({"grid": n, **row["slabs"][-1], "single_rank_ms": whole_ms}), flush=True)
        rows.append(row)
        del rhs, sol
        torch.cuda.empty_cache()
    return rows


def distributed(reps, steps):
    import torch.distributed as dist

    from sopht_mpi_b200.numeric.eulerian_grid_ops import UnboundedPoissonSolverMPI3D, poisson
    from sopht_mpi_b200.utils import MPIConstruct3D
    from sopht_mpi_b200.utils.device import DeviceField

    floor = poisson._SLAB_CUFFT_MIN_CELLS
    rows = []
    for n in LADDER:
        mc = MPIConstruct3D(*n, real_t=np.float32, rank_distribution=(0, 1, 1))
        size, rank = mc.size, mc.rank
        if n[0] % size or n[0] // size < 2 * GS:
            continue
        nzl = n[0] // size
        r_t = torch.rand((3, nzl + 2 * GS, n[1] + 2 * GS, n[2] + 2 * GS), device=mc.device)
        rhs, out = DeviceField(r_t), DeviceField(torch.zeros_like(r_t))
        row = {"grid": list(n), "ranks": size}
        for label, min_cells in (("replicated", 1 << 62), ("slabs", 0)):
            poisson._SLAB_CUFFT_MIN_CELLS = min_cells
            s = UnboundedPoissonSolverMPI3D(*n, mpi_construct=mc, ghost_size=GS, real_t=np.float32, backend="cufft")
            poisson._SLAB_CUFFT_MIN_CELLS = floor

            def solve():
                s.vector_field_solve(solution_vector_field=out, rhs_vector_field=rhs)

            dist.barrier()
            row[label] = {"replicated": s.replicated, "vector_solve_ms": timed(solve, reps),
                          "workspace_bytes": s.workspace_bytes}
            if not s.replicated:
                s.set_profiling(True)
                solve()
                row[label]["stage_ms"] = s.last_stage_ms()
                s.set_profiling(False)
                row[label]["exchange_bytes_per_component"] = int(s.lib.sb200_poisson_slab_buffer_bytes(s._handle, 1))
            s.close()
            del s
        rows.append(row)
        if rank == 0:
            print(json.dumps(row), flush=True)
    step = {}
    n = (768, 384, 384)
    if n[0] % dist.get_world_size() == 0:
        from sopht_mpi_b200.simulator import UnboundedFlowSimulator3D

        for label, min_cells in (("replicated", 1 << 62), ("slabs", 0)):
            poisson._SLAB_CUFFT_MIN_CELLS = min_cells
            sim = UnboundedFlowSimulator3D(grid_size=n, x_range=1.0, kinematic_viscosity=1e-3,
                                           flow_type="navier_stokes_with_forcing", real_t=np.float32,
                                           with_free_stream_flow=True, rank_distribution=(0, 1, 1))
            poisson._SLAB_CUFFT_MIN_CELLS = floor
            sim.vorticity_field[...] = 0.1
            u_inf = [1.0, 0.0, 0.0]

            def one():
                sim.time_step(dt=1e-4, free_stream_velocity=u_inf)

            step[label] = {"replicated": sim.unbounded_poisson_solver.replicated,
                           "step_ms": timed(one, max(steps, 1), warmup=3)}
            sim.unbounded_poisson_solver.close()
            del sim
    return rows, step


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--virtual", type=str, default=None, help="comma-separated rank counts, one GPU")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", type=str, required=True)
    args = ap.parse_args()
    if args.virtual:
        res = {"mode": "virtual ranks on one GPU", "card": card(), "dtype": "float32",
               "ladder": virtual_ladder([int(v) for v in args.virtual.split(",")], args.reps)}
        rank = 0
    else:
        from sopht_mpi_b200.utils import MPIConstruct3D  # noqa: F401  (sets up the process group)

        rows, step = distributed(args.reps, args.steps)
        import torch.distributed as dist

        rank = dist.get_rank()
        res = {"mode": f"{dist.get_world_size()} ranks", "card": card(), "dtype": "float32", "ladder": rows,
               "navier_stokes_with_forcing_768x384x384": step}
    if rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
        print("wrote", args.out)


if __name__ == "__main__":
    main()
