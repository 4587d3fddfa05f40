"""Two steps of bench.py's workload, built and stepped exactly as `bench.py main()` does, run by
test_gpu_slab_benchmark_grids.py.

One process (no WORLD_SIZE) is the single-GPU reference: it writes to SB200_BENCH_STEP_DIR what the
ranks compare against (per-plane digests of the fields after the initial compute_flow_velocity, step 1's
dt and Lagrangian arrays, the interiors of omega, u and psi after step 2, step 2's dt and Lagrangian
forcing).  A second single process finds the reference there and compares its own run with it
(single.json): the spreading adds with floating-point atomics, so two single-GPU runs of a step with a
body differ in the last bits.  As P z-slab ranks (gloo + every rank on cuda:0 with
SB200_TEST_SINGLE_DEVICE=1, or torchrun over NCCL) every rank runs the same steps, checks its own planes
and writes rank<r>.json there."""
import hashlib
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from harness import join_ranks, leave_ranks  # noqa: E402

FIELDS = ("vorticity_field", "velocity_field", "stream_func_field")


def _interior(sim, name):
    gs = sim.ghost_size
    return getattr(sim, name).tensor[:, gs:-gs, gs:-gs, gs:-gs]


def _plane_digests(t):
    """blake2b of every (component, z plane) of a (3, nz, ny, nx) device tensor: equal digests = equal bits"""
    out = []
    for c in range(t.shape[0]):
        host = t[c].cpu().numpy()
        out.append([hashlib.blake2b(host[z].tobytes(), digest_size=16).hexdigest() for z in range(host.shape[0])])
    return out


def _lag(interactor):
    return {"forcing": np.array(interactor.global_lag_grid_forcing_field),
            "velocity_mismatch": np.array(interactor.global_lag_grid_velocity_mismatch_field),
            "position_mismatch": np.array(interactor.global_lag_grid_position_mismatch_field)}


def run(name, device):
    """bench.py main(): the workload, the simulator on z-slabs, the interactor, then two of its steps"""
    from sopht_mpi_b200.simulator import PrescribedForcingGrid, RigidBodyFlowInteractionMPI, UnboundedFlowSimulator3D

    grid = list(bench.WORKLOADS[name][0])
    w = bench.workload_setup(name, grid)
    u_inf = w["u_inf"]
    sim = UnboundedFlowSimulator3D(
        grid_size=tuple(grid), x_range=w["x_range"], kinematic_viscosity=w["nu"], flow_type=w["flow_type"],
        real_t=w["real_t"], with_free_stream_flow=bool(w["body"]), use_fused_kernels=True, poisson_backend="auto",
        rank_distribution=(0, 1, 1), **w["sim_kw"])
    w0 = bench.initial_vorticity(w, sim.local_x, sim.local_y, sim.local_z)
    sim.vorticity_field[...] = torch.from_numpy(w0).pin_memory().to(device)
    del w0
    if dist.is_initialized():
        dist.barrier()  # (host set-up takes a different time on every rank; the solve waits on its peers)
    sim.compute_flow_velocity(free_stream_velocity=u_inf)
    interactor = None
    if w["body"]:
        pts = w["points"]

        class _Body:
            pass

        interactor = RigidBodyFlowInteractionMPI(
            mpi_construct=sim.mpi_construct, mpi_ghost_exchange_communicator=sim.mpi_ghost_exchange_communicator,
            rigid_body=_Body(), eul_grid_forcing_field=sim.eul_grid_forcing_field,
            eul_grid_velocity_field=sim.velocity_field, virtual_boundary_stiffness_coeff=w["k"],
            virtual_boundary_damping_coeff=w["c"], dx=sim.dx, grid_dim=3,
            forcing_grid_cls=lambda grid_dim, rigid_body: PrescribedForcingGrid(
                grid_dim, pts, velocity_field=w["lag_vel"], max_lag_grid_dx=w["dx"], static=True))
    out = {"init": {f: _plane_digests(_interior(sim, f)) for f in FIELDS}}
    for step in (1, 2):
        dt = sim.compute_stable_timestep(dt_prefac=0.5)
        if interactor is not None:
            for _ in range(w["substeps"]):
                interactor.compute_flow_forces_and_torques()
            interactor()
            lag = _lag(interactor)
            interactor.time_step(dt)
            lag["position_mismatch"] = np.array(interactor.global_lag_grid_position_mismatch_field)
            out[f"lag{step}"] = lag
        sim.time_step(dt=dt, free_stream_velocity=u_inf)
        out[f"dt{step}"] = float(dt)
    torch.cuda.synchronize()
    out["final"] = {f: _plane_digests(_interior(sim, f)) for f in FIELDS}
    return sim, interactor, out


def _rel(got, want, scale):
    return float(np.abs(np.asarray(got, np.float64) - np.asarray(want, np.float64)).max() / max(scale, 1e-300))


def write_reference(name, path, device):
    sim, interactor, out = run(name, device)
    meta = {"dt1": out["dt1"], "dt2": out["dt2"], "init": out["init"], "final": out["final"], "max_abs": {}}
    for f in FIELDS:
        t = _interior(sim, f)
        meta["max_abs"][f] = float(t.abs().max().item())
        a = np.lib.format.open_memmap(os.path.join(path, f + ".npy"), mode="w+", dtype=np.dtype(sim.real_t),
                                      shape=tuple(t.shape))
        for c in range(t.shape[0]):
            a[c] = t[c].cpu().numpy()
        a.flush()
        del a
    for step in (1, 2):
        for k, v in out.get(f"lag{step}", {}).items():
            np.save(os.path.join(path, f"lag{step}_{k}.npy"), v)
    with open(os.path.join(path, "reference.json"), "w") as fh:
        json.dump(meta, fh)


def check_rank(name, path, device, rank, size, result):
    sim, interactor, out = run(name, device)
    with open(os.path.join(path, "reference.json")) as fh:
        ref = json.load(fh)
    nzl = bench.WORKLOADS[name][0][0] // size
    planes = slice(rank * nzl, rank * nzl + nzl)
    res = {"rank": rank, "identical": {}, "rel": {}}
    for stage in ("init", "final"):
        for f in FIELDS:
            res["identical"][f"{stage}_{f}"] = all(out[stage][f][c] == ref[stage][f][c][planes] for c in range(3))
    res["identical"]["dt1"] = out["dt1"] == ref["dt1"]
    res["identical"]["dt2"] = out["dt2"] == ref["dt2"]
    res["rel"]["dt2"] = abs(out["dt2"] - ref["dt2"]) / ref["dt2"]
    for step in (1, 2):
        for k, v in out.get(f"lag{step}", {}).items():
            want = np.load(os.path.join(path, f"lag{step}_{k}.npy"))
            res["identical"][f"lag{step}_{k}"] = bool(np.array_equal(v, want))
            res["rel"][f"lag{step}_{k}"] = _rel(v, want, np.abs(want).max())
    res["where"] = {}
    for f in FIELDS:
        diff = np.abs(_interior(sim, f).cpu().numpy().astype(np.float64)
                      - np.load(os.path.join(path, f + ".npy"), mmap_mode="r")[:, planes])
        at = np.unravel_index(int(np.argmax(diff)), diff.shape)
        res["rel"][f] = float(diff[at]) / max(ref["max_abs"][f], 1e-300)
        res["where"][f] = [int(at[0]), int(at[1]) + rank * nzl, int(at[2]), int(at[3])]  # (c, global z, y, x)
    with open(os.path.join(path, result), "w") as fh:
        json.dump(res, fh)
    return sim, interactor


def main():
    name, path = os.environ["SB200_BENCH_STEP_WORKLOAD"], os.environ["SB200_BENCH_STEP_DIR"]
    if int(os.environ.get("WORLD_SIZE", "1")) == 1:
        torch.cuda.set_device(0)
        if os.path.exists(os.path.join(path, "reference.json")):
            check_rank(name, path, torch.device("cuda", 0), 0, 1, "single.json")
        else:
            write_reference(name, path, torch.device("cuda", 0))
        print("DIST_BENCH_STEP_REFERENCE_OK")
        return
    join_ranks()
    rank, size = dist.get_rank(), dist.get_world_size()
    device = torch.device("cuda", torch.cuda.current_device())
    sim, interactor = check_rank(name, path, device, rank, size, f"rank{rank}.json")
    closables = (sim.unbounded_poisson_solver, getattr(sim.mpi_construct, "_peer_halo", None))
    del sim, interactor
    leave_ranks("DIST_BENCH_STEP_WORKER_OK", *closables)


if __name__ == "__main__":
    main()
