"""Multi-GPU worker (one process per GPU, NCCL) run by test_gpu_multi.py through torchrun:
z-slab Poisson solve, halo exchange + fused step, IB ghost sum -- each rank checks its own slab
against the single-domain CPU oracle computed on identical global inputs."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

from harness import join_ranks, leave_ranks  # noqa: E402
from oracle.poisson import UnboundedPoissonSolverOracle3D  # noqa: E402
from oracle.simulator import FlowSimulatorOracle3D  # noqa: E402
from oracle import ib as ib_oracle  # noqa: E402


def rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    if b.size == 0:  # a rank that owns no Lagrangian point (8 slabs, one small body)
        return 0.0
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def main():
    join_ranks()
    from sopht_mpi_b200.numeric.eulerian_grid_ops import UnboundedPoissonSolverMPI3D
    from sopht_mpi_b200.simulator import UnboundedFlowSimulator3D
    from sopht_mpi_b200.utils import MPIConstruct3D
    from sopht_mpi_b200.utils.device import DeviceField

    gs = 2
    for real_t, tol in ((np.float64, 1e-10), (np.float32, 1e-5)):
        # ---------------- Poisson on slabs
        n = (32, 16, 32)
        mc = MPIConstruct3D(*n, real_t=real_t, rank_distribution=(0, 1, 1))
        rank, size = mc.rank, mc.size
        nzl = n[0] // size
        rng = np.random.default_rng(0)
        rhs = rng.uniform(size=(3, n[0] + 2 * gs, n[1] + 2 * gs, n[2] + 2 * gs)).astype(real_t)
        ref = np.zeros_like(rhs)
        UnboundedPoissonSolverOracle3D(*n, x_range=1.0, real_t=real_t).vector_field_solve(ref, rhs, gs)
        solver = UnboundedPoissonSolverMPI3D(*n, mpi_construct=mc, ghost_size=gs, x_range=1.0, real_t=real_t)
        loc = np.ascontiguousarray(rhs[:, rank * nzl:rank * nzl + nzl + 2 * gs])
        out = DeviceField(torch.zeros(loc.shape, dtype=torch.from_numpy(loc).dtype, device=mc.device))
        solver.vector_field_solve(solution_vector_field=out,
                                  rhs_vector_field=DeviceField(torch.from_numpy(loc).to(mc.device)))
        inner = (slice(None), slice(gs, -gs), slice(gs, -gs), slice(gs, -gs))
        err = rel(np.asarray(out)[inner], ref[:, rank * nzl + gs:rank * nzl + gs + nzl, gs:-gs, gs:-gs])
        assert err <= tol, ("poisson", real_t, err)
        getattr(solver, "_peer", None) and solver._peer.check()
        solver.close()

        # ---------------- full simulator steps on slabs vs single-domain oracle
        n = (32, 16, 32)
        # (Laplacian filter on: float64 runs order 1 multiplicative, float32 order 2 convolution)
        kw = dict(grid_size=n, x_range=1.0, kinematic_viscosity=1e-2, flow_type="navier_stokes_with_forcing",
                  real_t=real_t, with_free_stream_flow=True, filter_vorticity=True,
                  filter_setting_dict=({"order": 1, "type": "multiplicative"} if real_t == np.float64
                                       else {"order": 2, "type": "convolution"}))
        sim = UnboundedFlowSimulator3D(rank_distribution=(0, 1, 1), **kw)
        ora = FlowSimulatorOracle3D(**kw)
        zz, yy, xx = np.meshgrid(ora.local_z, ora.local_y, ora.local_x, indexing="ij")
        blob = np.exp(-((xx - 0.5) ** 2 + (yy - 0.25) ** 2 + (zz - 0.5) ** 2) / 0.01)
        w0 = np.stack([blob * (yy - 0.25) * 40, -blob * (xx - 0.5) * 40, 0.3 * blob]).astype(real_t)
        sl = slice(rank * nzl, rank * nzl + nzl + 2 * gs)
        ora.vorticity_field[...] = w0
        sim.vorticity_field[...] = np.ascontiguousarray(w0[:, sl])
        u_inf = [1.0, 0.0, 0.0]
        ora.compute_flow_velocity(u_inf)
        sim.compute_flow_velocity(free_stream_velocity=u_inf)
        for step in range(3):
            dt = ora.compute_stable_timestep(dt_prefac=0.5)
            dt_gpu = sim.compute_stable_timestep(dt_prefac=0.5)
            assert abs(dt_gpu - dt) <= 1e-5 * dt, ("dt", step, real_t, dt_gpu, dt)
            force = (0.5 * np.stack([blob, 0.5 * blob, -blob]) * np.cos(3.0 * step)).astype(real_t)
            force[:, :gs], force[:, -gs:] = 0, 0
            force[:, :, :gs], force[:, :, -gs:] = 0, 0
            force[:, :, :, :gs], force[:, :, :, -gs:] = 0, 0
            ora.eul_grid_forcing_field[...] = force
            sim.eul_grid_forcing_field[...] = np.ascontiguousarray(force[:, sl])
            ora.time_step(dt, free_stream_velocity=u_inf)
            sim.time_step(dt=dt, free_stream_velocity=u_inf)
        isl = slice(rank * nzl + gs, rank * nzl + gs + nzl)
        for name in ("vorticity_field", "velocity_field", "stream_func_field"):
            got = np.asarray(getattr(sim, name))[inner]
            want = getattr(ora, name)[:, isl, gs:-gs, gs:-gs]
            err = np.abs(got - want).max() / np.abs(getattr(ora, name)).max()
            assert err <= tol, (name, real_t, err)
        gmax = sim.get_max_vorticity()
        assert abs(gmax - ora.vorticity_field[:, gs:-gs, gs:-gs, gs:-gs].max()) <= 50 * tol
        sim.unbounded_poisson_solver.close()

    # ---------------- virtual boundary forcing across slabs: ownership, forces, spreading + ghost sum
    from sopht_mpi_b200.numeric.immersed_boundary_ops import VirtualBoundaryForcingMPI

    real_t = np.float32
    n = (32, 16, 32)
    mc = MPIConstruct3D(*n, real_t=real_t, rank_distribution=(0, 1, 1))
    rank, size = mc.rank, mc.size
    nzl = n[0] // size
    dx = real_t(1.0 / n[2])
    rng = np.random.default_rng(3)
    n_lag = 40
    pos = np.stack([rng.uniform(0.2, 0.8, n_lag), rng.uniform(0.15, 0.35, n_lag),
                    rng.uniform(0.1, 0.9, n_lag)])
    for k in range(1, size):  # points that straddle every slab face
        pos[2, 2 * k] = k * nzl * float(dx) + 0.3 * float(dx)
        pos[2, 2 * k + 1] = k * nzl * float(dx) - 0.3 * float(dx)
    vel = rng.uniform(-1, 1, size=pos.shape)
    u_glob = rng.uniform(size=(3, n[0] + 2 * gs, n[1] + 2 * gs, n[2] + 2 * gs)).astype(real_t)
    vbf_o = ib_oracle.VirtualBoundaryForcingOracle(-5.0, -0.7, 3, dx, real_t, np.float64, gs)
    f_glob = np.zeros_like(u_glob)
    vbf_o.compute_interaction_force_on_eul_and_lag_grid(f_glob, u_glob, pos, vel)
    vbf = VirtualBoundaryForcingMPI(mpi_construct=mc, ghost_size=gs, virtual_boundary_stiffness_coeff=-5.0,
                                    virtual_boundary_damping_coeff=-0.7, grid_dim=3, dx=dx,
                                    global_lag_grid_position_field=pos if rank == 0 else np.zeros((3, 0)))
    expect_addr = ib_oracle.lag_nodes_rank_address(pos, dx, real_t(dx / 2), mc.local_grid_size, mc.grid_topology)
    assert np.array_equal(vbf.mpi_lagrangian_field_communicator.rank_address, expect_addr)
    sl = slice(rank * nzl, rank * nzl + nzl + 2 * gs)
    u_loc = DeviceField(torch.from_numpy(np.ascontiguousarray(u_glob[:, sl])).to(mc.device))
    f_loc = DeviceField(torch.ones(u_loc.shape, dtype=torch.float32, device=mc.device))
    vbf.compute_interaction_forcing(local_eul_grid_forcing_field=f_loc, local_eul_grid_velocity_field=u_loc,
                                    global_lag_grid_position_field=pos if rank == 0 else None,
                                    global_lag_grid_velocity_field=vel if rank == 0 else None)
    if rank == 0:
        assert rel(vbf.global_lag_grid_forcing_field, vbf_o.forcing) <= 1e-5
    got = np.asarray(f_loc)[(slice(None), slice(gs, -gs), slice(gs, -gs), slice(gs, -gs))]
    want = f_glob[:, rank * nzl + gs:rank * nzl + gs + nzl, gs:-gs, gs:-gs]
    assert np.abs(got - want).max() / np.abs(f_glob).max() <= 1e-5
    assert float(np.abs(np.asarray(f_loc)[:, :gs]).max()) == 0.0  # ghosts cleared
    # device ownership = the reference's integers; the replicated state is the same on every rank
    assert np.array_equal(vbf._owner.cpu().numpy()[:n_lag], expect_addr)
    assert vbf.local_num_lag_nodes == int((expect_addr == rank).sum())
    assert rel(vbf.local_lag_grid_forcing_field, vbf_o.forcing[:, expect_addr == rank]) <= 1e-5
    # a second interaction after a step, with points that migrated across the slab faces
    vbf.time_step(0.1)
    vbf_o.time_step(0.1)
    pos2 = pos.copy()
    pos2[2] += 0.6 * float(dx) * np.where(np.arange(n_lag) % 2 == 0, 1.0, -1.0)
    f_glob[...] = 0
    vbf_o.compute_interaction_force_on_eul_and_lag_grid(f_glob, u_glob, pos2, vel)
    vbf.compute_interaction_forcing(local_eul_grid_forcing_field=f_loc, local_eul_grid_velocity_field=u_loc,
                                    global_lag_grid_position_field=pos2 if rank == 0 else None,
                                    global_lag_grid_velocity_field=vel if rank == 0 else None)
    addr2 = ib_oracle.lag_nodes_rank_address(pos2, dx, real_t(dx / 2), mc.local_grid_size, mc.grid_topology)
    assert np.any(addr2 != expect_addr) and np.array_equal(vbf._owner.cpu().numpy()[:n_lag], addr2)
    assert rel(vbf.global_lag_grid_forcing_field, vbf_o.forcing) <= 1e-5  # on every rank
    assert rel(vbf.global_lag_grid_position_mismatch_field, vbf_o.position_mismatch) <= 1e-5
    got = np.asarray(f_loc)[(slice(None), slice(gs, -gs), slice(gs, -gs), slice(gs, -gs))]
    want = f_glob[:, rank * nzl + gs:rank * nzl + gs + nzl, gs:-gs, gs:-gs]
    assert np.abs(got - want).max() / np.abs(f_glob).max() <= 1e-5

    check_replicated_solves(gs)
    leave_ranks("DIST_GPU_WORKER_OK")


def check_replicated_solves(gs):
    """Configurations outside the slab pipeline (a grid that is not a power of two; the 2D `-np P`
    case of BASELINE configs[0]) run replicated: same results as the single-domain oracle."""
    from oracle.poisson import UnboundedPoissonSolverOracle2D
    from oracle.simulator import FlowSimulatorOracle2D
    from sopht_mpi_b200.numeric.eulerian_grid_ops import UnboundedPoissonSolverMPI3D
    from sopht_mpi_b200.simulator import UnboundedFlowSimulator2D
    from sopht_mpi_b200.utils import MPIConstruct3D
    from sopht_mpi_b200.utils.device import DeviceField

    real_t = np.float64
    size = dist.get_world_size()
    n = (6 * size, 20, 36)
    mc = MPIConstruct3D(*n, real_t=real_t, rank_distribution=(0, 1, 1))
    rank = mc.rank
    nzl = n[0] // size
    rng = np.random.default_rng(4)
    rhs = rng.uniform(size=(3, n[0] + 2 * gs, n[1] + 2 * gs, n[2] + 2 * gs)).astype(real_t)
    ref = np.zeros_like(rhs)
    UnboundedPoissonSolverOracle3D(*n, x_range=1.0, real_t=real_t).vector_field_solve(ref, rhs, gs)
    solver = UnboundedPoissonSolverMPI3D(*n, mpi_construct=mc, ghost_size=gs, x_range=1.0, real_t=real_t)
    assert solver.replicated and solver.backend == "cufft"
    loc = np.ascontiguousarray(rhs[:, rank * nzl:rank * nzl + nzl + 2 * gs])
    out = DeviceField(torch.full(loc.shape, 7.0, dtype=torch.float64, device=mc.device))
    solver.vector_field_solve(solution_vector_field=out, rhs_vector_field=DeviceField(torch.from_numpy(loc).to(mc.device)))
    got = np.asarray(out)
    inner = (slice(None), slice(gs, -gs), slice(gs, -gs), slice(gs, -gs))
    assert rel(got[inner], ref[:, rank * nzl + gs:rank * nzl + gs + nzl, gs:-gs, gs:-gs]) <= 1e-10
    assert np.all(got[:, 0] == 7.0)  # ghosts untouched
    one = DeviceField(torch.zeros(loc.shape[1:], dtype=torch.float64, device=mc.device))
    solver.solve(solution_field=one, rhs_field=DeviceField(torch.from_numpy(np.ascontiguousarray(loc[1])).to(mc.device)))
    assert rel(np.asarray(one)[inner[1:]], ref[1, rank * nzl + gs:rank * nzl + gs + nzl, gs:-gs, gs:-gs]) <= 1e-10

    # 2D flow past a cylinder on y-slabs (BASELINE configs[0]: 2D, float64, mpirun -np 2)
    n2 = (16 * size, 64)
    kw = dict(grid_size=n2, x_range=1.0, kinematic_viscosity=3e-3, flow_type="navier_stokes_with_forcing",
              real_t=real_t, with_free_stream_flow=True)
    sim = UnboundedFlowSimulator2D(rank_distribution=(0, 1), **kw)
    ora = FlowSimulatorOracle2D(**kw)
    nyl = n2[0] // size
    sl = slice(rank * nyl, rank * nyl + nyl + 2 * gs)
    yy, xx = np.meshgrid(ora.local_y, ora.local_x, indexing="ij")
    blob = np.exp(-((xx - 0.3) ** 2 + (yy - 0.5 * ora.local_y[-gs - 1]) ** 2) / 0.004)
    ora.vorticity_field[...] = 3.0 * blob
    sim.vorticity_field[...] = np.ascontiguousarray((3.0 * blob)[sl])
    u_inf = [1.0, 0.0]
    for c in range(2):
        ora.velocity_field[c] += real_t(u_inf[c])
    sim.velocity_field[...] = np.ascontiguousarray(ora.velocity_field[:, sl])
    for step in range(3):
        dt = ora.compute_stable_timestep()
        assert abs(sim.compute_stable_timestep() - dt) <= 1e-10 * dt
        force = np.stack([blob, -0.5 * blob]) * np.cos(2.0 * step)
        force[:, :gs], force[:, -gs:], force[:, :, :gs], force[:, :, -gs:] = 0, 0, 0, 0
        ora.eul_grid_forcing_field[...] = force
        sim.eul_grid_forcing_field[...] = np.ascontiguousarray(force[:, sl])
        ora.time_step(dt, free_stream_velocity=u_inf)
        sim.time_step(dt=dt, free_stream_velocity=u_inf)
    isl = slice(rank * nyl + gs, rank * nyl + gs + nyl)
    for name in ("vorticity_field", "velocity_field", "stream_func_field"):
        got = np.asarray(getattr(sim, name))[..., gs:-gs, gs:-gs]
        want = getattr(ora, name)[..., isl, gs:-gs]
        assert np.abs(got - want).max() / np.abs(getattr(ora, name)).max() <= 1e-10, name


if __name__ == "__main__":
    main()
