"""Multi-rank worker for the z-slab mode of the cuFFT backend (a grid that is not a power of two, above the
size floor of the slab pipeline), run by test_gpu_slab_cufft.py through torchrun (one process per GPU) or with
every rank a process on one GPU: the vector Poisson solve and three navier_stokes_with_forcing steps, each rank
checking its own slab against the single-domain CPU oracle computed on identical global inputs."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

from harness import join_ranks, leave_ranks  # noqa: E402
from oracle.poisson import UnboundedPoissonSolverOracle3D  # noqa: E402
from oracle.simulator import FlowSimulatorOracle3D  # noqa: E402

# nz splits into 2, 3, 4, 6 and 8 slabs of at least 2 ghost_size planes; 276480 cells, above the floor
N = (48, 72, 80)


def main():
    join_ranks()
    from sopht_mpi_b200.numeric.eulerian_grid_ops import UnboundedPoissonSolverMPI3D
    from sopht_mpi_b200.simulator import UnboundedFlowSimulator3D
    from sopht_mpi_b200.utils import MPIConstruct3D
    from sopht_mpi_b200.utils.device import DeviceField

    gs = 2
    inner = (slice(None), slice(gs, -gs), slice(gs, -gs), slice(gs, -gs))
    for real_t, tol in ((np.float64, 1e-10), (np.float32, 1e-5)):
        # ---------------- vector Poisson solve on slabs
        mc = MPIConstruct3D(*N, real_t=real_t, rank_distribution=(0, 1, 1))
        rank, size = mc.rank, mc.size
        nzl = N[0] // size
        rng = np.random.default_rng(0)
        rhs = rng.uniform(size=(3, N[0] + 2 * gs, N[1] + 2 * gs, N[2] + 2 * gs)).astype(real_t)
        ref = np.zeros_like(rhs)
        UnboundedPoissonSolverOracle3D(*N, x_range=1.0, real_t=real_t).vector_field_solve(ref, rhs, gs)
        solver = UnboundedPoissonSolverMPI3D(*N, mpi_construct=mc, ghost_size=gs, x_range=1.0, real_t=real_t)
        assert solver.backend == "cufft" and not solver.replicated
        loc = np.ascontiguousarray(rhs[:, rank * nzl:rank * nzl + nzl + 2 * gs])
        out = DeviceField(torch.full(loc.shape, 7.0, dtype=torch.from_numpy(loc).dtype, device=mc.device))
        for _ in range(2):  # the second solve reuses the exchange buffers
            solver.vector_field_solve(solution_vector_field=out,
                                      rhs_vector_field=DeviceField(torch.from_numpy(loc).to(mc.device)))
        got = np.asarray(out)
        want = ref[:, rank * nzl + gs:rank * nzl + gs + nzl, gs:-gs, gs:-gs]
        err = np.abs(got[inner] - want).max() / np.abs(ref).max()
        assert err <= tol, ("poisson", real_t, err)
        assert np.all(got[:, :gs] == 7.0) and np.all(got[:, :, :, -gs:] == 7.0)  # ghosts untouched
        solver._peer.check()
        solver.close()

        # ---------------- flow steps on slabs vs the single-domain oracle
        kw = dict(grid_size=N, x_range=1.0, kinematic_viscosity=1e-2, flow_type="navier_stokes_with_forcing",
                  real_t=real_t, with_free_stream_flow=True)
        sim = UnboundedFlowSimulator3D(rank_distribution=(0, 1, 1), **kw)
        assert not sim.unbounded_poisson_solver.replicated
        ora = FlowSimulatorOracle3D(**kw)
        zz, yy, xx = np.meshgrid(ora.local_z, ora.local_y, ora.local_x, indexing="ij")
        body = np.exp(-((xx - 0.5) ** 2 + (yy - 0.45) ** 2 + (zz - 0.3) ** 2) / 0.01)
        w0 = np.stack([body * (yy - 0.45) * 40, -body * (xx - 0.5) * 40, 0.3 * body]).astype(real_t)
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
            force = (0.5 * np.stack([body, 0.5 * body, -body]) * np.cos(3.0 * step)).astype(real_t)
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
        sim.unbounded_poisson_solver.close()
    leave_ranks("DIST_SLAB_CUFFT_WORKER_OK")


if __name__ == "__main__":
    main()
