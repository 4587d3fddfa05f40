"""Parity of the BENCHMARKED code paths against the CPU oracle, at BASELINE.json sizes.

`test_gpu_parity.py` runs at n <= 32, which selects the run-time-plan FFT kernels; the grids that
are timed (256^3 / 512x256x256 / 512^3) dispatch the compile-time specialised 16- and
32-point-per-thread transforms, the thread-order Green's table and the packed f32x2 arithmetic.
Everything below goes through the public operator API -> C ABI -> those kernels, on ONE GPU:

  * vector Poisson solve at 256^3 float32 / 128^3 float64 against the scipy oracle
    (reference UnboundedPoissonSolverMPI3D.py:133-187), and the in-kernel FFT backend against the
    cuFFT backend up to 512^3;
  * full Navier-Stokes steps at 256^3 float32 (BASELINE configs[1]) and 128^3 float64;
  * BASELINE configs[2]/[3]: sphere at 512x256x256 float32 and a rod with the Laplacian filter,
    through RigidBodyFlowInteractionMPI + UnboundedFlowSimulator3D(navier_stokes_with_forcing);
  * Peskin weights and the divergence L2 norm;
  * the z-slab (distributed) Poisson entry points and the ghost sum with P VIRTUAL ranks on one
    device (the test performs the block exchanges), so the 1-GPU box covers SURVEY rows P4 / L9.

Tolerances (north star): relative L-inf <= 1e-5 (float32), <= 1e-10 (float64).
"""
import ctypes
import os

import numpy as np
import pytest
import torch

from harness import _Cuda, slab_poisson_solve
from oracle import ib as ib_oracle
from oracle import stencils as st
from oracle.poisson import UnboundedPoissonSolverOracle3D
from oracle.simulator import FlowSimulatorOracle3D

pytestmark = pytest.mark.gpu

TOL = {np.float64: 1e-10, np.float32: 1e-5}
CORES = os.cpu_count() or 1


def _rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from sopht_mpi_b200 import _lib

    _lib.load()  # fails loudly if the extension is missing
    return torch.device("cuda", 0)


def _construct(n, real_t, gs=2):
    from sopht_mpi_b200.utils import MPIConstruct3D, MPIGhostCommunicator3D

    mc = MPIConstruct3D(*n, real_t=real_t)
    return mc, MPIGhostCommunicator3D(ghost_size=gs, mpi_construct=mc)


def _ring(sim_like, real_t):
    """vortex ring of bench.py on the (possibly non-cubic) local grid of a simulator / oracle"""
    import bench

    nz, ny, nx = sim_like.grid_size
    x_range = float(sim_like.x_range)  # every axis scaled to the unit cube, as bench.py does
    x = sim_like.local_x[None, None, :].astype(np.float64) / x_range
    y = sim_like.local_y[None, :, None].astype(np.float64) / (x_range * ny / nx)
    z = sim_like.local_z[:, None, None].astype(np.float64) / (x_range * nz / nx)
    return bench.vortex_ring(x, y, z, real_t)


# ------------------------------------------------------------------------------ Poisson
@pytest.mark.parametrize("n,real_t", [((256, 256, 256), np.float32), ((128, 128, 128), np.float64),
                                      ((128, 256, 512), np.float32)],
                         ids=["256-f32", "128-f64", "128x256x512-f32"])
def test_specialised_poisson_kernels_against_oracle(cuda, n, real_t):
    """Vector and scalar solve on random data (what the reference's tests feed,
    test_unbounded_poisson_solver_mpi_3d.py) through the LOG2N-specialised transforms."""
    from sopht_mpi_b200.numeric.eulerian_grid_ops import UnboundedPoissonSolverMPI3D

    gs = 2
    rng = np.random.default_rng(11)
    shape = tuple(v + 2 * gs for v in n)
    mc, _ = _construct(n, real_t)
    solver = UnboundedPoissonSolverMPI3D(*n, mpi_construct=mc, ghost_size=gs, x_range=1.0, real_t=real_t)
    assert solver.backend == "fft"
    oracle = UnboundedPoissonSolverOracle3D(*n, x_range=1.0, real_t=real_t, workers=CORES)
    rhs = rng.uniform(size=(3,) + shape).astype(real_t)
    ref = np.zeros_like(rhs)
    oracle.vector_field_solve(ref, rhs, gs)
    d_rhs = torch.from_numpy(rhs).to(cuda)
    out = torch.full_like(d_rhs, 7.0)
    solver.vector_field_solve(solution_vector_field=out, rhs_vector_field=d_rhs)
    got = out.cpu().numpy()
    inner = (slice(None),) + (slice(gs, -gs),) * 3
    for c in range(3):
        assert _rel(got[c][inner[1:]], ref[c][inner[1:]]) <= TOL[real_t], c
    mask = np.ones(shape, bool)
    mask[gs:-gs, gs:-gs, gs:-gs] = False
    assert np.all(got[:, mask] == 7.0)  # ghosts of the solution are never written
    one = torch.zeros_like(d_rhs[0])
    solver.solve(solution_field=one, rhs_field=d_rhs[2])
    assert _rel(one.cpu().numpy()[inner[1:]], ref[2][inner[1:]]) <= TOL[real_t]


@pytest.mark.parametrize("n,real_t", [((256, 256, 256), np.float32), ((512, 512, 512), np.float32),
                                      ((256, 256, 256), np.float64), ((64, 128, 1024), np.float32)],
                         ids=["256-f32", "512-f32", "256-f64", "64x128x1024-f32"])
def test_fft_backend_against_cufft_backend(cuda, n, real_t):
    """Both backends of the library on the same right-hand side, up to the 512^3 grid of the
    north-star target (n = 1024 transforms: 32 points per thread in all three strided passes)."""
    from sopht_mpi_b200.numeric.eulerian_grid_ops import UnboundedPoissonSolverMPI3D

    gs = 2
    mc, _ = _construct(n, real_t)
    gen = torch.Generator(device=cuda).manual_seed(5)
    dt = torch.float32 if real_t == np.float32 else torch.float64
    rhs = torch.rand((3,) + tuple(v + 2 * gs for v in n), device=cuda, dtype=dt, generator=gen)
    sols = {}
    for backend in ("fft", "cufft"):
        solver = UnboundedPoissonSolverMPI3D(*n, mpi_construct=mc, ghost_size=gs, x_range=1.0, real_t=real_t,
                                             backend=backend)
        sols[backend] = torch.zeros_like(rhs)
        solver.vector_field_solve(solution_vector_field=sols[backend], rhs_vector_field=rhs)
        torch.cuda.synchronize()
        del solver
        torch.cuda.empty_cache()
    scale = sols["cufft"].abs().max().item()
    err = (sols["fft"] - sols["cufft"]).abs().max().item() / scale
    assert err <= (1e-5 if real_t == np.float32 else 1e-11), err


# ------------------------------------------------------------------------ full time steps
@pytest.mark.parametrize("n,real_t,steps", [((256, 256, 256), np.float32, 2), ((128, 128, 128), np.float64, 3)],
                         ids=["256-f32", "128-f64"])
def test_navier_stokes_steps_at_baseline_size(cuda, n, real_t, steps):
    """BASELINE configs[1]: vortex ring, flow_type navier_stokes, the fused kernels that bench.py
    times; omega, u, psi after `steps` steps (reference test_flow_simulators_3d.py:266-330 compares
    the same three fields against the hand-composed operator sequence)."""
    from sopht_mpi_b200.simulator import UnboundedFlowSimulator3D

    kw = dict(grid_size=n, x_range=1.0, kinematic_viscosity=1e-3, flow_type="navier_stokes", real_t=real_t)
    sim = UnboundedFlowSimulator3D(**kw)
    ora = FlowSimulatorOracle3D(fft_workers=CORES, **kw)
    w0 = _ring(ora, real_t)
    ora.vorticity_field[...] = w0
    sim.vorticity_field[...] = w0
    zero = [0.0, 0.0, 0.0]
    ora.compute_flow_velocity(zero)
    sim.compute_flow_velocity(free_stream_velocity=zero)
    for _ in range(steps):
        dt = ora.compute_stable_timestep()
        assert abs(sim.compute_stable_timestep() - dt) <= 1e-5 * dt
        ora.time_step(dt, zero)
        sim.time_step(dt=dt, free_stream_velocity=zero)
    tol = TOL[real_t]
    assert _rel(sim.vorticity_field, ora.vorticity_field) <= tol
    assert _rel(sim.velocity_field, ora.velocity_field) <= tol
    assert _rel(sim.stream_func_field, ora.stream_func_field) <= tol


def _sphere_points(centre, diameter, spacing):
    import bench

    return bench.sphere_points(centre, diameter, spacing)


class _Body:
    pass


def _fsi_pair(n, real_t, x_range, pts, lag_vel, k, c, **sim_kw):
    """GPU simulator + interactor and the composed CPU oracle for the same body"""
    from sopht_mpi_b200.simulator import (PrescribedForcingGrid, RigidBodyFlowInteractionMPI,
                                          UnboundedFlowSimulator3D)

    kw = dict(grid_size=n, x_range=x_range, kinematic_viscosity=2e-3, flow_type="navier_stokes_with_forcing",
              real_t=real_t, with_free_stream_flow=True, **sim_kw)
    sim = UnboundedFlowSimulator3D(**kw)
    ora = FlowSimulatorOracle3D(fft_workers=CORES, **kw)
    dx = float(sim.dx)
    interactor = RigidBodyFlowInteractionMPI(
        mpi_construct=sim.mpi_construct, mpi_ghost_exchange_communicator=sim.mpi_ghost_exchange_communicator,
        rigid_body=_Body(), eul_grid_forcing_field=sim.eul_grid_forcing_field,
        eul_grid_velocity_field=sim.velocity_field, virtual_boundary_stiffness_coeff=k,
        virtual_boundary_damping_coeff=c, dx=sim.dx, grid_dim=3,
        forcing_grid_cls=lambda grid_dim, rigid_body: PrescribedForcingGrid(
            grid_dim, pts, velocity_field=lag_vel, max_lag_grid_dx=dx))
    area = dx ** 2
    vbf_o = ib_oracle.VirtualBoundaryForcingOracle(k * area, c * area, 3, ora.dx, real_t, np.float64,
                                                   sim.ghost_size)
    return sim, ora, interactor, vbf_o


def test_sphere_fsi_512x256x256_through_the_interactor(cuda):
    """BASELINE configs[2] (flow past a sphere with virtual boundary forcing, 512x256x256 float32,
    flow_past_sphere_case.py:32-82 with a synthetic latitude-ring surface grid): interactor() ->
    interactor.time_step -> flow step, twice, against FlowSimulatorOracle3D +
    VirtualBoundaryForcingOracle."""
    n, real_t = (256, 256, 512), np.float32
    diameter = 0.4 * min(n[0], n[1]) / n[2]
    pts = _sphere_points((0.25, 0.25, 0.25), diameter, np.pi * diameter / 192)
    assert pts.shape[1] > 1e4
    vel = np.zeros_like(pts)
    sim, ora, interactor, vbf_o = _fsi_pair(n, real_t, 1.0, pts, vel, -6e5 / 4, -3.5e2 / 4)
    u_inf = [1.0, 0.0, 0.0]
    ora.compute_flow_velocity(u_inf)
    sim.compute_flow_velocity(free_stream_velocity=u_inf)
    for _ in range(2):
        dt = ora.compute_stable_timestep(dt_prefac=0.5)
        assert abs(sim.compute_stable_timestep(dt_prefac=0.5) - dt) <= 1e-5 * dt
        vbf_o.compute_interaction_force_on_eul_and_lag_grid(ora.eul_grid_forcing_field, ora.velocity_field, pts, vel)
        interactor()
        assert _rel(interactor.global_lag_grid_forcing_field, vbf_o.forcing) <= 1e-4
        vbf_o.time_step(dt)
        interactor.time_step(dt)
        ora.time_step(dt, free_stream_velocity=u_inf)
        sim.time_step(dt=dt, free_stream_velocity=u_inf)
    assert np.abs(ora.vorticity_field).max() > 1.0  # the body did shed vorticity
    tol = TOL[real_t]
    assert _rel(sim.vorticity_field, ora.vorticity_field) <= tol
    assert _rel(sim.velocity_field, ora.velocity_field) <= tol
    assert _rel(sim.stream_func_field, ora.stream_func_field) <= tol
    assert _rel(interactor.local_lag_grid_position_mismatch_field, vbf_o.position_mismatch) <= 1e-4
    assert float(np.abs(np.asarray(sim.eul_grid_forcing_field)).max()) == 0.0  # reset by the flow step


@pytest.mark.parametrize("real_t", [np.float32, np.float64], ids=["f32", "f64"])
def test_rod_fsi_with_filter_through_the_interactor(cuda, real_t):
    """BASELINE configs[3] at half size (256x128x128, x_range 1.8, order-1 multiplicative filter,
    flow_past_rod_case.py:24-25,40,106-116,261-271): three velocity-interpolation sub-steps
    (compute_flow_forces_and_torques) + one full interaction per flow step, moving points."""
    import bench

    n = (128, 128, 256)
    x_range = 1.8
    y_range = x_range * n[1] / n[2]
    z_range = x_range * n[0] / n[2]
    pts0 = bench.rod_surface_points(x_range, y_range, z_range, n_elem=80, n_ring=32)
    assert pts0.shape[1] > 2000
    rng = np.random.default_rng(1234)
    vel = 0.05 * rng.standard_normal(pts0.shape)
    pts = pts0.copy()
    sim, ora, interactor, vbf_o = _fsi_pair(n, real_t, x_range, pts, vel, -2e5, -1e2, filter_vorticity=True,
                                            filter_setting_dict={"order": 1, "type": "multiplicative"})
    grid = interactor.forcing_grid
    u_inf = [1.0, 0.0, 0.0]
    ora.compute_flow_velocity(u_inf)
    sim.compute_flow_velocity(free_stream_velocity=u_inf)
    for _ in range(3):
        dt = ora.compute_stable_timestep(dt_prefac=0.25)
        assert abs(sim.compute_stable_timestep(dt_prefac=0.25) - dt) <= 1e-5 * dt
        for _sub in range(3):
            grid.position_field += (dt / 3) * vel  # the body moves between sub-steps
            pts = grid.position_field.copy()
            vbf_o.compute_interaction_force_on_lag_grid(ora.velocity_field, pts, vel)
            interactor.compute_flow_forces_and_torques()
            assert _rel(interactor.global_lag_grid_forcing_field, vbf_o.forcing) <= 10 * TOL[real_t]
            assert np.allclose(interactor.body_flow_forces[:, 0], -vbf_o.forcing.sum(axis=1),
                               rtol=100 * TOL[real_t])
        vbf_o.compute_interaction_force_on_eul_and_lag_grid(ora.eul_grid_forcing_field, ora.velocity_field, pts, vel)
        interactor()
        vbf_o.time_step(dt)
        interactor.time_step(dt)
        ora.time_step(dt, free_stream_velocity=u_inf)
        sim.time_step(dt=dt, free_stream_velocity=u_inf)
    tol = TOL[real_t]
    assert _rel(sim.vorticity_field, ora.vorticity_field) <= tol
    assert _rel(sim.velocity_field, ora.velocity_field) <= tol
    assert _rel(sim.stream_func_field, ora.stream_func_field) <= tol
    assert abs(interactor.get_grid_deviation_error_l2_norm()
               - np.linalg.norm(vbf_o.position_mismatch) / np.sqrt(pts.shape[1])) <= 1e-6


# ---------------------------------------------------------------------- diagnostics, Peskin
def test_divergence_l2_norm_and_max_vorticity(cuda):
    """E10 / E12 (flow_simulators_mpi_3d.py:451-476) on the device: sb200_divergence +
    sb200_sum_squares, sb200_max."""
    from sopht_mpi_b200.simulator import UnboundedFlowSimulator3D

    for real_t in (np.float32, np.float64):
        n = (32, 48, 64)
        sim = UnboundedFlowSimulator3D(grid_size=n, x_range=1.0, kinematic_viscosity=1e-3,
                                       flow_type="navier_stokes", real_t=real_t)
        gs = sim.ghost_size
        rng = np.random.default_rng(3)
        w = (rng.uniform(size=sim.vorticity_field.shape) - 0.3).astype(real_t)
        sim.vorticity_field[...] = w
        div = np.zeros(w.shape[1:], real_t)
        st.divergence_mpi(div, w, real_t(1.0 / sim.dx), gs)
        ref = np.sqrt(np.sum(div[gs:-gs, gs:-gs, gs:-gs].astype(np.float64) ** 2)) * float(sim.dx) ** 1.5
        got = sim.get_vorticity_divergence_l2_norm()
        assert abs(got - ref) <= (1e-5 if real_t == np.float32 else 1e-11) * ref
        assert sim.get_max_vorticity() == w[:, gs:-gs, gs:-gs, gs:-gs].max()


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("lag_t", [np.float32, np.float64], ids=["lag32", "lag64"])
def test_peskin_weights_and_interpolation_on_gpu(cuda, dim, lag_t):
    """L5 Peskin kernel (EulerianLagrangianGridCommunicatorMPI3D.py:482-589) through the fused
    sb200_ib_interact_lag with kernel_type = 1, against the oracle restatement (golden-pinned for
    the cosine kernel; the Peskin formula is checked against the reference's numba kernel in
    tests/test_oracle_golden.py)."""
    from sopht_mpi_b200 import _lib
    from sopht_mpi_b200.utils.device import dptr

    lib = _lib.load()
    gs, w, n_local = 2, 2, 24
    real_t = np.float64 if lag_t == np.float64 else np.float32
    dx = real_t(1.0 / n_local)
    shift = real_t(dx / 2)
    rng = np.random.default_rng(8)
    n = 777
    pos = (0.15 + 0.7 * rng.uniform(size=(dim, n))).astype(lag_t)
    eul = rng.uniform(size=(dim,) + (n_local + 2 * gs,) * dim).astype(real_t)
    nearest, support = ib_oracle.support_and_nearest_index(pos, dx, shift, w, (0,) * dim, gs)
    weights = ib_oracle.peskin_weights(support, dx, real_t)
    ref = np.zeros((dim, n), lag_t)
    ib_oracle.eulerian_to_lagrangian(ref, eul, weights, nearest, dx, w)
    g = _lib.make_grid(dim, real_t, gs, (n_local,) * dim, [1] * (2 * dim))
    p = _lib.IBParams()
    p.lag_dtype, p.kernel_type, p.width = _lib.dtype_code(lag_t), 1, w
    p.dx, p.coord_shift = float(dx), float(shift)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda)  # noqa: E731
    near_d = torch.zeros((dim, n), dtype=torch.int64, device=cuda)
    w_d, u_d = t(np.zeros_like(weights)), t(np.zeros_like(pos))
    eul_d, pos_d = t(eul), t(pos)
    _lib.check(lib, lib.sb200_ib_interact_lag(ctypes.byref(g), ctypes.byref(p), n, dptr(eul_d), dptr(pos_d),
                                              None, None, dptr(near_d), dptr(w_d), dptr(u_d), None, None, None))
    torch.cuda.synchronize()
    tol = 1e-5 if lag_t == np.float32 else 1e-10
    assert np.array_equal(near_d.cpu().numpy(), nearest)
    assert _rel(w_d.cpu().numpy(), weights) <= tol
    assert _rel(u_d.cpu().numpy(), ref) <= tol
    # the delta function is a partition of unity: weights sum to 1 / dx^dim
    sums = w_d.cpu().numpy().reshape(-1, n).sum(axis=0) * float(dx) ** dim
    assert np.abs(sums - 1.0).max() <= 10 * tol


@pytest.mark.parametrize("name", ["ib_3d_f32_f64.npz", "ib_2d_f32_f64.npz"])
def test_peskin_weights_against_reference_golden(cuda, name):
    """Peskin weights of the fused kernel against vectors produced by the reference's own numba
    kernel (tests/golden/make_golden.py: generate_peskin_interpolation_weights_kernel)."""
    from sopht_mpi_b200 import _lib
    from sopht_mpi_b200.utils.device import dptr

    lib = _lib.load()
    gd = np.load(os.path.join(os.path.dirname(__file__), "golden", name))
    dim, gs, w = int(gd["dim"]), int(gd["gs"]), int(gd["width"])
    dx, shift, pos = gd["dx"][()], gd["shift"][()], gd["pos"]
    real_t = type(dx)
    n_local = gd["eul_vec"].shape[-1] - 2 * gs
    g = _lib.make_grid(dim, real_t, gs, (n_local,) * dim, [1] * (2 * dim))
    p = _lib.IBParams()
    p.lag_dtype, p.kernel_type, p.width = _lib.dtype_code(pos.dtype), 1, w
    p.dx, p.coord_shift = float(dx), float(shift)
    n = pos.shape[1]
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda)  # noqa: E731
    near_d = torch.zeros((dim, n), dtype=torch.int64, device=cuda)
    w_d, u_d = t(np.zeros_like(gd["w_pes"])), t(np.zeros_like(pos))
    eul_d, pos_d = t(gd["eul_vec"]), t(pos)
    _lib.check(lib, lib.sb200_ib_interact_lag(ctypes.byref(g), ctypes.byref(p), n, dptr(eul_d), dptr(pos_d),
                                              None, None, dptr(near_d), dptr(w_d), dptr(u_d), None, None, None))
    torch.cuda.synchronize()
    assert np.array_equal(near_d.cpu().numpy(), gd["nearest"])
    assert _rel(w_d.cpu().numpy(), gd["w_pes"]) <= (1e-5 if pos.dtype == np.float32 else 1e-10)


# ------------------------------------------------------ distributed entry points, virtual ranks
@pytest.mark.parametrize("n,real_t,nranks", [((64, 32, 64), np.float32, 2), ((64, 64, 32), np.float64, 4),
                                             ((256, 256, 256), np.float32, 8), ((256, 128, 512), np.float32, 4),
                                             ((128, 128, 128), np.float64, 2)],
                         ids=["64x32x64-f32-P2", "64x64x32-f64-P4", "256-f32-P8", "256x128x512-f32-P4",
                              "128-f64-P2"])
def test_slab_poisson_with_virtual_ranks_on_one_gpu(cuda, n, real_t, nranks):
    """SURVEY P4 (MPIDomainDoublingCommunicator3D + mpi4py-fft transposes,
    UnboundedPoissonSolverMPI3D.py:190-382) on a single GPU: the slab pipeline of every rank, with
    the transposes done by the test, must reproduce the single-domain solve."""
    from sopht_mpi_b200.numeric.eulerian_grid_ops import UnboundedPoissonSolverMPI3D

    gs, ncomp = 2, 3
    dt = torch.float32 if real_t == np.float32 else torch.float64
    gen = torch.Generator(device=cuda).manual_seed(21)
    rhs = torch.rand((ncomp,) + tuple(v + 2 * gs for v in n), device=cuda, dtype=dt, generator=gen)
    outs = slab_poisson_solve(_Cuda(), n, real_t, nranks, rhs, ncomp, backend=1)
    mc, _ = _construct(n, real_t)
    single = UnboundedPoissonSolverMPI3D(*n, mpi_construct=mc, ghost_size=gs, x_range=1.0, real_t=real_t)
    ref = torch.zeros_like(rhs)
    single.vector_field_solve(solution_vector_field=ref, rhs_vector_field=rhs)
    if max(n) <= 128:  # and the single-domain solve is the oracle's
        oracle = UnboundedPoissonSolverOracle3D(*n, x_range=1.0, real_t=real_t, workers=CORES)
        want = np.zeros(rhs.shape, real_t)
        oracle.vector_field_solve(want, rhs.cpu().numpy(), gs)
        inner = (slice(None),) + (slice(gs, -gs),) * 3
        assert _rel(ref.cpu().numpy()[inner], want[inner]) <= TOL[real_t]
    # the single-domain solve runs the same three stages on a one-rank layout: bit for bit the same result
    nzl = n[0] // nranks
    for r in range(nranks):
        got = outs[r][:, gs:-gs, gs:-gs, gs:-gs]
        want = ref[:, r * nzl + gs:r * nzl + gs + nzl, gs:-gs, gs:-gs]
        assert torch.equal(got, want), (r, (got - want).abs().max().item() / ref.abs().max().item())
        assert torch.all(outs[r][:, 0] == 7.0) and torch.all(outs[r][:, :, :, -1] == 7.0)  # ghosts untouched


@pytest.mark.parametrize("real_t", [np.float32, np.float64], ids=["f32", "f64"])
def test_ghost_sum_with_virtual_ranks_on_one_gpu(cuda, real_t):
    """SURVEY L9 (MPIGhostSumCommunicator3D.ghost_sum, ...MPI3D.py:677-792) for three virtual
    z-slabs: spreading onto each padded slab followed by the ghost sum (slabs travel to the z
    neighbours, sb200_ghost_sum_add_z, sb200_clear_ghost_cells) equals spreading onto the single
    domain."""
    from sopht_mpi_b200 import _lib
    from sopht_mpi_b200.utils.device import dptr

    lib = _lib.load()
    gs, nranks = 2, 3
    n = (24, 16, 20)
    nzl = n[0] // nranks
    dt = torch.float32 if real_t == np.float32 else torch.float64
    rng = np.random.default_rng(17)
    shape = tuple(v + 2 * gs for v in n)
    glob = torch.from_numpy(rng.uniform(size=(3,) + shape).astype(real_t)).to(cuda)
    # single domain: only the ghost clearing applies (every neighbour is PROC_NULL)
    ref = glob.clone()
    g1 = _lib.make_grid(3, real_t, gs, n, [1] * 6)
    _lib.check(lib, lib.sb200_clear_ghost_cells(ctypes.byref(g1), dptr(ref), 3, None))
    # virtual slabs: slab r holds the global planes [r nzl, r nzl + nzl + 2 gs); a cell of the global
    # field that two slabs cover is split between them so that the ghost sum has to reassemble it
    slabs = []
    for r in range(nranks):
        part = glob[:, r * nzl:r * nzl + nzl + 2 * gs].clone()
        if r > 0:
            part[:, :2 * gs] *= 0.25
        if r < nranks - 1:
            part[:, -2 * gs:] *= 0.75
        slabs.append(part.contiguous())
    jobs = []
    for r in range(nranks):
        phys = [int(r == 0), int(r == nranks - 1), 1, 1, 1, 1]
        g = _lib.make_grid(3, real_t, gs, (nzl, n[1], n[2]), phys)
        from_prev = slabs[r - 1][:, -gs:].contiguous() if r > 0 else None  # upper ghost slab of r - 1
        from_next = slabs[r + 1][:, :gs].contiguous() if r < nranks - 1 else None  # lower ghost slab of r + 1
        jobs.append((slabs[r], g, from_prev, from_next))
    outs = []
    for part, g, from_prev, from_next in jobs:
        out = part.clone()
        _lib.check(lib, lib.sb200_ghost_sum_add_z(ctypes.byref(g), dptr(out), 3, dptr(from_prev),
                                                  dptr(from_next), None))
        _lib.check(lib, lib.sb200_clear_ghost_cells(ctypes.byref(g), dptr(out), 3, None))
        outs.append(out)
    torch.cuda.synchronize()
    tol = 1e-6 if real_t == np.float32 else 1e-14
    for r, out in enumerate(outs):
        want = ref[:, r * nzl + gs:r * nzl + gs + nzl]
        assert (out[:, gs:-gs] - want).abs().max().item() <= tol, r
        assert float(out[:, :gs].abs().max()) == 0.0 and float(out[:, -gs:].abs().max()) == 0.0


# -------------------------------------------------------------- device-resident Lagrangian state
def test_device_rank_ownership_on_gpu_against_reference_golden(cuda):
    """SURVEY L1 on the GPU: sb200_ib_rank_address gives the integers of the reference's
    _compute_lag_nodes_rank_address (tests/golden/ownership.npz, produced by the reference function)."""
    from ib_helpers import rank_address
    from sopht_mpi_b200 import _lib
    from sopht_mpi_b200.utils.device import dptr

    lib = _lib.load()
    o = np.load(os.path.join(os.path.dirname(__file__), "golden", "ownership.npz"))

    def call(name, *a):
        _lib.check(lib, getattr(lib, name)(*a))

    to_dev = lambda a: torch.from_numpy(a).to(cuda)  # noqa: E731
    to_host = lambda t: t.cpu().numpy()  # noqa: E731
    for t in ("f64", "f32"):
        for d in ("3", "2"):
            addr, flag = rank_address(call, dptr, o[f"pos{d}_{t}"], o["dx"][()], o["shift"][()], o["local" + d],
                                      o["topo" + d], to_dev, to_host)
            assert np.array_equal(addr, o[f"addr{d}_{t}"]) and flag == 0
    # many random points incl. block boundaries, against the host twin of the reference expression
    rng = np.random.default_rng(2)
    dx, local, topo = np.float32(1.0 / 96), np.array([12, 48, 96]), np.array([8, 2, 1])
    shift = np.float32(dx / 2)
    pos = rng.uniform(0.0, 1.0, size=(3, 20000))
    pos[2] = rng.uniform(0.0, 1.0, size=20000)
    k = rng.integers(0, 8, size=2000)
    pos[2, :2000] = k * float(dx) * 12 + float(shift)  # exactly on slab boundaries
    want = ib_oracle.lag_nodes_rank_address(pos, dx, shift, local, topo)
    got, flag = rank_address(call, dptr, pos, dx, shift, local, topo, to_dev, to_host)
    assert np.array_equal(got, want) and flag == 0


def test_virtual_boundary_forcing_host_mirrors_follow_the_device(cuda):
    """The reference keeps the Lagrangian state in host arrays that callers read, write in place and
    assign (test_virtual_boundary_forcing_mpi_3d.py:1104-1109, the restart recipe); here they are lazy
    mirrors of device arrays: every access pattern must see reference semantics."""
    from sopht_mpi_b200.numeric.immersed_boundary_ops import VirtualBoundaryForcingMPI

    real_t, n_local, gs, dim = np.float64, 16, 2, 3
    mc, _ = _construct((n_local,) * 3, real_t)
    dx = real_t(1.0 / n_local)
    rng = np.random.default_rng(9)
    pos = 0.25 + 0.5 * rng.uniform(size=(dim, 33))
    vel = rng.uniform(size=(dim, 33))
    k, c = -3.0, -0.5
    vbf = VirtualBoundaryForcingMPI(mpi_construct=mc, ghost_size=gs, virtual_boundary_stiffness_coeff=k,
                                    virtual_boundary_damping_coeff=c, grid_dim=dim, dx=dx,
                                    global_lag_grid_position_field=pos)
    ora = ib_oracle.VirtualBoundaryForcingOracle(k, c, dim, dx, real_t, np.float64, gs)
    assert vbf.local_num_lag_nodes == 33 and vbf.global_num_lag_nodes == 33
    u_h = rng.uniform(size=(dim,) + (n_local + 2 * gs,) * dim)
    u = torch.from_numpy(u_h).to(cuda)
    f = torch.zeros_like(u)
    f_h = np.zeros_like(u_h)
    # 1. attribute assignment of the state, then a step (reference test :1104-1109)
    dpos0 = 0.01 * rng.uniform(size=(dim, 33))
    vbf.local_lag_grid_position_mismatch_field = dpos0.copy()
    ora._ensure(33)
    ora.position_mismatch[...] = dpos0
    held = vbf.global_lag_grid_forcing_field  # an IO object would keep this reference
    for step in range(3):
        vbf.compute_interaction_forcing(local_eul_grid_forcing_field=f, local_eul_grid_velocity_field=u,
                                        global_lag_grid_position_field=pos, global_lag_grid_velocity_field=vel)
        f_h[...] = 0
        ora.compute_interaction_force_on_eul_and_lag_grid(f_h, u_h, pos, vel)
        assert _rel(held, ora.forcing) <= 1e-12  # refreshed without being asked for again
        assert _rel(f.cpu().numpy(), f_h) <= 1e-12
        vbf.time_step(0.05)
        ora.time_step(0.05)
        last_pos = pos
        pos = pos + 0.002  # the body moves: fresh kinematics every interaction
        if step == 1:  # 2. in-place write through a temporary reference
            vbf.local_lag_grid_position_mismatch_field[...] *= 0.5
            ora.position_mismatch[...] *= 0.5
    assert _rel(vbf.local_lag_grid_position_mismatch_field, ora.position_mismatch) <= 1e-12
    assert _rel(vbf.global_lag_grid_velocity_mismatch_field, ora.velocity_mismatch) <= 1e-12
    assert _rel(vbf.local_lag_grid_flow_velocity_field, ora.flow_velocity) <= 1e-12
    assert np.array_equal(vbf.local_nearest_eul_grid_index_to_lag_grid, ora.nearest)
    assert _rel(vbf.local_interp_weights, ora.weights) <= 1e-12
    assert np.array_equal(vbf.local_lag_grid_position_field, last_pos)
    assert vbf.time == pytest.approx(0.15)
    # 3. restart recipe: re-map, re-initialise the local buffers, scatter the global state back
    saved = vbf.global_lag_grid_position_mismatch_field.copy()
    comm = vbf.mpi_lagrangian_field_communicator
    comm.map_lagrangian_nodes_based_on_position(pos)
    vbf.local_num_lag_nodes = comm.local_num_lag_nodes
    vbf._init_local_buffers(vbf.local_num_lag_nodes)
    comm.scatter_global_field(local_lag_field=vbf.local_lag_grid_position_mismatch_field, global_lag_field=saved)
    vbf.time_step(0.0)
    assert np.array_equal(vbf.local_lag_grid_position_mismatch_field, saved)
    # 4. a point outside the domain is reported (the reference aborts)
    bad = pos.copy()
    bad[0, 0] = 1.7
    vbf.compute_interaction_force_on_lag_grid(u, bad, vel)
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError):
        vbf.compute_interaction_force_on_lag_grid(u, pos, vel)


def test_flow_past_sphere_example_with_the_in_repo_forcing_grid(cuda):
    """The call sequence of examples/3d_examples/FlowPastSphereCase/flow_past_sphere_case.py:32-140
    (RigidBodyFlowInteractionMPI + SphereForcingGrid + navier_stokes_with_forcing), at 64x32x32, against
    the composed oracle; the sphere is at rest, so its kinematics are uploaded once."""
    import types

    from sopht_mpi_b200.simulator import RigidBodyFlowInteractionMPI, SphereForcingGrid, UnboundedFlowSimulator3D

    real_t, n, x_range = np.float32, (32, 32, 64), 1.0
    kw = dict(grid_size=n, x_range=x_range, kinematic_viscosity=2e-3, flow_type="navier_stokes_with_forcing",
              real_t=real_t, with_free_stream_flow=True)
    sim = UnboundedFlowSimulator3D(**kw)
    ora = FlowSimulatorOracle3D(**kw)
    diameter = 0.4 * min(n[0], n[1]) / n[2]
    sphere = types.SimpleNamespace(
        radius=diameter / 2, position_collection=np.array([[0.25], [0.5 * sim.y_range], [0.5 * sim.z_range]]),
        velocity_collection=np.zeros((3, 1)), omega_collection=np.zeros((3, 1)),
        director_collection=np.eye(3).reshape(3, 3, 1))
    interactor = RigidBodyFlowInteractionMPI(
        mpi_construct=sim.mpi_construct, mpi_ghost_exchange_communicator=sim.mpi_ghost_exchange_communicator,
        rigid_body=sphere, eul_grid_forcing_field=sim.eul_grid_forcing_field,
        eul_grid_velocity_field=sim.velocity_field, virtual_boundary_stiffness_coeff=-6e5 / 4,
        virtual_boundary_damping_coeff=-3.5e2 / 4, dx=sim.dx, grid_dim=3, master_rank=0,
        forcing_grid_cls=SphereForcingGrid,
        num_forcing_points_along_equator=int(1.875 * diameter / x_range * n[2]))
    grid = interactor.forcing_grid
    assert isinstance(grid, SphereForcingGrid) and grid.num_lag_nodes > 100
    area = grid.get_maximum_lagrangian_grid_spacing() ** 2
    vbf_o = ib_oracle.VirtualBoundaryForcingOracle(-6e5 / 4 * area, -3.5e2 / 4 * area, 3, ora.dx, real_t, np.float64,
                                                   sim.ghost_size)
    u_inf = [1.0, 0.0, 0.0]
    ora.compute_flow_velocity(u_inf)
    sim.compute_flow_velocity(free_stream_velocity=u_inf)
    uploads = []
    real_upload = interactor._upload_kinematics
    interactor._upload_kinematics = lambda p, v: (uploads.append(interactor._kin_i), real_upload(p, v))[1]
    for _ in range(4):
        dt = ora.compute_stable_timestep(dt_prefac=0.5)
        assert abs(sim.compute_stable_timestep(dt_prefac=0.5) - dt) <= 1e-5 * dt
        vbf_o.compute_interaction_force_on_eul_and_lag_grid(ora.eul_grid_forcing_field, ora.velocity_field,
                                                            grid.position_field, grid.velocity_field)
        interactor()
        vbf_o.time_step(dt)
        interactor.time_step(dt)
        ora.time_step(dt, free_stream_velocity=u_inf)
        sim.time_step(dt=dt, free_stream_velocity=u_inf)
    assert len(set(uploads[1:])) == 1  # the device copy of the kinematics was reused after the first upload
    tol = TOL[real_t]
    assert _rel(sim.vorticity_field, ora.vorticity_field) <= tol
    assert _rel(sim.velocity_field, ora.velocity_field) <= tol
    interactor.compute_flow_forces_and_torques()
    vbf_o.compute_interaction_force_on_lag_grid(ora.velocity_field, grid.position_field, grid.velocity_field)
    assert _rel(interactor.global_lag_grid_forcing_field, vbf_o.forcing) <= 1e-4
    want = -vbf_o.forcing.sum(axis=1)  # the transverse components cancel to rounding noise
    assert np.allclose(interactor.body_flow_forces[:, 0], want, rtol=1e-3, atol=1e-5 * np.abs(want).max())
