"""Distributed Poisson solve of grids that are not powers of two: the z-slab mode of the cuFFT backend.

* P VIRTUAL ranks on one device (the test moves the exchange blocks) against the single-rank cuFFT solve of
  the whole domain and the scipy oracle, on rank counts whose kx blocks end partially filled, hold only the
  Nyquist bin, or hold no bin at all;
* the sphere workload's 2:1:1 shape refined 1.5x (768 x 384 x 384) on 3 and 6 virtual ranks;
* ranks as processes on one GPU (real CUDA IPC exchanges) and on several GPUs: tests/dist_slab_cufft_worker.py.

Tolerances: relative L-inf <= 1e-5 (float32), <= 1e-10 (float64).
"""
import os
import types

import numpy as np
import pytest
import torch

from harness import _Cuda, run_ranks, slab_poisson_solve
from oracle.poisson import UnboundedPoissonSolverOracle3D

pytestmark = pytest.mark.gpu

TOL = {np.float64: 1e-10, np.float32: 1e-5}
GS = 2


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from sopht_mpi_b200 import _lib

    _lib.load()
    return torch.device("cuda", 0)


def _rel(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


def _single_rank_cufft(cuda, real_t, n, rhs):
    from sopht_mpi_b200.numeric.eulerian_grid_ops import UnboundedPoissonSolverMPI3D
    from sopht_mpi_b200.utils import MPIConstruct3D

    mc = MPIConstruct3D(*n, real_t=real_t)
    solver = UnboundedPoissonSolverMPI3D(*n, mpi_construct=mc, ghost_size=GS, x_range=1.0, real_t=real_t,
                                         backend="cufft")
    assert solver.backend == "cufft"
    ref = torch.zeros_like(rhs)
    if rhs.shape[0] == 3:
        solver.vector_field_solve(solution_vector_field=ref, rhs_vector_field=rhs)
    else:
        solver.solve(solution_field=ref[0], rhs_field=rhs[0])
    torch.cuda.synchronize()
    return ref


def _check_slabs(outs, ref, n, nranks, tol):
    nzl = n[0] // nranks
    for r in range(nranks):
        got = outs[r][:, GS:-GS, GS:-GS, GS:-GS]
        want = ref[:, r * nzl + GS:r * nzl + GS + nzl, GS:-GS, GS:-GS]
        assert _rel(got, want) <= tol, (r, _rel(got, want))
        # ghosts untouched
        assert torch.all(outs[r][:, :GS] == 7.0) and torch.all(outs[r][:, -GS:] == 7.0)
        assert torch.all(outs[r][:, :, :GS] == 7.0) and torch.all(outs[r][:, :, :, -GS:] == 7.0)


# (120, 72, 100), kxl per rank count: P = 2 -> 52, 3 -> 36, 5 -> 24 (last block partial), 6 -> 20 (rank 5 holds
# only the Nyquist bin 100), 8 -> 16 (rank 7 holds none).  (120, 48, 75), odd nx: P = 3 -> 28, 8 -> 12 (rank 7
# holds none).
CASES = [((120, 72, 100), np.float64, 2, 1), ((120, 72, 100), np.float64, 3, 3), ((120, 72, 100), np.float64, 5, 1),
         ((120, 72, 100), np.float64, 6, 3), ((120, 72, 100), np.float64, 8, 3), ((120, 48, 75), np.float32, 3, 1),
         ((120, 48, 75), np.float32, 8, 3)]


@pytest.mark.parametrize("n,real_t,nranks,ncomp", CASES,
                         ids=[f"{'x'.join(map(str, c[0]))}-{np.dtype(c[1]).name}-P{c[2]}-c{c[3]}" for c in CASES])
def test_cufft_slab_solve_with_virtual_ranks(cuda, n, real_t, nranks, ncomp):
    dt = torch.float32 if real_t == np.float32 else torch.float64
    gen = torch.Generator(device=cuda).manual_seed(5)
    rhs = torch.rand((ncomp,) + tuple(v + 2 * GS for v in n), device=cuda, dtype=dt, generator=gen)
    outs = slab_poisson_solve(_Cuda(), n, real_t, nranks, rhs, ncomp, backend=0)
    ref = _single_rank_cufft(cuda, real_t, n, rhs)
    _check_slabs(outs, ref, n, nranks, TOL[real_t])
    # and the single-rank solve is the oracle's
    oracle = UnboundedPoissonSolverOracle3D(*n, x_range=1.0, real_t=real_t, workers=os.cpu_count() or 1)
    want = np.zeros(rhs.shape, real_t)
    r_np = rhs.cpu().numpy()
    for c in range(ncomp):
        oracle.solve(want[c], r_np[c], GS)
    inner = (slice(None),) + (slice(GS, -GS),) * 3
    nzl = n[0] // nranks
    for r in range(nranks):
        got = outs[r][inner].cpu().numpy()
        w = want[:, r * nzl + GS:r * nzl + GS + nzl, GS:-GS, GS:-GS]
        assert np.abs(got - w).max() / np.abs(want[inner]).max() <= TOL[real_t], r


@pytest.mark.parametrize("nranks", [3, 6])
def test_cufft_slab_solve_at_the_refined_sphere_grid(cuda, nranks):
    """768 x 384 x 384 float32 (the sphere workload's 2:1:1 shape, 1.5x refined), a grid users distribute:
    the solver takes the slab pipeline there, and the slabs match the single-rank cuFFT solve."""
    from sopht_mpi_b200.numeric.eulerian_grid_ops import UnboundedPoissonSolverMPI3D

    n, real_t = (768, 384, 384), np.float32
    stand_in = types.SimpleNamespace(size=nranks, rank=0, device=cuda)  # the selection reads size, rank, device
    solver = UnboundedPoissonSolverMPI3D(*n, mpi_construct=stand_in, ghost_size=GS, x_range=1.0, real_t=real_t)
    assert solver.backend == "cufft" and not solver.replicated
    del solver
    gen = torch.Generator(device=cuda).manual_seed(9)
    rhs = torch.rand((3,) + tuple(v + 2 * GS for v in n), device=cuda, dtype=torch.float32, generator=gen)
    outs = slab_poisson_solve(_Cuda(), n, real_t, nranks, rhs, 3, backend=0)
    ref = _single_rank_cufft(cuda, real_t, n, rhs)
    _check_slabs(outs, ref, n, nranks, TOL[real_t])


@pytest.mark.parametrize("nranks", [2, 3, 4, 6, 8])
def test_small_grids_stay_replicated(cuda, nranks):
    """below the size floor the distributed cuFFT solve stays replicated (the grid of dist_gpu_worker.py's
    replicated check), at or above it the slab pipeline runs"""
    from sopht_mpi_b200.numeric.eulerian_grid_ops import UnboundedPoissonSolverMPI3D
    from sopht_mpi_b200.numeric.eulerian_grid_ops import poisson

    stand_in = types.SimpleNamespace(size=nranks, rank=0, device=cuda)
    small = UnboundedPoissonSolverMPI3D(6 * nranks, 20, 36, mpi_construct=stand_in, ghost_size=GS)
    assert small.replicated and small.backend == "cufft"
    n = (48, 72, 80)  # the grid of tests/dist_slab_cufft_worker.py
    assert n[0] * n[1] * n[2] >= poisson._SLAB_CUFFT_MIN_CELLS
    big = UnboundedPoissonSolverMPI3D(*n, mpi_construct=stand_in, ghost_size=GS)
    assert not big.replicated and big.backend == "cufft"


@pytest.mark.parametrize("size", [3, 6])
def test_cufft_slab_solve_and_steps_with_ranks_on_one_gpu(size):
    """tests/dist_slab_cufft_worker.py (vector solve and flow steps on slabs of a grid that is not a power of
    two, over the peer-memory all-to-all) with every rank a process on cuda:0"""
    run_ranks("dist_slab_cufft_worker.py", size, "DIST_SLAB_CUFFT_WORKER_OK", where="one_gpu")


@pytest.mark.parametrize("nproc", [2, 3, 4, 6, 8])
def test_cufft_slab_solve_and_steps_on_several_gpus(nproc):
    run_ranks("dist_slab_cufft_worker.py", nproc, "DIST_SLAB_CUFFT_WORKER_OK", where="gpus")
