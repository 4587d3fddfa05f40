"""world_size-2 gloo worker for the host-side distributed logic (run by test_host_logic.py
through torch.distributed.run).  Exits non-zero on failure."""
import os
import sys

import numpy as np
import torch.distributed as dist

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

from harness import join_ranks, leave_ranks  # noqa: E402
from oracle import ib as ib_oracle  # noqa: E402
from sopht_mpi_b200.utils import (MPIConstruct2D, MPIConstruct3D, MPIFieldCommunicator3D,  # noqa: E402
                                  MPIGhostCommunicator2D, MPIGhostCommunicator3D,
                                  MPILagrangianFieldCommunicator3D)


def check_halo_3d(periodic):
    gs = 2
    mc = MPIConstruct3D(8, 6, 10, periodic_domain=periodic, real_t=np.float64,
                        rank_distribution=(0, 1, 1))
    assert tuple(mc.grid_topology) == (2, 1, 1) and tuple(mc.local_grid_size) == (4, 6, 10)
    comm = MPIGhostCommunicator3D(ghost_size=gs, mpi_construct=mc)
    rng = np.random.default_rng(0)  # same global field on both ranks
    glob = rng.uniform(size=(8, 6, 10))
    z0 = mc.rank * 4
    local = np.zeros((4 + 2 * gs, 6 + 2 * gs, 10 + 2 * gs))
    local[gs:-gs, gs:-gs, gs:-gs] = glob[z0:z0 + 4]
    comm.exchange_scalar_field_init(local)
    comm.exchange_finalise()
    if periodic:
        padded = np.pad(glob, gs, mode="wrap")
        assert np.array_equal(local, padded[z0:z0 + 4 + 2 * gs])
    else:
        if mc.rank == 0:
            assert np.array_equal(local[-gs:, gs:-gs, gs:-gs], glob[4:4 + gs])
            assert np.all(local[:gs] == 0)
        else:
            assert np.array_equal(local[:gs, gs:-gs, gs:-gs], glob[4 - gs:4])
            assert np.all(local[-gs:] == 0)
    vec = np.stack([local, 2 * local, 3 * local])
    comm.exchange_vector_field_init(vec)
    comm.exchange_finalise()


def check_field_comm_and_lagrangian():
    gs = 2
    mc = MPIConstruct3D(8, 6, 10, real_t=np.float32, rank_distribution=(0, 1, 1))
    fc = MPIFieldCommunicator3D(ghost_size=gs, mpi_construct=mc, master_rank=0)
    rng = np.random.default_rng(1)
    glob = rng.uniform(size=(8, 6, 10)).astype(np.float32)
    local = np.zeros((4 + 2 * gs, 6 + 2 * gs, 10 + 2 * gs), np.float32)
    fc.scatter_global_scalar_field(local, glob if mc.rank == 0 else None)
    assert np.array_equal(local[fc.inner_idx], glob[mc.rank * 4:(mc.rank + 1) * 4])
    back = np.zeros_like(glob)
    fc.gather_local_scalar_field(back, local)
    if mc.rank == 0:
        assert np.array_equal(back, glob)
    # Lagrangian ownership: same integers as the oracle restatement of the reference
    dx = np.float32(1.0 / 10)
    shift = np.float32(dx / 2)
    lc = MPILagrangianFieldCommunicator3D(eul_grid_dx=dx, eul_grid_coord_shift=shift, mpi_construct=mc,
                                          master_rank=0, real_t=np.float64)
    pos = np.stack([rng.uniform(0.05, 0.95, 40), rng.uniform(0.05, 0.55, 40),
                    rng.uniform(0.05, 0.75, 40)])
    pos[2, 0] = 4 * float(dx) + float(shift)  # exactly on the slab boundary
    lc.map_lagrangian_nodes_based_on_position(pos if mc.rank == 0 else None)
    expect = ib_oracle.lag_nodes_rank_address(pos, dx, shift, mc.local_grid_size, mc.grid_topology)
    assert np.array_equal(lc.rank_address, expect)
    assert lc.local_num_lag_nodes == np.count_nonzero(expect == mc.rank)
    local_lag = np.zeros((3, lc.local_num_lag_nodes))
    lc.scatter_global_field(local_lag, pos if mc.rank == 0 else None)
    assert np.array_equal(local_lag, pos[:, expect == mc.rank])
    zlo = mc.rank * 4 * float(dx) + float(shift)
    assert np.all(local_lag[2] >= zlo - 1e-12) and np.all(local_lag[2] < zlo + 4 * float(dx))
    gathered = np.zeros_like(pos)
    lc.gather_local_field(gathered, 2.0 * local_lag)
    if mc.rank == 0:
        assert np.allclose(gathered, 2.0 * pos)
    assert mc.grid.allreduce(float(mc.rank + 1), op="sum") == 3.0
    assert mc.grid.allreduce(float(mc.rank + 1), op="min") == 1.0
    assert mc.grid.allreduce(mc.rank == 1, op="lor") is True


def check_halo_2d():
    gs = 2
    mc = MPIConstruct2D(8, 6, real_t=np.float64)
    assert tuple(mc.grid_topology) == (2, 1)
    comm = MPIGhostCommunicator2D(ghost_size=gs, mpi_construct=mc)
    glob = np.arange(48, dtype=np.float64).reshape(8, 6)
    local = np.zeros((4 + 2 * gs, 6 + 2 * gs))
    local[gs:-gs, gs:-gs] = glob[mc.rank * 4:(mc.rank + 1) * 4]
    comm.exchange_scalar_field_init(local)
    comm.exchange_finalise()
    if mc.rank == 0:
        assert np.array_equal(local[-gs:, gs:-gs], glob[4:6])
    else:
        assert np.array_equal(local[:gs, gs:-gs], glob[2:4])


def check_block_exchange():
    """PeerExchange on its collective (non-IPC) path: block q of rank r's source buffer must land
    in block r of rank q's destination buffer (the transposes of the distributed Poisson solve)."""
    import torch

    from sopht_mpi_b200.utils.peer import PeerExchange

    rank, size = dist.get_rank(), dist.get_world_size()
    ex = PeerExchange(2, 6 * size, torch.device("cpu"), rank, size)
    assert ex.mode == "nccl all-to-all"
    ex.local[0].copy_(torch.arange(6 * size, dtype=torch.float32) + 100 * rank)
    try:
        ex.exchange(1, 0)
    except RuntimeError as exc:  # gloo builds without all_to_all: nothing to check on this box
        if "alltoall" in str(exc).lower() or "all_to_all" in str(exc).lower():
            return
        raise
    got = ex.local[1].numpy().reshape(size, 6)
    for q in range(size):
        assert np.array_equal(got[q], np.arange(6) + 6 * rank + 100 * q), (rank, q, got[q])


if __name__ == "__main__":
    join_ranks()
    check_halo_3d(periodic=False)
    check_block_exchange()
    check_halo_3d(periodic=True)
    check_field_comm_and_lagrangian()
    check_halo_2d()
    leave_ranks("DIST_WORKER_OK")
