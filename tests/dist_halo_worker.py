"""Worker of tests/test_gpu_ranks_on_one_device.py: P processes that all use cuda:0 (gloo process group for the
host-side messages) exchange halo planes and ghost-sum slabs through the peer-memory mailboxes
(utils/peer.py:PeerHalo: CUDA IPC mappings, push kernel, epoch flags) and check them against the global
numpy arrays every rank can build for itself.  This is the path the multi-GPU runs use, exercised on one
device so that a single-GPU box covers it."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

from harness import join_ranks, leave_ranks  # noqa: E402


def main():
    join_ranks()
    from sopht_mpi_b200.numeric.immersed_boundary_ops.eulerian_lagrangian_grid_communicator import (
        MPIGhostSumCommunicator)
    from sopht_mpi_b200.utils import MPIConstruct3D, MPIGhostCommunicator3D
    from sopht_mpi_b200.utils.device import DeviceField
    from sopht_mpi_b200.utils.peer import peer_halo

    rank, size = dist.get_rank(), dist.get_world_size()
    gs = 2
    for real_t in (np.float32, np.float64):
        for periodic in (False, True):
            n = (8 * size, 8, 12)
            mc = MPIConstruct3D(*n, periodic_domain=periodic, real_t=real_t, rank_distribution=(0, 1, 1))
            assert mc.device.type == "cuda" and mc.size == size
            nzl = n[0] // size
            comm = MPIGhostCommunicator3D(ghost_size=gs, mpi_construct=mc)
            rng = np.random.default_rng(7)
            for it in range(9):  # several rounds: the four mailbox slots are reused
                glob = rng.standard_normal((3, n[0], n[1] + 2 * gs, n[2] + 2 * gs)).astype(real_t)
                scal = rng.standard_normal((n[0], n[1] + 2 * gs, n[2] + 2 * gs)).astype(real_t)

                def local_of(g, r):
                    loc = np.full(g.shape[:-3] + (nzl + 2 * gs,) + g.shape[-2:], -7.0, real_t)
                    loc[..., gs:-gs, :, :] = g[..., r * nzl:(r + 1) * nzl, :, :]
                    return loc

                def expected(g, r):
                    want = local_of(g, r)
                    lo, hi = r * nzl - gs, (r + 1) * nzl
                    if r > 0 or periodic:
                        want[..., :gs, :, :] = np.take(g, np.arange(lo, lo + gs) % n[0], axis=-3)
                    if r < size - 1 or periodic:
                        want[..., -gs:, :, :] = np.take(g, np.arange(hi, hi + gs) % n[0], axis=-3)
                    return want

                v = DeviceField(torch.from_numpy(local_of(glob, rank)).to(mc.device))
                s = DeviceField(torch.from_numpy(local_of(scal, rank)).to(mc.device))
                # two exchanges in flight (what the fused vorticity update does with omega and u)
                comm.exchange_vector_field_init(v)
                comm.exchange_scalar_field_init(s)
                halo = peer_halo(mc, 1)
                assert halo is not None and halo._in_flight == 2, "the exchange did not go through peer memory"
                comm.exchange_finalise()
                got_v, got_s = np.asarray(v), np.asarray(s)
                want_v, want_s = expected(glob, rank), expected(scal, rank)
                if periodic:  # the undivided axes wrap locally (reference mpi_utils_3d.py periodic branch)
                    inner = (Ellipsis, slice(gs, -gs), slice(gs, -gs))
                    got_v, got_s, want_v, want_s = got_v[inner], got_s[inner], want_v[inner], want_s[inner]
                assert np.array_equal(got_v, want_v), ("vector halo", real_t, periodic, it)
                assert np.array_equal(got_s, want_s), ("scalar halo", real_t, periodic, it)
            halo.check()

            if not periodic:
                # ghost sum: every rank's ghost slabs are added to the neighbours' boundary planes
                gsum = MPIGhostSumCommunicator(ghost_size=gs, mpi_construct=mc)
                for it in range(5):
                    rngs = [np.random.default_rng(100 * it + r) for r in range(size)]
                    locs = [g.standard_normal((3, nzl + 2 * gs, n[1] + 2 * gs, n[2] + 2 * gs)).astype(real_t)
                            for g in rngs]
                    f = DeviceField(torch.from_numpy(locs[rank].copy()).to(mc.device))
                    gsum.ghost_sum(f)
                    want = locs[rank].copy()
                    if rank > 0:
                        want[:, gs:2 * gs] += locs[rank - 1][:, -gs:]
                    if rank < size - 1:
                        want[:, -2 * gs:-gs] += locs[rank + 1][:, :gs]
                    keep = want[:, gs:-gs, gs:-gs, gs:-gs].copy()
                    want[...] = 0
                    want[:, gs:-gs, gs:-gs, gs:-gs] = keep
                    tol = 1e-6 if real_t == np.float32 else 1e-14
                    assert np.abs(np.asarray(f) - want).max() <= tol, ("ghost sum", real_t, it)
                halo.check()
            dist.barrier()
            mc._peer_halo.close()
            mc._peer_halo = None
    leave_ranks("DIST_HALO_WORKER_OK")


if __name__ == "__main__":
    main()
