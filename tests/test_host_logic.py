"""Host-side logic: topology, halo exchange, field scatter/gather, Lagrangian rank
ownership -- single process and world_size 2 over gloo."""
import os

import numpy as np
import pytest

from harness import run_ranks
from oracle import ib as ib_oracle
from sopht_mpi_b200.utils import (MPIConstruct2D, MPIConstruct3D, MPIGhostCommunicator3D,
                                  MPILagrangianFieldCommunicator2D, MPILagrangianFieldCommunicator3D,
                                  check_valid_ghost_size_and_kernel_support, get_real_t, get_test_tol)
from sopht_mpi_b200.utils.comm import compute_slab_topology
from sopht_mpi_b200.utils.device import DeviceField

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def test_single_rank_construct():
    mc = MPIConstruct3D(8, 6, 10, real_t=np.float32)
    assert mc.size == 1 and mc.rank == 0
    assert tuple(mc.grid_topology) == (1, 1, 1)
    assert all(mc.physical_faces)
    assert tuple(mc.local_grid_size) == (8, 6, 10)
    mc2 = MPIConstruct2D(8, 6)
    assert tuple(mc2.grid_topology) == (1, 1)


def test_slab_topology_rules():
    assert tuple(compute_slab_topology(4, [0, 1, 1])) == (4, 1, 1)
    assert tuple(compute_slab_topology(2, [0, 0, 1])) == (2, 1, 1)
    assert tuple(compute_slab_topology(8, [0, 1])) == (8, 1)
    with pytest.raises(RuntimeError):
        compute_slab_topology(2, [1, 0, 1])


def test_invalid_decomposition_and_kernel_support():
    with pytest.raises(ValueError):
        check_valid_ghost_size_and_kernel_support(ghost_size=1, kernel_support=2)
    check_valid_ghost_size_and_kernel_support(ghost_size=2, kernel_support=2)
    assert get_real_t("single") is np.float32 and get_real_t("double") is np.float64
    assert get_test_tol("double") < get_test_tol("single")


def test_periodic_single_rank_halo():
    gs = 2
    mc = MPIConstruct3D(6, 5, 7, periodic_domain=True)
    comm = MPIGhostCommunicator3D(ghost_size=gs, mpi_construct=mc)
    rng = np.random.default_rng(0)
    glob = rng.uniform(size=(6, 5, 7))
    local = np.zeros((6 + 2 * gs, 5 + 2 * gs, 7 + 2 * gs))
    local[gs:-gs, gs:-gs, gs:-gs] = glob
    comm.exchange_scalar_field_init(local)
    comm.exchange_finalise()
    assert np.array_equal(local, np.pad(glob, gs, mode="wrap"))


def test_rank_ownership_against_reference_golden():
    """same integers as the reference's _compute_lag_nodes_rank_address on a (4,2,1)
    topology is out of slab scope; check the slab-compatible 2D case and a 3D slab case."""
    o = np.load(os.path.join(GOLDEN, "ownership.npz"))

    class FakeGrid:
        def __init__(self, topo):
            self.topo = topo
            self.coords = np.zeros(len(topo), dtype=int)

        def Get_cart_rank(self, c):
            return int(np.ravel_multi_index(tuple(c), self.topo))

        def bcast(self, x, root=0):
            return x

    class FakeConstruct:
        def __init__(self, topo, local):
            self.grid_dim = len(topo)
            self.grid_topology = np.array(topo)
            self.local_grid_size = np.array(local)
            self.grid = FakeGrid(tuple(topo))
            self.rank = 0
            self.size = int(np.prod(topo))

    for t in ("f64", "f32"):
        lc = MPILagrangianFieldCommunicator2D(o["dx"][()], o["shift"][()],
                                              FakeConstruct(o["topo2"], o["local2"]),
                                              real_t=o["pos2_" + t].dtype)
        assert np.array_equal(lc._compute_lag_nodes_rank_address(o["pos2_" + t]), o["addr2_" + t])
        lc3 = MPILagrangianFieldCommunicator3D(o["dx"][()], o["shift"][()],
                                               FakeConstruct(o["topo3"], o["local3"]),
                                               real_t=o["pos3_" + t].dtype)
        assert np.array_equal(lc3._compute_lag_nodes_rank_address(o["pos3_" + t]), o["addr3_" + t])


def test_lagrangian_node_outside_domain_aborts():
    mc = MPIConstruct3D(8, 8, 8)
    lc = MPILagrangianFieldCommunicator3D(np.float64(1 / 8), np.float64(1 / 16), mc)
    pos = np.array([[0.5], [0.5], [1.2]])
    with pytest.raises(RuntimeError):
        lc.map_lagrangian_nodes_based_on_position(pos)


def test_device_field_facade_on_cpu_tensor():
    import torch

    f = DeviceField(torch.zeros(3, 4, 5, dtype=torch.float64))
    v = f.view()
    f[0] = np.ones((4, 5))
    assert v.version == 1 and np.asarray(v)[0].sum() == 20
    f += 2.0
    assert np.amax(f[1]) == 2.0 and f.shape == (3, 4, 5) and f.dtype == np.float64
    assert np.allclose(np.asarray(f[0][1:3, 2:4]), 3.0)
    g = f.copy()
    g[...] = 0.0
    assert np.asarray(f).sum() > 0


def test_two_rank_gloo_halo_fields_and_ownership():
    run_ranks("dist_worker.py", 2, "DIST_WORKER_OK", where="cpu", timeout=600)


def test_row_block_magic_division_is_exact():
    """`SbRowBlocks` (csrc/poisson_fft.cu) divides the bin index by the kx-block length with
    umulhi(k, ceil(2^32 / kxl)) on the GPU (the emulation uses `/`): exact for every bin of every
    supported row length and block length."""
    k = np.arange(0, 4098, dtype=np.uint64)
    for kxl in range(1, 4100):
        magic = np.uint64((0x100000000 + kxl - 1) // kxl)
        assert np.array_equal((k * magic) >> np.uint64(32), k // np.uint64(kxl)), kxl


def test_slab_kx_block_length_rule():
    """kx bins per rank: ceil((nx + 1) / P) rounded up to a multiple of 4, P blocks cover every bin."""
    for nx in (16, 64, 256, 512, 1024, 4096):
        for nranks in (2, 4, 8):
            kxl = (((nx + 1 + nranks - 1) // nranks) + 3) & ~3
            assert kxl % 4 == 0 and kxl * nranks >= nx + 1 and (kxl - 4) * nranks < nx + 1 + 3 * nranks
