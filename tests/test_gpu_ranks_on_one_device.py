"""Peer-memory halo exchange / ghost sum (utils/peer.py:PeerHalo) with three PROCESSES on ONE GPU: real CUDA
IPC mappings, push kernels and epoch flags, so the single-GPU GPUTEST covers SURVEY rows H1 and L9 on the
transport the multi-GPU runs use (tests/test_gpu_multi.py needs >= 2 devices)."""
import pytest

from harness import run_ranks

pytestmark = pytest.mark.gpu


def test_peer_halo_and_ghost_sum_with_three_processes_on_one_gpu():
    run_ranks("dist_halo_worker.py", 3, "DIST_HALO_WORKER_OK", where="one_gpu")


@pytest.mark.parametrize("size", [2, 4])
def test_slab_decomposition_with_all_ranks_on_one_gpu(size):
    """tests/dist_gpu_worker.py (slab Poisson solve over the peer-memory all-to-all, halo exchange + fused
    steps, IB ownership / forces / ghost sum against the single-domain oracle) with every rank on cuda:0"""
    # (ranks that share a device take the push-kernel transport; tests/test_gpu_multi.py runs the copy-engine
    # transport on 2 and 4 real GPUs)
    run_ranks("dist_gpu_worker.py", size, "DIST_GPU_WORKER_OK", where="one_gpu")
