"""Multi-GPU parity (z-slabs over NCCL): needs >= 2 visible GPUs (gpurun --gpus 2)."""
import pytest

from harness import run_ranks

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("nproc", [2, 4, 8])
def test_slab_decomposition_against_single_domain_oracle(nproc):
    run_ranks("dist_gpu_worker.py", nproc, "DIST_GPU_WORKER_OK", where="gpus")
