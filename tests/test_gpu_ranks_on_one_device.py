"""Peer-memory halo exchange / ghost sum (utils/peer.py:PeerHalo) with three PROCESSES on ONE GPU: real CUDA
IPC mappings, push kernels and epoch flags, so the single-GPU GPUTEST covers SURVEY rows H1 and L9 on the
transport the multi-GPU runs use (tests/test_gpu_multi.py needs >= 2 devices)."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _run_ranks_on_one_gpu(script, size, marker, extra_env=None):
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    procs = []
    for rank in range(size):
        # (ranks that time-share one device hand it to each other a time slice at a time: generous wait limit)
        env = dict(os.environ, RANK=str(rank), WORLD_SIZE=str(size), LOCAL_RANK="0", MASTER_ADDR="127.0.0.1",
                   SB200_PEER_WAIT_S="60",
                   MASTER_PORT=str(port), CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0])
        env.update(extra_env or {})
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", script)], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = []
    try:
        for p in procs:
            outs.append(p.communicate(timeout=900))
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
    text = "\n".join(o[0][-2000:] + o[1][-4000:] for o in outs)
    assert all(p.returncode == 0 for p in procs) and marker in outs[0][0], text


def test_peer_halo_and_ghost_sum_with_three_processes_on_one_gpu():
    _run_ranks_on_one_gpu("dist_halo_worker.py", 3, "DIST_HALO_WORKER_OK")


@pytest.mark.parametrize("size", [2, 4])
def test_slab_decomposition_with_all_ranks_on_one_gpu(size):
    """tests/dist_gpu_worker.py (slab Poisson solve over the peer-memory all-to-all, halo exchange + fused
    steps, IB ownership / forces / ghost sum against the single-domain oracle) with every rank on cuda:0"""
    # (ranks that share a device take the push-kernel transport; tests/test_gpu_multi.py runs the copy-engine
    # transport on 2 and 4 real GPUs)
    _run_ranks_on_one_gpu("dist_gpu_worker.py", size, "DIST_GPU_WORKER_OK", {"SB200_TEST_SINGLE_DEVICE": "1"})
