"""What several test modules and the multi-rank workers share.

* Buffer backends: the C ABI on numpy arrays through the host-thread emulation of the kernels (tests/emu),
  or on torch tensors through the CUDA library, so that one test case runs on either.
* The z-slab Poisson solve of P virtual ranks in one process, the test doing both all-to-alls.
* Ranks as processes: `run_ranks` starts them, and a worker joins and leaves the process group with
  `join_ranks` / `leave_ranks`."""
import ctypes
import gc
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import stencils as st  # noqa: E402
from sopht_mpi_b200 import _lib  # noqa: E402

f32, f64 = np.float32, np.float64
_emu = None


# ------------------------------------------------------------------------------------ buffer backends
def emu():
    """the host-thread emulation library, built on first use"""
    global _emu
    if _emu is None:
        sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
        import build_emu

        _emu = _lib.bind(build_emu.build())
    return _emu


class _Host:
    """Buffers of the emulation: numpy arrays on the host."""

    lib = property(lambda self: emu())

    def dev(self, a, offset=0):
        """a copy of `a` that starts `offset` elements after a 256-byte boundary (numpy itself only promises
        16 bytes, less than the 32 the double vector kernels need)"""
        buf = np.empty(a.nbytes + offset * a.itemsize + 256, np.uint8)
        start = -buf.ctypes.data % 256 + offset * a.itemsize
        out = buf[start:start + a.nbytes].view(a.dtype).reshape(a.shape)
        out[...] = a
        return out

    def ptr(self, a):
        return None if a is None else ctypes.c_void_p(a.ctypes.data)

    def host(self, a):
        return np.array(a)


class _Cuda:
    """Buffers of the CUDA library: torch tensors on cuda:0."""

    def __init__(self):
        self.torch = torch
        self.lib = _lib.load()

    def dev(self, a, offset=0):
        t = self.torch
        buf = t.empty(a.size + offset, dtype=t.float64 if a.dtype == f64 else t.float32 if a.dtype == f32 else
                      t.uint8, device="cuda")
        out = buf[offset:].view(a.shape)
        out.copy_(t.from_numpy(np.ascontiguousarray(a)))
        return out

    def ptr(self, a):
        return None if a is None else ctypes.c_void_p(a.data_ptr())

    def host(self, a):
        self.torch.cuda.synchronize()
        return a.cpu().numpy()


def _call(be, name, *args):
    _lib.check(be.lib, getattr(be.lib, name)(*args))


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return _Cuda()


def _free():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _fused_reference(w, u, gs):
    """cross product -> curl update -> diffusion, the oracle's three sweeps in float64"""
    ref = w.astype(f64)
    buf = np.zeros_like(ref)
    st.elementwise_cross_product(buf, u.astype(f64), ref)
    st.update_vorticity_from_velocity_forcing_mpi(ref, buf, 0.3, gs)
    st.diffusion_timestep_mpi(ref, np.zeros(ref.shape[1:]), 0.05, gs)
    return ref


# ------------------------------------------------------------------------- the benchmark's body
def _ib_setup(name):
    """bench.py's body on its grid: the product keeps the Lagrangian arrays in the dtype of the points
    (float64 here) on the float32 grid, with dx and the coordinate shift rounded to the grid's real_t"""
    import bench

    w = bench.workload_setup(name, bench.WORKLOADS[name][0])
    real_t, pts = w["real_t"], w["points"]
    assert real_t == f32 and pts.dtype == f64
    dx = real_t(w["dx"])
    shift = real_t(dx / 2)
    p = _lib.IBParams()
    p.lag_dtype, p.kernel_type, p.width = _lib.F64, 0, 2
    p.dx, p.coord_shift = float(dx), float(shift)
    area = w["dx"] ** 2  # the interactor's max_lag_grid_dx ** 2
    p.stiffness, p.damping = w["k"] * area, w["c"] * area
    g = _lib.make_grid(3, real_t, 2, w["grid"], (1,) * 6)  # the simulator's ghost size
    return w, g, p


def _spread(be, g, p, forcing_lag, pos, shape):
    """the product's spreading on one rank: scatter, then the ghost sum (which only clears the ghosts)"""
    eul = torch.zeros(shape, dtype=torch.float32, device="cuda")
    n = pos.shape[1]
    _call(be, "sb200_ib_spread_owned", ctypes.byref(g), ctypes.byref(p), n, be.ptr(eul), be.ptr(forcing_lag),
          be.ptr(pos), None, 0, None)
    _call(be, "sb200_clear_ghost_cells", ctypes.byref(g), be.ptr(eul), 3, None)
    return eul


# ------------------------------------------------------------------------------ virtual z-slab ranks
def slabs(glob, nranks, gs):
    """each rank's slab of a padded (..., z, y, x) field (numpy or torch), as a contiguous copy: its nzl
    interior planes and gs ghost planes on either side, filled from the neighbours (what the halo exchange
    leaves there)"""
    nzl = (glob.shape[-3] - 2 * gs) // nranks
    cut = [glob[..., r * nzl:r * nzl + nzl + 2 * gs, :, :] for r in range(nranks)]
    return [np.ascontiguousarray(s) if isinstance(s, np.ndarray) else s.contiguous() for s in cut]


def slab_poisson_solve(be, n, real_t, nranks, rhs, ncomp, *, backend, x_range=1.0, per_component=False):
    """The z-slab solve of `nranks` handles of `backend` in this process, on the padded global `rhs`
    ((ncomp,) z, y, x: numpy arrays on _Host, torch tensors on _Cuda).  Every rank runs the forward,
    spectral and backward slab stages on its own slab; the two all-to-alls are block copies, block q of
    rank r -> block r of rank q (NCCL's all_to_all_single with equal splits).
    per_component: one call of each stage per component with ncomp = 1 at the component's offset, as
    numeric/eulerian_grid_ops/poisson.py calls them, into exchange buffers of that call's size that are
    dropped afterwards; otherwise one call of each stage with `ncomp`.  Returns each rank's padded slab of
    the solution, pre-filled with 7.0 so that callers can check that no ghost cell was written."""
    xp = np if isinstance(rhs, np.ndarray) else torch
    gs = (rhs.shape[-1] - n[2]) // 2
    locs = slabs(rhs, nranks, gs)
    outs = [xp.full_like(loc, 7.0) for loc in locs]

    def all_to_all(dst, src):
        for r in range(nranks):
            for q in range(nranks):
                dst[q].reshape(nranks, -1)[r][...] = src[r].reshape(nranks, -1)[q]

    handles = []
    try:
        for r in range(nranks):
            h = ctypes.c_void_p()
            _call(be, "sb200_poisson_create", ctypes.byref(h), 3, _lib.dtype_code(real_t), *n, gs, x_range, r, nranks,
                  backend, None)
            handles.append(h)
        for c, k in [(c, 1) for c in range(ncomp)] if per_component else [(0, ncomp)]:
            nel = int(be.lib.sb200_poisson_slab_buffer_bytes(handles[0], k)) // rhs.itemsize
            assert nel % nranks == 0
            send = [xp.zeros(nel, dtype=rhs.dtype, device=rhs.device) for _ in range(nranks)]
            recv = [xp.zeros(nel, dtype=rhs.dtype, device=rhs.device) for _ in range(nranks)]
            for r in range(nranks):
                _call(be, "sb200_poisson_slab_forward", handles[r], be.ptr(locs[r].reshape(ncomp, -1)[c]), k,
                      be.ptr(send[r]), None)
            all_to_all(recv, send)
            for r in range(nranks):
                _call(be, "sb200_poisson_slab_spectral", handles[r], be.ptr(recv[r]), k, None)
            all_to_all(send, recv)
            for r in range(nranks):
                _call(be, "sb200_poisson_slab_backward", handles[r], be.ptr(outs[r].reshape(ncomp, -1)[c]), k,
                      be.ptr(send[r]), None)
            if xp is torch:
                torch.cuda.synchronize()
            del send, recv
    finally:
        for h in handles:
            be.lib.sb200_poisson_destroy(h)
    return outs


# ------------------------------------------------------------------------------- ranks as processes
def run_ranks(script, size, marker, *, where, env=None, timeout=900):
    """Run tests/<script> as `size` ranks; every process must return 0 and rank 0 must print `marker`.

    where="one_gpu": `size` processes on the first visible GPU with SB200_TEST_SINGLE_DEVICE=1 (see
    join_ranks); "gpus": torch.distributed.run, one process per GPU; "cpu": torch.distributed.run with no
    GPU visible.  `env` is added to the environment of every rank."""
    if where == "one_gpu" and not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    if where == "gpus" and (not torch.cuda.is_available() or torch.cuda.device_count() < size):
        pytest.skip(f"needs {size} GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = str(s.getsockname()[1])
    s.close()
    path = os.path.join(ROOT, "tests", script)
    base = dict(os.environ)
    if where == "one_gpu":
        # (ranks that time-share one device hand it to each other a time slice at a time: generous wait limit)
        base.update(SB200_TEST_SINGLE_DEVICE="1", SB200_PEER_WAIT_S="60")
    elif where == "cpu":
        base.update(CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS="1")
    base.update(env or {})
    if where == "one_gpu":
        first_gpu = os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]
        runs = [([sys.executable, path], dict(base, RANK=str(rank), WORLD_SIZE=str(size), LOCAL_RANK="0",
                                              MASTER_ADDR="127.0.0.1", MASTER_PORT=port,
                                              CUDA_VISIBLE_DEVICES=first_gpu)) for rank in range(size)]
    else:
        runs = [([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={size}",
                  "--master-addr", "127.0.0.1", "--master-port", port, path], base)]
    procs = [subprocess.Popen(cmd, env=e, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
             for cmd, e in runs]
    outs = []
    try:
        for p in procs:
            outs.append(p.communicate(timeout=timeout))
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
                p.wait()
    text = "\n".join(o[0][-3000:] + o[1][-5000:] for o in outs)
    assert all(p.returncode == 0 for p in procs) and marker in outs[0][0], text


def join_ranks():
    """Join the process group of a rank started by run_ranks.  Ranks that share one device
    (SB200_TEST_SINGLE_DEVICE) take gloo for the collectives, because NCCL cannot run several ranks on one
    device; their peer-memory exchanges are the same CUDA IPC transports as on several GPUs.  Otherwise
    the product's own start-up: NCCL with one GPU per rank, gloo on a machine without GPUs."""
    if os.environ.get("SB200_TEST_SINGLE_DEVICE"):
        torch.cuda.set_device(0)
        dist.init_process_group(backend="gloo")
    else:
        from sopht_mpi_b200.utils.comm import init_process_group_if_needed

        init_process_group_if_needed()


def leave_ranks(marker, *closables):
    """Close `closables` (solvers, peer halos; None is skipped) and release the CUDA IPC mappings of the
    other ranks' buffers before any rank exits, then print `marker` on rank 0 and leave the group."""
    for c in closables:
        if c is not None:
            c.close()
    gc.collect()
    if torch.cuda.is_initialized():
        torch.cuda.ipc_collect()
    dist.barrier()
    if dist.get_rank() == 0:
        print(marker)
    dist.destroy_process_group()
