"""One case per kernel instantiation the launchers can select, each against a float64 reference of the same
input, and a guard that the emulation suite launches every compiled instantiation.

The launchers pick a kernel, or a template instantiation of one, from the shape and dtype of the input: the
x pass specialises n = 256 / 512 / 1024 and runs every other length through a generic kernel, the strided y
and z passes specialise 256..1024 (double) and 256..2048 (float), with 32 points per thread for float 512 /
1024 and a fused z pass (bulk-copy tiles) for float 2 nz = 512 / 1024; the fused vorticity update takes
version 2 for float rows of even length and version 1 for odd ones; the velocity kernel takes four cells per
thread when rows are a multiple of 4 cells and the pointers are aligned.  Skinny grids give the pass under
test the long axis and keep the others at 8-16 cells.

The CPU tier runs the cases through the host-thread emulation (tests/emu); the `-m gpu` tier runs the same
cases, plus the 4096-point transforms that are too slow to emulate, through the CUDA library on one device.
The last test of this module compares the emulation's launch log with the kernel instantiations compiled
into the emulation library."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from emu_util import emu
from oracle import stencils as st
from oracle.poisson import UnboundedPoissonSolverOracle2D, UnboundedPoissonSolverOracle3D
from sopht_mpi_b200 import _lib
from test_emu_kernels import _slab_solve_emulated

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "sopht_mpi_b200", "csrc")
f32, f64 = np.float32, np.float64


def _rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def _tol(real_t):
    return 1e-13 if real_t == f64 else 2e-6


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
        import torch

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
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return _Cuda()


def _case_id(v):
    if isinstance(v, type):
        return v.__name__.replace("float", "f")
    if isinstance(v, tuple):
        return "x".join(map(str, v))
    return None


# ------------------------------------------------------------------------------------------- Poisson
def _poisson_case(be, real_t, n, gs=2, x_range=1.0):
    """Single-rank solve of one random scalar field: interior against the float64 oracle of the same
    (real_t) input, ghost cells of the solution never written."""
    dim = len(n)
    rng = np.random.default_rng(sum(n) + gs)
    shape = tuple(v + 2 * gs for v in n)
    rhs = rng.uniform(size=shape).astype(real_t)
    sol = be.dev(np.full(shape, 7.0, real_t))
    h = ctypes.c_void_p()
    nzyx = n if dim == 3 else (1,) + n
    _call(be, "sb200_poisson_create", ctypes.byref(h), dim, _lib.dtype_code(real_t), *nzyx, gs, x_range, 0, 1, 1,
          None)
    try:
        d_rhs = be.dev(rhs)
        _call(be, "sb200_poisson_solve", h, be.ptr(sol), be.ptr(d_rhs), 1, None)
        got = be.host(sol)
    finally:
        be.lib.sb200_poisson_destroy(h)
    oracle = (UnboundedPoissonSolverOracle3D if dim == 3 else UnboundedPoissonSolverOracle2D)(
        *n, x_range=x_range, real_t=f64)
    ref = np.zeros(shape)
    oracle.solve(ref, rhs.astype(f64), gs)
    inner = (slice(gs, -gs),) * dim
    err = _rel(got[inner], ref[inner])
    assert err < _tol(real_t), err
    ghosts = np.ones(shape, bool)
    ghosts[inner] = False
    assert np.all(got[ghosts] == 7.0)
    return err


# (real_t, (nz, ny, nx), gs, x_range)
POISSON_3D = [
    # x pass: the generic kernel, LOG2N = 8 / 9 / 10, and the generic kernel above 1024
    (f64, (8, 8, 32), 2, 1.0), (f32, (8, 8, 64), 2, 1.8),
    (f64, (8, 8, 256), 2, 1.0), (f32, (8, 8, 256), 2, 1.0),
    (f64, (8, 8, 512), 2, 1.0), (f32, (8, 8, 512), 2, 1.0),
    (f64, (8, 8, 1024), 2, 1.0), (f32, (8, 8, 1024), 2, 1.0),
    (f64, (8, 8, 2048), 2, 1.0), (f32, (8, 8, 2048), 2, 1.0),
    # y pass, 2 ny = 256 / 512 / 1024 (float: 32 points per thread at 512 and 1024) / 2048 (float only)
    (f64, (8, 128, 16), 2, 1.0), (f32, (8, 128, 16), 2, 1.0),
    (f64, (8, 256, 16), 2, 1.0), (f32, (8, 256, 16), 2, 1.0),
    (f64, (8, 512, 16), 2, 1.0), (f32, (8, 512, 16), 2, 1.0),
    (f32, (8, 1024, 16), 2, 1.0),
    # z pass, 2 nz = 256 / 512 / 1024 (float: the fused bulk-copy z kernel) / 2048 (float only); float 256 and
    # 2048 read the thread-order Green's table
    (f64, (128, 8, 16), 2, 1.0), (f32, (128, 8, 16), 2, 1.0),
    (f64, (256, 8, 16), 2, 1.0), (f32, (256, 8, 16), 2, 1.0),
    (f64, (512, 8, 16), 2, 1.0), (f32, (512, 8, 16), 2, 1.0),
    (f32, (1024, 8, 16), 2, 1.0),
    # ghost size 3
    (f32, (16, 8, 32), 3, 1.0), (f64, (8, 16, 32), 3, 1.8),
]
# generic 4096-point lines: too slow for the emulation, and no instantiation of their own
POISSON_3D_4096 = [(t, n, 2, 1.0) for n in ((8, 8, 4096), (8, 2048, 16), (2048, 8, 16)) for t in (f64, f32)]

# (real_t, (ny, nx), gs, x_range): the 2D y pass multiplies by the Green's function without the thread-order
# table (float 2 ny = 256 / 2048 strided, 512 / 1024 32 points per thread)
POISSON_2D = [
    (f64, (256, 512), 2, 1.0),  # the 512 x 256 cylinder grid of BASELINE.json
    (f32, (128, 16), 2, 1.0), (f32, (256, 16), 2, 1.0), (f32, (512, 16), 2, 1.0), (f32, (1024, 16), 2, 1.0),
    (f32, (16, 32), 3, 1.8),
]


@pytest.mark.parametrize("real_t,n,gs,x_range", POISSON_3D, ids=_case_id)
def test_poisson_3d_against_float64(real_t, n, gs, x_range):
    _poisson_case(_Host(), real_t, n, gs, x_range)


@pytest.mark.parametrize("real_t,n,gs,x_range", POISSON_2D, ids=_case_id)
def test_poisson_2d_against_float64(real_t, n, gs, x_range):
    _poisson_case(_Host(), real_t, n, gs, x_range)


@pytest.mark.parametrize("real_t,n", [(f64, (256, 8, 16)), (f32, (1024, 8, 16))], ids=_case_id)
def test_slab_poisson_against_float64(real_t, n):
    """The z-slab entry points on two emulated ranks: f64 2 nz = 512, f32 2 nz = 2048 (thread-order table
    columns offset by the rank's first kx bin)."""
    gs, ncomp, nranks = 2, 1, 2
    rng = np.random.default_rng(4)
    rhs = rng.uniform(size=(ncomp,) + tuple(v + 2 * gs for v in n)).astype(real_t)
    out = _slab_solve_emulated(emu(), real_t, n, nranks, rhs, gs, ncomp)
    ref = np.zeros(rhs.shape[1:])
    UnboundedPoissonSolverOracle3D(*n, x_range=1.0, real_t=f64).solve(ref, rhs[0].astype(f64), gs)
    nzl = n[0] // nranks
    scale = np.abs(ref).max()
    for r in range(nranks):
        got = out[r][0, gs:-gs, gs:-gs, gs:-gs]
        want = ref[r * nzl + gs:r * nzl + gs + nzl, gs:-gs, gs:-gs]
        assert np.abs(got - want).max() / scale < _tol(real_t), r
        assert np.all(out[r][:, 0] == 7.0) and np.all(out[r][:, :, :, -1] == 7.0)


# -------------------------------------------------------------------------------- fused vorticity update
def _fused_reference(w, u, gs):
    """cross product -> curl update -> diffusion, the oracle's three sweeps in float64"""
    ref = w.astype(f64)
    buf = np.zeros_like(ref)
    st.elementwise_cross_product(buf, u.astype(f64), ref)
    st.update_vorticity_from_velocity_forcing_mpi(ref, buf, 0.3, gs)
    st.diffusion_timestep_mpi(ref, np.zeros(ref.shape[1:]), 0.05, gs)
    return ref


def _fused_case(be, real_t, n, gs):
    rng = np.random.default_rng(sum(n))
    shape = tuple(v + 2 * gs for v in n)
    g = _lib.make_grid(3, real_t, gs, n, (1,) * 6)
    w = rng.uniform(size=(3,) + shape).astype(real_t)
    u = (rng.uniform(size=(3,) + shape) - 0.5).astype(real_t)
    out, d_w, d_u = be.dev(np.full_like(w, np.nan)), be.dev(w), be.dev(u)
    _call(be, "sb200_vorticity_rhs_fused_3d", ctypes.byref(g), be.ptr(out), be.ptr(d_w), be.ptr(d_u), None, 0.3, 0.05,
          None)
    got = be.host(out)
    assert not np.isnan(got).any()
    err = _rel(got, _fused_reference(w, u, gs))
    assert err < _tol(real_t), err
    return err


# (real_t, (nz, ny, nx), gs): row length mx = nx + 2 gs; float takes version 2 for even mx, version 1 for odd
FUSED = [
    (f32, (9, 17, 65), 2), (f32, (8, 40, 71), 2),  # version 1, several tiles along x and y
    (f32, (8, 30, 64), 3), (f32, (8, 30, 65), 3), (f64, (8, 20, 40), 3),  # ghost size 3: v2, v1, double
]


@pytest.mark.parametrize("real_t,n,gs", FUSED, ids=_case_id)
def test_fused_vorticity_update_against_float64(real_t, n, gs):
    _fused_case(_Host(), real_t, n, gs)


@pytest.mark.parametrize("real_t,gs", [(f32, 2), (f32, 3), (f64, 3)], ids=["f32", "f32-gs3", "f64-gs3"])
def test_fused_vorticity_update_odd_rows_on_virtual_z_slabs(real_t, gs):
    """Odd row length: three virtual z-slabs with exchanged ghost planes give the whole-domain result."""
    rng = np.random.default_rng(6)
    nzl, ny, nx, ranks = 8, 10, 13, 3
    gshape = (ranks * nzl + 2 * gs, ny + 2 * gs, nx + 2 * gs)
    assert gshape[2] % 2 == 1
    w = rng.uniform(size=(3,) + gshape).astype(real_t)
    u = (rng.uniform(size=(3,) + gshape) - 0.5).astype(real_t)
    ref = _fused_reference(w, u, gs)
    for r in range(ranks):
        g = _lib.make_grid(3, real_t, gs, (nzl, ny, nx), (r == 0, r == ranks - 1, 1, 1, 1, 1))
        lo = r * nzl
        wl = np.ascontiguousarray(w[:, lo:lo + nzl + 2 * gs])
        ul = np.ascontiguousarray(u[:, lo:lo + nzl + 2 * gs])
        out = np.full_like(wl, np.nan)
        be = _Host()
        _call(be, "sb200_vorticity_rhs_fused_3d", ctypes.byref(g), be.ptr(out), be.ptr(wl), be.ptr(ul), None, 0.3,
              0.05, None)
        assert _rel(out[:, gs:-gs], ref[:, lo + gs:lo + gs + nzl]) < _tol(real_t), r


@pytest.mark.parametrize("gs", [2, 3])
def test_fused_vorticity_update_odd_rows_by_plane_ranges(gs):
    """Version 1 (float, odd rows): interior planes, then the planes next to the slab faces, equal the
    whole-grid call bit for bit."""
    rng = np.random.default_rng(7)
    n = (20, 10, 67)
    shape = tuple(v + 2 * gs for v in n)
    assert shape[2] % 2 == 1
    g = _lib.make_grid(3, f32, gs, n, (0, 0, 1, 1, 1, 1))
    w = rng.uniform(size=(3,) + shape).astype(f32)
    u = (rng.uniform(size=(3,) + shape) - 0.5).astype(f32)
    be = _Host()
    whole = np.full_like(w, np.nan)
    _call(be, "sb200_vorticity_rhs_fused_3d", ctypes.byref(g), be.ptr(whole), be.ptr(w), be.ptr(u), None, 0.3, 0.05,
          None)
    parts = np.full_like(w, np.nan)
    mz, k = shape[0], 2 * gs
    for z0, z1 in ((k, mz - k), (0, k), (mz - k, mz)):
        _call(be, "sb200_vorticity_rhs_fused_3d_range", ctypes.byref(g), be.ptr(parts), be.ptr(w), be.ptr(u), 0.3,
              0.05, z0, z1, None)
    assert not np.isnan(parts).any() and np.array_equal(parts, whole)


# ------------------------------------------------------------------------ velocity from stream function
def _velocity_case(be, real_t, n, gs, offset=0, phys=(1,) * 6):
    """curl of psi + free stream (ring zeroed, forcing reset, max |u|) against the float64 oracle; `offset`
    starts the velocity one element into a larger buffer, which must take the scalar kernel"""
    rng = np.random.default_rng(sum(n) + offset)
    shape = tuple(v + 2 * gs for v in n)
    g = _lib.make_grid(3, real_t, gs, n, phys)
    psi = rng.uniform(size=(3,) + shape).astype(real_t)
    u0 = rng.uniform(size=(3,) + shape).astype(real_t)
    ref = u0.astype(f64)
    st.curl_mpi(ref, psi.astype(f64), 0.8, gs, phys)
    fs = np.array([1.0, 0.5, -0.25])
    for c in range(3):
        ref[c] += fs[c]
    u = be.dev(u0, offset)
    forcing = be.dev(rng.uniform(size=(3,) + shape).astype(real_t))
    vmax, d_psi = be.dev(np.zeros(1)), be.dev(psi)
    _call(be, "sb200_velocity_from_stream_function", ctypes.byref(g), be.ptr(u), be.ptr(d_psi), 0.8,
          fs.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), be.ptr(forcing), be.ptr(vmax), None)
    got = be.host(u)
    err = _rel(got, ref)
    assert err < _tol(real_t), err
    assert np.abs(be.host(forcing)).max() == 0
    inner = (slice(None),) + (slice(gs, -gs),) * 3
    assert np.isclose(be.host(vmax)[0], np.abs(ref[inner]).sum(axis=0).max(), rtol=_tol(real_t))
    return err


# (real_t, (nz, ny, nx), gs, velocity offset): mx % 4 == 0 and aligned pointers take four cells per thread
VELOCITY = [
    (f32, (6, 9, 10), 3, 0), (f64, (6, 9, 10), 3, 0),  # mx = 16: four cells per thread
    (f32, (6, 9, 11), 3, 0), (f64, (6, 9, 11), 3, 0),  # mx = 17: scalar kernel
    (f32, (6, 9, 12), 2, 1), (f64, (6, 9, 12), 2, 1),  # mx = 16, velocity misaligned: scalar kernel
]


@pytest.mark.parametrize("real_t,n,gs,offset", VELOCITY, ids=_case_id)
def test_velocity_from_stream_function_against_float64(real_t, n, gs, offset):
    _velocity_case(_Host(), real_t, n, gs, offset)


@pytest.mark.parametrize("real_t", [f64, f32], ids=["f64", "f32"])
@pytest.mark.parametrize("phys", [(0, 0, 1, 1, 1, 1), (0, 1, 1, 1, 1, 1)], ids=["inner", "last"])
def test_vectorised_velocity_on_slab_faces_against_float64(real_t, phys):
    """Four cells per thread on z-slabs whose z faces are not physical: cells on those faces keep their
    old value."""
    _velocity_case(_Host(), real_t, (10, 7, 12), 2, 0, phys)


# ------------------------------------------------------------------------------- other ghost-size cases
@pytest.mark.parametrize("real_t,gs", [(f64, 2), (f64, 3), (f32, 3)], ids=["f64", "f64-gs3", "f32-gs3"])
@pytest.mark.parametrize("dim", [3, 2])
def test_sparse_forcing_update_and_flagged_reset_against_float64(real_t, gs, dim):
    """sb200_update_vorticity_from_sparse_forcing equals the plain update bit for bit and the float64 oracle
    within rounding; sb200_clear_flagged_tiles leaves F == 0 and the flags cleared."""
    from oracle import stencils_2d as st2

    rng = np.random.default_rng(13)
    n = (10, 37, 45) if dim == 3 else (150, 200)
    shape = tuple(v + 2 * gs for v in n)
    g = _lib.make_grid(dim, real_t, gs, n, [1] * (2 * dim))
    w = rng.uniform(size=((3,) + shape) if dim == 3 else shape).astype(real_t)
    f = rng.uniform(-1, 1, size=(dim,) + shape).astype(real_t)
    mask = np.zeros(shape, bool)
    mask[(slice(4, 9),) * dim] = True
    mask[(-1,) * dim] = True
    f *= mask
    be = _Host()
    plain, got = w.copy(), w.copy()
    _call(be, "sb200_update_vorticity_from_velocity_forcing", ctypes.byref(g), be.ptr(plain), be.ptr(f), 0.37, None)
    work = np.zeros(int(be.lib.sb200_tile_flag_count(ctypes.byref(g))), np.uint8)
    _call(be, "sb200_update_vorticity_from_sparse_forcing", ctypes.byref(g), be.ptr(got), be.ptr(f), 0.37,
          be.ptr(work), None)
    assert np.array_equal(got, plain)
    ref = w.astype(f64)
    (st if dim == 3 else st2).update_vorticity_from_velocity_forcing_mpi(ref, f.astype(f64), 0.37, gs)
    assert _rel(got, ref) < _tol(real_t)
    assert work.view(np.int32)[-4] > 0  # tiles were flagged
    _call(be, "sb200_clear_flagged_tiles", ctypes.byref(g), be.ptr(f), dim, be.ptr(work), None)
    assert not f.any() and not work.any()


@pytest.mark.parametrize("real_t", [f64, f32], ids=["f64", "f32"])
def test_one_pass_filter_and_penalisation_with_ghost_size_3(real_t):
    """The one-pass order-1 filter and the boundary penalisation at gs = 3: bit for bit against the oracle in
    the same precision, and within rounding of the float64 oracle."""
    from sopht_mpi_b200.numeric.eulerian_grid_ops.ops import _penalise_factor_table

    rng = np.random.default_rng(8)
    gs, n = 3, (12, 19, 40)
    shape = tuple(v + 2 * gs for v in n)
    g = _lib.make_grid(3, real_t, gs, n, [1] * 6)
    be = _Host()
    w = rng.uniform(size=(3,) + shape).astype(real_t)
    fb0, bb0 = rng.uniform(size=shape).astype(real_t), rng.uniform(size=shape).astype(real_t)
    same, ref = w.copy(), w.astype(f64)
    fb1, bb1 = fb0.copy(), bb0.copy()
    st.laplacian_filter_mpi(same, fb0.copy(), bb0.copy(), 1, "multiplicative", gs)
    st.laplacian_filter_mpi(ref, fb0.astype(f64), bb0.astype(f64), 1, "multiplicative", gs)
    out = np.full_like(w, np.nan)
    _call(be, "sb200_laplacian_filter_order1_out_of_place", ctypes.byref(g), be.ptr(out), be.ptr(w), 3, be.ptr(fb1),
          be.ptr(bb1), None)
    assert np.array_equal(out, same)
    assert _rel(out, ref) < _tol(real_t)

    width, dx = 2, real_t(1.0 / n[2])

    def line(nl, t):
        return np.linspace(dx / 2 - gs * dx, nl * dx - dx / 2 + gs * dx, nl + 2 * gs).astype(t)

    same, ref = w.copy(), w.astype(f64)
    st.penalise_field_boundary_mpi(same, width, dx, line(n[2], real_t), line(n[1], real_t), line(n[0], real_t), gs)
    st.penalise_field_boundary_mpi(ref, width, f64(dx), line(n[2], f64), line(n[1], f64), line(n[0], f64), gs)
    tab = _penalise_factor_table(real_t, width, dx, gs, [line(n[0], real_t), line(n[1], real_t), line(n[2], real_t)])
    got = w.copy()
    _call(be, "sb200_penalise_field_boundary", ctypes.byref(g), be.ptr(got), 3, width, be.ptr(tab), None)
    assert np.array_equal(got, same)
    assert _rel(got, ref) < _tol(real_t)


@pytest.mark.parametrize("real_t", [f64, f32], ids=["f64", "f32"])
@pytest.mark.parametrize("ncomp", [1, 2, 3])
def test_reductions_by_component_count(real_t, ncomp):
    """max |sum of components|, max and sum of squares for every component count (1 and 3 are compiled
    apart, 2 takes the run-time count) against float64 numpy."""
    rng = np.random.default_rng(ncomp)
    gs, n = 2, (7, 9, 11)
    g = _lib.make_grid(3, real_t, gs, n, (1,) * 6)
    f = (rng.uniform(size=(ncomp,) + tuple(v + 2 * gs for v in n)) - 0.5).astype(real_t)
    inner = f[(slice(None),) + (slice(gs, -gs),) * 3].astype(f64)
    out, be = np.zeros(1), _Host()
    _call(be, "sb200_max_abs_sum", ctypes.byref(g), be.ptr(f), ncomp, be.ptr(out), None)
    assert np.isclose(out[0], np.abs(inner).sum(axis=0).max(), rtol=_tol(real_t))
    _call(be, "sb200_max", ctypes.byref(g), be.ptr(f), ncomp, be.ptr(out), None)
    assert out[0] == inner.max()
    _call(be, "sb200_sum_squares", ctypes.byref(g), be.ptr(f), ncomp, be.ptr(out), None)
    assert np.isclose(out[0], (inner ** 2).sum(), rtol=1e-12)


@pytest.mark.parametrize("real_t", [f64, f32], ids=["f64", "f32"])
def test_elementwise_and_slab_face_operators(real_t):
    """fill, add-fixed-value, cross product, filter flux along one axis, the ghost-plane sum of spreading
    across z-slab faces and the position-mismatch update, against float64 numpy."""
    rng = np.random.default_rng(10)
    gs, n = 2, (6, 7, 9)
    shape = tuple(v + 2 * gs for v in n)
    cells = int(np.prod(shape))
    code, be = _lib.dtype_code(real_t), _Host()
    a = rng.uniform(size=(3,) + shape).astype(real_t)
    b = rng.uniform(size=(3,) + shape).astype(real_t)
    got = a.copy()
    _call(be, "sb200_set_fixed_val", code, be.ptr(got), got.size, 0.75, None)
    assert np.all(got == real_t(0.75))
    got = a.copy()
    vals = np.array([0.5, -1.25, 2.0])
    _call(be, "sb200_add_fixed_val", code, be.ptr(got), 3, cells, vals.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
          None)
    assert _rel(got, a.astype(f64) + vals[:, None, None, None]) < _tol(real_t)
    _call(be, "sb200_elementwise_cross_product", code, be.ptr(got), be.ptr(a), be.ptr(b), cells, None)
    assert _rel(got, np.cross(a.astype(f64), b.astype(f64), axis=0)) < _tol(real_t)

    g = _lib.make_grid(3, real_t, gs, n, (1,) * 6)
    for axis in range(3):
        flux = b[0].copy()
        ref = b[0].astype(f64)
        st._laplacian_filter_axis_mpi(axis, a[0].astype(f64), ref, gs)  # the wrapper's regions, then its ring clear
        st.clear_physical_ring(ref, gs)
        _call(be, "sb200_laplacian_filter_axis", ctypes.byref(g), be.ptr(flux), be.ptr(a[0]), 2 - axis, None)
        assert _rel(flux, ref) < _tol(real_t), axis

    plane = shape[1] * shape[2]
    prev = rng.uniform(size=(3, gs * plane)).astype(real_t)
    nxt = rng.uniform(size=(3, gs * plane)).astype(real_t)
    got = a.copy()
    _call(be, "sb200_ghost_sum_add_z", ctypes.byref(g), be.ptr(got), 3, be.ptr(prev), be.ptr(nxt), None)
    ref = a.astype(f64)
    ref[:, gs:2 * gs] += prev.reshape(3, gs, *shape[1:])
    ref[:, -2 * gs:-gs] += nxt.reshape(3, gs, *shape[1:])
    assert _rel(got, ref) < _tol(real_t)

    dpos, dvel = a[0, 0].copy(), b[0, 0]
    _call(be, "sb200_ib_update_position_mismatch", code, be.ptr(dpos), be.ptr(dvel), dvel.size, 0.125, None)
    assert _rel(dpos, a[0, 0].astype(f64) + 0.125 * dvel) < _tol(real_t)


def test_ib_kernels_with_float_lagrangian_on_a_double_grid():
    """Lagrangian arrays in float, Eulerian grid in double: the same interpolation, forcing and spreading as
    the all-double kernels fed the same (float-representable) values, to float rounding."""
    rng = np.random.default_rng(15)
    dim, gs, width, n_local, n = 3, 2, 2, 12, 40
    dx, shift = 1.0 / n_local, 0.5 / n_local
    g = _lib.make_grid(dim, f64, gs, (n_local,) * dim, [1] * 6)
    eul = rng.uniform(size=(dim,) + (n_local + 2 * gs,) * dim)
    pos = (0.2 + 0.6 * rng.uniform(size=(dim, n))).astype(f32)
    vel, dpos = rng.uniform(size=(dim, n)).astype(f32), rng.uniform(size=(dim, n)).astype(f32)
    be, out = _Host(), {}
    for lag_t in (f64, f32):
        p = _lib.IBParams()
        p.lag_dtype, p.kernel_type, p.width = _lib.dtype_code(lag_t), 0, width
        p.dx, p.coord_shift, p.stiffness, p.damping = dx, shift, -2.0, -0.3
        x, v, dp = (a.astype(lag_t) for a in (pos, vel, dpos))
        u, dv, f = (np.zeros((dim, n), lag_t) for _ in range(3))
        _call(be, "sb200_ib_interact_lag", ctypes.byref(g), ctypes.byref(p), n, be.ptr(eul), be.ptr(x), be.ptr(v),
              be.ptr(dp), None, None, be.ptr(u), be.ptr(dv), be.ptr(f), None)
        spread = np.zeros_like(eul)
        fs = f.astype(f32).astype(lag_t)  # the same forcing values in both runs
        _call(be, "sb200_ib_spread", ctypes.byref(g), ctypes.byref(p), n, be.ptr(spread), be.ptr(fs), be.ptr(x), None)
        out[lag_t] = (u, f, spread)
    for got, want in zip(out[f32], out[f64]):
        assert _rel(got, want) < 2e-6


# ------------------------------------------------------------------------------ the same cases on a GPU
@pytest.mark.gpu
@pytest.mark.parametrize("real_t,n,gs,x_range", POISSON_3D + POISSON_3D_4096 + POISSON_2D, ids=_case_id)
def test_poisson_on_gpu_against_float64(cuda, real_t, n, gs, x_range, record_property):
    record_property("rel_linf", _poisson_case(cuda, real_t, n, gs, x_range))


@pytest.mark.gpu
@pytest.mark.parametrize("real_t,n,gs", FUSED, ids=_case_id)
def test_fused_vorticity_update_on_gpu_against_float64(cuda, real_t, n, gs, record_property):
    record_property("rel_linf", _fused_case(cuda, real_t, n, gs))


@pytest.mark.gpu
@pytest.mark.parametrize("real_t,n,gs,offset", VELOCITY, ids=_case_id)
def test_velocity_on_gpu_against_float64(cuda, real_t, n, gs, offset, record_property):
    record_property("rel_linf", _velocity_case(cuda, real_t, n, gs, offset))


# ------------------------------------------------------------------------------------ coverage guard
EMULATION_MODULES = ("test_emu_kernels.py", "test_emu_launch_coverage.py")

# compiled instantiations that no emulation test launches, and why
NOT_EMULATED = {
    "sb_push_blocks_kernel": "writes halo planes into another process's buffers through CUDA IPC mappings "
                             "(test_gpu_multi.py, test_gpu_ranks_on_one_device.py)",
    "sb_wait_flags_kernel": "spins on flags another process's push kernel sets (test_gpu_multi.py, "
                            "test_gpu_ranks_on_one_device.py)",
    "sb_flat_kernel<GreensFillOp": "the Green's function of the cuFFT backend, which has no emulation "
                                   "(test_gpu_parity_full.py::test_fft_backend_against_cufft_backend)",
}


def _global_kernel_names():
    """base names of the functions declared __global__ in the CUDA sources"""
    names = set()
    for f in sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".h"))):
        text = open(os.path.join(CSRC, f)).read()
        for m in re.finditer(r"__global__\s+void\s+", text):
            rest = text[m.end():]
            if rest.startswith("__launch_bounds__"):  # skip its balanced parentheses
                depth, i = 0, len("__launch_bounds__")
                while True:
                    depth += {"(": 1, ")": -1}.get(rest[i], 0)
                    i += 1
                    if depth == 0:
                        break
                rest = rest[i:]
            names.add(re.match(r"\s*(\w+)", rest).group(1))
    return names


def _kernel_instantiations(lib_path):
    """address -> demangled name of every defined function of the library whose base name is a kernel's, and
    the address of the launch-log export (to place the table at the library's load base)"""
    kernels = _global_kernel_names()
    out = subprocess.run(["nm", "-C", "--defined-only", lib_path], capture_output=True, text=True, check=True).stdout
    table, anchor = {}, None
    for line in out.splitlines():
        parts = line.split(None, 2)
        if len(parts) != 3 or parts[1] not in "TtWw":
            continue
        addr, name = int(parts[0], 16), parts[2]
        if name == "sb200_emu_launched_kernels":
            anchor = addr
        m = re.match(r"(?:void )?(\w+)(?:<.*>)?\(.*\)$", name)
        if m and m.group(1) in kernels:
            table[addr] = name
    return table, anchor


def test_every_compiled_kernel_instantiation_is_launched(request):
    """Every kernel instantiation in the emulation library has run in this session, except those listed in
    NOT_EMULATED.  Runs last among the emulation tests, and only when the session holds all of them."""
    from pathlib import Path

    wanted = set()
    for name in EMULATION_MODULES:
        mod = pytest.Module.from_parent(request.session, path=Path(HERE, name))
        wanted |= {it.nodeid for it in mod.collect() if not it.get_closest_marker("gpu")}
    missing = wanted - {it.nodeid for it in request.session.items}
    if missing:
        pytest.skip(f"the launch log is complete only when every emulation test runs ({len(missing)} not selected)")
    lib = emu()
    table, anchor = _kernel_instantiations(lib._name)
    base = ctypes.cast(lib.sb200_emu_launched_kernels, ctypes.c_void_p).value - anchor
    count = lib.sb200_emu_launched_kernels(None, 0)
    addrs = (ctypes.c_void_p * count)()
    lib.sb200_emu_launched_kernels(addrs, count)
    launched = {table.get(a - base, hex(a)) for a in addrs}
    assert launched <= set(table.values())  # every launched address names a kernel of the table
    never = sorted(name for name in set(table.values()) - launched
                   if not any(re.match(r"(?:void )?" + re.escape(k) + r"\b", name) for k in NOT_EMULATED))
    assert not never, "compiled kernel instantiations no emulation test launches:\n" + "\n".join(never)
