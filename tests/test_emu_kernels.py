"""Kernel LOGIC check in the GPU-less container: the CUDA sources compiled with
-DSB200_EMU (host-thread emulation, tests/emu) against the oracle.  This exercises
the same device code the GPU runs (write masks, ring zeroing, penalise gather,
warp-per-point IB kernels); the real parity tests are the `-m gpu` ones."""
import ctypes
import glob
import os

import numpy as np
import pytest

from harness import _call, _Host, emu, slab_poisson_solve
from ib_helpers import rank_address
from oracle import stencils as st
from sopht_mpi_b200 import _lib

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
_HOST = _Host()
ptr = _HOST.ptr


def call(fn_name, *args):
    _call(_HOST, fn_name, *args)


def _rel(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _tol(real_t):
    return 1e-13 if real_t == np.float64 else 2e-6


@pytest.fixture(params=[np.float64, np.float32], ids=["f64", "f32"])
def setup3d(request):
    real_t = request.param
    rng = np.random.default_rng(0)
    n, gs = (9, 11, 13), 2
    shape = tuple(v + 2 * gs for v in n)
    g = _lib.make_grid(3, real_t, gs, n, [1] * 6)
    return real_t, rng, n, gs, shape, g


def test_update_vorticity_and_curl(setup3d):
    real_t, rng, n, gs, shape, g = setup3d
    w = rng.uniform(size=(3,) + shape).astype(real_t)
    f = rng.uniform(size=(3,) + shape).astype(real_t)
    w0, w1 = w.copy(), w.copy()
    st.update_vorticity_from_velocity_forcing_mpi(w0, f, 0.37, gs)
    call("sb200_update_vorticity_from_velocity_forcing", ctypes.byref(g), ptr(w1), ptr(f), 0.37, None)
    assert _rel(w1, w0) < _tol(real_t)
    c0 = rng.uniform(size=(3,) + shape).astype(real_t)
    c1 = c0.copy()
    st.curl_mpi(c0, f, 0.8, gs)
    call("sb200_curl", ctypes.byref(g), ptr(c1), ptr(f), 0.8, None)
    assert _rel(c1, c0) < _tol(real_t)


def test_partial_physical_faces_match_virtual_rank_semantics(setup3d):
    """z faces NOT physical (inner slab of a z-slab decomposition): no z ring, no z penalty."""
    real_t, rng, n, gs, shape, _ = setup3d
    phys = (False, False, True, True, True, True)
    g = _lib.make_grid(3, real_t, gs, n, phys)
    f = rng.uniform(size=shape).astype(real_t)
    fl0 = rng.uniform(size=shape).astype(real_t)
    fl1 = fl0.copy()
    st.diffusion_flux_mpi(fl0, f, 0.1, gs, phys)
    call("sb200_diffusion_flux", ctypes.byref(g), ptr(fl1), ptr(f), 0.1, None)
    assert _rel(fl1, fl0) < _tol(real_t)


def test_diffusion_advection_divergence(setup3d):
    real_t, rng, n, gs, shape, g = setup3d
    w = rng.uniform(size=(3,) + shape).astype(real_t)
    vel = (rng.uniform(size=(3,) + shape) - 0.5).astype(real_t)
    a0, a1 = w.copy(), w.copy()
    b0 = rng.uniform(size=shape).astype(real_t)
    b1 = b0.copy()
    st.diffusion_timestep_mpi(a0, b0, 0.1, gs)
    call("sb200_diffusion_timestep", ctypes.byref(g), ptr(a1), 3, ptr(b1), 0.1, None)
    assert _rel(a1, a0) < _tol(real_t) and _rel(b1, b0) < _tol(real_t)
    a0, a1 = w.copy(), w.copy()
    b0 = np.ones(shape, real_t)
    b1 = b0.copy()
    st.advection_timestep_mpi(a0, b0, vel, 0.2, gs)
    call("sb200_advection_timestep_eno3", ctypes.byref(g), ptr(a1), 3, ptr(b1), ptr(vel), 0.2, None)
    assert _rel(a1, a0) < _tol(real_t) and _rel(b1, b0) < 10 * _tol(real_t)
    d0 = rng.uniform(size=shape).astype(real_t)
    d1 = d0.copy()
    st.divergence_mpi(d0, w, 3.0, gs)
    call("sb200_divergence", ctypes.byref(g), ptr(d1), ptr(w), 3.0, None)
    assert _rel(d1, d0) < _tol(real_t)


@pytest.mark.parametrize("order", [0, 1, 2, 3])
@pytest.mark.parametrize("phys", [(1,) * 6, (0, 0, 1, 1, 1, 1), (1, 0, 1, 1, 1, 1)], ids=["single", "inner", "first"])
@pytest.mark.parametrize("ftype,fname", [(0, "multiplicative"), (1, "convolution")])
def test_laplacian_filter(setup3d, ftype, fname, phys, order):
    """The out-of-place stage chain against the reference sequence (filter, ring clear, buffer copy per
    stage), including the stale flux values that survive in never-written ghost cells of inner slabs."""
    real_t, rng, n, gs, shape, _ = setup3d
    g = _lib.make_grid(3, real_t, gs, n, phys)
    w = rng.uniform(size=(3,) + shape).astype(real_t)
    a0, a1 = w.copy(), w.copy()
    fb0 = rng.uniform(size=shape).astype(real_t)
    fb1 = fb0.copy()
    bb0, bb1 = np.zeros(shape, real_t), np.zeros(shape, real_t)
    st.laplacian_filter_mpi(a0, fb0, bb0, order, fname, gs, phys)
    call("sb200_laplacian_filter", ctypes.byref(g), ptr(a1), 3, order, ftype, ptr(fb1), ptr(bb1), None)
    assert _rel(a1, a0) < _tol(real_t) and _rel(fb1, fb0) < _tol(real_t)


def test_penalise_is_bit_exact(setup3d):
    from sopht_mpi_b200.numeric.eulerian_grid_ops.ops import _penalise_factor_table

    real_t, rng, n, gs, shape, g = setup3d
    width = 2
    dx = real_t(1.0 / n[2])

    def line(nl):
        return np.linspace(dx / 2 - gs * dx, nl * dx - dx / 2 + gs * dx, nl + 2 * gs).astype(real_t)

    xg, yg, zg = line(n[2]), line(n[1]), line(n[0])
    w = rng.uniform(size=(3,) + shape).astype(real_t)
    a0, a1 = w.copy(), w.copy()
    st.penalise_field_boundary_mpi(a0, width, dx, xg, yg, zg, gs)
    tab = _penalise_factor_table(real_t, width, dx, gs, [zg, yg, xg])
    call("sb200_penalise_field_boundary", ctypes.byref(g), ptr(a1), 3, width, ptr(tab), None)
    assert np.array_equal(a1, a0)


def test_reductions_and_fused_velocity(setup3d):
    real_t, rng, n, gs, shape, g = setup3d
    vel = (rng.uniform(size=(3,) + shape) - 0.5).astype(real_t)
    inner = (slice(None),) + (slice(gs, -gs),) * 3
    out = np.zeros(1, np.float64)
    call("sb200_max_abs_sum", ctypes.byref(g), ptr(vel), 3, ptr(out), None)
    assert np.isclose(out[0], np.abs(vel[inner]).sum(axis=0).max(), rtol=1e-6)
    call("sb200_max", ctypes.byref(g), ptr(vel), 3, ptr(out), None)
    assert out[0] == vel[inner].max()
    call("sb200_sum_squares", ctypes.byref(g), ptr(vel), 3, ptr(out), None)
    assert np.isclose(out[0], (vel[inner].astype(np.float64) ** 2).sum(), rtol=1e-12)
    psi = rng.uniform(size=(3,) + shape).astype(real_t)
    u0 = rng.uniform(size=(3,) + shape).astype(real_t)
    u1 = u0.copy()
    st.curl_mpi(u0, psi, 0.8, gs)
    fs = np.array([1.0, 0.5, -0.25])
    for c in range(3):
        u0[c] += real_t(fs[c])
    forcing = rng.uniform(size=(3,) + shape).astype(real_t)
    call("sb200_velocity_from_stream_function", ctypes.byref(g), ptr(u1), ptr(psi), 0.8,
         fs.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), ptr(forcing), ptr(out), None)
    assert _rel(u1, u0) < _tol(real_t)
    assert np.abs(forcing).max() == 0
    assert np.isclose(out[0], np.abs(u0[inner]).sum(axis=0).max(), rtol=1e-6)


@pytest.mark.parametrize("real_t", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("phys", [(1,) * 6, (0, 0, 1, 1, 1, 1), (0, 1, 1, 1, 1, 1)], ids=["single", "inner", "last"])
def test_vectorised_velocity_kernel(real_t, phys):
    """Rows of a multiple of 4 cells take the 4-cells-per-thread kernel: same curl / ring / free stream /
    forcing reset / max as the composed oracle, including cells that keep their old value on slab faces."""
    rng = np.random.default_rng(9)
    n, gs = (10, 7, 12), 2
    shape = tuple(v + 2 * gs for v in n)
    assert shape[2] % 4 == 0
    g = _lib.make_grid(3, real_t, gs, n, phys)
    psi = rng.uniform(size=(3,) + shape).astype(real_t)
    u0 = rng.uniform(size=(3,) + shape).astype(real_t)
    u1 = u0.copy()
    st.curl_mpi(u0, psi, 0.8, gs, phys)
    fs = np.array([1.0, 0.5, -0.25])
    for c in range(3):
        u0[c] += real_t(fs[c])
    forcing = rng.uniform(size=(3,) + shape).astype(real_t)
    out = np.zeros(1, np.float64)
    call("sb200_velocity_from_stream_function", ctypes.byref(g), ptr(u1), ptr(psi), 0.8,
         fs.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), ptr(forcing), ptr(out), None)
    assert _rel(u1, u0) < _tol(real_t)
    assert np.abs(forcing).max() == 0
    inner = (slice(None),) + (slice(gs, -gs),) * 3
    assert np.isclose(out[0], np.abs(u0[inner]).sum(axis=0).max(), rtol=1e-6)


@pytest.mark.parametrize("real_t", [np.float64, np.float32], ids=["f64", "f32"])
def test_2d_operators(real_t):
    rng = np.random.default_rng(5)
    n, gs = (10, 14), 2
    shape = tuple(v + 2 * gs for v in n)
    g = _lib.make_grid(2, real_t, gs, n, [1] * 4)
    inner = (slice(gs, -gs),) * 2
    # outplane curl on the interior-of-interior, zero ring
    psi = rng.uniform(size=shape).astype(real_t)
    u = rng.uniform(size=(2,) + shape).astype(real_t)
    call("sb200_curl", ctypes.byref(g), ptr(u), ptr(psi), 0.5, None)
    ref = np.zeros_like(u)
    ref[0, 3:-3, 3:-3] = real_t(0.5) * (psi[4:-2, 3:-3] - psi[2:-4, 3:-3])
    ref[1, 3:-3, 3:-3] = -real_t(0.5) * (psi[3:-3, 4:-2] - psi[3:-3, 2:-4])
    assert _rel(u, ref) < _tol(real_t)
    # diffusion flux 5 point
    fl = np.zeros(shape, real_t)
    call("sb200_diffusion_flux", ctypes.byref(g), ptr(fl), ptr(psi), 0.25, None)
    ref = np.zeros(shape, real_t)
    ref[3:-3, 3:-3] = real_t(0.25) * (psi[3:-3, 4:-2] + psi[3:-3, 2:-4] + psi[4:-2, 3:-3]
                                      + psi[2:-4, 3:-3] - 4 * psi[3:-3, 3:-3])
    assert _rel(fl, ref) < _tol(real_t)
    # forcing update: omega += p (dFy/dx - dFx/dy) on [2:-2] cells (plus the ghost strips the slabs touch)
    w = np.zeros(shape, real_t)
    f = rng.uniform(size=(2,) + shape).astype(real_t)
    call("sb200_update_vorticity_from_velocity_forcing", ctypes.byref(g), ptr(w), ptr(f), 2.0, None)
    ref = real_t(2.0) * (f[1][2:-2, 3:-1] - f[1][2:-2, 1:-3] - f[0][3:-1, 2:-2] + f[0][1:-3, 2:-2])
    assert _rel(w[inner], ref) < _tol(real_t)


@pytest.mark.parametrize("real_t", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("phys", [(1, 1, 1, 1), (0, 1, 1, 1), (0, 0, 1, 1)], ids=["single", "first_slab", "inner_slab"])
def test_2d_operators_against_the_2d_wrapper_oracle(real_t, phys):
    """Every 2D operator of config 1 against oracle/stencils_2d.py (five wrapper regions, ring
    zeroing, x-then-y penalisation), on single-domain and y-slab face patterns."""
    from oracle import stencils_2d as st2
    from sopht_mpi_b200.numeric.eulerian_grid_ops.ops import _penalise_factor_table

    rng = np.random.default_rng(11)
    n, gs = (12, 17), 2
    shape = tuple(v + 2 * gs for v in n)
    g = _lib.make_grid(2, real_t, gs, n, phys)
    tol = _tol(real_t)
    w = rng.uniform(size=shape).astype(real_t)
    f = rng.uniform(size=(2,) + shape).astype(real_t)
    vel = (rng.uniform(size=(2,) + shape) - 0.5).astype(real_t)
    # forcing update
    a0, a1 = w.copy(), w.copy()
    st2.update_vorticity_from_velocity_forcing_mpi(a0, f, 0.37, gs)
    call("sb200_update_vorticity_from_velocity_forcing", ctypes.byref(g), ptr(a1), ptr(f), 0.37, None)
    assert _rel(a1, a0) < tol
    # out-of-plane curl + ring
    c0 = rng.uniform(size=(2,) + shape).astype(real_t)
    c1 = c0.copy()
    st2.outplane_field_curl_mpi(c0, w, 0.8, gs, phys)
    call("sb200_curl", ctypes.byref(g), ptr(c1), ptr(w), 0.8, None)
    assert _rel(c1, c0) < tol
    # diffusion time step (flux buffer holds garbage on entry)
    a0, a1 = w.copy(), w.copy()
    fl0, fl1 = np.ones(shape, real_t), np.ones(shape, real_t)
    st2.diffusion_timestep_mpi(a0, fl0, 0.1, gs, phys)
    call("sb200_diffusion_timestep", ctypes.byref(g), ptr(a1), 1, ptr(fl1), 0.1, None)
    assert _rel(a1, a0) < tol
    # ENO3 advection time step: compare where every operand is defined ([2:-2], like the reference tests)
    a0, a1 = w.copy(), w.copy()
    fl0, fl1 = np.ones(shape, real_t), np.ones(shape, real_t)
    st2.advection_timestep_mpi(a0, fl0, vel, 0.2, gs)
    call("sb200_advection_timestep_eno3", ctypes.byref(g), ptr(a1), 1, ptr(fl1), ptr(vel), 0.2, None)
    assert _rel(a1[2:-2, 2:-2], a0[2:-2, 2:-2]) < tol
    # penalisation is bit exact (tabulated sine factors)
    dx = real_t(1.0 / n[1])
    xg = ((np.arange(shape[1]) - gs + 0.5) * dx).astype(real_t)
    yg = ((np.arange(shape[0]) - gs + 0.5) * dx).astype(real_t)
    a0, a1 = w.copy(), w.copy()
    st2.penalise_field_boundary_mpi(a0, 3, dx, xg, yg, gs, phys)
    tab = _penalise_factor_table(real_t, 3, dx, gs, [yg, xg])
    call("sb200_penalise_field_boundary", ctypes.byref(g), ptr(a1), 1, 3, ptr(tab), None)
    assert np.array_equal(a0, a1)


IB_FILES = sorted(glob.glob(os.path.join(GOLDEN, "ib_*.npz")))


@pytest.mark.parametrize("path", IB_FILES, ids=[os.path.basename(p) for p in IB_FILES])
def test_ib_kernels_against_reference_golden(path):
    gd = np.load(path)
    dim, gs, w = int(gd["dim"]), int(gd["gs"]), int(gd["width"])
    dx, shift = gd["dx"][()], gd["shift"][()]
    real_t = type(dx)
    pos = gd["pos"]
    lag_t = pos.dtype.type
    n_local = gd["eul_vec"].shape[-1] - 2 * gs
    g = _lib.make_grid(dim, real_t, gs, (n_local,) * dim, [1] * (2 * dim))
    p = _lib.IBParams()
    p.lag_dtype = _lib.dtype_code(lag_t)
    p.kernel_type = 0
    p.width = w
    ss = list(gd["substart_xyz"]) + [0] * (3 - dim)
    for i in range(3):
        p.substart_xyz[i] = int(ss[i])
    p.dx, p.coord_shift, p.stiffness, p.damping = float(dx), float(shift), -3.0, -0.5
    n = pos.shape[1]
    near = np.zeros((dim, n), np.int64)
    wts = np.zeros(gd["w_cos"].shape, lag_t)
    u, dv, f = (np.zeros((dim, n), lag_t) for _ in range(3))
    vel = np.full((dim, n), 0.25, lag_t)
    dpos = np.full((dim, n), 0.01, lag_t)
    eul = np.ascontiguousarray(gd["eul_vec"])
    call("sb200_ib_interact_lag", ctypes.byref(g), ctypes.byref(p), n, ptr(eul), ptr(pos), ptr(vel),
         ptr(dpos), ptr(near), ptr(wts), ptr(u), ptr(dv), ptr(f), None)
    tol = 1e-6 if (lag_t == np.float32) else 1e-13
    assert np.array_equal(near, gd["nearest"])  # bit exact index work
    assert _rel(wts, gd["w_cos"]) < tol
    assert _rel(u, gd["e2l_vec"]) < tol
    assert _rel(f, -3.0 * dpos - 0.5 * (gd["e2l_vec"] - vel)) < 10 * tol
    p.kernel_type = 1
    wp = np.zeros_like(wts)
    call("sb200_ib_interact_lag", ctypes.byref(g), ctypes.byref(p), n, ptr(eul), ptr(pos), ptr(vel),
         ptr(dpos), ptr(near), ptr(wp), ptr(u), ptr(dv), ptr(f), None)
    assert _rel(wp, gd["w_pes"]) < max(tol, 1e-7 if real_t == np.float32 else 0)
    p.kernel_type = 0
    out = np.zeros_like(gd["l2e_vec"])
    lagv = np.ascontiguousarray(gd["lag_vec"])
    call("sb200_ib_spread", ctypes.byref(g), ctypes.byref(p), n, ptr(out), ptr(lagv), ptr(pos), None)
    assert _rel(out, gd["l2e_vec"]) < (1e-6 if out.dtype == np.float32 else 1e-13)
    call("sb200_clear_ghost_cells", ctypes.byref(g), ptr(out), dim, None)
    inner = (slice(None),) + (slice(gs, -gs),) * dim
    chk = gd["l2e_vec"].copy()
    keep = chk[inner].copy()
    chk[...] = 0
    chk[inner] = keep
    assert _rel(out, chk) < (1e-6 if out.dtype == np.float32 else 1e-13)


@pytest.mark.parametrize("real_t,n", [
    (np.float64, (8, 8, 16)), (np.float32, (16, 8, 32)), (np.float64, (8, 8, 256)),
    (np.float32, (8, 64, 16)), (np.float64, (128, 8, 16)), (np.float32, (8, 8, 1024)),
    (np.float32, (128, 8, 16)), (np.float32, (8, 128, 16)), (np.float32, (256, 8, 16)),
    (np.float32, (8, 256, 16)), (np.float32, (512, 8, 16)), (np.float64, (8, 128, 16)),
    (np.float32, (8, 512, 16)),
], ids=lambda v: str(v) if isinstance(v, tuple) else v.__name__)
def test_pruned_fft_poisson_pipeline_3d(real_t, n):
    """backend 1 (in-kernel pruned FFT pipeline): every Stockham plan shape up to n = 1024
    against the scipy.fft oracle (which is what the reference's FFT test pins to)."""
    from oracle.poisson import UnboundedPoissonSolverOracle3D

    lib = emu()
    gs = 2
    rng = np.random.default_rng(0)
    h = ctypes.c_void_p()
    _lib.check(lib, lib.sb200_poisson_create(ctypes.byref(h), 3, _lib.dtype_code(real_t), n[0], n[1], n[2],
                                             gs, 1.0, 0, 1, 1, None))
    shape = tuple(v + 2 * gs for v in n)
    rhs = rng.uniform(size=(2,) + shape).astype(real_t)
    sol = np.full_like(rhs, 7.0)
    _lib.check(lib, lib.sb200_poisson_solve(h, ptr(sol), ptr(rhs), 2, None))
    lib.sb200_poisson_destroy(h)
    oracle = UnboundedPoissonSolverOracle3D(*n, x_range=1.0, real_t=real_t)
    ref = np.zeros_like(rhs)
    for c in range(2):
        oracle.solve(ref[c], rhs[c], gs)
    inner = (slice(None),) + (slice(gs, -gs),) * 3
    assert _rel(sol[inner], ref[inner]) < (1e-13 if real_t == np.float64 else 2e-6)
    assert np.all(sol[:, 0] == 7.0) and np.all(sol[:, :, :, -1] == 7.0)  # ghosts untouched


@pytest.mark.parametrize("real_t,n,nranks", [
    (np.float64, (16, 8, 32), 2), (np.float64, (32, 16, 16), 4), (np.float32, (128, 8, 16), 2),
    (np.float32, (16, 128, 32), 2), (np.float32, (32, 8, 64), 8),
    # 2 nz = 512 / 1024: the tile-layout z kernel (sb_fft_zconvw_kernel)
    (np.float32, (256, 8, 16), 2), (np.float32, (512, 8, 16), 4),
], ids=lambda v: str(v) if not isinstance(v, type) else v.__name__)
def test_slab_decomposed_poisson_pipeline(real_t, n, nranks):
    """The distributed (z-slab) solve, all ranks emulated in one process, against the scipy oracle and,
    bit for bit, against the single-domain solve (the same three stages on a one-rank layout)."""
    from oracle.poisson import UnboundedPoissonSolverOracle3D

    lib = emu()
    gs, ncomp = 2, 2
    rng = np.random.default_rng(1)
    shape = tuple(v + 2 * gs for v in n)
    rhs = rng.uniform(size=(ncomp,) + shape).astype(real_t)
    out = slab_poisson_solve(_Host(), n, real_t, nranks, rhs, ncomp, backend=1)
    h = ctypes.c_void_p()
    _lib.check(lib, lib.sb200_poisson_create(ctypes.byref(h), 3, _lib.dtype_code(real_t), n[0], n[1], n[2],
                                             gs, 1.0, 0, 1, 1, None))
    single = np.full_like(rhs, 7.0)
    _lib.check(lib, lib.sb200_poisson_solve(h, ptr(single), ptr(rhs), ncomp, None))
    lib.sb200_poisson_destroy(h)
    oracle = UnboundedPoissonSolverOracle3D(*n, x_range=1.0, real_t=real_t)
    ref = np.zeros_like(rhs)
    for c in range(ncomp):
        oracle.solve(ref[c], rhs[c], gs)
    nzl = n[0] // nranks
    tol = 1e-13 if real_t == np.float64 else 2e-6
    scale = np.abs(ref).max()
    for r in range(nranks):
        got = out[r][:, gs:-gs, gs:-gs, gs:-gs]
        want = ref[:, r * nzl + gs:r * nzl + gs + nzl, gs:-gs, gs:-gs]
        assert np.abs(got - want).max() / scale < tol, (r, np.abs(got - want).max() / scale)
        assert np.array_equal(got, single[:, r * nzl + gs:r * nzl + gs + nzl, gs:-gs, gs:-gs]), r
        assert np.all(out[r][:, 0] == 7.0) and np.all(out[r][:, :, :, -1] == 7.0)  # ghosts untouched


# (256, 16): 2 ny = 512 runs the y pass through the 32-points-per-thread kernel (sb_fft_strided32_kernel)
@pytest.mark.parametrize("real_t, n", [(np.float64, (16, 32)), (np.float32, (16, 32)), (np.float32, (256, 16))],
                         ids=["f64", "f32", "f32-ny256"])
def test_pruned_fft_poisson_pipeline_2d(real_t, n):
    from oracle.poisson import UnboundedPoissonSolverOracle2D

    lib = emu()
    gs = 2
    rng = np.random.default_rng(0)
    h = ctypes.c_void_p()
    _lib.check(lib, lib.sb200_poisson_create(ctypes.byref(h), 2, _lib.dtype_code(real_t), 1, n[0], n[1], gs,
                                             1.0, 0, 1, 1, None))
    shape = tuple(v + 2 * gs for v in n)
    rhs = rng.uniform(size=shape).astype(real_t)
    sol = np.zeros_like(rhs)
    _lib.check(lib, lib.sb200_poisson_solve(h, ptr(sol), ptr(rhs), 1, None))
    lib.sb200_poisson_destroy(h)
    oracle = UnboundedPoissonSolverOracle2D(*n, x_range=1.0, real_t=real_t)
    ref = np.zeros_like(rhs)
    oracle.solve(ref, rhs, gs)
    inner = (slice(gs, -gs),) * 2
    assert _rel(sol[inner], ref[inner]) < (1e-13 if real_t == np.float64 else 2e-6)


@pytest.mark.parametrize("real_t", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("n", [(20, 24, 70), (9, 17, 66), (6, 60, 200)], ids=["a", "b", "interior-blocks"])
def test_fused_vorticity_update_equals_the_three_reference_sweeps(real_t, n):
    """csrc/fused.cu against cross product -> curl update -> diffusion composed from the
    oracle's restatement of the reference wrappers (bit-for-bit the same cells)."""
    rng = np.random.default_rng(0)
    gs = 2
    shape = tuple(v + 2 * gs for v in n)
    g = _lib.make_grid(3, real_t, gs, n, (1,) * 6)
    w = rng.uniform(size=(3,) + shape).astype(real_t)
    u = (rng.uniform(size=(3,) + shape) - 0.5).astype(real_t)
    ref = w.copy()
    buf = np.zeros_like(w)
    flux = np.zeros(shape, real_t)
    st.elementwise_cross_product(buf, u, ref)
    st.update_vorticity_from_velocity_forcing_mpi(ref, buf, 0.3, gs)
    st.diffusion_timestep_mpi(ref, flux, 0.05, gs)
    out = np.full_like(w, np.nan)
    call("sb200_vorticity_rhs_fused_3d", ctypes.byref(g), ptr(out), ptr(w), ptr(u), None, 0.3, 0.05, None)
    assert not np.isnan(out).any()
    assert _rel(out, ref) < _tol(real_t)


@pytest.mark.parametrize("real_t", [np.float64, np.float32], ids=["f64", "f32"])
def test_fused_vorticity_update_on_virtual_z_slabs(real_t):
    """Three virtual z-slabs with exchanged ghost planes: every slab's interior must equal
    the single-domain result (what the reference's MPI-vs-serial tests assert)."""
    rng = np.random.default_rng(1)
    gs, nzl, ny, nx, ranks = 2, 6, 10, 12, 3
    gshape = (ranks * nzl + 2 * gs, ny + 2 * gs, nx + 2 * gs)
    w = rng.uniform(size=(3,) + gshape).astype(real_t)
    u = (rng.uniform(size=(3,) + gshape) - 0.5).astype(real_t)
    ref = w.copy()
    buf = np.zeros_like(w)
    flux = np.zeros(gshape, real_t)
    st.elementwise_cross_product(buf, u, ref)
    st.update_vorticity_from_velocity_forcing_mpi(ref, buf, 0.3, gs)
    st.diffusion_timestep_mpi(ref, flux, 0.05, gs)
    for r in range(ranks):
        phys = (r == 0, r == ranks - 1, 1, 1, 1, 1)
        g = _lib.make_grid(3, real_t, gs, (nzl, ny, nx), phys)
        lo = r * nzl  # padded global index of the slab's first ghost plane
        wl = np.ascontiguousarray(w[:, lo:lo + nzl + 2 * gs])
        ul = np.ascontiguousarray(u[:, lo:lo + nzl + 2 * gs])
        out = np.full_like(wl, np.nan)
        call("sb200_vorticity_rhs_fused_3d", ctypes.byref(g), ptr(out), ptr(wl), ptr(ul), None, 0.3, 0.05,
             None)
        inner = (slice(None), slice(gs, -gs))
        assert _rel(out[inner], ref[:, lo + gs:lo + gs + nzl]) < _tol(real_t)


def test_device_rank_ownership_against_reference_golden():
    """SURVEY L1: the ownership kernel gives the integers of the reference's
    _compute_lag_nodes_rank_address (tests/golden/ownership.npz), any topology, both dtypes."""
    o = np.load(os.path.join(GOLDEN, "ownership.npz"))
    for t in ("f64", "f32"):
        for d in ("3", "2"):
            addr, flag = rank_address(call, ptr, o[f"pos{d}_{t}"], o["dx"][()], o["shift"][()],
                                                o["local" + d], o["topo" + d])
            assert np.array_equal(addr, o[f"addr{d}_{t}"]) and flag == 0
    # a point beyond the last block raises the flag (the reference aborts)
    pos = o["pos3_f64"].copy()
    pos[0, 0] = float(o["dx"][()]) * o["local3"][2] * o["topo3"][2] * 1.5
    _, flag = rank_address(call, ptr, pos, o["dx"][()], o["shift"][()], o["local3"], o["topo3"])
    assert flag == 1


@pytest.mark.parametrize("lag_t", [np.float64, np.float32], ids=["lag64", "lag32"])
def test_owner_filtered_ib_kernels_assemble_the_global_result(lag_t):
    """The replicated-state scheme of VirtualBoundaryForcingMPI: every virtual rank runs the
    interaction on the points it owns and writes zeros elsewhere; the SUM over the ranks equals the
    single-rank arrays, and the owner-filtered spreading contributions add up to the full spreading."""
    real_t = np.float32
    rng = np.random.default_rng(5)
    dim, gs, w, n_local, n = 3, 2, 2, 12, 40
    dx, shift = real_t(1.0 / n_local), real_t(0.5 / n_local)
    g = _lib.make_grid(dim, real_t, gs, (n_local,) * dim, [1] * 6)
    p = _lib.IBParams()
    p.lag_dtype, p.kernel_type, p.width = _lib.dtype_code(lag_t), 0, w
    p.dx, p.coord_shift, p.stiffness, p.damping = float(dx), float(shift), -2.0, -0.3
    pos = (0.2 + 0.6 * rng.uniform(size=(dim, n))).astype(lag_t)
    vel = rng.uniform(size=(dim, n)).astype(lag_t)
    dpos = rng.uniform(size=(dim, n)).astype(lag_t)
    eul = rng.uniform(size=(dim,) + (n_local + 2 * gs,) * dim).astype(real_t)
    owner = rng.integers(0, 3, size=n).astype(np.int32)

    def interact(owner_arr, rank):
        u, dv, f = (np.full((dim, n), 9.0, lag_t) for _ in range(3))
        call("sb200_ib_interact_owned", ctypes.byref(g), ctypes.byref(p), n, ptr(eul), ptr(pos), ptr(vel),
             ptr(dpos), None, None, ptr(u), ptr(dv), ptr(f), ptr(owner_arr) if owner_arr is not None else None,
             rank, None)
        return u, dv, f

    full = interact(None, 0)
    parts = [interact(owner, r) for r in range(3)]
    for k in range(3):
        assert np.array_equal(sum(part[k] for part in parts), full[k])
        for r in range(3):
            assert np.all(parts[r][k][:, owner != r] == 0)
    spread_full = np.zeros_like(eul)
    call("sb200_ib_spread_owned", ctypes.byref(g), ctypes.byref(p), n, ptr(spread_full), ptr(full[2]), ptr(pos),
         None, 0, None)
    acc = np.zeros_like(eul)
    for r in range(3):
        call("sb200_ib_spread_owned", ctypes.byref(g), ctypes.byref(p), n, ptr(acc), ptr(full[2]), ptr(pos),
             ptr(owner), r, None)
    assert _rel(acc, spread_full) < 1e-6


@pytest.mark.parametrize("dim", [3, 2])
@pytest.mark.parametrize("sparse", [True, False], ids=["sparse", "dense"])
def test_sparse_forcing_update_and_flagged_reset(dim, sparse):
    """sb200_update_vorticity_from_sparse_forcing == the plain update (bit for bit, for a forcing field
    that is zero almost everywhere as well as for a dense one); sb200_clear_flagged_tiles leaves F == 0
    and the flags cleared."""
    real_t = np.float32
    rng = np.random.default_rng(12)
    gs = 2
    n = (10, 37, 45) if dim == 3 else (150, 200)
    shape = tuple(v + 2 * gs for v in n)
    g = _lib.make_grid(dim, real_t, gs, n, [1] * (2 * dim))
    w = rng.uniform(size=((3,) + shape) if dim == 3 else shape).astype(real_t)
    f = rng.uniform(-1, 1, size=(dim,) + shape).astype(real_t)
    if sparse:
        mask = np.zeros(shape, bool)
        mask[(slice(4, 8),) * dim] = True
        mask[(-1,) * dim] = True  # a ghost corner cell too
        f *= mask
    ref, got = w.copy(), w.copy()
    call("sb200_update_vorticity_from_velocity_forcing", ctypes.byref(g), ptr(ref), ptr(f), 0.37, None)
    count = int(emu().sb200_tile_flag_count(ctypes.byref(g)))
    work = np.zeros(count, np.uint8)
    call("sb200_update_vorticity_from_sparse_forcing", ctypes.byref(g), ptr(got), ptr(f), 0.37, ptr(work), None)
    assert np.array_equal(got, ref)
    ints = work.view(np.int32)
    nchunks = (ints.size - 4) // 4
    n_flagged, n_active = int(ints[4 * nchunks]), int(ints[4 * nchunks + 1])
    assert n_flagged == int((ints[:nchunks] > 0).sum()) > 0
    assert n_active == int((ints[nchunks:2 * nchunks] > 0).sum()) >= n_flagged
    assert (n_active < nchunks) if sparse else (n_flagged == nchunks)
    call("sb200_clear_flagged_tiles", ctypes.byref(g), ptr(f), dim, ptr(work), None)
    assert not f.any() and not work.any()


def test_one_pass_order1_multiplicative_filter(setup3d):
    """sb200_laplacian_filter_order1_out_of_place == the reference's stage chain (field and both buffers)."""
    real_t, rng, n, gs, shape, g = setup3d
    w = rng.uniform(size=(3,) + shape).astype(real_t)
    ref = w.copy()
    fb0, bb0 = rng.uniform(size=shape).astype(real_t), rng.uniform(size=shape).astype(real_t)
    fb1, bb1 = fb0.copy(), bb0.copy()
    st.laplacian_filter_mpi(ref, fb0, bb0, 1, "multiplicative", gs)
    out = np.full_like(w, np.nan)
    call("sb200_laplacian_filter_order1_out_of_place", ctypes.byref(g), ptr(out), ptr(w), 3, ptr(fb1), ptr(bb1), None)
    assert np.array_equal(out, ref) and np.array_equal(fb1, fb0) and np.array_equal(bb1, bb0)
    big = (20, 19, 70)  # several tiles along every axis
    shape2 = tuple(v + 2 * gs for v in big)
    g2 = _lib.make_grid(3, real_t, gs, big, [1] * 6)
    w2 = rng.uniform(size=(3,) + shape2).astype(real_t)
    ref2 = w2.copy()
    a, b = np.zeros(shape2, real_t), np.zeros(shape2, real_t)
    st.laplacian_filter_mpi(ref2, a, b, 1, "multiplicative", gs)
    out2, a1, b1 = np.empty_like(w2), np.zeros(shape2, real_t), np.zeros(shape2, real_t)
    call("sb200_laplacian_filter_order1_out_of_place", ctypes.byref(g2), ptr(out2), ptr(w2), 3, ptr(a1), ptr(b1), None)
    assert np.array_equal(out2, ref2) and np.array_equal(a1, a)


def test_operators_outside_the_simulator_paths(setup3d):
    """Brinkmann penalisation, level set -> characteristic function, vorticity update from a penalised
    velocity (SURVEY 8(f)4) against their closed forms / the velocity-forcing update of the difference."""
    real_t, rng, n, gs, shape, g = setup3d
    code = _lib.dtype_code(real_t)
    cells = int(np.prod(shape))
    f = rng.uniform(size=(3,) + shape).astype(real_t)
    tgt = rng.uniform(size=(3,) + shape).astype(real_t)
    chi = rng.uniform(size=shape).astype(real_t)
    out = np.zeros_like(f)
    call("sb200_brinkmann_penalise", code, ptr(out), 7.5, ptr(chi), ptr(tgt), ptr(f), 3, cells, None)
    lam = real_t(7.5)
    assert _rel(out, (f + lam * chi * tgt) / (1 + lam * chi)) < _tol(real_t)
    ls = (rng.uniform(size=shape) - 0.5).astype(real_t)
    got = np.zeros_like(ls)
    call("sb200_char_func_from_level_set", code, ptr(got), ptr(ls), 0.2, cells, None)
    s = ls / real_t(0.2)
    want = np.where(ls > 0.2, 1.0, np.where(ls < -0.2, 0.0, 0.5 * (1 + s + np.sin(np.pi * s) / np.pi)))
    assert np.abs(got - want).max() < (1e-6 if real_t == np.float32 else 1e-14)
    assert got.min() >= -1e-6 and got.max() <= 1 + 1e-6
    w = rng.uniform(size=(3,) + shape).astype(real_t)
    up, u = tgt, f
    ref = w.copy()
    st.update_vorticity_from_velocity_forcing_mpi(ref, (up - u).astype(real_t), 0.4, gs)
    call("sb200_update_vorticity_from_penalised_velocity", ctypes.byref(g), ptr(w), ptr(up), ptr(u), 0.4, None)
    assert _rel(w, ref) < _tol(real_t)


@pytest.mark.parametrize("real_t", [np.float64, np.float32], ids=["f64", "f32"])
def test_fused_vorticity_update_by_plane_ranges(real_t):
    """The plane-range entry point (interior planes while the halo exchange is in flight, the planes next
    to the slab faces afterwards) assembles exactly the whole-grid result."""
    rng = np.random.default_rng(3)
    gs, n = 2, (20, 10, 66)
    shape = tuple(v + 2 * gs for v in n)
    g = _lib.make_grid(3, real_t, gs, n, (0, 0, 1, 1, 1, 1))  # an inner z-slab
    w = rng.uniform(size=(3,) + shape).astype(real_t)
    u = (rng.uniform(size=(3,) + shape) - 0.5).astype(real_t)
    whole = np.full_like(w, np.nan)
    call("sb200_vorticity_rhs_fused_3d", ctypes.byref(g), ptr(whole), ptr(w), ptr(u), None, 0.3, 0.05, None)
    parts = np.full_like(w, np.nan)
    mz = shape[0]
    for z0, z1 in ((4, mz - 4), (0, 4), (mz - 4, mz)):
        call("sb200_vorticity_rhs_fused_3d_range", ctypes.byref(g), ptr(parts), ptr(w), ptr(u), 0.3, 0.05, z0, z1, None)
    assert not np.isnan(parts).any() and np.array_equal(parts, whole)
