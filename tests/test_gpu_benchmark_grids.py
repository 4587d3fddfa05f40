"""The kernels of the benchmarked step against float64, at the grid sizes bench.py times.

At these sizes the launch geometry comes from the device and the grid: the z chunks of the marching fused
kernels follow from the SM count and occupancy, the persistent fused z pass of the Poisson solve starts one
block per resident slot and lets each block take several tiles, almost every block of fused v2 takes its
FAST body, and the IB kernels see ~131 k points with overlapping supports.  The skinny shapes of
test_emu_launch_coverage.py reach none of this.

Every case feeds a kernel random (or the benchmark's) input and compares it with a float64 computation of
the same operation on the same rounded input: relative L-inf <= 2e-6 for float32 and <= 1e-13 for float64,
measured for incremental updates against the largest reference increment.  Kernels without floating-point
atomics (all but IB spreading and the sum of squares) run twice on the same input and must give the same
bits.  The grids and set-up are bench.py's (`WORKLOADS`, `workload_setup`); the kernels are driven through
the C ABI on torch buffers."""
import ctypes
import math
import os

import numpy as np
import pytest
import torch

import bench
from oracle import ib as ib_oracle
from oracle import stencils as st
from oracle.poisson import UnboundedPoissonSolverOracle3D
from oracle.simulator import FlowSimulatorOracle3D
from sopht_mpi_b200 import _lib
from test_emu_launch_coverage import _call, _Cuda, _fused_reference

pytestmark = pytest.mark.gpu

f32, f64 = np.float32, np.float64
GS = 2  # the simulator's ghost size
CORES = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
GRID_512 = bench.WORKLOADS["fsi_512_f32"][0]
GRID_ROD = bench.WORKLOADS["rod_fsi_512x256x256_f32"][0]
GRID_256 = bench.WORKLOADS["vortex_ring_256_f32"][0]
assert bench.WORKLOADS["vortex_ring_256_f64"][0] == GRID_256
assert bench.WORKLOADS["sphere_vbf_512x256x256_f32"][0] == GRID_ROD


def _tol(real_t):
    return 1e-13 if real_t == f64 else 2e-6


def _rel(a, b):
    """relative L-inf of a against b (numpy or torch, computed in float64)"""
    if isinstance(b, torch.Tensor):
        a = a.to(b.device, torch.float64) if isinstance(a, torch.Tensor) else torch.from_numpy(a).to(b.device)
        return ((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-300)).item()
    return float(np.abs(np.asarray(a, f64) - b).max() / max(np.abs(b).max(), 1e-300))


def _check(record_property, name, err, tol):
    record_property(name, err)
    assert err <= tol, (name, err)


def _free():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


@pytest.fixture(scope="module")
def cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return _Cuda()


def _inner(ncomp=0):
    return (slice(None),) * ncomp + (slice(GS, -GS),) * 3


# ------------------------------------------------------------------------------- Poisson
def greens_spectrum_f64(n, x_range, device):
    """oracle/poisson.py's Green's function of the doubled domain and its spectrum times dx^3, in torch
    float64 on `device` (the scipy oracle needs too much host memory at 512^3)"""
    nz, ny, nx = n
    dx = x_range / nx
    ranges = (x_range * nz / nx, x_range * ny / nx, x_range)

    def axis(m, rng):
        c = torch.arange(2 * m, dtype=torch.float64, device=device) * dx
        return torch.minimum(c, 2 * rng - c) ** 2

    z, y, x = (axis(m, r) for m, r in zip(n, ranges))
    g = (x[None, None, :] + y[None, :, None]) + z[:, None, None]
    g = (1 / g.sqrt_()) / (4 * math.pi)
    g[0, 0, 0] = 1 / (4 * math.pi * dx)
    ghat = torch.fft.rfftn(g) * dx ** 3
    del g
    return ghat


def poisson_solve_f64(rhs_interior, ghat):
    """oracle/poisson.py's solve of one interior field (torch float64, on the device of ghat)"""
    nz, ny, nx = rhs_interior.shape
    doubled = torch.zeros((2 * nz, 2 * ny, 2 * nx), dtype=torch.float64, device=ghat.device)
    doubled[:nz, :ny, :nx] = rhs_interior
    back = torch.fft.irfftn(torch.fft.rfftn(doubled) * ghat, s=doubled.shape)
    return back[:nz, :ny, :nx].clone()


def test_torch_float64_poisson_reference_matches_the_scipy_oracle(cuda):
    n, x_range = (64, 32, 64), 1.8
    rhs = np.random.default_rng(1).uniform(size=tuple(v + 2 * GS for v in n))
    ref = np.zeros_like(rhs)
    UnboundedPoissonSolverOracle3D(*n, x_range=x_range, real_t=f64).solve(ref, rhs, GS)
    inner = _inner()
    ghat = greens_spectrum_f64(n, x_range, "cuda")
    got = poisson_solve_f64(torch.from_numpy(rhs[inner]).cuda(), ghat).cpu().numpy()
    assert _rel(got, ref[inner]) <= 1e-13


POISSON = [(GRID_512, f32, 1.0), (GRID_ROD, f32, 1.8), (GRID_256, f32, 1.0), (GRID_256, f64, 1.0)]


@pytest.mark.parametrize("n,real_t,x_range", POISSON, ids=["512-f32", "256x256x512-f32-rod", "256-f32", "256-f64"])
def test_vector_poisson_solve(cuda, n, real_t, x_range, record_property):
    """fft backend: each component against float64, ghost cells of the solution never written, and two
    solves of the same input give the same bits (the persistent z kernel hands out tiles dynamically)."""
    be, t = cuda, torch.float32 if real_t == f32 else torch.float64
    shape = (3,) + tuple(v + 2 * GS for v in n)
    gen = torch.Generator(device="cuda").manual_seed(sum(n))
    rhs = torch.rand(shape, generator=gen, dtype=t, device="cuda")
    sols = [torch.full_like(rhs, 7.0) for _ in range(2)]
    h = ctypes.c_void_p()
    _call(be, "sb200_poisson_create", ctypes.byref(h), 3, _lib.dtype_code(real_t), *n, GS, x_range, 0, 1, 1, None)
    try:
        for sol in sols:
            _call(be, "sb200_poisson_solve", h, be.ptr(sol), be.ptr(rhs), 3, None)
        torch.cuda.synchronize()
    finally:
        be.lib.sb200_poisson_destroy(h)
    assert torch.equal(sols[0], sols[1])
    got = sols[0]
    del sols
    ghost = torch.ones(shape[1:], dtype=torch.bool, device="cuda")
    ghost[_inner()] = False
    assert bool((got[:, ghost] == 7.0).all())
    del ghost
    inner = _inner()
    if n != GRID_512:  # the scipy oracle (doubled domains up to 512 x 512 x 1024)
        oracle = UnboundedPoissonSolverOracle3D(*n, x_range=x_range, real_t=f64, workers=CORES)
        host_rhs = rhs.cpu().numpy()
        errs = []
        for c in range(3):
            ref = np.zeros(shape[1:])
            oracle.solve(ref, host_rhs[c].astype(f64), GS)
            errs.append(_rel(got[c][inner].cpu().numpy(), ref[inner]))
    else:
        ghat = greens_spectrum_f64(n, x_range, "cuda")
        errs = [_rel(got[c][inner], poisson_solve_f64(rhs[c][inner].double(), ghat)) for c in range(3)]
        del ghat
    del rhs, got
    _free()
    _check(record_property, "rel_linf", max(errs), _tol(real_t))


# ------------------------------------------------------------------------ fused vorticity update
FUSED = [(GRID_512, f32), (GRID_ROD, f32), (GRID_256, f64)]


@pytest.mark.parametrize("n,real_t", FUSED, ids=["512-f32", "256x256x512-f32", "256-f64"])
def test_fused_vorticity_update(cuda, n, real_t, record_property):
    """v2 (float, even rows) and the double kernel on random omega and u: the increment out - omega against
    the float64 increment, the same bits twice, and at 512^3 the slab call pattern (interior planes, then
    the 2 gs planes at each face) equal to the whole-grid call bit for bit."""
    be = cuda
    rng = np.random.default_rng(sum(n) + 1)
    shape = (3,) + tuple(v + 2 * GS for v in n)
    g = _lib.make_grid(3, real_t, GS, n, (1,) * 6)
    w = rng.uniform(size=shape).astype(real_t)
    u = (rng.uniform(size=shape) - 0.5).astype(real_t)
    d_w, d_u = be.dev(w), be.dev(u)
    outs = [torch.full_like(d_w, float("nan")) for _ in range(2)]
    for out in outs:
        _call(be, "sb200_vorticity_rhs_fused_3d", ctypes.byref(g), be.ptr(out), be.ptr(d_w), be.ptr(d_u), None, 0.3,
              0.05, None)
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[1])
    if n == GRID_512:
        parts = outs[1].fill_(float("nan"))
        mz, k = shape[1], 2 * GS
        for z0, z1 in ((k, mz - k), (0, k), (mz - k, mz)):
            _call(be, "sb200_vorticity_rhs_fused_3d_range", ctypes.byref(g), be.ptr(parts), be.ptr(d_w), be.ptr(d_u),
                  0.3, 0.05, z0, z1, None)
        torch.cuda.synchronize()
        assert torch.equal(parts, outs[0])
    got = outs[0].cpu().numpy()
    del outs, d_w, d_u
    _free()
    assert not np.isnan(got).any()
    ref = _fused_reference(w, u, GS)
    del u
    w64 = w.astype(f64)
    ref -= w64
    got = got - w64
    del w64
    _check(record_property, "rel_linf", _rel(got, ref), _tol(real_t))


# ------------------------------------------------------------------ velocity from stream function
VELOCITY = [(GRID_512, f32), (GRID_256, f64)]


@pytest.mark.parametrize("n,real_t", VELOCITY, ids=["512-f32", "256-f64"])
def test_velocity_from_stream_function(cuda, n, real_t, record_property):
    """The four-cells-per-thread kernel (rows of 516 / 260 cells): u - free stream against the float64
    curl, max |u| (the stable-dt input) against the float64 max, the forcing zero everywhere, and the same
    bits twice."""
    be = cuda
    rng = np.random.default_rng(sum(n) + 2)
    shape = (3,) + tuple(v + 2 * GS for v in n)
    assert shape[-1] % 4 == 0
    g = _lib.make_grid(3, real_t, GS, n, (1,) * 6)
    prefactor = float(real_t(0.5 * n[2]))  # real_t(0.5 / dx) on the unit box
    fs = np.array([1.0, 0.5, -0.25])
    psi = rng.uniform(size=shape).astype(real_t)
    u0 = rng.uniform(size=shape).astype(real_t)
    d_psi = be.dev(psi)
    runs = []
    for _ in range(2):
        u, vmax = be.dev(u0), torch.zeros(1, dtype=torch.float64, device="cuda")
        forcing = be.dev(rng.uniform(size=shape).astype(real_t))
        _call(be, "sb200_velocity_from_stream_function", ctypes.byref(g), be.ptr(u), be.ptr(d_psi), prefactor,
              fs.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), be.ptr(forcing), be.ptr(vmax), None)
        torch.cuda.synchronize()
        assert forcing.abs().max().item() == 0
        del forcing
        runs.append((u, vmax.item()))
    assert torch.equal(runs[0][0], runs[1][0]) and runs[0][1] == runs[1][1]
    got, vmax = runs[0][0].cpu().numpy(), runs[0][1]
    del runs, d_psi
    _free()
    ref = u0.astype(f64)
    del u0
    st.curl_mpi(ref, psi.astype(f64), prefactor, GS)
    del psi
    got = got.astype(f64)
    for c in range(3):
        got[c] -= fs[c]
    err = _rel(got, ref)
    for c in range(3):
        ref[c] += fs[c]
    want = np.abs(ref[_inner(1)]).sum(axis=0).max()
    record_property("rel_max_abs_sum", abs(vmax - want) / want)
    _check(record_property, "rel_linf", err, _tol(real_t))
    assert abs(vmax - want) <= _tol(real_t) * want


# ------------------------------------------------------------------- immersed boundary
def _ib_setup(name):
    """bench.py's body on its grid: the product keeps the Lagrangian arrays in the dtype of the points
    (float64 here) on the float32 grid, with dx and the coordinate shift rounded to the grid's real_t"""
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
    g = _lib.make_grid(3, real_t, GS, w["grid"], (1,) * 6)
    return w, g, p


def _spread(be, g, p, forcing_lag, pos, shape):
    """the product's spreading on one rank: scatter, then the ghost sum (which only clears the ghosts)"""
    eul = torch.zeros(shape, dtype=torch.float32, device="cuda")
    n = pos.shape[1]
    _call(be, "sb200_ib_spread_owned", ctypes.byref(g), ctypes.byref(p), n, be.ptr(eul), be.ptr(forcing_lag),
          be.ptr(pos), None, 0, None)
    _call(be, "sb200_clear_ghost_cells", ctypes.byref(g), be.ptr(eul), 3, None)
    return eul


@pytest.mark.parametrize("name", ["fsi_512_f32", "rod_fsi_512x256x256_f32"])
def test_ib_interaction_and_spreading(cuda, name, record_property):
    """sb200_ib_interact_owned (nearest index, weights, E->L interpolation, mismatch, penalty force) and
    sb200_ib_spread_owned at the benchmark's points against oracle/ib.py in float64: indices exact,
    flow velocity, velocity mismatch and forcing within the bar, the spread field against a float64
    np.add.at scatter of the same forcing with the same weights; the interaction gives the same bits twice."""
    be = cuda
    w, g, p = _ib_setup(name)
    pos, vel = w["points"], w["lag_vel"]
    n = pos.shape[1]
    assert n > (1e5 if name == "fsi_512_f32" else 1e4)
    shape = (3,) + tuple(v + 2 * GS for v in w["grid"])
    rng = np.random.default_rng(n)
    eul = (rng.uniform(size=shape) - 0.5).astype(f32)
    dpos = 0.1 * w["dx"] * rng.standard_normal(pos.shape)
    d_eul, d_pos, d_vel, d_dpos = be.dev(eul), be.dev(pos), be.dev(vel), be.dev(dpos)
    runs = []
    for _ in range(2):
        near = torch.zeros((3, n), dtype=torch.int64, device="cuda")
        u, dv, f = (torch.zeros((3, n), dtype=torch.float64, device="cuda") for _ in range(3))
        _call(be, "sb200_ib_interact_owned", ctypes.byref(g), ctypes.byref(p), n, be.ptr(d_eul), be.ptr(d_pos),
              be.ptr(d_vel), be.ptr(d_dpos), be.ptr(near), None, be.ptr(u), be.ptr(dv), be.ptr(f), None, 0, None)
        runs.append((near, u, dv, f))
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(*runs))
    near, u, dv, f = (a.cpu().numpy() for a in runs[0])
    spread = _spread(be, g, p, runs[0][3], d_pos, shape).cpu().numpy()
    del runs, d_eul, d_pos, d_vel, d_dpos
    _free()

    ora = ib_oracle.VirtualBoundaryForcingOracle(p.stiffness, p.damping, 3, p.dx, f64, f64, GS,
                                                 eul_grid_coord_shift=p.coord_shift, fast=True)
    ora._ensure(n)
    ora.position_mismatch[...] = dpos
    ora.compute_interaction_force_on_lag_grid(eul.astype(f64), pos, vel)
    del eul
    assert np.array_equal(near, ora.nearest)
    errs = {"rel_flow_velocity": _rel(u, ora.flow_velocity), "rel_velocity_mismatch": _rel(dv, ora.velocity_mismatch),
            "rel_forcing": _rel(f, ora.forcing)}
    ref = np.zeros(shape)
    ib_oracle.lagrangian_to_eulerian_fast(ref, f, ora.weights, ora.nearest, 2)
    ib_oracle.clear_ghost_cells_nd(ref, GS, 3)
    errs["rel_spread"] = _rel(spread, ref)
    for k, v in errs.items():
        record_property(k, v)
    _check(record_property, "rel_linf", max(errs.values()), 2e-6)


def test_sparse_forcing_update_and_flagged_reset(cuda, record_property):
    """The forcing of the fsi_512_f32 sphere (its points spread onto the 512^3 float32 grid, a thin shell
    over thousands of 1024-cell chunks): the sparse update equals the dense update bit for bit, twice, its
    increment matches float64, and sb200_clear_flagged_tiles leaves F == 0 everywhere and the flags
    cleared."""
    be = cuda
    w, g, p = _ib_setup("fsi_512_f32")
    pos = w["points"]
    shape = (3,) + tuple(v + 2 * GS for v in w["grid"])
    rng = np.random.default_rng(3)
    lag_f = be.dev(rng.uniform(-1, 1, size=pos.shape))
    d_f = _spread(be, g, p, lag_f, be.dev(pos), shape)
    del lag_f
    omega = rng.uniform(size=shape).astype(f32)
    d_w = be.dev(omega)
    plain = d_w.clone()
    prefactor = 0.37
    _call(be, "sb200_update_vorticity_from_velocity_forcing", ctypes.byref(g), be.ptr(plain), be.ptr(d_f), prefactor,
          None)
    nflags = int(be.lib.sb200_tile_flag_count(ctypes.byref(g)))
    for _ in range(2):
        got = d_w.clone()
        work = torch.zeros(nflags, dtype=torch.uint8, device="cuda")
        _call(be, "sb200_update_vorticity_from_sparse_forcing", ctypes.byref(g), be.ptr(got), be.ptr(d_f), prefactor,
              be.ptr(work), None)
        torch.cuda.synchronize()
        assert torch.equal(got, plain)
    flagged = int(work.view(torch.int32)[-4].item())
    record_property("flagged_chunks", flagged)
    assert flagged > 1000
    f_host = d_f.cpu().numpy()
    _call(be, "sb200_clear_flagged_tiles", ctypes.byref(g), be.ptr(d_f), 3, be.ptr(work), None)
    torch.cuda.synchronize()
    assert d_f.abs().max().item() == 0 and work.max().item() == 0
    got = got.cpu().numpy()
    del d_w, plain, d_f, work
    _free()
    ref = omega.astype(f64)
    st.update_vorticity_from_velocity_forcing_mpi(ref, f_host.astype(f64), prefactor, GS)
    del f_host
    w64 = omega.astype(f64)
    ref -= w64
    got = got - w64
    _check(record_property, "rel_linf", _rel(got, ref), 2e-6)


# ------------------------------------------------------------------ rod: filter and penalisation
def test_rod_filter_and_penalisation(cuda, record_property):
    """The rod workload's one-pass order-1 multiplicative filter and the boundary penalisation on its
    256 x 256 x 512 grid (x_range 1.8): bit for bit against the float32 oracle, within the bar of the
    float64 oracle, the same bits twice."""
    from sopht_mpi_b200.numeric.eulerian_grid_ops.ops import _penalise_factor_table

    be = cuda
    name = "rod_fsi_512x256x256_f32"
    wl = bench.workload_setup(name, bench.WORKLOADS[name][0])
    assert wl["sim_kw"]["filter_setting_dict"] == {"order": 1, "type": "multiplicative"}
    n, real_t = wl["grid"], wl["real_t"]
    sim_dx = real_t(wl["x_range"] / n[2])
    g = _lib.make_grid(3, real_t, GS, n, (1,) * 6)
    shape = (3,) + tuple(v + 2 * GS for v in n)
    rng = np.random.default_rng(8)
    w = rng.uniform(size=shape).astype(real_t)
    d_w = be.dev(w)
    outs = []
    for _ in range(2):
        out = torch.full_like(d_w, float("nan"))
        fb, bb = torch.zeros_like(d_w[0]), torch.zeros_like(d_w[0])
        _call(be, "sb200_laplacian_filter_order1_out_of_place", ctypes.byref(g), be.ptr(out), be.ptr(d_w), 3,
              be.ptr(fb), be.ptr(bb), None)
        outs.append(out)
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[1])
    got = outs[0].cpu().numpy()
    del outs
    same, ref = w.copy(), w.astype(f64)
    zeros = np.zeros(shape[1:], real_t)
    st.laplacian_filter_mpi(same, zeros.copy(), zeros.copy(), 1, "multiplicative", GS)
    st.laplacian_filter_mpi(ref, zeros.astype(f64), zeros.astype(f64), 1, "multiplicative", GS)
    assert np.array_equal(got, same)
    err_filter = _rel(got, ref)

    width = 2  # the simulator's penalty_zone_width

    def line(nl, t):  # FlowSimulatorOracle3D.local_x / _y / _z
        dx = t(sim_dx)
        return np.linspace(dx / 2.0 - GS * dx, nl * dx - dx / 2.0 + GS * dx, nl + 2 * GS).astype(t)

    tab = be.dev(_penalise_factor_table(real_t, width, sim_dx, GS, [line(n[0], real_t), line(n[1], real_t),
                                                                     line(n[2], real_t)]))
    outs = []
    for _ in range(2):
        out = d_w.clone()
        _call(be, "sb200_penalise_field_boundary", ctypes.byref(g), be.ptr(out), 3, width, be.ptr(tab), None)
        outs.append(out)
    torch.cuda.synchronize()
    assert torch.equal(outs[0], outs[1])
    got = outs[0].cpu().numpy()
    del outs, d_w, tab
    _free()
    same, ref = w.copy(), w.astype(f64)
    st.penalise_field_boundary_mpi(same, width, sim_dx, line(n[2], real_t), line(n[1], real_t), line(n[0], real_t),
                                   GS)
    # (the float64 run takes the float32 coordinate lines: near the faces x - x_start is a difference of
    # two numbers ~1, so recomputing the lines in float64 would change the input by several ppm of the factor)
    st.penalise_field_boundary_mpi(ref, width, f64(sim_dx), *(line(m, real_t).astype(f64) for m in n[::-1]), GS)
    assert np.array_equal(got, same)
    err_pen = _rel(got, ref)
    record_property("rel_filter", err_filter)
    record_property("rel_penalise", err_pen)
    _check(record_property, "rel_linf", max(err_filter, err_pen), 2e-6)


# ---------------------------------------------------------------------------------- reductions
def test_reductions_at_512(cuda, record_property):
    """max |sum of components| and max against numpy float64 (the same bits twice), sum of squares to
    rtol 1e-12, on the 512^3 float32 grid."""
    be = cuda
    g = _lib.make_grid(3, f32, GS, GRID_512, (1,) * 6)
    shape = (3,) + tuple(v + 2 * GS for v in GRID_512)
    f = (np.random.default_rng(12).uniform(size=shape) - 0.5).astype(f32)
    d_f = be.dev(f)
    got = {}
    for name, runs in (("sb200_max_abs_sum", 2), ("sb200_max", 2), ("sb200_sum_squares", 1)):
        vals = []
        for _ in range(runs):
            out = torch.zeros(1, dtype=torch.float64, device="cuda")
            _call(be, name, ctypes.byref(g), be.ptr(d_f), 3, be.ptr(out), None)
            vals.append(out.item())
        assert len(set(vals)) == 1, (name, vals)
        got[name] = vals[0]
    del d_f
    _free()
    inner = f[_inner(1)].astype(f64)
    del f
    want = np.abs(inner).sum(axis=0).max()
    err = abs(got["sb200_max_abs_sum"] - want) / want
    assert got["sb200_max"] == inner.max()
    sq = float(np.sum(inner * inner))
    record_property("rel_sum_squares", abs(got["sb200_sum_squares"] - sq) / sq)
    assert abs(got["sb200_sum_squares"] - sq) <= 1e-12 * sq
    _check(record_property, "rel_linf", err, 2e-6)


# ----------------------------------------------------------------------------- one whole step
def test_one_fsi_step_through_the_interactor(cuda, record_property):
    """One step of fsi_256_f32 as bench.py runs it (dt, interactor(), interactor.time_step, flow step)
    against FlowSimulatorOracle3D + VirtualBoundaryForcingOracle in float64, both starting from the same
    float32 state.  (The float64 oracle at 512^3 would need about 70 GB of host memory.)

    The velocity has a wider bound: it is the curl of psi, a difference of neighbouring values over 2 dx,
    so the float32 error of the solved psi (~5e-7 of max |psi|) comes out about four times larger
    relative to max |u|.  The curl kernel itself is within 1e-7 of float64 on the same psi
    (test_velocity_from_stream_function)."""
    from sopht_mpi_b200.simulator import PrescribedForcingGrid, RigidBodyFlowInteractionMPI, UnboundedFlowSimulator3D

    name = "fsi_256_f32"
    wl = bench.workload_setup(name, bench.WORKLOADS[name][0])
    n, u_inf = wl["grid"], wl["u_inf"]
    kw = dict(grid_size=n, x_range=wl["x_range"], kinematic_viscosity=wl["nu"], flow_type=wl["flow_type"],
              with_free_stream_flow=True)
    sim = UnboundedFlowSimulator3D(real_t=f32, **kw)
    pts, vel = wl["points"], wl["lag_vel"]

    class _Body:
        pass

    interactor = RigidBodyFlowInteractionMPI(
        mpi_construct=sim.mpi_construct, mpi_ghost_exchange_communicator=sim.mpi_ghost_exchange_communicator,
        rigid_body=_Body(), eul_grid_forcing_field=sim.eul_grid_forcing_field,
        eul_grid_velocity_field=sim.velocity_field, virtual_boundary_stiffness_coeff=wl["k"],
        virtual_boundary_damping_coeff=wl["c"], dx=sim.dx, grid_dim=3,
        forcing_grid_cls=lambda grid_dim, rigid_body: PrescribedForcingGrid(
            grid_dim, pts, velocity_field=vel, max_lag_grid_dx=wl["dx"], static=True))
    sim.vorticity_field[...] = bench.initial_vorticity(wl, sim.local_x, sim.local_y, sim.local_z)
    sim.compute_flow_velocity(free_stream_velocity=u_inf)

    ora = FlowSimulatorOracle3D(real_t=f64, fft_workers=CORES, **kw)
    for field in ("vorticity_field", "velocity_field", "stream_func_field"):
        getattr(ora, field)[...] = np.asarray(getattr(sim, field))
    area = wl["dx"] ** 2
    vbf = ib_oracle.VirtualBoundaryForcingOracle(wl["k"] * area, wl["c"] * area, 3, f64(sim.dx), f64, f64, GS,
                                                 eul_grid_coord_shift=f64(f32(sim.dx / 2)), fast=True)

    dt = ora.compute_stable_timestep(dt_prefac=0.5)
    errs = {"rel_dt": abs(float(sim.compute_stable_timestep(dt_prefac=0.5)) - dt) / dt}
    vbf.compute_interaction_force_on_eul_and_lag_grid(ora.eul_grid_forcing_field, ora.velocity_field, pts, vel)
    interactor()
    errs["rel_lag_forcing"] = _rel(interactor.global_lag_grid_forcing_field, vbf.forcing)
    vbf.time_step(dt)
    interactor.time_step(dt)
    ora.time_step(dt, free_stream_velocity=u_inf)
    sim.time_step(dt=dt, free_stream_velocity=u_inf)
    assert np.abs(ora.eul_grid_forcing_field).max() == 0
    for field in ("vorticity_field", "velocity_field", "stream_func_field"):
        errs["rel_" + field] = _rel(np.asarray(getattr(sim, field)), getattr(ora, field))
    errs["rel_position_mismatch"] = _rel(interactor.local_lag_grid_position_mismatch_field, vbf.position_mismatch)
    for k, v in errs.items():
        record_property(k, v)
    del sim, interactor
    _free()
    assert errs.pop("rel_velocity_field") <= 5e-6
    _check(record_property, "rel_linf", max(errs.values()), 2e-6)
