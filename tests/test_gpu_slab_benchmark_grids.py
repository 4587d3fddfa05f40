"""The z-slab step of the strong-scaled benchmark against the single-GPU step, at the grids bench.py times.

`bench.py --gpus N` runs its workloads on N z-slabs.  At the benchmarked sizes the slab path takes launch
geometry that the small slab tests never reach: at 512^3 on 8 ranks the doubled x axis has 513 kx bins,
cut into kx slabs of 68 bins padded to 72 lines, the last of which holds only 37 real bins; the x pass
at n = 512 writes blocks for 8 destinations; the 1024-point y and z passes run on those slabs; the slab
faces z = 128 ... 320 cut the sphere, so the sparse forcing update, the IB interaction and the spreading
all see slab faces inside the body.

The slab solve runs the same three stages as the single-GPU solve, and the other slab kernels compute
each cell from the same inputs as on the whole grid, so most of the slab path must equal the
single-GPU path bit for bit.  That bar is stronger than a tolerance, needs no float64 reference at
512^3, and composes with test_gpu_benchmark_grids.py, which ties the single-GPU kernels to float64 at
these grids.  Only the spreading (floating-point atomics) and the ghost sum that follows it are held
to the float64 bar of that module instead.

Part 1 drives P virtual ranks on one GPU through the C ABI: every rank has its own handles and slab
allocations of nzl + 2 gs planes, and the test moves blocks and ghost planes between the ranks with
torch copies, as the product's exchanges do.  Part 2 runs the real slab step of bench.py as P processes
on one GPU (tests/dist_bench_step_worker.py) against a single-process run of the same steps."""
import ctypes
import json
import math
import os

import numpy as np
import pytest
import torch

import bench
from harness import _call, _free, _ib_setup, _spread, cuda, run_ranks, slab_poisson_solve, slabs  # noqa: F401
from oracle import ib as ib_oracle
from sopht_mpi_b200 import _lib

pytestmark = pytest.mark.gpu

f32, f64 = np.float32, np.float64
GS = 2  # the simulator's ghost size
GRID_512, GRID_ROD, GRID_256 = (bench.WORKLOADS[k][0] for k in ("fsi_512_f32", "rod_fsi_512x256x256_f32",
                                                                 "vortex_ring_256_f64"))
PS = (2, 4, 8)
# (grid, real_t, x_range): fsi_512_f32; the rod grid (sphere_vbf_512x256x256_f32 is the same shape with
# x_range 1.0); vortex_ring_256_f64
GRIDS = {"512-f32": (GRID_512, f32, 1.0), "256x256x512-f32-rod": (GRID_ROD, f32, 1.8),
         "256-f64": (GRID_256, f64, 1.0)}
IB_WORKLOADS = {"512-f32": "fsi_512_f32", "256x256x512-f32-rod": "rod_fsi_512x256x256_f32"}


def _torch_t(real_t):
    return torch.float32 if real_t == f32 else torch.float64


def _rows(glob, r, nzl):
    """the global planes that are rank r's interior planes"""
    return glob[..., GS + r * nzl:GS + r * nzl + nzl, :, :]


def _interior_planes(slab):
    return slab[..., GS:-GS, :, :]


def _slab_grid(real_t, n, nranks, r):
    """the sb200_grid_t of rank r: physical z faces only on the first and the last rank"""
    return _lib.make_grid(3, real_t, GS, (n[0] // nranks, n[1], n[2]), (int(r == 0), int(r == nranks - 1), 1, 1, 1, 1))


def _mismatch(got, want):
    """0.0 when the bits agree, otherwise the relative L-inf difference (inf when NaNs differ)"""
    if torch.equal(got, want):
        return 0.0
    d = (got.double() - want.double()).abs().max().item()
    return d / max(want.double().abs().max().item(), 1e-300) if math.isfinite(d) else math.inf


def _coefficients(n, real_t, x_range):
    """the prefactors of the flow step at a stable dt of the benchmark (CFL 0.1, dt_prefac 0.5, |u| ~ 1)"""
    dx = real_t(x_range / n[2])
    dt = 0.5 * 0.1 * float(dx)
    return float(real_t(dt / (2 * dx))), float(real_t(1e-3 * dt / dx / dx))


def _report(record_property, results):
    """results: {P: relative difference (0.0 = bit-identical)}; every P is reported before any assert"""
    for nranks, err in results.items():
        record_property(f"P{nranks}", "bit-identical" if err == 0.0 else err)
    bad = {p: e for p, e in results.items() if e != 0.0}
    assert not bad, f"slab results differ from the single-GPU results: {bad}"


# ------------------------------------------------------------------------------- Poisson
def _single_solve(be, n, real_t, x_range, rhs, ncomp):
    sol = torch.full_like(rhs, 7.0)
    h = ctypes.c_void_p()
    _call(be, "sb200_poisson_create", ctypes.byref(h), 3, _lib.dtype_code(real_t), *n, GS, x_range, 0, 1, 1, None)
    try:
        _call(be, "sb200_poisson_solve", h, be.ptr(sol), be.ptr(rhs), ncomp, None)
        torch.cuda.synchronize()
    finally:
        be.lib.sb200_poisson_destroy(h)
    return sol


def _ghosts_untouched(out):
    inner = torch.zeros(out.shape[-3:], dtype=torch.bool, device=out.device)
    inner[GS:-GS, GS:-GS, GS:-GS] = True
    return bool((out[..., ~inner] == 7.0).all())


@pytest.mark.parametrize("grid", list(GRIDS))
def test_slab_poisson_solve_like_the_product(cuda, grid, record_property):
    """Per component with ncomp = 1, as the product calls the slab stages: every rank's interior equals
    the single-GPU vector solve of the same padded rhs bit for bit, the ghost cells of the solution keep
    their sentinel, one call with ncomp = 3 gives the same bits, and a scalar solve equals the single-GPU
    scalar solve."""
    be = cuda
    n, real_t, x_range = GRIDS[grid]
    t = _torch_t(real_t)
    gen = torch.Generator(device="cuda").manual_seed(sum(n) + 11)
    rhs = torch.rand((3,) + tuple(v + 2 * GS for v in n), generator=gen, dtype=t, device="cuda")
    ref = _single_solve(be, n, real_t, x_range, rhs, 3)
    ref1 = _single_solve(be, n, real_t, x_range, rhs[1], 1)
    results, problems = {}, []
    for nranks in PS:
        nzl = n[0] // nranks
        outs = slab_poisson_solve(be, n, real_t, nranks, rhs, 3, backend=1, x_range=x_range, per_component=True)
        err = max(_mismatch(_interior_planes(o)[..., GS:-GS, GS:-GS], _rows(ref, r, nzl)[..., GS:-GS, GS:-GS])
                  for r, o in enumerate(outs))
        if not all(_ghosts_untouched(o) for o in outs):
            problems.append(f"P{nranks}: a ghost cell of the solution was written")
        batched = slab_poisson_solve(be, n, real_t, nranks, rhs, 3, backend=1, x_range=x_range)
        if not all(torch.equal(a, b) for a, b in zip(outs, batched)):
            problems.append(f"P{nranks}: ncomp = 3 differs from three ncomp = 1 calls")
        del outs, batched
        scalar = slab_poisson_solve(be, n, real_t, nranks, rhs[1], 1, backend=1, x_range=x_range, per_component=True)
        err1 = max(_mismatch(_interior_planes(o)[..., GS:-GS, GS:-GS], _rows(ref1, r, nzl)[..., GS:-GS, GS:-GS])
                   for r, o in enumerate(scalar))
        if not all(_ghosts_untouched(o) for o in scalar):
            problems.append(f"P{nranks}: a ghost cell of the scalar solution was written")
        del scalar
        results[nranks] = max(err, err1)
    del rhs, ref, ref1
    _free()
    assert not problems, problems
    _report(record_property, results)


# ------------------------------------------------------------------------ fused vorticity update
@pytest.mark.parametrize("grid", list(GRIDS))
def test_slab_fused_vorticity_update(cuda, grid, record_property):
    """The product's calls on slab allocations (_fused_vorticity_update): the interior range
    [reach, mz - reach) with reach = 2 + gs, then the two face ranges, with lo = 0 on rank 0 and
    hi = mz on rank P-1.  Every slab's interior planes equal the rows of the whole-grid
    sb200_vorticity_rhs_fused_3d bit for bit."""
    be = cuda
    n, real_t, x_range = GRIDS[grid]
    t = _torch_t(real_t)
    p, d = _coefficients(n, real_t, x_range)
    gen = torch.Generator(device="cuda").manual_seed(sum(n) + 12)
    shape = (3,) + tuple(v + 2 * GS for v in n)
    w = torch.rand(shape, generator=gen, dtype=t, device="cuda")
    u = torch.rand(shape, generator=gen, dtype=t, device="cuda") - 0.5
    g = _lib.make_grid(3, real_t, GS, n, (1,) * 6)
    whole = torch.full_like(w, float("nan"))
    _call(be, "sb200_vorticity_rhs_fused_3d", ctypes.byref(g), be.ptr(whole), be.ptr(w), be.ptr(u), None, p, d, None)
    torch.cuda.synchronize()
    results = {}
    reach = 2 + GS
    for nranks in PS:
        nzl = n[0] // nranks
        ws, us = slabs(w, nranks, GS), slabs(u, nranks, GS)
        err = 0.0
        for r in range(nranks):
            gr = _slab_grid(real_t, n, nranks, r)
            out = torch.full_like(ws[r], float("nan"))
            mz = out.shape[1]
            lo = 0 if r == 0 else reach
            hi = mz if r == nranks - 1 else mz - reach
            for z0, z1 in ((lo, hi), (0, lo), (hi, mz)):
                if z1 > z0:
                    _call(be, "sb200_vorticity_rhs_fused_3d_range", ctypes.byref(gr), be.ptr(out), be.ptr(ws[r]),
                          be.ptr(us[r]), p, d, z0, z1, None)
            torch.cuda.synchronize()
            err = max(err, _mismatch(_interior_planes(out), _rows(whole, r, nzl)))
            del out
        results[nranks] = err
        del ws, us
    del w, u, whole
    _free()
    _report(record_property, results)


# ------------------------------------------------------------------ velocity from stream function
@pytest.mark.parametrize("grid", list(GRIDS))
def test_slab_velocity_from_stream_function(cuda, grid, record_property):
    """sb200_velocity_from_stream_function with a free stream and the forcing reset on each slab (psi's
    ghost planes from the neighbours): every slab's interior planes equal the whole-grid velocity bit for
    bit, the maximum over the ranks of the per-rank max |u| equals the whole-grid scalar exactly, and the
    forcing is zero on every slab afterwards."""
    be = cuda
    n, real_t, x_range = GRIDS[grid]
    t = _torch_t(real_t)
    prefactor = float(real_t(0.5 / real_t(x_range / n[2])))
    fs = (ctypes.c_double * 3)(1.0, 0.5, -0.25)
    gen = torch.Generator(device="cuda").manual_seed(sum(n) + 13)
    shape = (3,) + tuple(v + 2 * GS for v in n)
    psi = torch.rand(shape, generator=gen, dtype=t, device="cuda")
    u0 = torch.rand(shape, generator=gen, dtype=t, device="cuda")
    g = _lib.make_grid(3, real_t, GS, n, (1,) * 6)
    whole = u0.clone()
    forcing = torch.rand(shape, generator=gen, dtype=t, device="cuda")
    vmax = torch.zeros(1, dtype=torch.float64, device="cuda")
    _call(be, "sb200_velocity_from_stream_function", ctypes.byref(g), be.ptr(whole), be.ptr(psi), prefactor, fs,
          be.ptr(forcing), be.ptr(vmax), None)
    torch.cuda.synchronize()
    assert forcing.abs().max().item() == 0
    del forcing
    vmax = vmax.item()
    results, problems = {}, []
    for nranks in PS:
        nzl = n[0] // nranks
        psis, us = slabs(psi, nranks, GS), slabs(u0, nranks, GS)
        err, vmaxes = 0.0, []
        for r in range(nranks):
            gr = _slab_grid(real_t, n, nranks, r)
            f = torch.rand(us[r].shape, generator=gen, dtype=t, device="cuda") + 0.5
            vm = torch.zeros(1, dtype=torch.float64, device="cuda")
            _call(be, "sb200_velocity_from_stream_function", ctypes.byref(gr), be.ptr(us[r]), be.ptr(psis[r]),
                  prefactor, fs, be.ptr(f), be.ptr(vm), None)
            torch.cuda.synchronize()
            err = max(err, _mismatch(_interior_planes(us[r]), _rows(whole, r, nzl)))
            vmaxes.append(vm.item())
            if f.abs().max().item() != 0:
                problems.append(f"P{nranks} rank {r}: forcing not reset")
            del f
        if max(vmaxes) != vmax:
            problems.append(f"P{nranks}: max over ranks of max |u| {max(vmaxes)!r} != whole grid {vmax!r}")
        results[nranks] = err
        del psis, us
    del psi, u0, whole
    _free()
    assert not problems, problems
    _report(record_property, results)


# ------------------------------------------------------------------ sparse forcing update
def _body_forcing(be, name):
    """the body's spread forcing on the whole grid, built as test_gpu_benchmark_grids.py builds it"""
    w, g, p = _ib_setup(name)
    pos = w["points"]
    shape = (3,) + tuple(v + 2 * GS for v in w["grid"])
    rng = np.random.default_rng(3)
    lag_f = be.dev(rng.uniform(-1, 1, size=pos.shape))
    return w, g, _spread(be, g, p, lag_f, be.dev(pos), shape)


@pytest.mark.parametrize("grid", list(IB_WORKLOADS))
def test_slab_sparse_forcing_update(cuda, grid, record_property):
    """The body's spread forcing F on slabs, F's ghost planes filled from the neighbours as
    ctx.exchange_vector(f) does before the update: every slab's vorticity equals the whole-grid sparse
    update bit for bit; after sb200_clear_flagged_tiles F is zero on every slab, ghost planes included,
    and the flag buffer is zeroed."""
    be = cuda
    name = IB_WORKLOADS[grid]
    w, g, d_f = _body_forcing(be, name)
    n, real_t = w["grid"], w["real_t"]
    prefactor, _ = _coefficients(n, real_t, w["x_range"])
    gen = torch.Generator(device="cuda").manual_seed(sum(n) + 14)
    omega = torch.rand(d_f.shape, generator=gen, dtype=torch.float32, device="cuda")
    whole = omega.clone()
    work = torch.zeros(int(be.lib.sb200_tile_flag_count(ctypes.byref(g))), dtype=torch.uint8, device="cuda")
    _call(be, "sb200_update_vorticity_from_sparse_forcing", ctypes.byref(g), be.ptr(whole), be.ptr(d_f), prefactor,
          be.ptr(work), None)
    torch.cuda.synchronize()
    assert not torch.equal(whole, omega)
    del work
    results, problems = {}, []
    zlo, zhi = (float(w["points"][2].min()) / w["dx"], float(w["points"][2].max()) / w["dx"])
    record_property("body_planes", f"{zlo:.0f}-{zhi:.0f}")
    for nranks in PS:
        nzl = n[0] // nranks
        ws, fs = slabs(omega, nranks, GS), slabs(d_f, nranks, GS)
        err = 0.0
        for r in range(nranks):
            gr = _slab_grid(real_t, n, nranks, r)
            flags = torch.zeros(int(be.lib.sb200_tile_flag_count(ctypes.byref(gr))), dtype=torch.uint8,
                                device="cuda")
            _call(be, "sb200_update_vorticity_from_sparse_forcing", ctypes.byref(gr), be.ptr(ws[r]), be.ptr(fs[r]),
                  prefactor, be.ptr(flags), None)
            _call(be, "sb200_clear_flagged_tiles", ctypes.byref(gr), be.ptr(fs[r]), 3, be.ptr(flags), None)
            torch.cuda.synchronize()
            err = max(err, _mismatch(_interior_planes(ws[r]), _rows(whole, r, nzl)))
            if fs[r].abs().max().item() != 0:
                problems.append(f"P{nranks} rank {r}: F not zero after the reset")
            if flags.max().item() != 0:
                problems.append(f"P{nranks} rank {r}: flags not cleared")
        results[nranks] = err
        del ws, fs
    del omega, whole, d_f
    _free()
    assert not problems, problems
    _report(record_property, results)


# ------------------------------------------------------------------- immersed boundary
def _slab_params(p, z0):
    """the IB parameters of a slab whose first interior plane is global plane z0"""
    q = _lib.IBParams.from_buffer_copy(p)
    q.substart_xyz[2] = z0
    return q


def _f64_spread(be, w, p, lag_f, shape):
    """float64 scatter of the same forcing with the oracle's nearest indices and cosine weights, ghost
    cells cleared (on the device: the 512^3 float64 field is 3.3 GB)"""
    pos = w["points"]
    near, support = ib_oracle.support_and_nearest_index(pos, p.dx, p.coord_shift, 2, (0, 0, 0), GS)
    weights = ib_oracle.cosine_weights(support, p.dx, f64)  # (4, 4, 4, N), array axes (z, y, x)
    del support
    mz, my, mx = shape[1:]
    off = np.arange(-1, 3)
    z = near[2][None, None, None, :] + off[:, None, None, None]
    y = near[1][None, None, None, :] + off[None, :, None, None]
    x = near[0][None, None, None, :] + off[None, None, :, None]
    flat = torch.from_numpy(((z * my + y) * mx + x).reshape(-1)).cuda()
    wt = torch.from_numpy(weights.reshape(-1)).cuda()
    del weights
    ref = torch.zeros(shape, dtype=torch.float64, device="cuda")
    f = lag_f.double()
    npts = f.shape[1]
    for c in range(3):
        vals = (wt.view(-1, npts) * f[c][None, :]).reshape(-1)
        ref[c].view(-1).index_add_(0, flat, vals)
    ref[:, :GS], ref[:, -GS:] = 0, 0
    ref[:, :, :GS], ref[:, :, -GS:] = 0, 0
    ref[:, :, :, :GS], ref[:, :, :, -GS:] = 0, 0
    return ref


@pytest.mark.parametrize("grid", list(IB_WORKLOADS))
def test_slab_ib_interaction_and_spreading(cuda, grid, record_property):
    """The benchmark's body on slabs:
    - sb200_ib_rank_address gives the integers of oracle.ib.lag_nodes_rank_address;
    - sb200_ib_interact_owned on each slab (velocity ghost planes from the neighbours), summed over the
      ranks as the all-reduce of virtual_boundary_forcing.py does, equals the single-domain interaction
      bit for bit (the weights come from the global floor index, evaluated in double), and every rank
      writes zeros for the points it does not own;
    - sb200_ib_spread_owned on each slab, then the ghost sum (sb200_ghost_sum_add_z with the neighbours'
      ghost planes, sb200_clear_ghost_cells), matches the float64 spread within the bar of
      test_gpu_benchmark_grids.py (relative to max |F|; the spread uses atomics)."""
    be = cuda
    name = IB_WORKLOADS[grid]
    w, g, p = _ib_setup(name)
    pos, vel = w["points"], w["lag_vel"]
    n, npts = w["grid"], pos.shape[1]
    dx32 = f32(w["dx"])
    shape = (3,) + tuple(v + 2 * GS for v in n)
    rng = np.random.default_rng(npts)
    gen = torch.Generator(device="cuda").manual_seed(npts)
    eul = torch.rand(shape, generator=gen, dtype=torch.float32, device="cuda") - 0.5
    dpos = 0.1 * w["dx"] * rng.standard_normal(pos.shape)
    d_pos, d_vel, d_dpos = be.dev(pos), be.dev(vel), be.dev(dpos)

    def interact(grid_t, params, field, owner=None, rank=0):
        u, dv, f = (torch.full((3, npts), float("nan"), dtype=torch.float64, device="cuda") for _ in range(3))
        _call(be, "sb200_ib_interact_owned", ctypes.byref(grid_t), ctypes.byref(params), npts, be.ptr(field),
              be.ptr(d_pos), be.ptr(d_vel), be.ptr(d_dpos), None, None, be.ptr(u), be.ptr(dv), be.ptr(f),
              be.ptr(owner), rank, None)
        return torch.stack((u, dv, f))

    single = interact(g, p, eul)
    spread_single = _spread(be, g, p, single[2], d_pos, shape)
    ref = _f64_spread(be, w, p, single[2], shape)
    scale = ref.abs().max().item()
    err_single = ((spread_single.double() - ref).abs().max().item()) / scale
    record_property("rel_spread_single_gpu", err_single)
    results, problems, spread_errs = {}, [], {}
    for nranks in PS:
        nzl = n[0] // nranks
        local = (nzl, n[1], n[2])
        sub_dx = (ctypes.c_double * 3)(*(float(v) for v in dx32 * np.asarray(local)))
        topo = (ctypes.c_int32 * 3)(nranks, 1, 1)
        owner = torch.full((npts,), -1, dtype=torch.int32, device="cuda")
        flag = torch.zeros(1, dtype=torch.int32, device="cuda")
        _call(be, "sb200_ib_rank_address", _lib.F64, 3, npts, be.ptr(d_pos), float(f32(dx32 / 2)), sub_dx, topo,
              be.ptr(owner), be.ptr(flag), None)
        want = ib_oracle.lag_nodes_rank_address(pos, dx32, f32(dx32 / 2), local, (nranks, 1, 1))
        own = owner.cpu().numpy()
        if not np.array_equal(own, want) or flag.item() != 0:
            problems.append(f"P{nranks}: rank address differs from the oracle's")
        owners = sorted(set(own.tolist()))
        record_property(f"P{nranks}_owning_ranks", ",".join(map(str, owners)))
        us = slabs(eul, nranks, GS)
        total = torch.zeros_like(single)
        for r in range(nranks):
            part = interact(_slab_grid(f32, n, nranks, r), _slab_params(p, r * nzl), us[r], owner, r)
            if not bool((part[:, :, owner != r] == 0).all()):
                problems.append(f"P{nranks} rank {r}: non-zero values at points it does not own")
            total += part
        err = _mismatch(total, single)
        # spreading, then the ghost sum over the slab faces
        fs = []
        for r in range(nranks):
            f = torch.zeros_like(us[r])
            _call(be, "sb200_ib_spread_owned", ctypes.byref(_slab_grid(f32, n, nranks, r)),
                  ctypes.byref(_slab_params(p, r * nzl)), npts,
                  be.ptr(f), be.ptr(single[2]), be.ptr(d_pos), be.ptr(owner), r, None)
            fs.append(f)
        from_prev = [fs[r - 1][:, -GS:].contiguous() if r > 0 else None for r in range(nranks)]
        from_next = [fs[r + 1][:, :GS].contiguous() if r < nranks - 1 else None for r in range(nranks)]
        serr = 0.0
        for r in range(nranks):
            gr = _slab_grid(f32, n, nranks, r)
            _call(be, "sb200_ghost_sum_add_z", ctypes.byref(gr), be.ptr(fs[r]), 3, be.ptr(from_prev[r]),
                  be.ptr(from_next[r]), None)
            _call(be, "sb200_clear_ghost_cells", ctypes.byref(gr), be.ptr(fs[r]), 3, None)
            torch.cuda.synchronize()
            serr = max(serr, (_interior_planes(fs[r]).double() - _rows(ref, r, nzl)).abs().max().item() / scale)
            if fs[r][:, :GS].abs().max().item() != 0 or fs[r][:, -GS:].abs().max().item() != 0:
                problems.append(f"P{nranks} rank {r}: ghost planes of the spread forcing not cleared")
        spread_errs[nranks] = serr
        record_property(f"P{nranks}_rel_spread", serr)
        results[nranks] = err
        del us, fs, from_prev, from_next, total
    del eul, single, spread_single, ref, d_pos, d_vel, d_dpos
    _free()
    assert not problems, problems
    assert max(spread_errs.values()) <= 2e-6, spread_errs
    _report(record_property, results)


# ------------------------------------------------- part 2: the real slab step as processes on one GPU
STEP_CASES = [("fsi_512_f32", 2), ("fsi_512_f32", 4), ("fsi_512_f32", 8), ("rod_fsi_512x256x256_f32", 4),
              ("vortex_ring_256_f64", 4)]
# whole-step bars of test_one_fsi_step_through_the_interactor (float32 error of a step against float64).
# Two single-GPU runs of these steps already differ, by the order of the spreading's atomic adds: at
# 512^3 by ~5e-6 of max |u| (the forcing's curl makes |omega| ~ 900 next to the sphere, where u peaks at
# ~6.4), which is the velocity bar itself.  So each quantity is held to the larger of its bar and twice
# the difference between two single-GPU runs, measured in the same test.
STEP_BARS = {"vorticity_field": 2e-6, "stream_func_field": 2e-6, "lag2_forcing": 2e-6, "dt2": 2e-6,
             "velocity_field": 5e-6}


def _step_env(name, path):
    return {"SB200_BENCH_STEP_WORKLOAD": name, "SB200_BENCH_STEP_DIR": str(path)}


def _bench_step_single_gpu_runs(name, path):
    """the reference run, then a second single-GPU run that compares itself with it (single.json)"""
    for _ in range(2):
        run_ranks("dist_bench_step_worker.py", 1, "DIST_BENCH_STEP_REFERENCE_OK", where="one_gpu",
                  env=_step_env(name, path))


def _check_bench_step(name, nranks, path, record_property):
    """every rank: bit-identical up to the first spreading (the fields of the initial
    compute_flow_velocity, step 1's dt, Lagrangian forcing and mismatches); after it within the
    whole-step bars of the single-GPU step, or within twice the difference of two single-GPU runs where
    that is larger; without a body bit-identical throughout"""
    body = bench.WORKLOADS[name][2] is not None
    ranks = []
    for r in range(nranks):
        with open(os.path.join(path, f"rank{r}.json")) as fh:
            ranks.append(json.load(fh))
    with open(os.path.join(path, "single.json")) as fh:
        single = json.load(fh)
    exact = ["dt1"] + [f"init_{f}" for f in ("vorticity_field", "velocity_field", "stream_func_field")]
    if body:
        exact += ["lag1_forcing", "lag1_velocity_mismatch", "lag1_position_mismatch"]
    else:
        exact += [k for k in ranks[0]["identical"]]
    differ = sorted({k for res in ranks + [single] for k in exact if not res["identical"][k]})
    worst = {k: max(res["rel"][k] for res in ranks) for k in ranks[0]["rel"]}
    for k, v in sorted(worst.items()):
        identical = all(res["identical"][f"final_{k}" if k.endswith("_field") else k] for res in ranks)
        record_property(k, "bit-identical" if identical else v)
        record_property("single_gpu_rerun_" + k, single["rel"][k])
    assert not differ, f"differ from the single-GPU step: {differ}"
    if body:
        over = {k: (worst[k], bar, single["rel"][k]) for k, bar in STEP_BARS.items()
                if not worst[k] <= max(bar, 2 * single["rel"][k])}
        assert not over, over


@pytest.mark.parametrize("name,nranks", STEP_CASES, ids=[f"{n}-P{p}" for n, p in STEP_CASES])
def test_bench_step_with_ranks_on_one_gpu(name, nranks, tmp_path, record_property):
    """Two steps of bench.py's step sequence as `nranks` processes on one GPU (gloo for the collectives,
    the push transport of the peer-memory exchanges) against the same steps in one process."""
    try:
        _bench_step_single_gpu_runs(name, tmp_path)
        run_ranks("dist_bench_step_worker.py", nranks, "DIST_BENCH_STEP_WORKER_OK", where="one_gpu",
                  env=dict(_step_env(name, tmp_path), SB200_PEER_WAIT_S="300"))
        _check_bench_step(name, nranks, tmp_path, record_property)
    finally:
        for f in tmp_path.iterdir():  # (about 5 GB at 512^3)
            f.unlink()


@pytest.mark.parametrize("name,nranks", STEP_CASES, ids=[f"{n}-P{p}" for n, p in STEP_CASES])
def test_bench_step_on_gpus(name, nranks, tmp_path, record_property):
    """The same steps with one GPU per rank under torch.distributed.run: NCCL and the default transport
    of the exchanges (the copy-engine transport on 2 and 4 ranks)."""
    if not torch.cuda.is_available() or torch.cuda.device_count() < nranks:
        pytest.skip(f"needs {nranks} GPUs")  # before the single-GPU runs
    try:
        _bench_step_single_gpu_runs(name, tmp_path)
        run_ranks("dist_bench_step_worker.py", nranks, "DIST_BENCH_STEP_WORKER_OK", where="gpus",
                  env=_step_env(name, tmp_path))
        _check_bench_step(name, nranks, tmp_path, record_property)
    finally:
        for f in tmp_path.iterdir():
            f.unlink()
