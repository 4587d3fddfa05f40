"""Eulerian <-> Lagrangian grid communicators.

Mirrors ``sopht_mpi/numeric/immersed_boundary_ops/EulerianLagrangianGridCommunicatorMPI3D.py:7-113``
(and the 2D twin).  The hot path used by the virtual-boundary forcing goes through
the fused warp-per-point kernels of ``libsophtb200`` (``interact`` / ``spread``);
the reference's five granular kernel attributes are kept for API compatibility and
run on the device as well.
"""
import ctypes

import numpy as np
import torch

from ... import _lib
from ...utils.device import Staged, current_stream_ptr, dptr, torch_dtype


class MPIGhostSumCommunicator:
    """Ghost-sum for slab decompositions (reference ``MPIGhostSumCommunicator3D``
    ``...MPI3D.py:592-792``): ghost slabs go to the leading-axis neighbours and are
    added to their first / last interior layers; then every ghost cell is zeroed."""

    def __init__(self, ghost_size, mpi_construct):
        if ghost_size < 0 and not isinstance(ghost_size, int):
            raise ValueError(
                f"Ghost size {ghost_size} needs to be an integer >= 0 for field communication.")
        self.ghost_size = ghost_size
        self.mpi_construct = mpi_construct
        self.lib = _lib.load()
        self.grid = _lib.make_grid(mpi_construct.grid_dim, mpi_construct.real_t, ghost_size,
                                   mpi_construct.local_grid_size, mpi_construct.physical_faces)
        self._bufs = {}

    def ghost_sum(self, local_field):
        mc = self.mpi_construct
        dim = mc.grid_dim
        st = Staged(mc.device)
        f = st(local_field, out=True)
        ncomp = 1 if f.ndim == dim else f.shape[0]
        gs = self.ghost_size
        stream = current_stream_ptr(mc.device)
        if mc.size > 1:
            comps = [f] if ncomp == 1 else [f[c] for c in range(ncomp)]
            key = (ncomp, f.dtype)
            if key not in self._bufs:
                shape = (ncomp, gs) + tuple(comps[0].shape[1:])
                self._bufs[key] = (torch.zeros(shape, dtype=f.dtype, device=f.device),
                                   torch.zeros(shape, dtype=f.dtype, device=f.device))
            recv_prev, recv_next = self._bufs[key]
            from ...utils.peer import peer_halo

            up, down = [t[-gs:] for t in comps], [t[:gs] for t in comps]
            halo = peer_halo(mc, up[0].numel() * up[0].element_size())
            # the add kernel reads the received slabs where they are (mailbox or receive buffer)
            from_prev, from_next = halo.finish(halo.start(up, down, list(recv_prev), list(recv_next)))
            _lib.check(self.lib, self.lib.sb200_ghost_sum_add_z(
                ctypes.byref(self.grid), dptr(f), ncomp,
                ctypes.c_void_p(from_prev[0]) if from_prev else None,
                ctypes.c_void_p(from_next[0]) if from_next else None, stream))
        _lib.check(self.lib, self.lib.sb200_clear_ghost_cells(ctypes.byref(self.grid), dptr(f), ncomp,
                                                             stream))
        st.finish()

    def clear_ghost_cells(self, field):
        st = Staged(self.mpi_construct.device)
        f = st(field, out=True)
        ncomp = 1 if f.ndim == self.mpi_construct.grid_dim else f.shape[0]
        _lib.check(self.lib, self.lib.sb200_clear_ghost_cells(
            ctypes.byref(self.grid), dptr(f), ncomp, current_stream_ptr(self.mpi_construct.device)))
        st.finish()


class _EulerianLagrangianGridCommunicatorMPI:
    def __init__(self, grid_dim, dx, eul_grid_coord_shift, interp_kernel_width, real_t, mpi_construct,
                 ghost_size, n_components=1, interp_kernel_type="cosine"):
        if ghost_size < interp_kernel_width:
            raise ValueError(
                f"ghost size ({ghost_size}) needs to be >= interp kernel width "
                f"({interp_kernel_width})")
        assert n_components == 1 or n_components == grid_dim, \
            "invalid number of components for interpolation!"
        if interp_kernel_type not in ("cosine", "peskin"):
            raise ValueError(
                "Invalid interpolation kernel type. Currently supported types are"
                "'cosine' and 'peskin'.")
        assert interp_kernel_width == 2, \
            "Interpolation kernel inconsistent with interpolation kernel width!"
        self.lib = _lib.load()
        self.grid_dim = grid_dim
        self.dx = dx
        self.eul_grid_coord_shift = eul_grid_coord_shift
        self.interp_kernel_width = interp_kernel_width
        self.real_t = real_t
        self.mpi_construct = mpi_construct
        self.ghost_size = ghost_size
        self.n_components = n_components
        self.interp_kernel_type = interp_kernel_type
        self.device = mpi_construct.device
        self.mpi_ghost_sum_comm = MPIGhostSumCommunicator(ghost_size=ghost_size,
                                                          mpi_construct=mpi_construct)
        self.mpi_substart_idx = np.flip(mpi_construct.grid.coords * mpi_construct.local_grid_size)
        self.mpi_local_substart_coord_shift = self.mpi_substart_idx - ghost_size
        self.grid = _lib.make_grid(grid_dim, real_t, ghost_size, mpi_construct.local_grid_size,
                                   mpi_construct.physical_faces)
        self.eulerian_grid_ghost_sum = self.mpi_ghost_sum_comm.ghost_sum

    # ---- fused device path -------------------------------------------------
    def ib_params(self, lag_dtype, stiffness=0.0, damping=0.0):
        p = _lib.IBParams()
        p.lag_dtype = _lib.dtype_code(lag_dtype)
        p.kernel_type = 0 if self.interp_kernel_type == "cosine" else 1
        p.width = int(self.interp_kernel_width)
        sub = [int(v) for v in self.mpi_substart_idx] + [0] * (3 - self.grid_dim)
        for i in range(3):
            p.substart_xyz[i] = sub[i]
        p.dx = float(self.dx)
        p.coord_shift = float(self.eul_grid_coord_shift)
        p.stiffness = float(stiffness)
        p.damping = float(damping)
        return p

    def interact(self, params, n, eul_velocity, pos, vel, dpos, nearest, weights, flow_vel, dvel, force):
        """steps 1-5 of ``compute_interaction_force_on_lag_grid`` in one launch"""
        _lib.check(self.lib, self.lib.sb200_ib_interact_lag(
            ctypes.byref(self.grid), ctypes.byref(params), int(n), dptr(eul_velocity), dptr(pos),
            dptr(vel), dptr(dpos), dptr(nearest), dptr(weights), dptr(flow_vel), dptr(dvel), dptr(force),
            current_stream_ptr(self.device)))

    def spread(self, params, n, eul_forcing, lag_forcing, pos):
        _lib.check(self.lib, self.lib.sb200_ib_spread(
            ctypes.byref(self.grid), ctypes.byref(params), int(n), dptr(eul_forcing), dptr(lag_forcing),
            dptr(pos), current_stream_ptr(self.device)))

    # ---- the reference's granular kernels (device tensors, torch plumbing) --
    def _offsets(self):
        w = self.interp_kernel_width
        return torch.arange(-w + 1, w + 1, device=self.device)

    def local_eulerian_grid_support_of_lagrangian_grid_kernel(
            self, local_eul_grid_support_of_lag_grid, nearest_eul_grid_index_to_lag_grid, lag_positions):
        st = Staged(self.device)
        sup = st(local_eul_grid_support_of_lag_grid, out=True)
        near = st(nearest_eul_grid_index_to_lag_grid, out=True)
        pos = st(lag_positions)
        dim = self.grid_dim
        shift = torch.as_tensor(np.ascontiguousarray(self.mpi_local_substart_coord_shift),
                                device=self.device).reshape(dim, 1)
        ct = torch.promote_types(pos.dtype, torch_dtype(self.real_t))
        dx = torch.tensor(float(self.dx), dtype=ct, device=self.device)
        a = pos.to(ct) - float(self.eul_grid_coord_shift)
        # numpy floor_divide semantics (fmod based)
        mod = torch.fmod(a, dx)
        div = (a - mod) / dx
        neg = (mod != 0) & ((dx < 0) != (mod < 0))
        div = torch.where(neg, div - 1, div)
        fl = torch.floor(div)
        fl = torch.where(div - fl > 0.5, fl + 1, fl)
        near.copy_(fl.to(torch.int64) - shift)
        off = self._offsets()
        k = 2 * self.interp_kernel_width
        n = pos.shape[1]
        for d in range(dim):
            shape = [1] * dim + [1]
            shape[dim - 1 - d] = k  # component d varies along array axis dim-1-d
            o = off.reshape(shape)
            val = ((near[d].reshape([1] * dim + [n]) + o + shift[d]).to(torch.float64) * float(self.dx)
                   + float(self.eul_grid_coord_shift) - pos[d].to(torch.float64).reshape([1] * dim + [n]))
            sup[d].copy_(val.expand(sup[d].shape).to(sup.dtype))
        st.finish()

    def interpolation_weights_kernel(self, interp_weights, local_eul_grid_support_of_lag_grid):
        st = Staged(self.device)
        w, sup = st(interp_weights, out=True), st(local_eul_grid_support_of_lag_grid, out=True)
        dim = self.grid_dim
        rt = np.dtype(self.real_t).type
        if self.interp_kernel_type == "cosine":
            sup.div_(float(self.dx))
            res = torch.full_like(sup[0], float(rt((0.25 / float(self.dx)) ** dim)))
            for d in range(dim):
                res = res * (1.0 + torch.cos(float(rt(0.5 * np.pi)) * sup[d]))
        else:
            sup.copy_(torch.abs(sup) / float(self.dx))
            res = torch.full_like(sup[0], (0.125 / float(self.dx)) ** dim)
            for d in range(dim):
                r = sup[d]
                a = (r < 1.0) * (3.0 - 2 * r + torch.sqrt(torch.abs(1 + 4 * r - 4 * r ** 2)))
                b = ((r >= 1.0) & (r < 2.0)) * (5.0 - 2 * r - torch.sqrt(torch.abs(-7 + 12 * r - 4 * r ** 2)))
                res = res * (a + b)
        w.copy_(res.to(w.dtype))
        st.finish()

    def _window_index(self, near):
        dim = self.grid_dim
        off = self._offsets()
        k = 2 * self.interp_kernel_width
        n = near.shape[1]
        idx = []
        for ax in range(dim):  # array axis order
            d = dim - 1 - ax
            shape = [1] * dim + [1]
            shape[ax] = k
            idx.append((near[d].reshape([1] * dim + [n]) + off.reshape(shape)).expand([k] * dim + [n]))
        return tuple(idx)

    def eulerian_to_lagrangian_grid_interpolation_kernel(
            self, lag_grid_field, eul_grid_field, interp_weights, nearest_eul_grid_index_to_lag_grid):
        st = Staged(self.device)
        lag = st(lag_grid_field, out=True)
        eul, w, near = st(eul_grid_field), st(interp_weights), st(nearest_eul_grid_index_to_lag_grid)
        idx = self._window_index(near)
        dim = self.grid_dim
        dxp = float(np.dtype(self.real_t).type(self.dx) ** dim)
        sum_axes = tuple(range(dim))
        if self.n_components == 1:
            lag.copy_(((eul[idx].to(torch.float64) * w.to(torch.float64)).sum(sum_axes) * dxp).to(lag.dtype))
        else:
            for c in range(dim):
                lag[c].copy_(((eul[c][idx].to(torch.float64) * w.to(torch.float64)).sum(sum_axes)
                              * dxp).to(lag.dtype))
        st.finish()

    def lagrangian_to_eulerian_grid_interpolation_kernel_without_ghost_sum(
            self, eul_grid_field, lag_grid_field, interp_weights, nearest_eul_grid_index_to_lag_grid):
        st = Staged(self.device)
        eul = st(eul_grid_field, out=True)
        lag, w, near = st(lag_grid_field), st(interp_weights), st(nearest_eul_grid_index_to_lag_grid)
        idx = self._window_index(near)
        if self.n_components == 1:
            eul.index_put_(idx, (lag * w).to(eul.dtype), accumulate=True)
        else:
            for c in range(self.grid_dim):
                eul[c].index_put_(idx, (lag[c] * w).to(eul.dtype), accumulate=True)
        st.finish()

    def lagrangian_to_eulerian_grid_interpolation_kernel(
            self, eul_grid_field, lag_grid_field, interp_weights, nearest_eul_grid_index_to_lag_grid):
        self.lagrangian_to_eulerian_grid_interpolation_kernel_without_ghost_sum(
            eul_grid_field, lag_grid_field, interp_weights, nearest_eul_grid_index_to_lag_grid)
        self.eulerian_grid_ghost_sum(local_field=eul_grid_field)


class EulerianLagrangianGridCommunicatorMPI3D(_EulerianLagrangianGridCommunicatorMPI):
    def __init__(self, dx, eul_grid_coord_shift, interp_kernel_width, real_t, mpi_construct, ghost_size,
                 n_components=1, interp_kernel_type="cosine"):
        super().__init__(3, dx, eul_grid_coord_shift, interp_kernel_width, real_t, mpi_construct,
                         ghost_size, n_components, interp_kernel_type)


class EulerianLagrangianGridCommunicatorMPI2D(_EulerianLagrangianGridCommunicatorMPI):
    def __init__(self, dx, eul_grid_coord_shift, interp_kernel_width, real_t, mpi_construct, ghost_size,
                 n_components=1, interp_kernel_type="cosine"):
        super().__init__(2, dx, eul_grid_coord_shift, interp_kernel_width, real_t, mpi_construct,
                         ghost_size, n_components, interp_kernel_type)
