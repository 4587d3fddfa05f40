"""Unbounded Poisson solvers with the reference's class names and methods
(``sopht_mpi/numeric/eulerian_grid_ops/poisson_solver_3d/UnboundedPoissonSolverMPI3D.py:14-187``,
``poisson_solver_2d/UnboundedPoissonSolverMPI2D.py:12-153``)."""
import ctypes

import numpy as np

from ... import _lib
from ...utils.device import Staged, current_stream_ptr, dptr


def _is_pow2(n):
    return n > 0 and (n & (n - 1)) == 0


# Smallest 3D grid (cells) whose cuFFT solve runs on z-slabs when distributed; smaller grids stay replicated.
# A tiny solve is bound by launches and latency, so the two exchanges per component of the slab pipeline
# (six per vector solve) cost more than one all-gather there.  PROVISIONAL: the crossover has not been
# measured on several GPUs.  2^18 cells (64^3) keeps the small grids the replicated path serves, e.g.
# (6P, 20, 36) on up to 8 ranks (<= 34560 cells), replicated; DESIGN section 5 gives the reasoning and
# tools/bench_slab_cufft.py is the measurement to set it from.
_SLAB_CUFFT_MIN_CELLS = 1 << 18


class _UnboundedPoissonSolver:
    def __init__(self, dim, grid_size, mpi_construct, ghost_size, x_range, real_t, backend):
        self.lib = _lib.load()
        self.dim = dim
        self.mpi_construct = mpi_construct
        self.ghost_size = ghost_size
        self.x_range = x_range
        self.real_t = real_t
        gs3 = [1] * (3 - dim) + [int(g) for g in grid_size]
        self.grid_size_z, self.grid_size_y, self.grid_size_x = gs3
        self.y_range = x_range * (self.grid_size_y / self.grid_size_x)
        if dim == 3:
            self.z_range = x_range * (self.grid_size_z / self.grid_size_x)
        self.dx = real_t(x_range / self.grid_size_x)
        self.device = mpi_construct.device
        if self.device.type != "cuda":
            raise _lib.SophtB200Error("the Poisson solver needs a CUDA device (no CPU fallback)")
        if backend == "auto":
            pow2 = all(_is_pow2(int(g)) for g in grid_size)
            big_enough = gs3[2] >= 16 and gs3[1] >= 8 and (dim == 2 or gs3[0] >= 8)
            small_enough = gs3[2] <= 4096 and gs3[1] <= 2048 and gs3[0] <= 2048
            backend = ("fft" if (pow2 and big_enough and small_enough
                                 and _fft_backend_available(self.lib)) else "cufft")
        # Distributed solve.  The slab pipeline (transposes over NVLink, see _solve_slabs) covers 3D grids
        # split into leading-axis slabs at least 2 ghost_size thick: power-of-two grids on 2, 4 or 8 ranks
        # through the in-kernel transforms, every other grid through the cuFFT backend's z-slab mode on any
        # rank count, once the grid reaches _SLAB_CUFFT_MIN_CELLS.  Everything else the reference's
        # mpi4py-fft path accepts (2D decompositions such as BASELINE configs[0]'s `-np 2` cylinder, small
        # grids) runs REPLICATED: the slab interiors are all-gathered over NCCL, every GPU solves the whole
        # (then small) domain with the single-rank solver and keeps its own slab.
        self.replicated = False
        if mpi_construct.size > 1:
            size = mpi_construct.size
            lead = gs3[3 - dim]
            slab_ok = (dim == 3 and lead % size == 0 and lead // size >= 2 * ghost_size
                       and ((backend == "fft" and size in (2, 4, 8))
                            or (backend == "cufft" and gs3[0] * gs3[1] * gs3[2] >= _SLAB_CUFFT_MIN_CELLS)))
            if not slab_ok:
                self.replicated = True
                if backend == "fft" and not all(_is_pow2(int(g)) for g in grid_size):
                    backend = "cufft"
        self.backend = backend
        self._slab_bufs = []
        self._slab_events = None
        self._handle = ctypes.c_void_p()
        lib_rank, lib_size = (0, 1) if self.replicated else (mpi_construct.rank, mpi_construct.size)
        _lib.check(self.lib, self.lib.sb200_poisson_create(
            ctypes.byref(self._handle), dim, _lib.dtype_code(real_t), gs3[0], gs3[1], gs3[2],
            ghost_size, float(x_range), lib_rank, lib_size,
            1 if backend == "fft" else 0, current_stream_ptr(self.device)))

    def __del__(self):
        try:
            if getattr(self, "_handle", None):
                self.lib.sb200_poisson_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    def close(self):
        """Release the exchange buffers shared with the other ranks (collective: call it on every rank
        before the process group goes away)."""
        peer = getattr(self, "_peer", None)
        if peer is not None:
            peer.close(collective=True)
            self._peer = None
            self._slab_bufs = []

    @property
    def workspace_bytes(self):
        return int(self.lib.sb200_poisson_workspace_bytes(self._handle))

    STAGE_NAMES = ("x_r2c", "y_forward", "z_fused_forward_green_inverse", "y_inverse", "x_c2r")

    SLAB_STAGE_NAMES = ("local_x_r2c", "all_to_all_z_to_kx", "y_forward_z_fused_y_inverse",
                        "all_to_all_kx_to_z", "local_x_c2r")

    def set_profiling(self, enable=True):
        """Record CUDA events around the launches of a solve (single rank: the five kernels, inside
        the library; z-slabs: the three local stages and the two all-to-alls, on the torch stream)."""
        if self.mpi_construct.size == 1:
            _lib.check(self.lib, self.lib.sb200_poisson_set_profiling(self._handle, int(bool(enable))))
        self._slab_events = [] if enable else None

    def last_stage_ms(self):
        """Device time (ms) of each stage of the last profiled solve."""
        if self.mpi_construct.size == 1:
            out = (ctypes.c_float * 5)()
            _lib.check(self.lib, self.lib.sb200_poisson_last_stage_ms(self._handle, out, 5))
            return dict(zip(self.STAGE_NAMES, (float(v) for v in out)))
        ev = self._slab_events
        ev[-1].synchronize()
        return {name: ev[i].elapsed_time(ev[i + 1]) for i, name in enumerate(self.SLAB_STAGE_NAMES)}

    def _solve(self, solution, rhs, ncomp):
        st = Staged(self.device)
        s, r = st(solution, out=True), st(rhs)
        stream = current_stream_ptr(self.device)
        if self.mpi_construct.size == 1:
            _lib.check(self.lib, self.lib.sb200_poisson_solve(self._handle, dptr(s), dptr(r), ncomp, stream))
        elif self.replicated:
            self._solve_replicated(s, r, ncomp, stream)
        else:
            self._solve_slabs(s, r, ncomp, stream)
        st.finish()

    def _solve_replicated(self, s, r, ncomp, stream):
        """all-gather the slab interiors -> whole-domain solve on every GPU -> keep the own slab"""
        import torch
        import torch.distributed as dist

        mc, gs, dim = self.mpi_construct, self.ghost_size, self.dim
        size, rank = mc.size, mc.rank
        inner = (slice(None),) + (slice(gs, -gs),) * dim
        r_v = r if r.dim() == dim + 1 else r.unsqueeze(0)
        s_v = s if s.dim() == dim + 1 else s.unsqueeze(0)
        local = r_v[inner].contiguous()                    # (ncomp, n_lead / P, ...)
        if getattr(self, "_rep_bufs", None) is None or self._rep_bufs[0].shape[1] != ncomp:
            glob_shape = (ncomp,) + tuple(int(g) + 2 * gs for g in
                                          (self.grid_size_z, self.grid_size_y, self.grid_size_x)[3 - dim:])
            self._rep_bufs = (torch.empty((size,) + tuple(local.shape), dtype=local.dtype, device=local.device),
                              torch.zeros(glob_shape, dtype=local.dtype, device=local.device),
                              torch.zeros(glob_shape, dtype=local.dtype, device=local.device))
        gathered, g_rhs, g_sol = self._rep_bufs
        dist.all_gather_into_tensor(gathered.view(-1), local.view(-1))  # (flat: the form every backend takes)
        n_lead = local.shape[1]
        # (P, ncomp, n_lead_local, ...) -> (ncomp, P * n_lead_local, ...): slabs stack along the leading axis
        g_rhs[inner].copy_(gathered.transpose(0, 1).reshape((ncomp, size * n_lead) + tuple(local.shape[2:])))
        _lib.check(self.lib, self.lib.sb200_poisson_solve(self._handle, dptr(g_sol), dptr(g_rhs), ncomp, stream))
        own = (slice(None), slice(gs + rank * n_lead, gs + (rank + 1) * n_lead)) + (slice(gs, -gs),) * (dim - 1)
        s_v[inner].copy_(g_sol[own])

    def _solve_slabs(self, s, r, ncomp, stream):
        """z-slab solve: local x pass, all-to-all (z-slabs <-> kx-slabs, on the x-pass output: the
        smallest array of the pipeline), y / fused z / inverse y passes on the kx-slab, all-to-all
        back, local inverse x pass.  The transposes replace mpi4py-fft's and the domain-doubling
        copies (reference ``UnboundedPoissonSolverMPI3D.py:190-382``, ``fft_mpi_3d.py:27-48``).

        The components are software-pipelined: each has its own pair of exchange buffers, the
        kernels run on the caller's stream and the NCCL all-to-alls on a second stream, so the
        exchange of component c overlaps the transforms of component c +- 1 (events order them).
        With profiling on, the stages run back to back instead so that each can be timed."""
        import torch
        import torch.distributed as dist

        lib, h = self.lib, self._handle
        if not self._slab_bufs:
            from ...utils.peer import PeerExchange

            nfloat = int(lib.sb200_poisson_slab_buffer_bytes(h, 1)) // 4
            # per component a (send, recv) pair, visible to the other ranks through CUDA IPC
            self._peer = PeerExchange(6, nfloat, self.device, self.mpi_construct.rank, self.mpi_construct.size)
            self.exchange_mode = self._peer.mode
            self._slab_bufs = [(self._peer.local[2 * c], self._peer.local[2 * c + 1]) for c in range(3)]
            # high priority: the NCCL kernels must get SMs while a transform kernel still has blocks queued
            self._comm_stream = torch.cuda.Stream(device=self.device, priority=-1)
        main = torch.cuda.current_stream(self.device)
        comm = self._comm_stream
        vol = r.numel() // ncomp if r.dim() == 4 else r.numel()
        esize = r.element_size()
        rp, sp = dptr(r), dptr(s)

        def comp_ptr(base, c):
            return ctypes.c_void_p(base.value + c * vol * esize)

        events = getattr(self, "_slab_events", None)
        if events is not None:  # serial, timed stages (profiling)
            events.clear()

            def mark():
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                events.append(ev)

            mark()
            for c in range(ncomp):
                _lib.check(lib, lib.sb200_poisson_slab_forward(h, comp_ptr(rp, c), 1, dptr(self._slab_bufs[c][0]),
                                                               stream))
            mark()
            for c in range(ncomp):
                self._peer.exchange(2 * c + 1, 2 * c)
            mark()
            for c in range(ncomp):
                _lib.check(lib, lib.sb200_poisson_slab_spectral(h, dptr(self._slab_bufs[c][1]), 1, stream))
            mark()
            for c in range(ncomp):
                self._peer.exchange(2 * c, 2 * c + 1)
            mark()
            for c in range(ncomp):
                _lib.check(lib, lib.sb200_poisson_slab_backward(h, comp_ptr(sp, c), 1,
                                                                dptr(self._slab_bufs[c][0]), stream))
            mark()
            return

        def after(ev_stream):
            ev = torch.cuda.Event()
            ev.record(ev_stream)
            return ev

        # the exchange buffers may still be in use by the previous solve's last transfers
        comm.wait_stream(main)
        fwd, a2a1, spec, a2a2 = [], [], [], []
        for c in range(ncomp):
            send, _ = self._slab_bufs[c]
            _lib.check(lib, lib.sb200_poisson_slab_forward(h, comp_ptr(rp, c), 1, dptr(send), stream))
            fwd.append(after(main))
        for c in range(ncomp):
            send, recv = self._slab_bufs[c]
            with torch.cuda.stream(comm):
                comm.wait_event(fwd[c])
                self._peer.exchange(2 * c + 1, 2 * c)
                a2a1.append(after(comm))
        for c in range(ncomp):
            send, recv = self._slab_bufs[c]
            main.wait_event(a2a1[c])
            _lib.check(lib, lib.sb200_poisson_slab_spectral(h, dptr(recv), 1, stream))
            spec.append(after(main))
            with torch.cuda.stream(comm):
                comm.wait_event(spec[c])
                self._peer.exchange(2 * c, 2 * c + 1)
                a2a2.append(after(comm))
        for c in range(ncomp):
            send, _ = self._slab_bufs[c]
            main.wait_event(a2a2[c])
            _lib.check(lib, lib.sb200_poisson_slab_backward(h, comp_ptr(sp, c), 1, dptr(send), stream))

    def solve(self, solution_field, rhs_field):
        """-del^2(solution_field) = rhs_field on the unbounded domain; padded local
        fields, only interiors are read / written."""
        self._solve(solution_field, rhs_field, 1)


_FFT_AVAILABLE = None


def _fft_backend_available(lib):
    return bool(lib.sb200_poisson_fft_available())


class UnboundedPoissonSolverMPI3D(_UnboundedPoissonSolver):
    def __init__(self, grid_size_z, grid_size_y, grid_size_x, mpi_construct, ghost_size,
                 x_range=1.0, real_t=np.float64, backend="auto"):
        super().__init__(3, (grid_size_z, grid_size_y, grid_size_x), mpi_construct, ghost_size,
                         x_range, real_t, backend)

    def vector_field_solve(self, solution_vector_field, rhs_vector_field):
        """three component solves (reference :169-187), batched in one call"""
        self._solve(solution_vector_field, rhs_vector_field, 3)


class UnboundedPoissonSolverMPI2D(_UnboundedPoissonSolver):
    def __init__(self, grid_size_y, grid_size_x, mpi_construct, ghost_size, x_range=1.0,
                 real_t=np.float64, backend="auto"):
        super().__init__(2, (grid_size_y, grid_size_x), mpi_construct, ghost_size, x_range, real_t,
                         backend)
