"""Domain decomposition and communication: the distributed backend of the path.

Replaces the reference's mpi4py layer (``sopht_mpi/utils/mpi_utils_3d.py`` /
``mpi_utils_2d.py``) with one process per GPU over ``torch.distributed``
(NCCL for device tensors, a gloo side group for small host objects).

Decomposition: slabs along the LEADING array axis (z in 3D, y in 2D), i.e.
``grid_topology = (P, 1, 1)`` / ``(P, 1)``: halo planes are contiguous in memory, so
one send/recv per direction moves whole padded planes with no pack kernel and the
face exchange already carries edge/corner ghosts.
"""
import os

import numpy as np
import torch
import torch.distributed as dist

from .device import DeviceField
from .logger import logger


class MPI:
    """Names the reference's call sites use (``MPI.MIN`` ... ``MPI.PROC_NULL``)."""

    MIN = "min"
    MAX = "max"
    SUM = "sum"
    LOR = "lor"
    LAND = "land"
    PROC_NULL = -1


_host_group = None


def init_process_group_if_needed():
    """Join the process group described by the torchrun environment (if any)."""
    if dist.is_available() and not dist.is_initialized() and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        backend = "nccl" if torch.cuda.is_available() else "gloo"
        if torch.cuda.is_available():
            torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dist.init_process_group(backend=backend)


def world_size():
    return dist.get_world_size() if dist.is_initialized() else 1


def world_rank():
    return dist.get_rank() if dist.is_initialized() else 0


def host_group():
    """gloo group for small host-side messages (scalars, rank address arrays)."""
    global _host_group
    if not dist.is_initialized():
        return None
    if _host_group is None:
        if dist.get_backend() == "gloo":
            _host_group = dist.group.WORLD
        else:
            _host_group = dist.new_group(backend="gloo")
    return _host_group


class CartGrid:
    """Cartesian communicator of the slab topology with the small part of the
    mpi4py ``Cartcomm`` interface the reference touches
    (``coords``, ``allreduce``, ``bcast``, ``reduce``, ``Get_cart_rank`` ...)."""

    def __init__(self, topology, periodic):
        self.topology = np.asarray(topology, dtype=int)
        self.periodic = bool(periodic)
        self.size = world_size()
        self.rank = world_rank()
        self.coords = np.array(np.unravel_index(self.rank, self.topology), dtype=int)

    def Get_size(self):
        return self.size

    def Get_rank(self):
        return self.rank

    def Get_cart_rank(self, coords):
        return int(np.ravel_multi_index(tuple(int(c) for c in coords), self.topology))

    def Get_coords(self, rank):
        return np.array(np.unravel_index(int(rank), self.topology), dtype=int)

    def Shift(self, dim, disp):
        out = []
        for d in (-disp, disp):
            c = self.coords.copy()
            c[dim] += d
            if 0 <= c[dim] < self.topology[dim]:
                out.append(self.Get_cart_rank(c))
            elif self.periodic:
                c[dim] %= self.topology[dim]
                out.append(self.Get_cart_rank(c))
            else:
                out.append(MPI.PROC_NULL)
        return tuple(out)

    # ---- small host collectives
    def allreduce(self, value, op=MPI.SUM):
        if self.size == 1:
            return value
        if op in (MPI.LOR, MPI.LAND):
            t = torch.tensor([1.0 if value else 0.0], dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX if op == MPI.LOR else dist.ReduceOp.MIN,
                            group=host_group())
            return bool(t.item() > 0.5)
        t = torch.tensor([float(value)], dtype=torch.float64)
        red = {MPI.MIN: dist.ReduceOp.MIN, MPI.MAX: dist.ReduceOp.MAX, MPI.SUM: dist.ReduceOp.SUM}[op]
        dist.all_reduce(t, op=red, group=host_group())
        return type(value)(t.item()) if isinstance(value, (float, np.floating)) else t.item()

    def reduce(self, value, op=MPI.SUM, root=0):
        r = self.allreduce(value, op=op)
        return r if self.rank == root else None

    def bcast(self, obj, root=0):
        if self.size == 1:
            return obj
        box = [obj]
        dist.broadcast_object_list(box, src=root, group=host_group())
        return box[0]

    def allgather(self, obj):
        if self.size == 1:
            return [obj]
        out = [None] * self.size
        dist.all_gather_object(out, obj, group=host_group())
        return out

    def Barrier(self):
        if self.size > 1:
            dist.barrier(group=host_group())

    def Abort(self):
        raise RuntimeError("Abort called on the process grid")


def compute_slab_topology(size, rank_distribution):
    """Slab version of ``MPI.Compute_dims(size, dims=rank_distribution)``
    (reference ``mpi_utils_3d.py:46-48``): 0 = free, 1 = not distributed.  All ranks
    go to the leading array axis; other free axes stay undivided."""
    dims = [int(d) for d in rank_distribution]
    topo = [1] * len(dims)
    if size == 1:
        return np.array(topo)
    fixed = int(np.prod([d for d in dims if d > 0]))
    if dims[0] != 0 or size % fixed:
        raise RuntimeError(
            f"rank_distribution {rank_distribution} cannot be realised with leading-axis slabs "
            f"on {size} ranks")
    for i, d in enumerate(dims):
        if d > 0:
            topo[i] = d
    topo[0] = size // fixed
    if any(d == 0 for d in dims[1:]):
        logger.warning(
            "rank_distribution leaves more than one axis free; this build decomposes along the "
            f"leading axis only (slabs): topology {topo}")
    if fixed != 1:
        raise RuntimeError("only leading-axis slab decompositions are supported")
    return np.array(topo)


class MPIConstruct:
    """Topology + local sizes (reference ``MPIConstruct3D`` ``mpi_utils_3d.py:7-83``,
    ``MPIConstruct2D`` ``mpi_utils_2d.py:9-84``)."""

    def __init__(self, grid_dim, global_grid_size, periodic_domain=False, real_t=np.float64,
                 rank_distribution=None):
        init_process_group_if_needed()
        self.grid_dim = grid_dim
        self.real_t = real_t
        self.periodic_domain = periodic_domain
        if rank_distribution is None:
            self.rank_distribution = [0] * grid_dim
            self.rank_distribution[-1] = 1
        else:
            self.rank_distribution = list(rank_distribution)
        if 1 not in self.rank_distribution:
            logger.warning(
                f"Rank distribution {self.rank_distribution} needs to be "
                "aligned in at least one direction for fft")
        self.grid_topology = compute_slab_topology(world_size(), self.rank_distribution)
        self.global_grid_size = np.array(global_grid_size)
        if np.any(self.global_grid_size % self.grid_topology):
            logger.error(
                "Cannot divide grid evenly to processors in x, y and/or z directions!\n"
                f"{self.global_grid_size / self.grid_topology} x {self.grid_topology} "
                f"!= {self.global_grid_size}")
            raise RuntimeError("Invalid domain decomposition")
        self.local_grid_size = (self.global_grid_size / self.grid_topology).astype(int)
        self.grid = CartGrid(self.grid_topology, periodic_domain)
        self.world = self.grid
        self.previous_grid_along = np.zeros(grid_dim).astype(int)
        self.next_grid_along = np.zeros(grid_dim).astype(int)
        for d in range(grid_dim):
            self.previous_grid_along[d], self.next_grid_along[d] = self.grid.Shift(d, 1)
        self.size = self.grid.Get_size()
        self.rank = self.grid.Get_rank()
        self.device = (torch.device("cuda", torch.cuda.current_device())
                       if torch.cuda.is_available() else torch.device("cpu"))
        logger.debug(
            f"Initializing a {grid_dim}D simulation with\n"
            f"global_grid_size : {self.global_grid_size.tolist()}\n"
            f"processes : {self.grid_topology}\n"
            f"local_grid_size : {self.local_grid_size.tolist()}\n")

    @property
    def physical_faces(self):
        """2*dim flags, array order (z_prev,z_next,y_prev,...): neighbour is PROC_NULL."""
        flags = []
        for d in range(self.grid_dim):
            flags += [self.previous_grid_along[d] == MPI.PROC_NULL,
                      self.next_grid_along[d] == MPI.PROC_NULL]
        return flags

    @property
    def substart_idx(self):
        """global index of the first local interior cell, array order."""
        return self.grid.coords * self.local_grid_size


def _tensor_of(field):
    if isinstance(field, DeviceField):
        return field.tensor, None
    if isinstance(field, torch.Tensor):
        return field, None
    host = np.asarray(field)
    return torch.from_numpy(host), host  # shares memory with the numpy array


class MPIGhostCommunicator:
    """Halo exchange (reference ``MPIGhostCommunicator3D`` ``mpi_utils_3d.py:86-1142``,
    2D ``mpi_utils_2d.py:87-420``): non-blocking init calls accumulate requests that
    ``exchange_finalise`` completes, so interior work can overlap the transfer."""

    def __init__(self, ghost_size, mpi_construct, full_exchange=True):
        if ghost_size <= 0 and not isinstance(ghost_size, int):
            raise ValueError(
                f"Ghost size {ghost_size} needs to be an integer > 0"
                "for calling ghost communication.")
        self.ghost_size = ghost_size
        self.mpi_construct = mpi_construct
        self.full_exchange = full_exchange
        self.grid_coord = np.array(mpi_construct.grid.coords)
        self.comm_requests = []  # (neighbour exchange, its pending exchange, fields) per started exchange
        # fields whose ghost planes are known to be current: (data_ptr, host-write version) of the last
        # exchange; the owner of a field drops the entry when a kernel rewrites it (``mark_stale``)
        self._fresh = {}

    # -- local periodic wrap of the undivided axes (only for periodic domains)
    def _wrap_local_axes(self, t):
        gs = self.ghost_size
        for ax in range(t.ndim - 1, 0, -1):
            lo = [slice(None)] * t.ndim
            hi = [slice(None)] * t.ndim
            src_lo = [slice(None)] * t.ndim
            src_hi = [slice(None)] * t.ndim
            lo[ax], src_lo[ax] = slice(0, gs), slice(-2 * gs, -gs)
            hi[ax], src_hi[ax] = slice(-gs, None), slice(gs, 2 * gs)
            t[tuple(lo)] = t[tuple(src_lo)].clone()
            t[tuple(hi)] = t[tuple(src_hi)].clone()

    def _exchange_init(self, fields):
        mc = self.mpi_construct
        gs = self.ghost_size
        if mc.periodic_domain:
            for t in fields:
                self._wrap_local_axes(t)
        if mc.size == 1:
            if mc.periodic_domain:
                for t in fields:
                    t[:gs] = t[-2 * gs:-gs].clone()
                    t[-gs:] = t[gs:2 * gs].clone()
            return
        from .peer import peer_halo

        # boundary planes to the neighbours (their mailboxes, or messages straight into the ghost planes)
        up, down = [t[-2 * gs:-gs] for t in fields], [t[gs:2 * gs] for t in fields]
        halo = peer_halo(mc, up[0].numel() * up[0].element_size())
        pending = halo.start(up, down, [t[:gs] for t in fields], [t[-gs:] for t in fields])
        self.comm_requests.append((halo, pending, list(fields)))

    def exchange_scalar_field_init(self, local_field):
        t, _ = _tensor_of(local_field)
        self._exchange_init([t])

    # the reference exposes the three flavours separately; with slab planes they coincide
    exchange_scalar_field_faces_init = exchange_scalar_field_init
    exchange_scalar_field_full_init = exchange_scalar_field_init

    def exchange_vector_field_init(self, local_vector_field):
        t, _ = _tensor_of(local_vector_field)
        self._exchange_init([t[c] for c in range(t.shape[0])])
        if isinstance(local_vector_field, DeviceField):
            self.mark_fresh(local_vector_field)

    def exchange_finalise(self):
        gs = self.ghost_size
        for halo, pending, fields in self.comm_requests:
            from_prev, from_next = halo.finish(pending)
            dst, src = [], []
            for c, t in enumerate(fields):
                for received, ghost in ((from_prev, t[:gs]), (from_next, t[-gs:])):
                    if received and received[c] != ghost.data_ptr():  # (not yet in the ghost plane)
                        dst.append(ghost.data_ptr())
                        src.append(received[c])
            halo.copy_blocks(dst, src, fields[0][:gs].numel() * fields[0].element_size())
        self.comm_requests = []

    # ---- ghost freshness (B200 build): lets the simulator skip an exchange of a field whose ghost
    # planes were filled since it was last written (the interactor exchanges the velocity right before
    # the flow step exchanges it again)
    @staticmethod
    def _fresh_key(field):
        t = getattr(field, "tensor", field)
        return (t.data_ptr() if isinstance(t, torch.Tensor) else id(t), getattr(field, "version", None))

    def mark_fresh(self, field):
        ptr, version = self._fresh_key(field)
        self._fresh[ptr] = version

    def mark_stale(self, field):
        self._fresh.pop(self._fresh_key(field)[0], None)

    def is_fresh(self, field):
        ptr, version = self._fresh_key(field)
        return ptr in self._fresh and self._fresh[ptr] == version and version is not None


class MPIFieldCommunicator:
    """Scatter / gather of whole fields between the master rank and the slabs
    (reference ``MPIFieldCommunicator3D`` ``mpi_utils_3d.py:1145-1306``); a test and
    IO helper, off the hot path."""

    def __init__(self, ghost_size, mpi_construct, master_rank=0):
        if ghost_size < 0 and not isinstance(ghost_size, int):
            raise ValueError(
                f"Ghost size {ghost_size} needs to be an integer >= 0"
                "for field IO communication.")
        self.ghost_size = ghost_size
        self.mpi_construct = mpi_construct
        self.master_rank = master_rank
        if ghost_size == 0:
            self.inner_idx = ...
        else:
            self.inner_idx = (slice(ghost_size, -ghost_size),) * mpi_construct.grid_dim

    def _block(self, rank):
        mc = self.mpi_construct
        coords = mc.grid.Get_coords(rank)
        return tuple(slice(int(c * n), int((c + 1) * n)) for c, n in zip(coords, mc.local_grid_size))

    def gather_local_scalar_field(self, global_field, local_field):
        mc = self.mpi_construct
        local = np.asarray(local_field[self.inner_idx])
        blocks = mc.grid.allgather(local)
        if mc.rank == self.master_rank:
            for r, b in enumerate(blocks):
                global_field[self._block(r)] = b

    def scatter_global_scalar_field(self, local_field, global_field):
        mc = self.mpi_construct
        g = mc.grid.bcast(np.asarray(global_field) if mc.rank == self.master_rank else None,
                          root=self.master_rank)
        local_field[self.inner_idx] = np.ascontiguousarray(g[self._block(mc.rank)])

    def gather_local_vector_field(self, global_vector_field, local_vector_field):
        for c in range(self.mpi_construct.grid_dim):
            self.gather_local_scalar_field(
                global_vector_field[c] if global_vector_field is not None else None,
                local_vector_field[c])

    def scatter_global_vector_field(self, local_vector_field, global_vector_field):
        for c in range(self.mpi_construct.grid_dim):
            self.scatter_global_scalar_field(
                local_vector_field[c],
                global_vector_field[c] if global_vector_field is not None else None)


class MPILagrangianFieldCommunicator:
    """Lagrangian node -> rank ownership and scatter/gather of ``(dim, N)`` fields
    (reference ``MPILagrangianFieldCommunicator3D`` ``mpi_utils_3d.py:1309-1459``,
    2D ``mpi_utils_2d.py:571-712``).  Host-side numpy: identical integer results."""

    def __init__(self, eul_grid_dx, eul_grid_coord_shift, mpi_construct, master_rank=0,
                 real_t=np.float64):
        self.grid_dim = mpi_construct.grid_dim
        self.mpi_construct = mpi_construct
        self.master_rank = master_rank
        self.rank = mpi_construct.rank
        self.eul_subblock_dx = eul_grid_dx * mpi_construct.local_grid_size
        self.eul_grid_coord_shift = eul_grid_coord_shift
        self.real_t = real_t
        topo = tuple(int(t) for t in mpi_construct.grid_topology)
        self.rank_map = np.zeros(topo, dtype=np.int32)
        for idx in np.ndindex(*topo):
            self.rank_map[idx] = mpi_construct.grid.Get_cart_rank(idx)

    def _compute_lag_nodes_rank_address(self, global_lag_positions):
        """block coordinate = ((pos - shift) / (dx * n_local)).astype(int32): truncation,
        in the dtype of the positions (reference ``mpi_utils_3d.py:1357-1384``)."""
        dim = self.grid_dim
        coords = []
        for ax in range(dim):  # array axis order; positions are x,y,z
            pos = global_lag_positions[dim - 1 - ax, ...]
            coords.append(((pos - self.eul_grid_coord_shift) / self.eul_subblock_dx[ax]).astype(np.int32))
        if any(np.any(coords[ax] >= self.mpi_construct.grid_topology[ax]) for ax in range(dim)):
            logger.error("Lagrangian node is found outside of Eulerian domain!")
            self.mpi_construct.grid.Abort()
        return self.rank_map[tuple(coords)]

    def map_lagrangian_nodes_based_on_position(self, global_lag_positions):
        # a body that did not move keeps its ownership map (same positions -> same integers): one
        # array comparison on the master instead of the mapping and its broadcast
        if self.mpi_construct.size == 1 and getattr(self, "_last_positions", None) is not None:
            if (self._last_positions.shape == np.shape(global_lag_positions)
                    and np.array_equal(self._last_positions, global_lag_positions)):
                return
        if self.mpi_construct.size == 1:
            self._last_positions = np.array(global_lag_positions, copy=True)
        if self.rank == self.master_rank:
            if global_lag_positions.shape[0] != self.grid_dim:
                logger.error(f"global_lag_positions needs to be shape ({self.grid_dim}, ...)")
                self.mpi_construct.grid.Abort()
            rank_address = self._compute_lag_nodes_rank_address(global_lag_positions)
        else:
            rank_address = None
        self.rank_address = self.mpi_construct.grid.bcast(rank_address, root=self.master_rank)
        # ownership lists are derived once per mapping (vectorised: the reference's python-level
        # ``set(rank_address)`` costs milliseconds for 1e4-1e5 points)
        owned = self.rank_address == self.rank
        self.local_nodes_idx = np.where(owned)
        self._local_idx = self.local_nodes_idx[0]
        self.local_num_lag_nodes = int(self._local_idx.size)
        self._all_local = self.local_num_lag_nodes == self.rank_address.shape[-1]
        self.slave_ranks_containing_lag_nodes = (
            set(np.unique(self.rank_address).tolist()) - set([self.master_rank]))

    def _idx_of(self, rank):
        return self._local_idx if rank == self.rank else np.where(self.rank_address == rank)[0]

    def scatter_global_field(self, local_lag_field, global_lag_field):
        mc = self.mpi_construct
        if mc.size == 1:
            if self._all_local:
                local_lag_field[...] = global_lag_field
            else:
                local_lag_field[...] = global_lag_field[:, self._local_idx]
            return
        g = mc.grid.bcast(np.asarray(global_lag_field) if self.rank == self.master_rank else None,
                          root=self.master_rank)
        idx = self._local_idx
        if idx.size or self.rank == self.master_rank:
            local_lag_field[...] = g[:, idx]

    def gather_local_field(self, global_lag_field, local_lag_field):
        mc = self.mpi_construct
        if mc.size == 1:
            if self._all_local:
                global_lag_field[...] = local_lag_field
            else:
                global_lag_field[:, self._local_idx] = local_lag_field
            return
        parts = mc.grid.allgather(np.asarray(local_lag_field))
        if self.rank == self.master_rank:
            for r, part in enumerate(parts):
                idx = self._idx_of(r)
                if idx.size:
                    global_lag_field[:, idx] = part.reshape(self.grid_dim, idx.size)
