"""Exchanges over NVLink peer memory (one process per GPU, one node): the all-to-all of the slab Poisson
solve (``PeerExchange``) and the z-neighbour exchange of halo planes and ghost-sum slabs (``PeerHalo``).

Every rank allocates its exchange buffers (plain device allocations of ``libsophtb200``), publishes
their CUDA IPC handles and opens the handles of the ranks it sends to WHILE ITS OWN DEVICE IS CURRENT, so
the mappings live in its compute context (``_IpcBuffers``, which also owns the teardown).  A push is then
ONE small kernel (``sb200_peer_push_blocks``) whose thread blocks store every destination block straight
into the destination rank's buffer, all peers concurrently through the NVSwitch.  "All blocks have
landed" is signalled through peer memory too: the last thread block of every destination raises an epoch
flag in the destination's memory, and a one-warp kernel on the destination's stream waits for the flags
(bounded spin), so no collective sits on the critical path.

The all-to-all replaces the MPI ``Alltoallw`` inside mpi4py-fft's transposes (reference
``poisson_solver_3d/fft_mpi_3d.py:27-48``).  It uses the copy engines (one ``cudaMemcpyPeerAsync`` per
destination on the stream + a one-element all-reduce as the barrier) when at most 4 ranks each have a GPU
of their own, the push kernel otherwise.  Without CUDA IPC (different nodes, no peer access, CPU tensors)
the all-to-all is a ``torch.distributed`` collective and the neighbour exchange point-to-point messages.
"""
import ctypes

import torch
import torch.distributed as dist

from .. import _lib
from .comm import host_group
from .device import current_stream_ptr
from .logger import logger


class _RawDeviceArray:
    """``__cuda_array_interface__`` view of a raw device allocation (so torch can alias it)"""

    def __init__(self, ptr, count, typestr):
        self.__cuda_array_interface__ = {"shape": (int(count),), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2}


def _on_every_rank(ok):
    """host collective: whether ``ok`` holds on every rank"""
    flag = torch.tensor([1.0 if ok else 0.0], dtype=torch.float64)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=host_group())
    return flag.item() > 0.5


class _IpcBuffers:
    """Device allocations of this rank that other ranks map through CUDA IPC, and this rank's mappings of
    theirs.  No allocation may be freed while a peer still maps it, which fixes the order of ``close``."""

    def __init__(self, device):
        self.device = device
        self.lib = _lib.load() if device.type == "cuda" else None
        self._raw = []     # own allocations
        self._opened = []  # mappings of other ranks' allocations

    def alloc(self, nbytes):
        """a zeroed allocation (``sb200_peer_alloc`` synchronises the device before it returns, so a peer's
        first flag cannot be wiped by a fill still in flight); returns its address"""
        ptr = ctypes.c_void_p()
        _lib.check(self.lib, self.lib.sb200_peer_alloc(int(nbytes), ctypes.byref(ptr)))
        self._raw.append(ptr.value)
        return ptr.value

    def map_peers(self, peers):
        """Collective: export the handles of every allocation, all-gather them with the device index of every
        rank on the host group, and open those of the ranks in ``peers``.  Returns ``{rank: [address of each
        allocation]}`` (this rank's own addresses for itself) and the list of device indices."""
        lib = self.lib
        mine = []
        for p in self._raw:
            handle = ctypes.create_string_buffer(64)
            _lib.check(lib, lib.sb200_ipc_export(ctypes.c_void_p(p), handle))
            mine.append(handle.raw)
        device = self.device.index if self.device.index is not None else torch.cuda.current_device()
        gathered = [None] * dist.get_world_size()
        dist.all_gather_object(gathered, (mine, device), group=host_group())
        addresses = {}
        for q in peers:
            if q == dist.get_rank():
                addresses[q] = list(self._raw)
                continue
            addresses[q] = []
            for raw in gathered[q][0]:
                p = ctypes.c_void_p()
                _lib.check(lib, lib.sb200_ipc_open(ctypes.create_string_buffer(raw, 64), ctypes.byref(p)))
                self._opened.append(p.value)
                addresses[q].append(p.value)
        return addresses, [g[1] for g in gathered]

    def close(self, collective=True):
        """Unmap the peers' allocations, then free the own ones.  With ``collective`` (call it on every rank)
        a barrier separates the two; without it a peer may still map the own allocations, so they are left
        to process exit."""
        if not self._raw:
            return
        torch.cuda.synchronize(self.device)
        for p in self._opened:
            self.lib.sb200_ipc_close(ctypes.c_void_p(p))
        self._opened = []
        if not (collective and dist.is_initialized()):
            return
        dist.barrier(group=host_group())
        for p in self._raw:
            self.lib.sb200_peer_free(ctypes.c_void_p(p))
        self._raw = []


class PeerExchange:
    def __init__(self, n_buffers, n_float32, device, rank, nranks):
        self.rank, self.nranks, self.device = rank, nranks, device
        self.n_buffers, self.n_float32 = n_buffers, int(n_float32)
        # thread blocks per destination: ~32 blocks of 512 threads saturate one NVLink port pair
        # (tools/ubench/peer_copy.py: 8 -> 364, 16 -> 630, 32 -> 658 GB/s); with P - 1 destinations in
        # flight the egress limit is shared, so fewer blocks per destination leave more SMs to the
        # transform kernels the exchange overlaps
        self.blocks_per_peer = max(4, -(-40 // max(nranks - 1, 1)))
        self._ipc = _IpcBuffers(device)
        self._lib = self._ipc.lib
        self.peer_ptr = None    # [rank][buffer] -> base address of that rank's buffer
        self.peer_flag_ptr = None
        self._plans = {}
        self._epoch = [0] * n_buffers
        use_ipc = nranks > 1 and device.type == "cuda"
        if use_ipc:
            def shared(count, typestr):
                return torch.as_tensor(_RawDeviceArray(self._ipc.alloc(4 * count), count, typestr), device=device)

            # zero-initialised (the padding bins of the last kx block are never written)
            self.local = [shared(n_float32, "<f4") for _ in range(n_buffers)]
            # epoch flags [buffer][source rank] (written by the peers)
            self.flags = shared(n_buffers * nranks, "<i4").view(n_buffers, nranks)
        else:
            self.local = [torch.zeros(n_float32, dtype=torch.float32, device=device) for _ in range(n_buffers)]
            self.flags = torch.zeros((n_buffers, max(nranks, 1)), dtype=torch.int32, device=device)
        self._flag = torch.zeros(1, dtype=torch.float32, device=device)
        self._done = torch.zeros((n_buffers, 8), dtype=torch.int32, device=device)  # arrival counters
        self._err = torch.zeros(1, dtype=torch.int32, device=device)
        if use_ipc:
            ok = False
            try:
                self._map_peers()
                ok = True
            except Exception as exc:  # pragma: no cover - depends on the node
                logger.warning(f"CUDA IPC peer mapping unavailable ({type(exc).__name__}: {exc}); "
                               "the transposes use NCCL all-to-all")
            if not _on_every_rank(ok):
                self.peer_ptr = None

    # ------------------------------------------------------------------ set-up
    def _map_peers(self):
        addresses, self._peer_dev = self._ipc.map_peers(range(self.nranks))
        self._dev = self._peer_dev[self.rank]
        # measured on the 512^3 step (profiles/r02_exchange_transports.txt): inside the component pipeline
        # the copy engines win on 2 and 4 ranks (few, large copies; no SM or load/store-path interference with
        # the transform kernels the exchange overlaps), the push kernel on 8 (seven destinations at once).
        # Ranks that share a device push: copies between two contexts of one device are not what the copy
        # engines are for.  The device list is the same on every rank, and so is the choice, which matters
        # because the two transports complete differently (all-reduce against peer flags).
        own_devices = len(set(self._peer_dev)) == self.nranks
        self.transport = "copy" if self.nranks <= 4 and own_devices else "push"
        self.peer_ptr = [addresses[q][:-1] for q in range(self.nranks)]
        self.peer_flag_ptr = [addresses[q][-1] for q in range(self.nranks)]
        if self.transport == "copy":
            lib = self._lib
            for q in range(self.nranks):
                if q != self.rank:
                    # copy engines: without the reverse mapping the driver stages the copy through the
                    # host (25 GB/s instead of ~640 GB/s, profiles/r01_peer_copy.txt)
                    _lib.check(lib, lib.sb200_enable_peer_access(self._dev, self._peer_dev[q]))
                    _lib.check(lib, lib.sb200_enable_peer_access(self._peer_dev[q], self._dev))

    def close(self, collective=True):
        """Release the buffers shared with the other ranks (``collective``: see ``_IpcBuffers.close``)."""
        self.peer_ptr = None
        self._ipc.close(collective)
        if collective:
            self.local, self.flags = [], None

    def __del__(self):
        try:
            self._ipc.close(collective=False)
        except Exception:
            pass

    @property
    def mode(self):
        if self.peer_ptr is None:
            return "nccl all-to-all"
        return "cuda-ipc push kernel" if self.transport == "push" else "cuda-ipc peer copies"

    # ------------------------------------------------------------------ the exchange
    def exchange(self, dst, src):
        """Block q of this rank's buffer `src` -> block `rank` of rank q's buffer `dst`, for every q
        (buffers are addressed by their index in ``self.local``).  Runs on the current stream."""
        nranks, rank = self.nranks, self.rank
        s_blocks = self.local[src].chunk(nranks)
        if self.peer_ptr is None:
            d_blocks = self.local[dst].chunk(nranks)
            d_blocks[rank].copy_(s_blocks[rank])
            empty = self.local[dst][:0]
            dist.all_to_all([empty if q == rank else d_blocks[q] for q in range(nranks)],
                            [empty if q == rank else s_blocks[q] for q in range(nranks)])
            return
        lib = self._lib
        stream = current_stream_ptr(self.device)
        plan = self._plans.get((dst, src))
        if plan is None:  # pointer tables of this (dst, src) pair, built once
            order = [(rank + k) % nranks for k in range(nranks)]  # local block first, then the ring
            nbytes = s_blocks[0].numel() * 4
            dptr = (ctypes.c_void_p * nranks)(*[self.peer_ptr[q][dst] + rank * nbytes for q in order])
            ddev = (ctypes.c_int * nranks)(*[self._peer_dev[q] for q in order])
            sptr = (ctypes.c_void_p * nranks)(*[s_blocks[q].data_ptr() for q in order])
            # where to signal on each destination: its flags[dst][this rank]
            fptr = (ctypes.c_void_p * nranks)(*[self.peer_flag_ptr[q] + 4 * (dst * nranks + rank) for q in order])
            plan = self._plans[(dst, src)] = (dptr, ddev, sptr, nbytes, fptr)
        dptr, ddev, sptr, nbytes, fptr = plan
        if self.transport == "push":
            self._epoch[dst] += 1
            epoch = self._epoch[dst]
            _lib.check(lib, lib.sb200_peer_push_blocks(
                nranks, dptr, sptr, nbytes, self.blocks_per_peer, fptr, epoch,
                ctypes.c_void_p(self._done[dst].data_ptr()), stream))
            _lib.check(lib, lib.sb200_peer_wait_flags(
                ctypes.c_void_p(self.flags[dst].data_ptr()), nranks, epoch, ctypes.c_void_p(self._err.data_ptr()),
                stream))
            return
        _lib.check(lib, lib.sb200_peer_copy_blocks(nranks, dptr, ddev, sptr, self._dev, nbytes, stream))
        # all ranks' copies precede their all-reduce in stream order: past this point every block of
        # `dst` has landed here, and every rank has finished reading the `src` blocks it was sent
        dist.all_reduce(self._flag)

    def check(self):
        """raise if a wait ever timed out (synchronises)"""
        if int(self._err.item()) != 0:
            raise _lib.SophtB200Error("peer exchange: a rank did not deliver its blocks in time")


class PeerHalo:
    """Neighbour exchange of contiguous plane blocks (halo planes, ghost-sum slabs): ``start`` sends,
    ``finish`` waits and says where the received blocks are.

    Every rank owns a MAILBOX (raw device allocation, CUDA IPC) of ``4 slots x 2 directions x capacity``
    bytes plus epoch flags, and maps the mailboxes of its two z neighbours.  On that path ``start`` is ONE
    small kernel (``sb200_peer_push_blocks``) that stores this rank's boundary planes into the neighbours'
    mailboxes over NVLink and raises their flags, and ``finish`` a one-warp kernel per direction on the
    receiving stream.  All launches go through the C ABI (~10 us of host time per exchange against
    ~150-200 us for an NCCL ``batch_isend_irecv`` group, which made the slab steps host bound:
    profiles/r02_trace_*).  Blocks the mailboxes cannot take (no CUDA IPC, host tensors, not 16-byte
    granular, too large, too many exchanges in flight) go as point-to-point messages instead.

    Mailbox exchanges are numbered identically on all ranks (SPMD order); exchange e uses slot e % 4 and at
    most TWO exchanges may be in flight (started, not yet finished) at a time.  Before a rank pushes
    exchange x it has waited for every exchange <= x - 2, in particular for its neighbour's push of x - 2,
    and that neighbour had unpacked every exchange <= x - 4 before issuing it (stream order): slot x % 4 is
    free.  Replaces the ``Isend / Irecv`` pairs of the reference's ``MPIGhostCommunicator`` /
    ``MPIGhostSumCommunicator`` (``sopht_mpi/utils/mpi_utils_3d.py:275-740``,
    ``numeric/immersed_boundary_ops/EulerianLagrangianGridCommunicatorMPI3D.py``).
    """

    MAX_BLOCKS = 4  # blocks (components) per direction
    SLOTS, MAX_IN_FLIGHT = 4, 2
    THREAD_BLOCKS_PER_BLOCK = 8  # of the push and unpacking launches

    def __init__(self, mpi_construct, capacity_bytes):
        from .comm import MPI  # (PROC_NULL)

        mc = mpi_construct
        self.device = mc.device
        prev, nxt = int(mc.previous_grid_along[0]), int(mc.next_grid_along[0])
        self.prev = None if prev == MPI.PROC_NULL else prev
        self.next = None if nxt == MPI.PROC_NULL else nxt
        self.capacity = (int(capacity_bytes) + 255) // 256 * 256
        self._ipc = _IpcBuffers(self.device)
        self._lib = self._ipc.lib
        self._epoch = 0
        self._in_flight = 0
        self._done = torch.zeros(8, dtype=torch.int32, device=self.device)
        self._err = torch.zeros(1, dtype=torch.int32, device=self.device)
        ok = False
        if self.device.type == "cuda":
            self.mailbox = self._ipc.alloc(2 * self.SLOTS * self.capacity)  # [slot][direction][capacity]
            self.flags = self._ipc.alloc(4 * 2 * 8)                         # int32 [direction][8]
            try:
                self._peer, _ = self._ipc.map_peers(sorted({self.prev, self.next} - {None}))
                ok = True
            except Exception as exc:  # pragma: no cover - depends on the node
                logger.warning(f"CUDA IPC peer mapping unavailable for halos ({type(exc).__name__}: {exc}); "
                               "halo exchanges use NCCL send / recv")
        self.ok = _on_every_rank(ok)

    def close(self):
        """collective: unmap the neighbours' mailboxes, then free the own one"""
        self.ok = False
        self._ipc.close()

    # ------------------------------------------------------------------ the exchange
    def _fits_mailbox(self, blocks, n_per_direction):
        """contiguous device blocks of one size, 16-byte granular, that fit a mailbox direction"""
        if not self.ok or n_per_direction > self.MAX_BLOCKS or self._in_flight >= self.MAX_IN_FLIGHT:
            return False
        nbytes = blocks[0].numel() * blocks[0].element_size()
        return (all(b.is_cuda and b.is_contiguous() and b.numel() * b.element_size() == nbytes
                    and b.data_ptr() % 16 == 0 for b in blocks)
                and nbytes % 16 == 0 and nbytes * n_per_direction <= self.capacity)

    def _region(self, base, slot, direction):
        return base + (2 * slot + direction) * self.capacity

    def start(self, up, down, recv_prev, recv_next):
        """``up[c]`` -> the next rank, ``down[c]`` -> the previous rank (lists of one block per component,
        equally sized contiguous tensors; nothing goes where there is no neighbour).  The messages of the
        fallback land in ``recv_prev[c]`` (from the previous rank) and ``recv_next[c]``.  Runs on the
        current stream; returns what ``finish`` takes."""
        ncomp = len(up)
        nbytes = up[0].numel() * up[0].element_size()
        requests, epoch = [], None
        if self._fits_mailbox(list(up) + list(down), ncomp):
            self._epoch += 1
            self._in_flight += 1
            epoch, slot = self._epoch, self._epoch % self.SLOTS
            src, dst, flg = [], [], []
            if self.next is not None:
                box, flags = self._peer[self.next]
                src += up
                dst += [self._region(box, slot, 0) + c * nbytes for c in range(ncomp)]
                flg += [flags + 4 * c for c in range(ncomp)]
            if self.prev is not None:
                box, flags = self._peer[self.prev]
                src += down
                dst += [self._region(box, slot, 1) + c * nbytes for c in range(ncomp)]
                flg += [flags + 4 * (8 + c) for c in range(ncomp)]
            n = len(src)
            _lib.check(self._lib, self._lib.sb200_peer_push_blocks(
                n, (ctypes.c_void_p * n)(*dst), (ctypes.c_void_p * n)(*[b.data_ptr() for b in src]), nbytes,
                self.THREAD_BLOCKS_PER_BLOCK, (ctypes.c_void_p * n)(*flg), epoch,
                ctypes.c_void_p(self._done.data_ptr()), current_stream_ptr(self.device)))
            from_prev = [self._region(self.mailbox, slot, 0) + c * nbytes for c in range(ncomp)]
            from_next = [self._region(self.mailbox, slot, 1) + c * nbytes for c in range(ncomp)]
        else:
            # "up" messages and "down" messages carry different tags, and every rank posts them in the same
            # order: the two directions stay apart even when prev == next (a periodic domain on two ranks)
            ops = []
            for c in range(ncomp):
                if self.next is not None:
                    ops.append(dist.P2POp(dist.isend, up[c], self.next, tag=2 * c))
                if self.prev is not None:
                    ops.append(dist.P2POp(dist.irecv, recv_prev[c], self.prev, tag=2 * c))
                    ops.append(dist.P2POp(dist.isend, down[c], self.prev, tag=2 * c + 1))
                if self.next is not None:
                    ops.append(dist.P2POp(dist.irecv, recv_next[c], self.next, tag=2 * c + 1))
            requests = dist.batch_isend_irecv(ops) if ops else []
            from_prev, from_next = [t.data_ptr() for t in recv_prev], [t.data_ptr() for t in recv_next]
        return (requests, epoch, from_prev if self.prev is not None else [],
                from_next if self.next is not None else [])

    def finish(self, pending):
        """Wait (on the current stream) for the blocks of the exchange ``pending``; returns the addresses of
        the blocks received from the previous and from the next rank (one per component, none where there
        is no neighbour): in the local mailbox, or in the receive tensors given to ``start``."""
        requests, epoch, from_prev, from_next = pending
        for req in requests:
            req.wait()
        if epoch is None:
            return from_prev, from_next
        self._in_flight -= 1
        stream = current_stream_ptr(self.device)
        for direction, blocks in enumerate((from_prev, from_next)):
            if blocks:
                _lib.check(self._lib, self._lib.sb200_peer_wait_flags(
                    ctypes.c_void_p(self.flags + 4 * 8 * direction), len(blocks), epoch,
                    ctypes.c_void_p(self._err.data_ptr()), stream))
        return from_prev, from_next

    def copy_blocks(self, dst_ptrs, src_ptrs, nbytes):
        """local block copies (the unpacking of a halo exchange) in one launch"""
        n = len(dst_ptrs)
        if n:
            _lib.check(self._lib, self._lib.sb200_peer_push_blocks(
                n, (ctypes.c_void_p * n)(*dst_ptrs), (ctypes.c_void_p * n)(*src_ptrs), nbytes,
                self.THREAD_BLOCKS_PER_BLOCK, None, 0, None, current_stream_ptr(self.device)))

    def check(self):
        if int(self._err.item()) != 0:
            raise _lib.SophtB200Error("peer halo exchange: a neighbour did not deliver its planes in time")


def peer_halo(mpi_construct, block_bytes):
    """The process-wide neighbour exchange of ``mpi_construct`` (more than one rank), with mailboxes for
    ``MAX_BLOCKS`` blocks of ``block_bytes`` per direction (created, or grown, collectively: every rank asks
    for the same sizes in the same order)."""
    mc = mpi_construct
    nbytes_per_direction = PeerHalo.MAX_BLOCKS * int(block_bytes)
    halo = getattr(mc, "_peer_halo", None)
    if halo is not None and halo.capacity < nbytes_per_direction and halo.ok:
        halo.close()
        halo = None
    if halo is None:
        halo = mc._peer_halo = PeerHalo(mc, max(int(nbytes_per_direction), 1 << 20))
    return halo
