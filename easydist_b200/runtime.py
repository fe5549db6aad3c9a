"""Process-level runtime: symmetric heap, peer mapping, groups, tensor views.

Python stays the orchestrator (as in the reference, where everything above the collectives is
Python); this module owns the one-time bootstrap that ProcessGroupNCCL does for the reference:
exchange of the CUDA-IPC handles of every rank's slab over torch.distributed, group creation for
the mesh dims (reference: easydist/torch/device_mesh.py:129-150 + sharding.py:729-730 rank lists).
"""
import ctypes
import os
from ctypes import byref, c_int, c_int64, c_size_t, c_uint64, c_void_p

import torch

from . import _lib
from ._lib import check

_DEFAULT_HEAP = int(os.environ.get("EDB_HEAP_BYTES", str(8 << 30)))


class _CudaArray:
    """Minimal __cuda_array_interface__ holder so torch can view the slab without owning it."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {
            "shape": (int(nbytes),),
            "typestr": "|u1",
            "data": (int(ptr), False),
            "version": 3,
            "strides": None,
        }


class SymmBuffer:
    """A buffer in the symmetric heap, named by its offset (same offset on every rank)."""

    __slots__ = ("offset", "nbytes", "_rt")

    def __init__(self, rt, offset, nbytes):
        self._rt = rt
        self.offset = int(offset)
        self.nbytes = int(nbytes)

    def tensor(self, dtype, shape):
        numel = 1
        for s in shape:
            numel *= int(s)
        nbytes = numel * torch.empty((), dtype=dtype).element_size()
        assert nbytes <= self.nbytes, (nbytes, self.nbytes)
        flat = self._rt.slab[self.offset:self.offset + nbytes]
        return flat.view(dtype).view(tuple(int(s) for s in shape))

    def sub(self, delta, nbytes):
        """The sub-range [delta, delta + nbytes) of this buffer as a buffer of its own."""
        assert 0 <= delta and delta + nbytes <= self.nbytes
        return SymmBuffer(self._rt, self.offset + int(delta), nbytes)

    @property
    def ptr(self):
        return self._rt.heap_base + self.offset


class Runtime:
    """One per process (one process per GPU)."""

    def __init__(self, rank, world, device, heap_bytes=None):
        self.lib = _lib.load()
        self.rank, self.world, self.device_index = int(rank), int(world), int(device)
        heap_bytes = int(heap_bytes or _DEFAULT_HEAP)
        check(self.lib.edb_init(self.rank, self.world, self.device_index, heap_bytes))
        base, nbytes, user = c_void_p(), c_size_t(), c_size_t()
        check(self.lib.edb_heap_info(byref(base), byref(nbytes), byref(user)))
        self.heap_base, self.heap_bytes, self.user_offset = base.value, nbytes.value, user.value
        self.device = torch.device("cuda", self.device_index)
        self._holder = _CudaArray(self.heap_base, self.heap_bytes)
        self.slab = torch.as_tensor(self._holder, device=self.device)
        assert self.slab.data_ptr() == self.heap_base and self.slab.numel() == self.heap_bytes
        self._groups = {}       # tuple(ranks) -> gid
        self._group_meta = {}   # gid -> (n, my_index, ranks)
        # dynamic staging ring: the upper quarter of the heap; the rest is the static arena
        self._ring_size = (self.heap_bytes - self.user_offset) // 4 // 256 * 256
        self._ring_base = self.heap_bytes - self._ring_size
        self._ring_pos = 0
        self._static_limit = self._ring_base
        self._attached = self.world == 1
        # a peer that stays away longer than this is fatal (the waiting kernel traps): same role as
        # the NCCL watchdog timeout of the reference's process groups
        self.set_option("spin_timeout_ms", int(os.environ.get("EDB_SPIN_TIMEOUT_MS", "120000")))
        for opt in ("push_sync", "comm_ctas"):
            if os.environ.get("EDB_" + opt.upper()) is not None:
                self.set_option(opt, int(os.environ["EDB_" + opt.upper()]))

    # ---- bootstrap -------------------------------------------------------------------------
    def attach_peers(self, process_group=None):
        """Exchange IPC handles over torch.distributed and map every peer slab."""
        if self._attached:
            return
        import torch.distributed as dist
        buf = ctypes.create_string_buffer(64)
        check(self.lib.edb_ipc_export(buf))
        mine = bytes(buf.raw)
        handles = [None] * self.world
        dist.all_gather_object(handles, (self.rank, mine), group=process_group)
        for r, h in handles:
            if r != self.rank:
                check(self.lib.edb_ipc_attach(int(r), ctypes.create_string_buffer(h, 64)))
        dist.barrier(group=process_group)
        self._attached = True
        self._pg = process_group

    def host_barrier(self):
        """Host-level rendezvous (torch.distributed): used once after compilation so that no rank
        starts its first step — whose kernels wait on peers with a finite, fatal timeout — while
        another rank is still tracing / re-homing parameter shards."""
        if self.world <= 1:
            return
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            torch.cuda.synchronize(self.device)
            # the symmetric heap is only symmetric if every rank made the same allocations: compare
            # the bump pointers (uneven shards / a rank-dependent branch would otherwise make peers
            # read and write each other's buffers at the wrong offsets, silently)
            marks = None
            try:
                marks = [None] * self.world
                dist.all_gather_object(marks, (self.rank, self.mark()),
                                       group=getattr(self, "_pg", None))
            except Exception as e:  # noqa: BLE001 — the check is a diagnostic, the barrier is what matters
                import logging
                logging.getLogger(__name__).warning("symmetric-heap check skipped: %r", e)
                marks = None
            if marks is not None and len({m for _, m in marks}) != 1:
                raise _lib.EdbError(_lib.EDB_E_STATE,
                                    f"symmetric heap diverged across ranks after compilation: {marks}")
            dist.barrier(group=getattr(self, "_pg", None))

    def group(self, ranks, slot=None):
        """gid of the group of global `ranks` (mesh-dim order); created on first use.

        Slots are assigned in creation order; SPMD programs create their groups in the same
        order on every member (mesh dim 0, 1, ... then the world group), which keeps them equal.
        """
        members = tuple(int(r) for r in ranks)
        gid = self._groups.get(members)
        if gid is not None:
            return gid
        if not self._attached:
            self.attach_peers()
        if slot is None:
            slot = len(self._groups)
        out = c_int()
        check(self.lib.edb_group_create(_lib.int_array(members), len(members), int(slot), byref(out)))
        n, me = c_int(), c_int()
        check(self.lib.edb_group_info(out.value, byref(n), byref(me)))
        self._groups[members] = out.value
        self._group_meta[out.value] = (n.value, me.value, members)
        return out.value

    def group_size(self, gid):
        return self._group_meta[gid][0]

    def group_index(self, gid):
        return self._group_meta[gid][1]

    # ---- symmetric memory ------------------------------------------------------------------
    def alloc(self, nbytes, align=256):
        """Static symmetric allocation (bump; deterministic across ranks)."""
        off = c_uint64()
        check(self.lib.edb_symm_alloc(max(16, int(nbytes)), int(align), byref(off)))
        if off.value + nbytes > self._static_limit:
            raise _lib.EdbError(_lib.EDB_E_STATE,
                                "static symmetric arena exhausted; raise EDB_HEAP_BYTES")
        return SymmBuffer(self, off.value, max(16, int(nbytes)))

    def mark(self):
        m = c_uint64()
        check(self.lib.edb_symm_mark(byref(m)))
        return m.value

    def reset(self, mark):
        check(self.lib.edb_symm_reset(int(mark)))

    def ring_alloc(self, nbytes):
        """Dynamic staging buffer from the ring (valid until the ring wraps around)."""
        nbytes = (max(16, int(nbytes)) + 255) // 256 * 256
        if nbytes > self._ring_size:
            raise _lib.EdbError(_lib.EDB_E_STATE,
                                f"staging buffer of {nbytes} bytes exceeds the dynamic ring "
                                f"({self._ring_size}); raise EDB_HEAP_BYTES")
        if self._ring_pos + nbytes > self._ring_size:
            self._ring_pos = 0
        off = self._ring_base + self._ring_pos
        self._ring_pos += nbytes
        return SymmBuffer(self, off, nbytes)

    # ---- misc --------------------------------------------------------------------------------
    def stream(self):
        return c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def launch_count(self):
        return int(self.lib.edb_launch_count())

    def health(self):
        """Raise if a collective of this process timed out on a peer (the kernel trapped; the
        record lives in pinned host memory, so this works without touching the dead context)."""
        check(self.lib.edb_health())

    def error_flags(self):
        """Op numbers whose spin waits timed out, per group slot (all zero when healthy)."""
        torch.cuda.synchronize(self.device)
        words = self.slab[:64 * 1024].view(torch.int64).view(-1, 128)
        return [int(words[s, 28]) for s in range(len(self._groups))]

    def set_option(self, name, value):
        check(self.lib.edb_set_option(name.encode(), int(value)))

    def get_option(self, name):
        v = c_int64()
        check(self.lib.edb_get_option(name.encode(), byref(v)))
        return v.value

    def finalize(self):
        self.slab = None
        self._holder = None
        check(self.lib.edb_finalize())


_runtime = None


def init(rank=None, world=None, device=None, heap_bytes=None):
    """Create the process runtime (idempotent). Reads RANK/WORLD_SIZE/LOCAL_RANK by default."""
    global _runtime
    if _runtime is not None:
        return _runtime
    if not torch.cuda.is_available():
        raise _lib.EdbError(_lib.EDB_E_STATE, "easydist_b200 needs a CUDA device (no CPU fallback)")
    if rank is None:
        rank = int(os.environ.get("RANK", "0"))
    if world is None:
        world = int(os.environ.get("WORLD_SIZE", "1"))
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", str(rank % max(1, torch.cuda.device_count()))))
    torch.cuda.set_device(device)
    _runtime = Runtime(rank, world, device, heap_bytes)
    if world > 1:
        _runtime.attach_peers()
    return _runtime


def get_runtime():
    if _runtime is None:
        raise _lib.EdbError(_lib.EDB_E_STATE, "easydist_b200.runtime.init() has not been called")
    return _runtime


def is_initialized():
    return _runtime is not None


def shutdown():
    global _runtime
    if _runtime is not None:
        _runtime.finalize()
        _runtime = None
