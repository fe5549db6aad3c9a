"""TEST INFRASTRUCTURE: the ten reshard callables over torch.distributed (gloo) so that the
host-side logic (lowering, data-parallel rewrites, executor) can be exercised with world_size 2 on
CPU.  Semantics follow the oracle / the reference (sharding.py:94-163); the product binds
easydist_b200.reshard (libedb.so) instead and has no CPU path."""
from typing import List

import torch
import torch.distributed as dist
from torch._subclasses.fake_tensor import FakeTensor

from easydist_b200.reshard import all_reduce_push_sizes  # noqa: E402,F401  (pure host arithmetic)

_GROUPS = {}


def init_groups(mesh):
    """dist.new_group is collective over the WORLD: create every mesh-dim sub-group on every rank
    in one global order before any op needs it (mesh: numpy array of ranks)."""
    import numpy as np
    mesh = np.asarray(mesh)
    for mdim in range(mesh.ndim):
        moved = np.moveaxis(mesh, mdim, -1).reshape(-1, mesh.shape[mdim])
        for row in moved:
            key = tuple(int(r) for r in row)
            if key not in _GROUPS:
                _GROUPS[key] = dist.new_group(list(key), backend="gloo")


def _pg(ranks):
    key = tuple(ranks)
    if key not in _GROUPS:
        if len(key) != dist.get_world_size():
            raise RuntimeError(f"group {key} was not created by init_groups(mesh)")
        _GROUPS[key] = dist.new_group(list(ranks), backend="gloo")
    return _GROUPS[key]


def _fake(t):
    return isinstance(t, FakeTensor) or t.is_meta


_OPS = {"sum": dist.ReduceOp.SUM, "max": dist.ReduceOp.MAX, "min": dist.ReduceOp.MIN,
        "avg": dist.ReduceOp.SUM}


def all_reduce_start(self, reduceOp: str, group: List[int], tag: str = "", *, _buf=None):
    if _fake(self):
        return torch.empty_like(self)
    out = self.contiguous().clone()
    acc = out.float() if out.dtype in (torch.bfloat16, torch.float16) else out
    dist.all_reduce(acc, op=_OPS[reduceOp], group=_pg(group))
    if reduceOp == "avg":
        acc = acc * (1.0 / len(group))
    return acc.to(self.dtype)


def all_reduce_end(self, reduceOp, group, tag=""):
    return self


def all_gather_start(self, gather_dim: int, group: List[int], tag: str = "", *, _buf=None):
    n = len(group)
    shape = list(self.shape)
    shape[gather_dim] *= n
    if _fake(self):
        return self.new_empty(shape)
    parts = [torch.empty_like(self.contiguous()) for _ in range(n)]
    dist.all_gather(parts, self.contiguous(), group=_pg(group))
    return torch.cat(parts, dim=gather_dim)


def all_gather_end(self, gather_dim, group, tag=""):
    return self


def scatter_wrapper(tensor, num_chunks, dim, indice):
    return torch.ops.aten.chunk(tensor, num_chunks, dim)[indice].contiguous()


def copy_wrapper(self, other):
    return torch.ops.aten.copy_.default(self, other)


def reduce_scatter_start(self, reduceOp: str, scatter_dim: int, group: List[int], tag: str = "", *,
                         _buf=None, _scale=1.0, _out_dtype=None):
    n = len(group)
    assert self.size(scatter_dim) % n == 0
    shape = list(self.shape)
    shape[scatter_dim] //= n
    if _fake(self):
        return self.new_empty(shape, dtype=_out_dtype or self.dtype)
    red = all_reduce_start(self, reduceOp, group)
    me = list(group).index(dist.get_rank())
    out = torch.chunk(red, n, scatter_dim)[me].contiguous()
    if _scale != 1.0:
        out = out * _scale
    return out.to(_out_dtype or self.dtype)


def reduce_scatter_end(self, reduceOp, scatter_dim, group, tag=""):
    return self


def all_to_all_start(tensor, gather_dim, scatter_dim, num_chunks, indice, ranks, tag="", *,
                     _buf=None):
    g = all_gather_start(tensor, gather_dim, ranks)
    if _fake(tensor):
        shape = list(g.shape)
        shape[scatter_dim] //= num_chunks
        return tensor.new_empty(shape)
    return scatter_wrapper(g, num_chunks, scatter_dim, indice)


def all_to_all_end(tensor, gather_dim, scatter_dim, num_chunks, indice, ranks, tag=""):
    return tensor


# fused ops (semantics of easydist_b200.reshard.ag_mm / mm_push / rs_finish) for CPU tests of the
# fusion rewrite


_EPOCHS = {"barriers": 0, "open_pushes": 0}


def epoch_barrier(x, group):
    """CPU stand-in of reshard.epoch_barrier: a real gloo barrier, counted; pushes issued since
    the previous barrier become reducible."""
    if _fake(x) or len(group) <= 1:
        return x
    dist.barrier(group=_pg(group))
    _EPOCHS["barriers"] += 1
    _EPOCHS["open_pushes"] = 0
    return x


def ag_prefetch(x, group, *, _items=None):
    return x


def gathered(w_shard, group, *deps, _buf=None):
    """CPU stand-in of reshard.gathered: a real all-gather at every use."""
    if _fake(w_shard):
        return w_shard.new_empty((len(group) * w_shard.numel(),))
    return all_gather_start(w_shard.reshape(-1), 0, group)


def mm_push(a, b, group, *, _buf=None):
    """CPU stand-in of reshard.mm_push (epoch mode): the token carries the partial product."""
    if _fake(a):
        return a.new_empty((a.shape[0], b.shape[1]))
    _EPOCHS["open_pushes"] += 1
    return a @ b


def ag_mm(x, w_shard, group, n_out, k_in, bias=None, *, _buf=None, _epoch=1):
    if _fake(x):
        return x.new_empty((x.shape[0], n_out)), w_shard.new_empty((n_out, k_in))
    w = all_gather_start(w_shard.reshape(-1), 0, group).view(n_out, k_in)
    out = x @ w.t()
    if bias is not None:
        out = out + bias
    return out, w


def rs_finish(tokens, group, *, _bufs=None, _numels=None, _scale=1.0, _out_dtype=None):
    n = len(group)
    if tokens and _fake(tokens[0]):
        return [t.new_empty((int(k),), dtype=_out_dtype or t.dtype) for t, k in zip(tokens, _numels)]
    # epoch protocol: a barrier must separate the pushes from their reduction
    assert _EPOCHS["open_pushes"] == 0, "rs_finish without an epoch barrier in front"
    me = list(group).index(dist.get_rank())
    outs = []
    for t in tokens:
        red = all_reduce_start(t.flatten(), "sum", group)
        outs.append((torch.chunk(red, n, 0)[me].contiguous() * _scale).to(_out_dtype or t.dtype))
    return outs


def box_exchange(tensor, dst_shape, boxes, peer_src_shapes, group, *, _buf=None):
    """Partition P2P redistribution over gloo: every member publishes its source partition, each
    rank copies the boxes it needs (semantics of reshard.box_exchange / sharding.py:427-474)."""
    if _fake(tensor):
        return tensor.new_empty([int(s) for s in dst_shape])
    n = len(group)
    parts = [torch.empty([int(v) for v in shp], dtype=tensor.dtype) for shp in peer_src_shapes]
    # partitions differ in shape: exchange them one broadcast per member
    me = list(group).index(dist.get_rank())
    for i, r in enumerate(group):
        buf = tensor.contiguous().clone() if i == me else parts[i]
        if buf.numel():
            dist.broadcast(buf, src=r, group=_pg(group))
        parts[i] = buf
    out = tensor.new_empty([int(s) for s in dst_shape])
    for (p_idx, s_start, d_start, ext) in boxes:
        ssl = tuple(slice(a, a + e) for a, e in zip(s_start, ext))
        dsl = tuple(slice(a, a + e) for a, e in zip(d_start, ext))
        out[dsl] = parts[p_idx][ssl]
    return out


class FakeSymmRuntime:
    """Stands in for easydist_b200.runtime.Runtime in the fusion pass (offsets only)."""

    class _Buf:
        def __init__(self, offset, nbytes):
            self.offset, self.nbytes = offset, nbytes

        def tensor(self, dtype, shape):
            return torch.empty(shape, dtype=dtype)

        def sub(self, delta, nbytes):
            return FakeSymmRuntime._Buf(self.offset + delta, nbytes)

    def __init__(self):
        self._off = 1 << 20

    def get_option(self, name):
        return {"allreduce_oneshot_bytes": 512 * 1024}[name]

    def alloc(self, nbytes, align=256):
        off = (self._off + align - 1) // align * align
        self._off = off + nbytes
        return FakeSymmRuntime._Buf(off, nbytes)


FUSED_FUNCS = [ag_mm, mm_push, rs_finish, epoch_barrier, ag_prefetch, gathered]
COMM_FUNCS = [all_reduce_start, all_gather_start, reduce_scatter_start, all_to_all_start]
COMM_SYNC_FUNCS = [all_reduce_end, all_gather_end, reduce_scatter_end, all_to_all_end]
CUSTOM_FUNCS = COMM_FUNCS + COMM_SYNC_FUNCS + [scatter_wrapper, copy_wrapper]
