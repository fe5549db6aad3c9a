"""Host-side mirror of the reference's reshard operator interface, backed by libedb.so.

Same names, argument meaning and error behaviour as the ten FX `call_function` targets of
easydist/torch/passes/sharding.py:94-168 (`all_reduce_start/end`, `all_gather_start/end`,
`reduce_scatter_start/end`, `all_to_all_start/end`, `scatter_wrapper`, `copy_wrapper`) plus the
registries other passes key on (`COMM_FUNCS`, `COMM_SYNC_FUNCS`, `CUSTOM_FUNCS`,
sharding.py:166-168), so they can be bound in place of the reference's callables.

Differences that are the point of this backend:
  * every `*_start` is ONE CUDA kernel over peer memory (no NCCL, no funcol, no wait_tensor);
    the matching `*_end` is the identity because the work is stream-ordered;
  * non-dim-0 gathers/scatters need no chunk+cat copy: the dim is folded into the box indexing;
  * `all_to_all` moves 1/n of the bytes (the reference all-gathers and slices, sharding.py:155-163);
  * an optional keyword `_buf=(offset, nbytes[, offset2])` names static symmetric buffers chosen at
    lowering time; without it a staging ring is used and results are copied to torch-owned memory.
There is no CPU path: tensors must live on the runtime's CUDA device (FakeTensors are accepted so
that FX meta propagation works, mirroring how the reference's passes call these ops on fakes).
"""
from ctypes import byref, c_int64
from typing import List

import ctypes

import torch
from torch.fx.node import has_side_effect
from torch._subclasses.fake_tensor import FakeTensor

from . import _lib
from ._lib import DTYPE_CODES, REDOP_CODES, check, i64_array
from .runtime import SymmBuffer, get_runtime

_TORCH_DTYPE_CODE = {
    torch.float32: DTYPE_CODES["float32"],
    torch.bfloat16: DTYPE_CODES["bfloat16"],
    torch.float16: DTYPE_CODES["float16"],
    torch.float64: DTYPE_CODES["float64"],
    torch.int32: DTYPE_CODES["int32"],
    torch.int64: DTYPE_CODES["int64"],
}


def _is_fake(t):
    return isinstance(t, FakeTensor) or (isinstance(t, torch.Tensor) and t.is_meta)


def _require_cuda(t, what):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{what}: expected a tensor, got {type(t)}")
    if not t.is_cuda:
        raise _lib.EdbError(_lib.EDB_E_INVALID,
                            f"{what}: tensor is on {t.device}; easydist_b200 has no CPU path")


def _dtype_code(t, what):
    code = _TORCH_DTYPE_CODE.get(t.dtype)
    if code is None:
        raise _lib.EdbError(_lib.EDB_E_UNSUPPORTED, f"{what}: dtype {t.dtype} cannot be reduced")
    return code


def _redop(name, what):
    try:
        return REDOP_CODES[name]
    except KeyError:
        raise _lib.EdbError(_lib.EDB_E_INVALID, f"{what}: unknown reduceOp {name!r}") from None


def _norm_dim(dim, ndim):
    return dim + ndim if dim < 0 else dim


def _group(group):
    rt = get_runtime()
    gid = rt.group(group)
    return rt, gid, rt.group_size(gid), rt.group_index(gid)


def _buffers(rt, _buf, sizes):
    """Resolve static (`_buf`) or ring staging buffers for the byte sizes in `sizes`."""
    if _buf is not None:
        offs = [_buf[0]] + list(_buf[2:])
        return [SymmBuffer(rt, o, s) for o, s in zip(offs, sizes)], True
    return [rt.ring_alloc(s) for s in sizes], False


# ---- all_reduce -------------------------------------------------------------------------------------


def all_reduce_push_sizes(nbytes, numel, elem_size, n, oneshot_bytes):
    """(receive bytes, result bytes) of edb_all_reduce_push — same rule as the C side."""
    two_shot = nbytes > oneshot_bytes * (8 if n == 2 else 1) and numel % (16 // elem_size * n) == 0
    return (nbytes if two_shot else n * nbytes), nbytes


def all_reduce_start(self: torch.Tensor, reduceOp: str, group: List[int], tag: str = "", *,
                     _buf=None, _push=0):
    """P(op) -> R. Reference: sharding.py:94-98 (c10d_functional.all_reduce).
    `_push=1` (set by lowering.assign_static_buffers for graphs that end with an epoch barrier):
    the push protocol, _buf = (receive offset, size, result offset); the result is a view of the
    static symmetric result buffer."""
    if _is_fake(self):
        return torch.empty_like(self, memory_format=torch.contiguous_format)
    _require_cuda(self, "all_reduce_start")
    rt, gid, n, _ = _group(group)
    x = self.contiguous()
    if _push and _buf is not None and n > 1 and x.numel() > 0:
        recv_off, out_off = int(_buf[0]), int(_buf[2])
        check(rt.lib.edb_all_reduce_push(gid, out_off, recv_off, x.data_ptr(), x.numel(),
                                         _dtype_code(x, "all_reduce_start"),
                                         _redop(reduceOp, "all_reduce_start"), rt.stream()))
        return SymmBuffer(rt, out_off, x.numel() * x.element_size()).tensor(x.dtype, x.shape)
    out = torch.empty_like(x)
    nbytes = x.numel() * x.element_size()
    if nbytes == 0:
        return out
    two_shot = n > 1 and nbytes > rt.get_option("allreduce_oneshot_bytes")
    sizes = [nbytes, nbytes] if two_shot else [nbytes]
    if n > 1:
        bufs, _ = _buffers(rt, _buf, sizes)
        s1 = bufs[0].offset
        s2 = bufs[1].offset if two_shot else 0
    else:
        s1 = s2 = 0
    check(rt.lib.edb_all_reduce(gid, out.data_ptr(), s1, s2, x.data_ptr(), x.numel(),
                                _dtype_code(x, "all_reduce_start"),
                                _redop(reduceOp, "all_reduce_start"), rt.stream()))
    return out


def all_reduce_end(self: torch.Tensor, reduceOp: str, group: List[int], tag: str = ""):
    """Reference: sharding.py:101-102 (wait_tensor). Identity: the start is stream-ordered."""
    return self


# ---- all_gather --------------------------------------------------------------------------------------


def all_gather_start(self: torch.Tensor, gather_dim: int, group: List[int], tag: str = "", *,
                     _buf=None, _push=0):
    """S(gather_dim) -> R. Reference: sharding.py:105-111 gathers along dim 0 and leaves the
    chunk+cat to all_gather_end (:114-119); here the result is already laid out along
    `gather_dim`."""
    n_hint = len(group)
    ndim = self.dim()
    dim = _norm_dim(gather_dim, ndim)
    out_shape = list(self.shape)
    out_shape[dim] = out_shape[dim] * n_hint
    if _is_fake(self):
        return self.new_empty(out_shape)
    _require_cuda(self, "all_gather_start")
    rt, gid, n, _ = _group(group)
    x = self.contiguous()
    nbytes = x.numel() * x.element_size() * n
    if nbytes == 0:
        return x.new_empty(out_shape)
    (buf,), static = _buffers(rt, _buf, [nbytes])
    fn = rt.lib.edb_all_gather_push if (_push and static) else rt.lib.edb_all_gather
    check(fn(gid, buf.offset, x.data_ptr(), i64_array(x.shape), ndim, dim, x.element_size(),
             rt.stream()))
    out = buf.tensor(x.dtype, out_shape)
    return out if static else out.clone()


def all_gather_end(self: torch.Tensor, gather_dim: int, group: List[int], tag: str = ""):
    """Reference: sharding.py:114-119. Identity: all_gather_start already produced the layout."""
    return self


# ---- local ops ---------------------------------------------------------------------------------------


def scatter_wrapper(tensor, num_chunks, dim, indice):
    """R -> S(dim), local. Reference: sharding.py:122-123 `aten.chunk(t, n, dim)[i].contiguous()`
    (torch.chunk = ceil-div blocks; an index past the last chunk raises IndexError there too)."""
    ndim = tensor.dim()
    d = _norm_dim(dim, ndim)
    size = tensor.shape[d]
    block = -(-size // num_chunks) if size > 0 else 0
    n_actual = -(-size // block) if block > 0 else num_chunks  # size 0: n empty chunks
    if indice >= n_actual or indice < 0:
        raise IndexError("tuple index out of range")
    lo = min(size, block * indice)
    hi = min(size, block * (indice + 1))
    out_shape = list(tensor.shape)
    out_shape[d] = hi - lo
    if _is_fake(tensor):
        return tensor.new_empty(out_shape)
    _require_cuda(tensor, "scatter_wrapper")
    rt = get_runtime()
    x = tensor.contiguous()
    out = x.new_empty(out_shape)
    if out.numel():
        ext = c_int64()
        check(rt.lib.edb_scatter(out.data_ptr(), x.data_ptr(), i64_array(x.shape), ndim, d,
                                 int(num_chunks), int(indice), x.element_size(), byref(ext),
                                 rt.stream()))
    return out


def copy_wrapper(self, other):
    """State write-back. Reference: sharding.py:126-127 `aten.copy_(self, other)`; returns self."""
    if _is_fake(self) or _is_fake(other):
        return self
    _require_cuda(self, "copy_wrapper")
    if (other.is_cuda and self.shape == other.shape and self.dtype == other.dtype
            and self.is_contiguous() and other.is_contiguous()):
        if self.numel() and self.data_ptr() != other.data_ptr():
            rt = get_runtime()
            check(rt.lib.edb_copy(self.data_ptr(), other.data_ptr(),
                                  self.numel() * self.element_size(), rt.stream()))
        return self
    return torch.ops.aten.copy_.default(self, other)  # broadcasting / dtype-converting copies


# ---- reduce_scatter ----------------------------------------------------------------------------------


def reduce_scatter_start(self: torch.Tensor, reduceOp: str, scatter_dim: int, group: List[int],
                         tag: str = "", *, _buf=None, _scale: float = 1.0, _out_dtype=None,
                         _push=0):
    """P(op) -> S(scatter_dim). Reference: sharding.py:130-144 (pre-permute copy for dim != 0 and
    reduce_scatter_tensor). `_scale`/`_out_dtype` fuse the gradient scale / cast into the kernel."""
    n = len(group)
    ndim = self.dim()
    dim = _norm_dim(scatter_dim, ndim)
    assert self.size(dim) % n == 0, (
        f"input dimension 0 ({self.size(0)} must be a multiple of group_size {n}")
    out_shape = list(self.shape)
    out_shape[dim] //= n
    out_dtype = _out_dtype or self.dtype
    if _is_fake(self):
        return self.new_empty(out_shape, dtype=out_dtype)
    _require_cuda(self, "reduce_scatter_start")
    rt, gid, n, _ = _group(group)
    x = self.contiguous()
    out = x.new_empty(out_shape, dtype=out_dtype)
    nbytes = x.numel() * x.element_size()
    if nbytes == 0:
        return out
    stage, static = 0, False
    if n > 1:
        (buf,), static = _buffers(rt, _buf, [nbytes])
        stage = buf.offset
    fn = rt.lib.edb_reduce_scatter_push if (_push and static) else rt.lib.edb_reduce_scatter
    check(fn(gid, out.data_ptr(), stage, x.data_ptr(),
             i64_array(x.shape), ndim, dim, _dtype_code(x, "reduce_scatter_start"),
             _redop(reduceOp, "reduce_scatter_start"), float(_scale),
             _TORCH_DTYPE_CODE[out_dtype], rt.stream()))
    return out


def reduce_scatter_end(self: torch.Tensor, reduceOp: str, scatter_dim: int, group: List[int],
                       tag: str = ""):
    """Reference: sharding.py:147-152 (wait_tensor). Identity: the start is stream-ordered."""
    return self


# ---- all_to_all --------------------------------------------------------------------------------------


def all_to_all_start(tensor, gather_dim, scatter_dim, num_chunks, indice, ranks, tag: str = "", *,
                     _buf=None, _push=0):
    """S(gather_dim) -> S(scatter_dim). Reference: sharding.py:155-163 (all-gather + local chunk,
    n x over-communication); here a true all-to-all: each rank pulls only its slice."""
    n = len(ranks)
    ndim = tensor.dim()
    g, s = _norm_dim(gather_dim, ndim), _norm_dim(scatter_dim, ndim)
    out_shape = list(tensor.shape)
    out_shape[g] *= n
    if out_shape[s] % n != 0:
        raise _lib.EdbError(_lib.EDB_E_INVALID,
                            f"all_to_all: dim {s} of size {out_shape[s]} not divisible by {n}")
    out_shape[s] //= n
    if _is_fake(tensor):
        return tensor.new_empty(out_shape)
    _require_cuda(tensor, "all_to_all_start")
    rt, gid, n, me = _group(ranks)
    assert me == indice, f"all_to_all: indice {indice} is not this rank's coordinate {me}"
    x = tensor.contiguous()
    nbytes = x.numel() * x.element_size()
    if _push and _buf is not None and n > 1 and nbytes > 0:
        # push protocol: every member writes its pieces straight into the static result buffers
        check(rt.lib.edb_all_to_all_push(gid, int(_buf[0]), x.data_ptr(), i64_array(x.shape), ndim,
                                         g, s, x.element_size(), rt.stream()))
        return SymmBuffer(rt, int(_buf[0]), nbytes).tensor(x.dtype, out_shape)
    out = x.new_empty(out_shape)
    if nbytes == 0:
        return out
    stage = 0
    if n > 1:
        (buf,), _ = _buffers(rt, _buf, [nbytes])
        stage = buf.offset
    check(rt.lib.edb_all_to_all(gid, out.data_ptr(), stage, x.data_ptr(), i64_array(x.shape), ndim,
                                g, s, x.element_size(), rt.stream()))
    return out


def all_to_all_end(tensor, gather_dim, scatter_dim, num_chunks, indice, ranks, tag: str = ""):
    """Reference: sharding.py:160-163. Identity: all_to_all_start already sliced."""
    return tensor


# ---- extras beyond the ten callables -----------------------------------------------------------------


def halo_exchange(tensor, dim, halo, group, *, _buf=None):
    """S(dim) with halo: concat(prev[-halo:], x, next[:halo]) along dim — the lowering of
    metashard/halo.py:33-55 halo_padding that the reference never emits."""
    ndim = tensor.dim()
    d = _norm_dim(dim, ndim)
    if _is_fake(tensor):
        raise NotImplementedError("halo_exchange on fake tensors needs the rank coordinate")
    _require_cuda(tensor, "halo_exchange")
    rt, gid, n, me = _group(group)
    if halo > tensor.shape[d]:
        raise RuntimeError("Cannot halo padding for this sharded_tensor")  # halo.py:47-48
    x = tensor.contiguous()
    out_shape = list(x.shape)
    out_shape[d] += (halo if me > 0 else 0) + (halo if me < n - 1 else 0)
    out = x.new_empty(out_shape)
    nbytes = x.numel() * x.element_size()
    if nbytes == 0:
        return out
    stage = 0
    if n > 1:
        (buf,), _ = _buffers(rt, _buf, [nbytes])
        stage = buf.offset
    check(rt.lib.edb_halo_exchange(gid, out.data_ptr(), stage, x.data_ptr(), i64_array(x.shape),
                                   ndim, d, int(halo), x.element_size(), rt.stream()))
    return out


def box_exchange(tensor, dst_shape, boxes, peer_src_shapes, group, *, _buf=None):
    """Partition P2P redistribution (reference: do_p2p_comm_wrapper, sharding.py:595-612).

    `boxes`: list of (member_index, src_start, dst_start, extents) for THIS rank's destination;
    `peer_src_shapes`: source-partition shape of every group member."""
    if _is_fake(tensor):
        return tensor.new_empty([int(s) for s in dst_shape])
    _require_cuda(tensor, "box_exchange")
    rt, gid, n, me = _group(group)
    x = tensor.contiguous()
    ndim = x.dim()
    out = x.new_empty([int(s) for s in dst_shape])
    if not boxes and n == 1:
        return out
    nbytes = x.numel() * x.element_size()
    stage = 0
    if n > 1:
        (buf,), _ = _buffers(rt, _buf, [max(16, nbytes)])
        stage = buf.offset
    peers = _lib.int_array([b[0] for b in boxes])
    flat = lambda k: i64_array([v for b in boxes for v in b[k]])
    shapes = i64_array([v for s in peer_src_shapes for v in s])
    check(rt.lib.edb_box_exchange(gid, out.data_ptr(), i64_array(out.shape), stage,
                                  x.data_ptr() if x.numel() else None, i64_array(x.shape), ndim,
                                  x.element_size(), len(boxes), peers, flat(1), flat(2), flat(3),
                                  shapes, rt.stream()))
    return out


# ---- fused compute + collective (one kernel each) -----------------------------------------------------


@has_side_effect
def epoch_barrier(x, group):
    """Pass-through that runs the group-wide epoch barrier on the stream (edb_epoch_barrier).
    The fused kernels (`ag_mm`, `mm_push`) read peers' parameter shards and
    write peers' receive slots without any per-op handshake; two of these per train step — one in
    front of the optimizer, one behind it — are the only cross-rank rendezvous left
    (reference: one NCCL rendezvous per collective, sharding.py:94-152)."""
    if _is_fake(x) or len(group) <= 1:
        return x
    rt, gid, n, _ = _group(group)
    check(rt.lib.edb_epoch_barrier(gid, rt.stream()))
    return x


@has_side_effect
def ag_prefetch(x, group, *, _items):
    """Stand-alone all-gather prefetch (edb_ag_prefetch): for every item (src_off, dst_off, bytes,
    dst_stride) and every member p, copy p's symmetric range into local dst_off + p*dst_stride.
    Epoch mode: the start-of-step gathers (embeddings, first layer) that have no earlier GEMM to
    ride on.  Pass-through of `x`."""
    if _is_fake(x) or len(group) <= 1 or not _items:
        return x
    from . import gemm as _gemm
    _gemm.prefetch_standalone({"group": list(group), "items": list(_items)}, x.device)
    return x


def gathered(w_shard, group, *deps, _buf):
    """The dim-0 all-gather of parameter shard `w_shard` (all_gather_start/_end of the zero3 /
    auto-SPMD graphs, sharding.py:105-119) in epoch mode: the data was already put into the
    symmetric buffer at _buf[1] by prefetches earlier on the stream (`deps`: the nodes that
    carried them), so this is a zero-copy view — n * numel(w_shard) elements, flat."""
    n = len(group)
    if _is_fake(w_shard):
        return w_shard.new_empty((n * w_shard.numel(),))
    _require_cuda(w_shard, "gathered")
    rt = get_runtime()
    assert w_shard.data_ptr() == rt.heap_base + int(_buf[0]), "shard is not at its symmetric offset"
    nbytes = w_shard.numel() * w_shard.element_size()
    return SymmBuffer(rt, int(_buf[1]), n * nbytes).tensor(w_shard.dtype, (n * w_shard.numel(),))


def ag_mm(x, w_shard, group, n_out, k_in, bias=None, *, _buf, _epoch=1):
    """all_gather(weight shard, dim 0) fused into the consuming GEMM (all_gather_end -> aten.mm /
    addmm of the sharded graph).  `w_shard`: this rank's rows [n_out/n, k_in] (flat or 2-D) living
    at symmetric offset _buf[0]; _buf[1] = offset of the gathered [n_out, k_in] buffer that the
    kernel's copy CTAs fill while the MMA CTAs already run.  Returns (x @ W^T (+ bias), W_full).
    Epoch protocol: an epoch barrier earlier on the stream made every member's shard final, and
    none is modified before the next one.  That is the only protocol, so `_epoch` accepts only 1;
    the keyword is kept for existing callers that pass it."""
    if _epoch != 1:
        raise ValueError("ag_mm: only the epoch protocol (_epoch=1) is supported")
    n = len(group)
    if _is_fake(x):
        return (x.new_empty((x.shape[0], n_out)), w_shard.new_empty((n_out, k_in)))
    _require_cuda(x, "ag_mm")
    rt, gid, n, me = _group(group)
    shard_off, full_off = int(_buf[0]), int(_buf[1])
    assert w_shard.data_ptr() == rt.heap_base + shard_off, "weight shard is not at its symmetric offset"
    xc = x if (x.stride(1) == 1 and x.stride(0) % 8 == 0 and x.data_ptr() % 16 == 0) else x.contiguous()
    M, K = xc.shape
    assert K == k_in
    out = torch.empty((M, n_out), dtype=torch.bfloat16, device=x.device)
    from . import gemm as _gemm
    _gemm.note_fused_call("ag", M, n_out, K, True, True, xc.stride(), (1, k_in), group, _buf)
    check(rt.lib.edb_ag_gemm_epoch_bf16(gid, out.data_ptr(), xc.data_ptr(),
                                        bias.data_ptr() if bias is not None else None, shard_off,
                                        full_off, M, n_out, K, xc.stride(0), n_out, rt.stream()))
    w_full = SymmBuffer(rt, full_off, n_out * k_in * 2).tensor(torch.bfloat16, (n_out, k_in))
    return out, w_full


def mm_push(a, b, group, *, _buf):
    """aten.mm whose result is reduce-scattered over its rows (mm -> flatten ->
    reduce_scatter_start of the zero2/zero3 graphs), push half: a @ b on the regular GEMM path
    (cta_group::2 pairs, split-K) with every row block stored into its owner's receive slot over
    NVLink; no flags at all — the epoch barrier in front of `rs_finish` makes the slots complete.
    _buf = (symmetric offset of the n receive slots,).  Returns an empty token for graph ordering."""
    if _is_fake(a):
        return a.new_empty((0,))
    _require_cuda(a, "mm_push")
    from . import gemm as _gemm
    rt, gid, n, me = _group(group)
    M, K = a.shape
    N = b.shape[1]
    pa, pb = _gemm._prepare(a, 1), _gemm._prepare(b, 0)
    if pa is None or pb is None:
        raise _lib.EdbUnsupported(_lib.EDB_E_UNSUPPORTED, "mm_push: operand layout")
    (ta, a_k, lda), (tb, b_k, ldb) = pa, pb
    check(rt.lib.edb_gemm_push_bf16(gid, int(_buf[0]), ta.data_ptr(), tb.data_ptr(), M, N, K, lda,
                                    ldb, 1 if a_k else 0, 1 if b_k else 0, rt.stream()))
    _gemm.note_fused_call("push", M, N, K, a_k, b_k, a.stride(), b.stride(), group, _buf)
    return torch.empty((0,), dtype=a.dtype, device=a.device)


def rs_finish(tokens, group, *, _bufs, _numels, _scale=1.0, _out_dtype=None):
    """Reduce the receive slots of the pushed GEMMs `tokens` came from, all in one kernel:
    item i -> flat shard of _numels[i] elements = sum over ranks (rank order, fp32) * _scale.
    _bufs[i] = the (_buf) given to mm_push i.  The caller puts an epoch barrier in front: every
    slot is complete, nothing to wait for."""
    out_dtype = _out_dtype or torch.bfloat16
    if tokens and _is_fake(tokens[0]):
        return [tokens[0].new_empty((int(k),), dtype=out_dtype) for k in _numels]
    rt, gid, n, me = _group(group)
    dev = tokens[0].device
    outs = [torch.empty((int(k),), dtype=out_dtype, device=dev) for k in _numels]
    cnt = len(outs)
    dsts = (ctypes.c_void_p * cnt)(*[o.data_ptr() for o in outs])
    recv = (ctypes.c_uint64 * cnt)(*[int(b[0]) for b in _bufs])
    chunk = (ctypes.c_int64 * cnt)(*[int(k) * 2 for k in _numels])  # slots hold bf16
    check(rt.lib.edb_rs_finish_local(gid, cnt, dsts, recv, chunk, float(_scale),
                                     _TORCH_DTYPE_CODE[out_dtype], rt.stream()))
    return outs


COMM_FUNCS = [all_reduce_start, all_gather_start, reduce_scatter_start, all_to_all_start]
COMM_SYNC_FUNCS = [all_reduce_end, all_gather_end, reduce_scatter_end, all_to_all_end]
CUSTOM_FUNCS = COMM_FUNCS + COMM_SYNC_FUNCS + [scatter_wrapper, copy_wrapper]
FUSED_FUNCS = [ag_mm, mm_push, rs_finish, epoch_barrier, ag_prefetch, gathered]
