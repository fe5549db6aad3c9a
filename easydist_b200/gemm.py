"""Sharded-op kernel dispatch for dense contractions.

The sharded FX graph the reference executes calls ATen for every compute node
(easydist/torch/compile_auto.py:752-756 runs the GraphModule op by op; the Linear layers are
`aten.mm` / `aten.addmm`).  Here bf16 `aten.mm` / `aten.addmm` nodes are dispatched to the
hand-written tcgen05 GEMM of libedb.so:

  * all four operand layouts (row/column-major A and B) map to kernel variants, so Linear forward,
    dgrad and wgrad need no transposes;
  * the bias of `addmm` is added in the kernel epilogue;
  * operands whose leading dimension breaks TMA's 16-byte stride rule (e.g. the GPT-2 LM head,
    vocab 50257) are copied once into a padded buffer by the box-copy kernel, outputs with an
    unaligned N are produced into a padded buffer and returned as a narrowed view — the alternative
    is cuBLAS falling back to sm_75-class `align1` kernels (measured 3.7 ms vs ~0.5 ms per GEMM).

Whatever still cannot run natively (non-bf16, degenerate strides) goes to ATen and is counted, so
the share of native GEMMs is visible in `stats()`.
"""
import torch
from torch._subclasses.fake_tensor import FakeTensor

from . import _lib
from ._lib import check, i64_array

_stats = {"edb_gemm": 0, "aten_mm": 0, "padded_operands": 0, "unsupported": {}}
_calls = []  # (M, N, K, a_kmajor, b_kmajor, a.stride(), b.stride()) of the native launches since reset_stats()


def stats():
    return {"edb_gemm": _stats["edb_gemm"], "aten_mm": _stats["aten_mm"],
            "edb_gemm_epi": _stats.get("edb_gemm_epi", 0),
            "padded_operands": _stats["padded_operands"], "unsupported": dict(_stats["unsupported"])}


def reset_stats():
    _stats["edb_gemm"] = 0
    _stats["edb_gemm_epi"] = 0
    _stats["aten_mm"] = 0
    _stats["padded_operands"] = 0
    _stats["unsupported"] = {}
    del _calls[:]
    del _fused_calls[:]
    _pf_calls.clear()


def recorded_calls():
    return list(_calls)


_pf_calls = {}  # index into _calls -> prefetch descriptor carried by that launch
_fused_calls = []  # dicts: kind ("ag" | "push"), M, N, K, layouts / strides, group, _buf


def note_fused_call(kind, M, N, K, a_k, b_k, a_stride, b_stride, group, buf):
    """Fused collective GEMMs (reshard.ag_mm / mm_push) report here so that the bench can replay the
    step's complete GEMM launch list — the fused kernels are the dominant ones at N > 1."""
    if len(_fused_calls) < 8192:
        _fused_calls.append({"kind": kind, "M": int(M), "N": int(N), "K": int(K), "a_k": bool(a_k),
                             "b_k": bool(b_k), "a_stride": tuple(a_stride),
                             "b_stride": tuple(b_stride), "group": list(group),
                             "buf": tuple(int(b) for b in buf)})


def recorded_fused_calls():
    return list(_fused_calls)


def _stream(t):
    return torch.cuda.current_stream(t.device).cuda_stream


def _padded_copy(t):
    """t: 2-D bf16 with unit stride along dim 1 -> same values in a buffer whose row stride is a
    multiple of 8 elements (and 16-byte aligned base)."""
    rows, cols = t.shape
    ld = (cols + 7) // 8 * 8
    buf = torch.empty((rows, ld), dtype=t.dtype, device=t.device)
    lib = _lib.load()
    check(lib.edb_box_copy_local(buf.data_ptr(), i64_array([ld * 2, 2]), t.data_ptr(),
                                 i64_array([t.stride(0) * 2, 2]), i64_array([rows, cols]), 2, 2,
                                 _stream(t)))
    _stats["padded_operands"] += 1
    return buf[:, :cols]


def _prepare(t, unit_dim):
    """Return (tensor, kmajor_flag_for_that_unit_dim, ld) with a TMA-legal layout, or None.
    `unit_dim` semantics: for A=[M,K] K-major means stride(1)==1; for B=[K,N] 'K-major' means
    stride(0)==1 (stored [N,K])."""
    if t.shape[0] == 1 or t.shape[1] == 1:
        return None  # degenerate strides: leave to ATen
    s0, s1 = t.stride()
    if s1 == 1:
        rowmajor = t
    elif s0 == 1:
        rowmajor = t.t()  # a view with unit stride along its dim 1
    else:
        return None
    ld = rowmajor.stride(0)
    if ld % 8 or rowmajor.data_ptr() % 16:
        rowmajor = _padded_copy(rowmajor)
        ld = rowmajor.stride(0)
    unit_is_dim1 = (s1 == 1)
    kmajor = unit_is_dim1 if unit_dim == 1 else not unit_is_dim1
    return rowmajor, kmajor, ld


def _pf_arrays(pf):
    import ctypes
    items = pf["items"]
    k = len(items)
    # item = (src_off, dst_off, bytes, dst_stride[, src_stride])
    return (k, (ctypes.c_uint64 * k)(*[int(i[0]) for i in items]),
            (ctypes.c_uint64 * k)(*[int(i[1]) for i in items]),
            (ctypes.c_int64 * k)(*[int(i[2]) for i in items]),
            (ctypes.c_int64 * k)(*[int(i[3]) for i in items]),
            (ctypes.c_int64 * k)(*[int(i[4]) if len(i) > 4 else 0 for i in items]))


def prefetch_standalone(pf, device):
    """The all-gather prefetch `pf` as its own launch (edb_ag_prefetch)."""
    from .runtime import get_runtime
    rt = get_runtime()
    gid = rt.group(pf["group"])
    k, src, dst, nbytes, stride, sstride = _pf_arrays(pf)
    check(rt.lib.edb_ag_prefetch(gid, k, src, dst, nbytes, stride, sstride, rt.stream()))


EPI_ADD, EPI_GELU_BWD = 1, 2


def _launch(a, b, bias, pf=None, epi=None):
    pa = _prepare(a, 1)
    pb = _prepare(b, 0)
    if pa is None or pb is None:
        return None
    (ta, a_k, lda), (tb, b_k, ldb) = pa, pb
    M, K = a.shape
    N = b.shape[1]
    ldc = (N + 7) // 8 * 8
    out = torch.empty((M, ldc), dtype=torch.bfloat16, device=a.device)
    if bias is not None and (N % 8 or bias.data_ptr() % 16 or not bias.is_contiguous()):
        return None
    lib = _lib.load()
    if epi is not None:
        op, aux = epi
        if N % 8 or aux.dtype != torch.bfloat16 or aux.shape != (M, N) or aux.stride(1) != 1 or \
                aux.stride(0) % 8 or aux.data_ptr() % 16:
            return None
        import ctypes
        if pf:
            from .runtime import get_runtime
            gid = get_runtime().group(pf["group"])
            k, src, dst, nbytes, stride, sstride = _pf_arrays(pf)
        else:
            gid, k, src, dst, nbytes, stride, sstride = 0, 0, None, None, None, None, None
        check(lib.edb_gemm_epi_bf16(out.data_ptr(), ta.data_ptr(), tb.data_ptr(),
                                    bias.data_ptr() if bias is not None else None,
                                    aux.data_ptr(), aux.stride(0), int(op), M, N, K, lda, ldb, ldc,
                                    1 if a_k else 0, 1 if b_k else 0, gid, k, src, dst, nbytes,
                                    stride, sstride, _stream(a)))
        _stats["edb_gemm_epi"] = _stats.get("edb_gemm_epi", 0) + 1
    elif pf:
        # the GEMM carries an all-gather prefetch for a later kernel (lowering.prefetch_param_gathers)
        from .runtime import get_runtime
        gid = get_runtime().group(pf["group"])
        k, src, dst, nbytes, stride, sstride = _pf_arrays(pf)
        check(lib.edb_gemm_pf_bf16(out.data_ptr(), ta.data_ptr(), tb.data_ptr(),
                                   bias.data_ptr() if bias is not None else None, M, N, K, lda,
                                   ldb, ldc, 1 if a_k else 0, 1 if b_k else 0, gid, k, src, dst,
                                   nbytes, stride, sstride, _stream(a)))
    else:
        check(lib.edb_gemm_bf16(out.data_ptr(), ta.data_ptr(), tb.data_ptr(),
                                bias.data_ptr() if bias is not None else None, M, N, K, lda, ldb,
                                ldc, 1 if a_k else 0, 1 if b_k else 0, 0, _stream(a)))
    _stats["edb_gemm"] += 1
    if len(_calls) < 8192:
        _calls.append((M, N, K, bool(a_k), bool(b_k), tuple(a.stride()), tuple(b.stride())))
        if pf:
            _pf_calls[len(_calls) - 1] = pf
    return out if ldc == N else out[:, :N]


def _eligible(a, b):
    return (a.is_cuda and a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16
            and a.dim() == 2 and b.dim() == 2 and a.numel() > 0 and b.numel() > 0)


def _count_unsupported(a, b):
    key = (tuple(a.shape), tuple(a.stride()), tuple(b.shape), tuple(b.stride()), str(a.dtype))
    _stats["unsupported"][key] = _stats["unsupported"].get(key, 0) + 1
    _stats["aten_mm"] += 1


def mm(a, b, *, _pf=None):
    """aten.mm.default(a, b) with bf16 operands on the tcgen05 kernel.
    `_pf`: all-gather prefetch carried by this launch ({"group": ranks, "items": [(src_off,
    dst_off, bytes, dst_stride), ...]}, see edb_gemm_pf_bf16)."""
    if isinstance(a, FakeTensor) or isinstance(b, FakeTensor) or a.is_meta:
        return torch.ops.aten.mm.default(a, b)
    out = _launch(a, b, None, _pf) if _eligible(a, b) else None
    if out is None:
        if _pf:
            prefetch_standalone(_pf, a.device)  # the gather must happen whoever runs the GEMM
        _count_unsupported(a, b)
        return torch.ops.aten.mm.default(a, b)
    return out


def recorded_prefetches():
    return dict(_pf_calls)


def mm_add(a, b, res, bias=None, *, _pf=None):
    """res + (a @ b [+ bias]) in one kernel: the residual add behind a Linear fused into the GEMM
    epilogue (aten.add.Tensor(res, aten.addmm(bias, a, b)) of the traced graph)."""
    if isinstance(a, FakeTensor) or isinstance(b, FakeTensor) or a.is_meta:
        y = torch.ops.aten.mm.default(a, b) if bias is None else torch.ops.aten.addmm.default(bias, a, b)
        return torch.ops.aten.add.Tensor(res, y)
    ok_bias = bias is None or (bias.dim() == 1 and bias.dtype == torch.bfloat16 and
                               bias.shape[0] == b.shape[1])
    if _eligible(a, b) and ok_bias and isinstance(res, torch.Tensor) and res.dim() == 2:
        out = _launch(a, b, bias, _pf, (EPI_ADD, res))
        if out is not None:
            return out
    y = mm(a, b, _pf=_pf) if bias is None else addmm(bias, a, b, _pf=_pf)
    return torch.ops.aten.add.Tensor(res, y)


def mm_gelu_bwd(a, b, pre, *, _pf=None):
    """aten.gelu_backward(a @ b, pre, approximate='tanh') in one kernel (GEMM epilogue)."""
    if isinstance(a, FakeTensor) or isinstance(b, FakeTensor) or a.is_meta:
        return torch.ops.aten.gelu_backward.default(torch.ops.aten.mm.default(a, b), pre,
                                                    approximate="tanh")
    if _eligible(a, b) and isinstance(pre, torch.Tensor) and pre.dim() == 2:
        out = _launch(a, b, None, _pf, (EPI_GELU_BWD, pre))
        if out is not None:
            return out
    return torch.ops.aten.gelu_backward.default(mm(a, b, _pf=_pf), pre, approximate="tanh")


def addmm(bias, a, b, *, _pf=None):
    """aten.addmm.default(bias, a, b) = bias + a @ b, bias added in the GEMM epilogue."""
    if isinstance(a, FakeTensor) or isinstance(b, FakeTensor) or a.is_meta:
        return torch.ops.aten.addmm.default(bias, a, b)
    if _eligible(a, b) and bias.dim() == 1 and bias.dtype == torch.bfloat16 and \
            bias.shape[0] == b.shape[1]:
        out = _launch(a, b, bias, _pf)
        if out is not None:
            return out
    if _eligible(a, b):
        out = _launch(a, b, None, _pf)
        if out is not None:
            return torch.ops.aten.add.Tensor(out, bias)
    if _pf:
        prefetch_standalone(_pf, a.device)
    _count_unsupported(a, b)
    return torch.ops.aten.addmm.default(bias, a, b)
