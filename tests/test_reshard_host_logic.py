"""Host side of easydist_b200.reshard with the C-ABI mocked out: which entry point each of the
reference-signature callables reaches, with which arguments (shapes, dims, dtype / redop codes,
symmetric offsets, group ids), what it returns, and the errors it raises — no GPU, no compute.
(The kernels behind the entry points are checked by the -m gpu tests.)"""
import ctypes

import pytest
import torch

from easydist_b200 import _lib, reshard
from easydist_b200.runtime import SymmBuffer


class _FakeLib:
    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        if not name.startswith("edb_"):
            raise AttributeError(name)

        def fn(*args):
            self.calls.append((name, args))
            if name == "edb_scatter":
                pass
            return 0
        return fn


class _FakeRuntime:
    def __init__(self, world=2, me=0):
        self.lib = _FakeLib()
        self.world, self.me = world, me
        self.slab = torch.zeros(1 << 22, dtype=torch.uint8)
        self.groups = {}
        self._ring = 1 << 16
        self.options = {"allreduce_oneshot_bytes": 512 * 1024}

    def group(self, ranks, slot=None):
        return self.groups.setdefault(tuple(ranks), len(self.groups))

    def group_size(self, gid):
        return self.world

    def group_index(self, gid):
        return self.me

    def get_option(self, name):
        return self.options[name]

    def stream(self):
        return ctypes.c_void_p(0)

    def ring_alloc(self, nbytes):
        off = self._ring
        self._ring += (nbytes + 255) // 256 * 256
        return SymmBuffer(self, off, nbytes)


@pytest.fixture
def rt(monkeypatch):
    fake = _FakeRuntime()
    monkeypatch.setattr(reshard, "get_runtime", lambda: fake)
    monkeypatch.setattr(reshard, "_require_cuda", lambda t, what: None)
    return fake


def _i64(arr, n):
    return [arr[i] for i in range(n)]


def test_all_gather_reaches_the_abi_with_local_shape_and_returns_gathered_view(rt):
    x = torch.arange(24, dtype=torch.float32).view(2, 3, 4)
    out = reshard.all_gather_start(x, 1, [0, 1], _buf=(4096, 2 * x.numel() * 4))
    (name, args), = rt.lib.calls
    assert name == "edb_all_gather"
    gid, off, ptr, shape, ndim, dim, esize, _ = args
    assert (gid, off, ptr, ndim, dim, esize) == (0, 4096, x.data_ptr(), 3, 1, 4)
    assert _i64(shape, 3) == [2, 3, 4]
    assert out.shape == (2, 6, 4) and out.dtype == x.dtype
    assert out.data_ptr() == rt.slab.data_ptr() + 4096          # zero-copy view of the static buffer
    assert reshard.all_gather_end(out, 1, [0, 1]) is out
    # negative dims, non-contiguous input (sharding.py:106-107 contiguous-ises too)
    rt.lib.calls.clear()
    reshard.all_gather_start(x.transpose(0, 2), -1, [0, 1])
    (_, args), = rt.lib.calls
    assert args[5] == 2 and _i64(args[3], 3) == [4, 3, 2]


def test_reduce_scatter_codes_scale_and_divisibility(rt):
    x = torch.ones(4, 6, dtype=torch.bfloat16)
    out = reshard.reduce_scatter_start(x, "avg", 1, [0, 1], _scale=0.5, _out_dtype=torch.float32)
    (name, args), = rt.lib.calls
    assert name == "edb_reduce_scatter"
    assert args[5:7] == (2, 1)                                   # ndim, dim
    assert args[7] == _lib.DTYPE_CODES["bfloat16"] and args[8] == _lib.REDOP_CODES["avg"]
    assert args[9] == 0.5 and args[10] == _lib.DTYPE_CODES["float32"]
    assert out.shape == (4, 3) and out.dtype == torch.float32
    assert reshard.reduce_scatter_end(out, "avg", 1, [0, 1]) is out
    with pytest.raises(AssertionError):                          # sharding.py:136-137
        reshard.reduce_scatter_start(torch.ones(3, 5), "sum", 0, [0, 1])
    with pytest.raises(_lib.EdbError):
        reshard.reduce_scatter_start(torch.ones(4, 4), "prod", 0, [0, 1])


def test_all_reduce_one_and_two_shot_buffers(rt):
    small = torch.ones(1024)
    out = reshard.all_reduce_start(small, "sum", [0, 1])
    assert reshard.all_reduce_end(out, "sum", [0, 1]) is out
    big = torch.ones(1 << 18)                                    # 1 MiB > one-shot threshold
    reshard.all_reduce_start(big, "max", [0, 1])
    (_, a_small), (_, a_big) = rt.lib.calls
    assert a_small[2] != 0 and a_small[3] == 0                   # one staging buffer
    assert a_big[2] != 0 and a_big[3] != 0 and a_big[2] != a_big[3]
    assert a_big[7] == _lib.REDOP_CODES["max"]
    with pytest.raises(_lib.EdbError):
        reshard.all_reduce_start(torch.ones(4, dtype=torch.bool), "sum", [0, 1])


def test_scatter_wrapper_chunks_like_torch_chunk(rt):
    x = torch.arange(10.0).view(5, 2)
    out = reshard.scatter_wrapper(x, 2, 0, 1)
    (name, args), = rt.lib.calls
    assert name == "edb_scatter" and out.shape == (2, 2)         # ceil-div blocks: 3 + 2 rows
    assert args[3:7] == (2, 0, 2, 1)                              # ndim, dim, chunks, index
    with pytest.raises(IndexError):                               # past the last torch.chunk piece
        reshard.scatter_wrapper(torch.ones(2, 2), 4, 0, 3)
    assert reshard.scatter_wrapper(torch.ones(0, 4), 2, 0, 1).shape == (0, 4)


def test_all_to_all_shape_and_coordinate_checks(rt):
    x = torch.ones(2, 8, 4)
    out = reshard.all_to_all_start(x, 0, 1, 2, 0, [0, 1])
    assert out.shape == (4, 4, 4) and rt.lib.calls[-1][0] == "edb_all_to_all"
    with pytest.raises(_lib.EdbError):
        reshard.all_to_all_start(torch.ones(2, 3), 0, 1, 2, 0, [0, 1])   # 3 not divisible by 2
    with pytest.raises(AssertionError):
        reshard.all_to_all_start(x, 0, 1, 2, 1, [0, 1])                   # not this rank's coordinate


def test_product_path_has_no_cpu_fallback():
    with pytest.raises(_lib.EdbError, match="no CPU path"):
        reshard.all_gather_start(torch.ones(2, 2), 0, [0, 1])
    with pytest.raises(_lib.EdbError, match="no CPU path"):
        reshard.scatter_wrapper(torch.ones(2, 2), 2, 0, 0)


def test_runtime_group_registry():
    """Runtime.group: one C-ABI group per set of ranks, created on first use and cached; slots
    follow creation order."""
    from easydist_b200.runtime import Runtime

    class Lib:
        def __init__(self):
            self.created = []

        def edb_group_create(self, ranks, n, slot, out):
            self.created.append(([ranks[i] for i in range(n)], slot))
            out._obj.value = len(self.created) - 1
            return 0

        def edb_group_info(self, gid, n, me):
            n._obj.value = len(self.created[gid][0])
            me._obj.value = 1
            return 0

    rt = object.__new__(Runtime)
    rt.lib, rt._groups, rt._group_meta, rt._attached = Lib(), {}, {}, True
    g0 = rt.group([0, 1])
    assert rt.group((0, 1)) == g0                                            # cached
    g1 = rt.group([0, 2])
    g2 = rt.group([0, 1, 2, 3])
    assert len({g0, g1, g2}) == 3
    assert rt.lib.created == [([0, 1], 0), ([0, 2], 1), ([0, 1, 2, 3], 2)]
    assert rt.group_size(g1) == 2 and rt.group_index(g1) == 1
    assert rt.group_size(g2) == 4 and rt.group_index(g2) == 1
    assert rt.group([0, 2]) == g1 and rt.group([0, 1, 2, 3]) == g2
