"""Multi-GPU parity worker: one process per GPU (torchrun), compares every reshard kernel with the
oracle on the same seeded inputs, bit for bit.  Launched by tests/test_gpu_multi.py and directly:

    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29531 \
        tests/mgpu_worker.py [--bench]
"""
import argparse
import os
import sys
import zlib

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from easydist_b200 import reshard, runtime  # noqa: E402
from oracle import reshard_oracle as O  # noqa: E402  (tests may use the oracle as the checker)

TORCH_DT = {"float32": torch.float32, "int64": torch.int64, "float16": torch.float16,
            "bfloat16": torch.bfloat16, "int32": torch.int32, "uint8": torch.uint8,
            "float64": torch.float64}


def inputs_for(key, shape, dtype, world, lo=-8, hi=9):
    """Integer-valued inputs of every rank (known to all ranks) so reductions are exact."""
    out = []
    for r in range(world):
        rng = np.random.RandomState(zlib.crc32(key.encode()) % (2 ** 31 - 100000) + 1000 * r)
        out.append(rng.randint(lo, hi, size=shape).astype(np.float32 if dtype == "bfloat16"
                                                          else dtype))
    return out


def to_dev(x, dtype):
    x = np.asarray(x)
    t = torch.from_numpy(np.ascontiguousarray(x)).reshape(x.shape).cuda()
    return t.to(TORCH_DT[dtype])


def check_equal(got, want, what):
    g = got.float().cpu().numpy() if got.dtype in (torch.bfloat16, torch.float16) else \
        got.cpu().numpy()
    w = want.astype(np.float32) if got.dtype in (torch.bfloat16, torch.float16) else want
    if g.shape != tuple(w.shape) or not np.array_equal(g, w):
        raise AssertionError(f"{what}: mismatch shape {g.shape} vs {w.shape}; "
                             f"max|d|={np.abs(g.astype(np.float64) - w).max() if g.shape == w.shape else 'n/a'}")


def run_cases(rank, world, group, tag=""):
    n_ok = 0
    shapes_ag = [((3, 4), 0), ((3, 4), 1), ((2, 3, 5), 2), ((7,), 0), ((64, 1024), 0),
                 ((64, 1024), 1), ((5, 33), 1), ((2, 16, 128, 32), 2), ((1, 1, 16, 128), 2)]
    for dtype in ("float32", "int64", "bfloat16", "uint8"):
        for shape, dim in shapes_ag:
            key = f"ag{tag}_{shape}_{dim}_{dtype}"
            xs = inputs_for(key, shape, dtype, world, 0 if dtype == "uint8" else -8)
            want = O.all_gather(xs, dim)[rank]
            got = reshard.all_gather_start(to_dev(xs[rank], dtype), dim, group)
            check_equal(got, want, key)
            n_ok += 1
    a2a = [((2, 4 * world), 0, 1), ((2 * world, 3), 1, 0), ((2, 3, 2 * world), 0, 2),
           ((2, world, 5), 2, 1), ((2, 128, 16 * world), 0, 2), ((2 * world, 16, 8 * world), 2, 0),
           ((2, 32 * world, 128, 32), 0, 1), ((64 * world, 64), 1, 0)]
    for dtype in ("float32", "bfloat16", "int64"):
        for shape, g, s in a2a:
            key = f"a2a{tag}_{shape}_{g}_{s}_{dtype}"
            xs = inputs_for(key, shape, dtype, world)
            want = O.all_to_all(xs, g, s)[rank]
            got = reshard.all_to_all_start(to_dev(xs[rank], dtype), g, s, world, rank, group)
            check_equal(got, want, key)
            n_ok += 1
    red_shapes = [((2 * world, 3), 0), ((3, 2 * world), 1), ((2, 3, world), 2),
                  ((64 * world, 256), 0), ((16, 8 * world, 32), 1), ((1, 1024 * world), 1)]
    for dtype in ("float32", "bfloat16", "float16", "int64", "int32", "float64"):
        ops = ("sum", "max", "min") + (() if dtype.startswith("int") else ("avg",))
        for op in ops:
            for shape, dim in red_shapes:
                key = f"rs{tag}_{shape}_{dim}_{dtype}_{op}"
                # avg: multiples of `world` keep sum/world exact in every float dtype
                xs = inputs_for(key, shape, dtype, world)
                if op == "avg":
                    xs = [x * world for x in xs]
                want = O.reduce_scatter(xs, op, dim)[rank]
                got = reshard.reduce_scatter_start(to_dev(xs[rank], dtype), op, dim, group)
                check_equal(got, want, key)
                n_ok += 1
            for shape in [(5, 3), (), (1024,), (300, 1000), (1 << 20,)]:
                key = f"ar{tag}_{shape}_{dtype}_{op}"
                xs = inputs_for(key, shape, dtype, world)
                if op == "avg":
                    xs = [x * world for x in xs]
                want = O.all_reduce(xs, op)[rank]
                got = reshard.all_reduce_start(to_dev(xs[rank], dtype), op, group)
                check_equal(got, want, key)
                n_ok += 1
    # fused scale + cast on reduce-scatter (gradient averaging into fp32)
    xs = inputs_for("rs_cast", (8 * world, 64), "bfloat16", world)
    want = O.reduce_scatter([x.astype(np.float32) for x in xs], "sum", 0)[rank] * 0.5
    got = reshard.reduce_scatter_start(to_dev(xs[rank], "bfloat16"), "sum", 0, group, _scale=0.5,
                                       _out_dtype=torch.float32)
    check_equal(got, want, "rs_cast")
    # halo exchange vs halo_padding (metashard/halo.py:33-55)
    for shape, dim, halo in [((6, 5), 0, 2), ((4, 6, 3), 1, 1), ((3, 64), 1, 16)]:
        xs = inputs_for(f"halo_{shape}", shape, "float32", world)
        want = O.halo_padding(xs, halo, dim)[rank]
        got = reshard.halo_exchange(to_dev(xs[rank], "float32"), dim, halo, group)
        check_equal(got, want, f"halo {shape} {dim} {halo}")
        n_ok += 1
    return n_ok


def run_randn_cases(rank, world, group, ops=None, device="cuda"):
    """SURVEY.md section 8(d) config 5's second input class: `randn` with seed 1234 + rank (the
    integer-valued batteries above make reductions exact; here they round).  Data movement stays
    bit-exact; fp32 reductions within 1e-5 of the oracle relative to the largest element (both sum
    in fp32, the kernel in rank order); bf16 reductions within one bf16 ulp of the fp32 sum at the
    largest element (fp32 accumulation, one rounding).  `ops` defaults to the libedb callables; the
    CPU suite passes the gloo stand-ins to check this checker."""
    ops = ops or reshard
    n_ok = 0

    def inputs(shape, dtype):
        out = []
        for r in range(world):
            g = torch.Generator().manual_seed(1234 + r)
            x = torch.randn(shape, generator=g)
            if dtype == "bfloat16":
                x = x.bfloat16().float()   # the values the kernel sees
            out.append(x.numpy())
        return out

    def dev(x, dtype):
        return torch.from_numpy(np.ascontiguousarray(x)).to(device=device, dtype=TORCH_DT[dtype])

    def close(got, want, dtype, what):
        g = got.float().cpu().numpy().astype(np.float64)
        w = np.asarray(want, dtype=np.float64)
        assert g.shape == w.shape, f"{what}: shape {g.shape} vs {w.shape}"
        top = float(np.abs(w).max()) if w.size else 0.0
        tol = 1e-5 * top if dtype == "float32" else 2.0 ** (np.floor(np.log2(max(top, 1e-30))) - 7)
        err = float(np.abs(g - w).max()) if w.size else 0.0
        if err > tol:
            raise AssertionError(f"{what}: max |d| {err:.3e} > {tol:.3e}")

    for dtype in ("float32", "bfloat16"):
        for shape, dim in [((64, 1024), 0), ((64, 1024), 1), ((2, 16, 128, 32), 2)]:
            xs = inputs(shape, dtype)
            got = ops.all_gather_start(dev(xs[rank], dtype), dim, group)
            check_equal(got, O.all_gather(xs, dim)[rank], f"randn ag {shape} {dim} {dtype}")
            n_ok += 1
        for shape, g_, s_ in [((2, 128, 16 * world), 0, 2), ((64 * world, 64), 1, 0)]:
            xs = inputs(shape, dtype)
            got = ops.all_to_all_start(dev(xs[rank], dtype), g_, s_, world, rank, group)
            check_equal(got, O.all_to_all(xs, g_, s_)[rank], f"randn a2a {shape} {dtype}")
            n_ok += 1
        for shape, dim in [((64 * world, 256), 0), ((16, 8 * world, 32), 1), ((1, 1024 * world), 1)]:
            xs = inputs(shape, dtype)
            got = ops.reduce_scatter_start(dev(xs[rank], dtype), "sum", dim, group)
            close(got, O.reduce_scatter([x.astype(np.float32) for x in xs], "sum", dim)[rank], dtype,
                  f"randn rs {shape} {dim} {dtype}")
            n_ok += 1
        for shape in [(1024,), (300, 1000), (1 << 20,)]:
            xs = inputs(shape, dtype)
            got = ops.all_reduce_start(dev(xs[rank], dtype), "sum", group)
            close(got, O.all_reduce([x.astype(np.float32) for x in xs], "sum")[rank], dtype,
                  f"randn ar {shape} {dtype}")
            n_ok += 1
    return n_ok


def run_push_cases(rank, world, group, passes=4, big=True):
    """The push-protocol collectives (edb_*_push: static per-node buffers, one flag per peer, an
    epoch barrier between reuses of a buffer) bit for bit against the oracle: every op, the LL
    threshold switched off for half of the passes so that the push kernels themselves run on the
    small shapes too, random rank skew, buffers reused after a barrier (as a compiled step does)."""
    rt = runtime.get_runtime()
    n_ok = 0
    oneshot = rt.get_option("allreduce_oneshot_bytes")
    ll_saved = rt.get_option("ll_max_bytes")
    x0 = to_dev(np.zeros(1, dtype=np.float32), "float32")
    ag_cases = [((3, 4), 0), ((3, 4), 1), ((2, 3, 5), 2), ((7,), 0), ((64, 1024), 0), ((64, 1024), 1),
                ((5, 33), 1), ((2, 16, 128, 32), 2), ((512, 2048), 0)]
    a2a_cases = [((2, 4 * world), 0, 1), ((2 * world, 3), 1, 0), ((2, 3, 2 * world), 0, 2),
                 ((2, 128, 16 * world), 0, 2), ((2 * world, 16, 8 * world), 2, 0),
                 ((64 * world, 1024), 1, 0)]
    red_cases = [((2 * world, 3), 0), ((3, 2 * world), 1), ((2, 3, world), 2), ((64 * world, 256), 0),
                 ((16, 8 * world, 32), 1), ((512 * world, 1024), 0)]
    ar_cases = [(5, 3), (), (1024,), (300, 1000), (1 << 20,), (world * 1024 * 512,)]
    if not big:
        # bench.py's pre-timing battery: the host-side oracle work of the world-scaled shapes
        # (numpy over `world` ranks' inputs) would take minutes at 8 GPUs
        ag_cases, a2a_cases = ag_cases[:-1], a2a_cases[:-1]
        red_cases, ar_cases = red_cases[:-1], ar_cases[:-2] + [(256 * 1024,)]
    for pas in range(passes):
        rt.set_option("ll_max_bytes", ll_saved if pas % 2 == 0 else 0)
        mark = rt.mark()
        if rank % 2 == pas % 2:
            torch.cuda._sleep(2_000_000)  # skew: half of the ranks arrive late
        for dtype in ("float32", "bfloat16", "int64"):
            es = torch.empty((), dtype=TORCH_DT[dtype]).element_size()
            for shape, dim in ag_cases:
                key = f"pag{pas}_{shape}_{dim}_{dtype}"
                xs = inputs_for(key, shape, dtype, world)
                nb = int(np.prod(shape)) * es * world
                buf = rt.alloc(nb)
                got = reshard.all_gather_start(to_dev(xs[rank], dtype), dim, group,
                                               _buf=(buf.offset, nb), _push=1)
                check_equal(got, O.all_gather(xs, dim)[rank], key)
                n_ok += 1
            for shape, g, s_ in a2a_cases:
                key = f"pa2a{pas}_{shape}_{g}_{s_}_{dtype}"
                xs = inputs_for(key, shape, dtype, world)
                nb = int(np.prod(shape)) * es
                buf = rt.alloc(nb)
                got = reshard.all_to_all_start(to_dev(xs[rank], dtype), g, s_, world, rank, group,
                                               _buf=(buf.offset, nb), _push=1)
                check_equal(got, O.all_to_all(xs, g, s_)[rank], key)
                n_ok += 1
        for dtype in ("float32", "bfloat16", "int32", "float64"):
            es = torch.empty((), dtype=TORCH_DT[dtype]).element_size()
            ops_ = ("sum", "max") + (() if dtype.startswith("int") else ("avg",))
            for op in ops_:
                for shape, dim in red_cases:
                    key = f"prs{pas}_{shape}_{dim}_{dtype}_{op}"
                    xs = inputs_for(key, shape, dtype, world)
                    if op == "avg":
                        xs = [x * world for x in xs]
                    nb = int(np.prod(shape)) * es
                    buf = rt.alloc(nb)
                    got = reshard.reduce_scatter_start(to_dev(xs[rank], dtype), op, dim, group,
                                                       _buf=(buf.offset, nb), _push=1)
                    check_equal(got, O.reduce_scatter(xs, op, dim)[rank], key)
                    n_ok += 1
                for shape in ar_cases:
                    key = f"par{pas}_{shape}_{dtype}_{op}"
                    xs = inputs_for(key, shape, dtype, world)
                    if op == "avg":
                        xs = [x * world for x in xs]
                    numel = int(np.prod(shape)) if shape else 1
                    rb, ob = reshard.all_reduce_push_sizes(numel * es, numel, es, world, oneshot)
                    recv, outb = rt.alloc(rb), rt.alloc(ob)
                    got = reshard.all_reduce_start(to_dev(xs[rank], dtype), op, group,
                                                   _buf=(recv.offset, rb, outb.offset), _push=1)
                    check_equal(got, O.all_reduce(xs, op)[rank], key)
                    n_ok += 1
        # fused scale + cast
        xs = inputs_for(f"prs_cast{pas}", (8 * world, 64), "bfloat16", world)
        nb = 8 * world * 64 * 2
        buf = rt.alloc(nb)
        got = reshard.reduce_scatter_start(to_dev(xs[rank], "bfloat16"), "sum", 0, group, _scale=0.5,
                                           _out_dtype=torch.float32, _buf=(buf.offset, nb), _push=1)
        check_equal(got, O.reduce_scatter([x.astype(np.float32) for x in xs], "sum", 0)[rank] * 0.5,
                    "push rs_cast")
        n_ok += 1
        # the buffers are reused by the next pass: the barrier a compiled step ends with
        torch.cuda.synchronize()
        reshard.epoch_barrier(x0, group)
        rt.reset(mark)
    rt.set_option("ll_max_bytes", ll_saved)
    # CUDA-graph replay of a push sequence with changing inputs
    mark = rt.mark()
    xin = torch.zeros(64 * world, 256, device="cuda")
    nb = xin.numel() * 4
    b1, b2, b3, b4 = rt.alloc(nb * world), rt.alloc(nb), rt.alloc(nb * world), rt.alloc(nb)

    def seq():
        a = reshard.all_gather_start(xin, 0, group, _buf=(b1.offset, nb * world), _push=1)
        r_ = reshard.reduce_scatter_start(xin, "sum", 0, group, _buf=(b2.offset, nb), _push=1)
        ar = reshard.all_reduce_start(xin, "sum", group, _buf=(b3.offset, nb * world, b4.offset), _push=1)
        reshard.epoch_barrier(xin, group)
        return a, r_, ar

    for _ in range(2):
        seq()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = seq()
    for it in range(4):
        xs = inputs_for(f"pgraph{it}", (64 * world, 256), "float32", world)
        xin.copy_(to_dev(xs[rank], "float32"))
        graph.replay()
        torch.cuda.synchronize()
        check_equal(outs[0], O.all_gather(xs, 0)[rank], f"push graph ag {it}")
        check_equal(outs[1], O.reduce_scatter(xs, "sum", 0)[rank], f"push graph rs {it}")
        check_equal(outs[2], O.all_reduce(xs, "sum")[rank], f"push graph ar {it}")
        n_ok += 3
    reshard.epoch_barrier(x0, group)
    rt.reset(mark)
    rt.health()
    return n_ok


def run_p2p(rank, world, group):
    """Partition P2P redistribution vs the oracle's restatement of sharding.py:336-474."""
    n_ok = 0
    mesh = np.arange(world).reshape(world)
    g = np.arange(16 * 24, dtype=np.float32).reshape(16, 24)
    for src, dst in [((O.S(0),), (O.S(1),)), ((O.S(1),), (O.S(0),)), ((O.S(0),), (O.R,)),
                     ((O.R,), (O.S(1),))]:
        loc = O.make_locals(g, mesh, src)
        want = O.p2p_redistribute(loc, g.shape, mesh, src, dst)[rank]
        sp = O.partitions_from_spec(src, g.shape, mesh)
        tp = O.partitions_from_spec(dst, g.shape, mesh)
        recv = O.gen_recv_meta(sp, tp).get(rank, [])
        boxes = []
        for it in recv:
            s_part, t_part = sp[it.rank], tp[rank]
            boxes.append((it.rank, [a - b for a, b in zip(it.start, s_part.start)],
                          [a - b for a, b in zip(it.start, t_part.start)],
                          [e - s for s, e in zip(it.start, it.end)]))
        shapes = [[e - s for s, e in zip(p.start, p.end)] for p in sp]
        dshape = [e - s for s, e in zip(tp[rank].start, tp[rank].end)]
        got = reshard.box_exchange(to_dev(loc[rank], "float32"), dshape, boxes, shapes, group)
        check_equal(got, want, f"p2p {src}->{dst}")
        n_ok += 1
    return n_ok


def run_graph(rank, world, group, rows=64):
    """CUDA-graph capture + replay: epoch flags must keep working with static parameters
    (rows=64: flag protocol, 64 KiB messages; rows=4: low-latency packet protocol when enabled)."""
    rt = runtime.get_runtime()
    x = torch.zeros(rows, 256, device="cuda")
    buf_ag = rt.alloc(x.numel() * 4 * world)
    buf_rs = rt.alloc(x.numel() * 4 * world)
    buf_ar = rt.alloc(x.numel() * 4)

    def step():
        g = reshard.all_gather_start(x, 0, group, _buf=(buf_ag.offset, buf_ag.nbytes))
        r = reshard.reduce_scatter_start(g, "sum", 0, group, _buf=(buf_rs.offset, buf_rs.nbytes))
        a = reshard.all_reduce_start(r, "max", group, _buf=(buf_ar.offset, buf_ar.nbytes))
        return g, r, a

    def expect(vals):
        g = np.concatenate([np.full((rows, 256), v, np.float32) for v in vals])
        return g, g[rank * rows:(rank + 1) * rows] * world, np.full((rows, 256),
                                                                    max(vals) * world, np.float32)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        x.fill_(float(rank + 1))
        step()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = step()
    for it in range(5):
        x.fill_(float(rank + 1 + it))
        graph.replay()
        torch.cuda.synchronize()
        for o, w in zip(outs, expect([r + 1 + it for r in range(world)])):
            check_equal(o, w, f"graph replay {it}")
    return 5


def run_epoch(rank, world, group):
    """Epoch protocol (edb_epoch_barrier + flag-free fused kernels): a miniature train step

        AG+GEMM (epoch) x k  ->  push GEMM x k  ->  barrier -> rs_finish (local)  ->  in-place
        update of the symmetric weight shards ("optimizer")  ->  barrier

    repeated eagerly and from a replayed CUDA graph, with artificial rank skew (busy-wait kernels
    on alternating ranks) so that a missing rendezvous shows up as stale data.  Checked (i) bit for
    bit against the unfused kernels of this library (plain GEMM without split-K, like the fused
    kernel; GEMM -> reduce_scatter(avg) with the per-op flag protocol) and (ii) against a plain
    fp32 PyTorch computation of the same products (relative L2 error <= 6e-3: one bf16 rounding of
    the product / of each rank's partial product, 2^-9 rms).  The shapes include a K tail
    (K = 1000) and a reduce-scatter whose rows per rank are not a multiple of the tile pair."""
    from easydist_b200 import gemm
    rt = runtime.get_runtime()
    torch.manual_seed(4321)  # same on every rank: every rank knows every rank's operands
    ag_cases = [(M, N, K, wb) for (M, N, K, wb) in
                [(512, 256 * world, 256, False), (4096, 1024, 1024, True), (4096, 4096, 1024, True),
                 (4096, 3072, 1024, True), (384, 128 * world, 1000, False)]
                if N % world == 0 and N % 128 == 0 and (N // world) % 8 == 0]
    rs_cases = [(M, N, K) for (M, N, K) in
                [(128 * world, 256, 512), (1024, 1024, 4096), (4096, 1024, 4096), (1024, 4096, 4096),
                 (3072, 1024, 4096), (256 * world, 4096, 1024)] if (M // world) % 128 == 0]
    ag = []
    for (M, N, K, with_bias) in ag_cases:
        W = (torch.randn(N, K, device="cuda") * 0.1).bfloat16()
        x = torch.randn(M, K, device="cuda").bfloat16()
        bias = torch.randn(N, device="cuda").bfloat16() if with_bias else None
        rows = N // world
        shard_buf = rt.alloc(rows * K * 2, align=1024)
        full_buf = rt.alloc(N * K * 2, align=1024)
        w_shard = shard_buf.tensor(torch.bfloat16, (rows, K))
        w_shard.copy_(W[rank * rows:(rank + 1) * rows])
        ag.append((W, x, bias, shard_buf, full_buf, w_shard))
    rs = []
    g = torch.Generator(device="cuda").manual_seed(55)
    for (M, N, K) in rs_cases:
        a_all = [torch.randn(K, M, device="cuda", generator=g).bfloat16() for _ in range(world)]
        b_all = [torch.randn(K, N, device="cuda", generator=g).bfloat16() for _ in range(world)]
        recv = rt.alloc(M * N * 2, align=1024)
        stage = rt.alloc(M * N * 2, align=1024)
        rs.append((a_all, b_all, recv, stage))
    factor = torch.ones((), device="cuda", dtype=torch.bfloat16)  # the "step number", on device
    skew = [0]

    def maybe_sleep(parity):
        if skew[0] and rank % 2 == parity:
            torch.cuda._sleep(3_000_000)  # ~1.5 ms of busy waiting on half of the ranks

    def step():
        outs, fulls, toks, wants = [], [], [], []
        maybe_sleep(0)
        for (N_, (W, x, bias, shard_buf, full_buf, w_shard)) in zip(ag_cases, ag):
            M, N, K, _ = N_
            o, wf = reshard.ag_mm(x, w_shard, group, N, K, bias,
                                  _buf=(shard_buf.offset, full_buf.offset))
            outs.append(o)
            fulls.append(wf.clone())
        maybe_sleep(1)
        for (M, N, K), (a_all, b_all, recv, stage) in zip(rs_cases, rs):
            a, b = a_all[rank].t(), b_all[rank] * factor
            toks.append(reshard.mm_push(a, b, group, _buf=(recv.offset,)))
            part = gemm.mm(a, b)
            wants.append(reshard.reduce_scatter_start(part.flatten(), "avg", 0, group,
                                                      _buf=(stage.offset, M * N * 2)))
        maybe_sleep(0)
        toks[0] = reshard.epoch_barrier(toks[0], group)
        reds = reshard.rs_finish(toks, group, _bufs=[(r_[2].offset,) for r_ in rs],
                                 _numels=[M // world * N for (M, N, K) in rs_cases],
                                 _scale=1.0 / world)
        maybe_sleep(1)
        # the "optimizer": every rank rewrites its symmetric weight shard in place
        factor.add_(1)
        for (W, x, bias, shard_buf, full_buf, w_shard) in ag:
            rows = w_shard.shape[0]
            w_shard.copy_(W[rank * rows:(rank + 1) * rows] * factor)
        reshard.epoch_barrier(factor, group)
        return outs, fulls, reds, wants

    def check(it_factor, outs, fulls, reds, wants, what):
        n = 0
        for (M, N, K, with_bias), (W, x, bias, *_), o, wf in zip(ag_cases, ag, outs, fulls):
            Wi = (W * torch.tensor(it_factor, dtype=torch.bfloat16, device="cuda"))
            assert torch.equal(wf, Wi), f"{what}: epoch ag_mm gathered weight {(M, N, K)} x{it_factor}"
            # the fused kernel never splits K: neither may its reference
            rt.set_option("gemm_splitk", 0)
            try:
                ref = gemm.addmm(bias, x, Wi.t()) if with_bias else gemm.mm(x, Wi.t())
            finally:
                rt.set_option("gemm_splitk", 1)
            assert torch.equal(o, ref), f"{what}: epoch ag_mm {(M, N, K)} x{it_factor}: " \
                f"{(o.float() - ref.float()).abs().max()}"
            f32 = x.float() @ Wi.float().t() + (bias.float() if with_bias else 0.0)
            e = float((o.float() - f32).norm() / f32.norm())
            assert e <= 6e-3, f"{what}: epoch ag_mm vs fp32 {(M, N, K)}: rel l2 {e}"
            n += 2
        for (M, N, K), (a_all, b_all, *_), r_, w_ in zip(rs_cases, rs, reds, wants):
            assert torch.equal(r_, w_), f"{what}: push+rs_finish vs GEMM->reduce_scatter {(M, N, K)} " \
                f"x{it_factor}: {(r_.float() - w_.float()).abs().max()}"
            rows = M // world
            f32 = torch.zeros(rows, N, device="cuda")
            fb = torch.tensor(it_factor, dtype=torch.bfloat16, device="cuda")
            for r2 in range(world):
                f32 += a_all[r2].float().t()[rank * rows:(rank + 1) * rows] @ (b_all[r2] * fb).float()
            f32 /= world
            e = float((r_.float().view(rows, N) - f32).norm() / f32.norm())
            assert e <= 6e-3, f"{what}: push+rs_finish vs fp32 {(M, N, K)}: rel l2 {e}"
            n += 2
        return n

    n_ok = 0
    reshard.epoch_barrier(factor, group)  # shards initialised everywhere
    for it in range(4):
        skew[0] = it % 2
        f_before = float(factor)
        res = step()
        torch.cuda.synchronize()
        n_ok += check(f_before, *res, what=f"eager it {it}")
    skew[0] = 1
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        res = step()
    for it in range(4):
        f_before = float(factor)
        graph.replay()
        torch.cuda.synchronize()
        n_ok += check(f_before, *res, what=f"graph replay {it}")
    rt.health()
    return n_ok


def run_prefetch(rank, world, group):
    """All-gather as a prefetch: stand-alone (edb_ag_prefetch) and riding on a GEMM
    (edb_gemm_pf_bf16) — gathered bytes bit-exact vs the oracle's all_gather of the same shards
    (odd sizes, several items per launch, items that are sub-ranges of a shard), and the carrying
    GEMM bit-identical to the same GEMM without passengers."""
    from easydist_b200 import gemm
    rt = runtime.get_runtime()
    n_ok = 0
    rng = np.random.RandomState(2024)
    sizes = [16, 4096, 16384, 16400, 262144, 1048576 + 48, 6 * 1048576]
    shards, fulls, data = [], [], []
    for i, nbytes in enumerate(sizes):
        sb = rt.alloc(nbytes, align=1024)
        fb = rt.alloc(nbytes * world, align=1024)
        allv = [np.random.RandomState(1000 * i + r).randint(0, 256, size=nbytes).astype(np.uint8)
                for r in range(world)]
        sb.tensor(torch.uint8, (nbytes,)).copy_(torch.from_numpy(allv[rank]))
        shards.append(sb)
        fulls.append(fb)
        data.append(allv)
    x = to_dev(np.zeros(1, dtype=np.float32), "float32")
    reshard.epoch_barrier(x, group)  # every member's shards are in place

    def wipe():
        for fb, nbytes in zip(fulls, sizes):
            fb.tensor(torch.uint8, (nbytes * world,)).fill_(0xEE)

    def check_all(what):
        k = 0
        for fb, nbytes, allv in zip(fulls, sizes, data):
            got = fb.tensor(torch.uint8, (nbytes * world,)).cpu().numpy()
            want = O.all_gather([v for v in allv], 0)[rank]
            assert np.array_equal(got, want), f"{what}: gathered bytes differ (shard {nbytes} B)"
            k += 1
        return k

    # (1) stand-alone, all items in one call (the entry point chunks them by 4)
    wipe()
    items = [(sb.offset, fb.offset, nb, nb) for sb, fb, nb in zip(shards, fulls, sizes)]
    reshard.ag_prefetch(x, group, _items=items)
    torch.cuda.synchronize()
    n_ok += check_all("ag_prefetch")
    # (2) riding on GEMMs: items split into sub-ranges over several carriers
    wipe()
    split = []
    for sb, fb, nb in zip(shards, fulls, sizes):
        if nb >= 32768:
            cut = (nb // 2) // 16384 * 16384
            split += [(sb.offset, fb.offset, cut, nb), (sb.offset + cut, fb.offset + cut, nb - cut, nb)]
        else:
            split.append((sb.offset, fb.offset, nb, nb))
    torch.manual_seed(7)
    shapes = [(4096, 1024, 1024), (512, 256, 4096), (4096, 4096, 1024), (1024, 1024, 4096)]
    for gi in range(0, len(split), 3):
        M, N, K = shapes[(gi // 3) % len(shapes)]
        a = torch.randn(M, K, device="cuda").bfloat16()
        b = torch.randn(K, N, device="cuda").bfloat16()
        ref = gemm.mm(a, b)
        out = gemm.mm(a, b, _pf={"group": group, "items": split[gi:gi + 3]})
        assert torch.equal(out, ref), f"carrying GEMM {(M, N, K)} differs from the plain one"
        n_ok += 1
    torch.cuda.synchronize()
    n_ok += check_all("gemm_pf")
    reshard.epoch_barrier(x, group)
    # (3) in-place layout: every member's shard lives in its own slot of the gathered buffer
    # (src_off == dst_off, src_stride == dst_stride): only the n-1 remote ranges are copied
    for fb, nb, allv in zip(fulls, sizes, data):
        t = fb.tensor(torch.uint8, (nb * world,))
        t.fill_(0xEE)
        t[rank * nb:(rank + 1) * nb].copy_(torch.from_numpy(allv[rank]))
    reshard.epoch_barrier(x, group)
    inpl = [(fb.offset, fb.offset, nb, nb, nb) for fb, nb in zip(fulls, sizes)]
    reshard.ag_prefetch(x, group, _items=inpl[:3])
    a = torch.randn(2048, 1024, device="cuda").bfloat16()
    b = torch.randn(1024, 1024, device="cuda").bfloat16()
    ref = gemm.mm(a, b)
    out = gemm.mm(a, b, _pf={"group": group, "items": inpl[3:]})
    assert torch.equal(out, ref), "carrying GEMM (in-place items) differs from the plain one"
    torch.cuda.synchronize()
    n_ok += check_all("in-place prefetch") + 1
    reshard.epoch_barrier(x, group)
    return n_ok


def run_train_parity(rank, world):
    """The benchmarked path end to end: zero3 + epoch-mode AG+GEMM / push GEMM + rs_finish +
    re-homed shards + bucketed small gradients + fused SGD, through easydist_compile (eager and
    CUDA graph), against vanilla fp32 PyTorch on the same global batches: loss of every call, every
    parameter and every momentum buffer (tools/parity.py; tolerances calibrated by vanilla bf16)."""
    import dataclasses
    from easydist_b200.api import easydist_compile
    from easydist_b200.device_mesh import set_device_mesh
    from easydist_b200.workloads import GPT2, GPT2Config, gpt2_train_step, synthetic_tokens
    from tools import parity as P
    set_device_mesh(list(range(world)), ["dp"], rank=rank)
    # vocab 2000: not a multiple of 128, so (as with GPT-2's 50257) the tied embedding / LM head
    # stays on the unfused all-gather / reduce-scatter kernels
    cfg = GPT2Config(n_layer=2, n_head=8, n_embd=1024, vocab_size=2000, block_size=64)
    B, S, n_calls = 2, 64, 3
    n_ok = 0
    for cuda_graph in (False, True):
        torch.manual_seed(0)
        model = GPT2(cfg).to(device="cuda", dtype=torch.bfloat16)
        state0 = {k: v.detach().clone() for k, v in model.state_dict().items()}
        opt = torch.optim.SGD(model.parameters(), lr=1e-2, momentum=0.9, foreach=True)
        mk_opt = lambda ps: torch.optim.SGD(ps, lr=1e-2, momentum=0.9, foreach=True)
        batches = [[synthetic_tokens(cfg, B, S, seed=500 + 100 * b + r) for r in range(world)]
                   for b in range(n_calls)]
        step = easydist_compile(gpt2_train_step, parallel_mode="zero3", tracing_mode="fake",
                                cuda_graph=cuda_graph)
        losses = []
        for b in range(n_calls):
            t, y = batches[b][rank]
            losses.append(float(step(t.cuda(), y.cuda(), model, opt)))
        info = step.compiled_func.info
        if world > 1:
            # 8 Linear weights + token and position embeddings gathered by prefetch; 8 wgrad pushes
            assert info["fused"]["ag_pf"] == 10 and info["fused"]["mm_rs"] == 8, info
            assert info["comm_nodes"].get("epoch_barrier") == 2, info
        sched = ([0, 0] if cuda_graph else [0]) + list(range(1, n_calls))
        steps = [batches[b] for b in sched]
        ref_l, ref_p, ref_s = P.vanilla_run(lambda: GPT2(cfg), state0, steps, mk_opt, torch.float32, "cuda")
        van_l, van_p, van_s = P.vanilla_run(lambda: GPT2(cfg), state0, steps, mk_opt, torch.bfloat16, "cuda")
        got_p, got_s = P.compiled_state(step.compiled_func, ref_p, ref_s, world)
        ours = P.compare(got_p, got_s, ref_p, ref_s, low_precision=True)
        van = P.compare({k: v.bfloat16() for k, v in van_p.items()},
                        {k: {kk: vv.bfloat16() for kk, vv in st.items()} for k, st in van_s.items()},
                        ref_p, ref_s, low_precision=True)
        idx = [1 if cuda_graph else 0] + list(range(2 if cuda_graph else 1, len(sched)))
        for l, i in zip(losses, idx):
            want = ref_l[i][rank]
            assert abs(l - want) <= 2e-2 * abs(want), f"train parity loss {losses} vs {ref_l}"
        tol_state = max(2e-2, 2.0 * van["state_rel_l2"])
        tol_ulp = max(2.0, 2.0 * van["param_max_ulp"])
        assert ours["state_rel_l2"] <= tol_state, (ours, van)
        assert ours["param_max_ulp"] <= tol_ulp, (ours, van)
        n_ok += ours["checks"] + len(losses)
        if rank == 0:
            print(f"TRAIN_PARITY_OK world={world} cuda_graph={cuda_graph} checks={ours['checks']} "
                  f"momentum_rel_l2={ours['state_rel_l2']:.3e} (vanilla bf16 {van['state_rel_l2']:.3e}) "
                  f"param_ulp={ours['param_max_ulp']:.2f} (vanilla bf16 {van['param_max_ulp']:.2f}) "
                  f"fused={info.get('fused')}", flush=True)
    return n_ok


def bench_fused(rank, world, group):
    from easydist_b200 import gemm
    rt = runtime.get_runtime()
    _t = _graph_timer(world)
    timeit = lambda f: _t(f) * 1e3

    for (M, N, K) in [(4096, 1024, 1024), (4096, 4096, 1024), (4096, 1024, 4096), (4096, 3072, 1024)]:
        rows = N // world
        x = torch.randn(M, K, device="cuda").bfloat16()
        shard_buf, full_buf = rt.alloc(rows * K * 2, align=1024), rt.alloc(N * K * 2, align=1024)
        ag_buf = rt.alloc(N * K * 2, align=1024)
        w_shard = shard_buf.tensor(torch.bfloat16, (rows, K))
        w_shard.normal_()
        t_fused = timeit(lambda: reshard.ag_mm(x, w_shard, group, N, K, None,
                                                _buf=(shard_buf.offset, full_buf.offset), _epoch=1))

        def unfused():
            w = reshard.all_gather_start(w_shard, 0, group, _buf=(ag_buf.offset, N * K * 2))
            return gemm.mm(x, w.t())
        t_unf = timeit(unfused)
        t_gemm = timeit(lambda: gemm.mm(x, full_buf.tensor(torch.bfloat16, (N, K)).t()))
        # wgrad-like: dW[N,K] = dy^T[N,M] @ x[M,K], reduce-scattered over N
        dy = torch.randn(M, N, device="cuda").bfloat16()
        stage = rt.alloc(N * K * 2, align=1024)
        t_wg = timeit(lambda: gemm.mm(dy.t(), x))

        def unfused_rs():
            part = gemm.mm(dy.t(), x)
            return reshard.reduce_scatter_start(part.flatten(), "avg", 0, group,
                                                _buf=(stage.offset, N * K * 2))
        t_rs_u = timeit(unfused_rs)
        if rank == 0:
            print(f"FUSED M{M} N{N} K{K}: ag+gemm fused {t_fused:.1f}us unfused {t_unf:.1f}us "
                  f"(gemm alone {t_gemm:.1f}us) | gemm+rs unfused {t_rs_u:.1f}us "
                  f"(wgrad gemm alone {t_wg:.1f}us)", flush=True)


def run_auto_bundle(rank, world):
    """Auto-SPMD on real GPUs: graph + plan solved by the unmodified reference (recorded in
    tests/golden/auto_foo_mesh*.json), lowered by easydist_b200.lowering.sharding_transform and
    executed with the libedb kernels; outputs vs vanilla PyTorch on the same GPU, rtol 1e-4 (the
    reference's comparator, tests/test_torch/test_spmd.py:67)."""
    from tests.test_auto_bundle_cpu import run_bundle
    mesh_shape = {2: (2,), 4: (2, 2)}.get(world)
    if mesh_shape is None:
        return 0
    ok, msg, hist = run_bundle(rank, world, mesh_shape, reshard, True, "cuda")
    assert ok, f"auto bundle mesh {mesh_shape}: {msg}"
    if rank == 0:
        print(f"AUTO_BUNDLE_OK mesh={mesh_shape} comm={hist}", flush=True)
    return 1


def _graph_timer(world):
    """Time `f` as the average of 10 captured calls per CUDA-graph replay (no Python / launch
    overhead in the measurement), max over ranks."""

    def timeit(f, reps=5):
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                f()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        dist.barrier()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(10):
                f()
        g.replay()
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / (reps * 10)], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()  # ms per op
    return timeit


def bench(rank, world, group):
    """Reshard microbench (BASELINE.json config 5): bus bandwidth (nccl-tests convention) of the
    libedb kernels vs NCCL on the same GPUs, bf16, CUDA-graph replay timing."""
    rt = runtime.get_runtime()
    timeit = _graph_timer(world)
    res = []
    sizes = [1 << k for k in range(10, 31, 2)]
    for nbytes in sizes:
        if nbytes * 4 > rt.heap_bytes // 2:
            break
        mark = rt.mark()
        numel = nbytes // 2
        shard = torch.randn(max(1, numel // world), device="cuda").bfloat16()
        full = torch.randn(numel, device="cuda").bfloat16()
        b1, b2, b3 = rt.alloc(nbytes), rt.alloc(nbytes), rt.alloc(nbytes)
        nccl_out = torch.empty(shard.numel() * world, device="cuda", dtype=torch.bfloat16)
        nccl_rs = torch.empty(numel // world, device="cuda", dtype=torch.bfloat16)
        a2a_in = full.view(world, -1)
        a2a_out = torch.empty_like(a2a_in)
        row = {"bytes": nbytes}
        f = (world - 1) / world
        t = timeit(lambda: reshard.all_gather_start(shard, 0, group, _buf=(b1.offset, nbytes)))
        row["ag_edb_GBs"], row["ag_edb_us"] = nbytes * f / t / 1e6, t * 1e3
        t = timeit(lambda: dist.all_gather_into_tensor(nccl_out, shard))
        row["ag_nccl_GBs"], row["ag_nccl_us"] = nbytes * f / t / 1e6, t * 1e3
        t = timeit(lambda: reshard.reduce_scatter_start(full, "sum", 0, group,
                                                        _buf=(b2.offset, nbytes)))
        row["rs_edb_GBs"], row["rs_edb_us"] = nbytes * f / t / 1e6, t * 1e3
        t = timeit(lambda: dist.reduce_scatter_tensor(nccl_rs, full))
        row["rs_nccl_GBs"], row["rs_nccl_us"] = nbytes * f / t / 1e6, t * 1e3
        t = timeit(lambda: reshard.all_reduce_start(full, "sum", group,
                                                    _buf=(b2.offset, nbytes, b3.offset)))
        row["ar_edb_GBs"], row["ar_edb_us"] = 2 * nbytes * f / t / 1e6, t * 1e3
        t = timeit(lambda: dist.all_reduce(full))
        row["ar_nccl_GBs"], row["ar_nccl_us"] = 2 * nbytes * f / t / 1e6, t * 1e3
        if numel % (world * world) == 0 and numel >= world * world:
            x2 = full.view(world, -1)  # S(0) local [world, c] -> S(1): true all-to-all
            t = timeit(lambda: reshard.all_to_all_start(x2, 0, 1, world, rank, group,
                                                        _buf=(b1.offset, nbytes)))
            row["a2a_edb_GBs"], row["a2a_edb_us"] = nbytes * f / t / 1e6, t * 1e3
            t = timeit(lambda: dist.all_to_all_single(a2a_out, a2a_in))
            row["a2a_nccl_GBs"], row["a2a_nccl_us"] = nbytes * f / t / 1e6, t * 1e3
        res.append(row)
        rt.reset(mark)
        if rank == 0:
            print("BENCH " + " ".join(f"{k}={v:.1f}" if isinstance(v, float) else f"{k}={v}"
                                      for k, v in row.items()), flush=True)
    return res


def _ref_wrappers(world, rank, group_pg=None):
    """The reference's own communication wrappers restated over NCCL (easydist/torch/passes/
    sharding.py:94-163): all-gather along dim 0 + chunk/cat for other dims, pre-permute copy +
    reduce_scatter_tensor, all-to-all as all-gather + local chunk (its TODO), blocking each."""
    def ag(x, dim):
        x = x.contiguous()
        out = torch.empty((x.shape[0] * world,) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
        dist.all_gather_into_tensor(out, x)
        if dim != 0:
            out = torch.cat(torch.chunk(out, world, dim=0), dim=dim)
        return out

    def rs(x, dim):
        if dim != 0:
            x = torch.cat(torch.chunk(x, world, dim=dim))
        out = torch.empty((x.shape[0] // world,) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
        dist.reduce_scatter_tensor(out, x.contiguous())
        return out

    def ar(x):
        y = x.clone()
        dist.all_reduce(y)
        return y

    def a2a(x, g, s_):
        return torch.chunk(ag(x, g), world, s_)[rank].contiguous()

    return ag, rs, ar, a2a


def bench2(rank, world, group, sizes=None, dtypes=("bfloat16", "float32"), quiet=False):
    """Reshard microbench, BASELINE.json config 5 / SURVEY.md §8(d): all-gather, reduce-scatter(sum),
    all-reduce, all-to-all; total bytes 1 KB ... 1 GB (x4); bf16 and fp32; dims {0, last}; three
    arms on the same GPUs — this library (push protocol with static buffers + an epoch barrier per
    replayed batch of 10 ops, as in a compiled step), raw NCCL, and the reference's wrappers over
    NCCL.  Bus bandwidth in the nccl-tests convention; CUDA-graph replay timing, max over ranks."""
    rt = runtime.get_runtime()
    timeit = _graph_timer(world)
    r_ag, r_rs, r_ar, r_a2a = _ref_wrappers(world, rank)
    sizes = sizes or [1 << k for k in range(10, 31, 2)]
    oneshot = rt.get_option("allreduce_oneshot_bytes")
    f = (world - 1) / world
    rows_out = []
    for dtype in dtypes:
        tdt = TORCH_DT[dtype]
        es = torch.empty((), dtype=tdt).element_size()
        for dim_kind in ("0", "last"):
            for nbytes in sizes:
                if nbytes * (world + 3) > rt.heap_bytes // 2:
                    break
                cols = 1024 if nbytes // es >= 1024 * world * world else world
                rows = nbytes // es // cols
                if rows < world or rows % world:
                    rows = max(world, rows // world * world)
                full_shape = (rows, cols)
                numel = rows * cols
                nb = numel * es
                dim = 0 if dim_kind == "0" else 1
                if full_shape[dim] % world:
                    continue
                shard_shape = list(full_shape)
                shard_shape[dim] //= world
                mark = rt.mark()
                shard = torch.randn(shard_shape, device="cuda").to(tdt)
                full = torch.randn(full_shape, device="cuda").to(tdt)
                # static buffers may only be reused after a group barrier.  Up to 16 MiB ten buffer
                # sets rotate and ONE barrier follows every tenth call (a compiled step has two
                # barriers for hundreds of edges); above that a single set + a barrier per call
                # (a few us against milliseconds)
                K = 10 if nb <= (16 << 20) else 1
                rb, ob = reshard.all_reduce_push_sizes(nb, numel, es, world, oneshot)
                sets = [(rt.alloc(nb), rt.alloc(nb), rt.alloc(rb), rt.alloc(ob), rt.alloc(nb))
                        for _ in range(K)]
                row = {"dtype": dtype, "dim": dim_kind, "bytes": nb}

                def edb(fn):
                    cnt = [0]

                    def run():
                        i = cnt[0] % K
                        cnt[0] += 1
                        fn(sets[i])
                        if i == K - 1:
                            reshard.epoch_barrier(shard, group)
                    return run
                t = timeit(edb(lambda b_: reshard.all_gather_start(shard, dim, group, _buf=(b_[0].offset, nb), _push=1)))
                row["ag_edb_us"], row["ag_edb_GBs"] = t * 1e3, nb * f / t / 1e6
                t = timeit(lambda: dist.all_gather_into_tensor(torch.empty(numel, dtype=tdt, device="cuda"), shard.view(-1)))
                row["ag_nccl_us"] = t * 1e3
                t = timeit(lambda: r_ag(shard, dim))
                row["ag_ref_us"] = t * 1e3
                t = timeit(edb(lambda b_: reshard.reduce_scatter_start(full, "sum", dim, group, _buf=(b_[1].offset, nb), _push=1)))
                row["rs_edb_us"], row["rs_edb_GBs"] = t * 1e3, nb * f / t / 1e6
                t = timeit(lambda: dist.reduce_scatter_tensor(torch.empty(numel // world, dtype=tdt, device="cuda"), full.view(-1)))
                row["rs_nccl_us"] = t * 1e3
                t = timeit(lambda: r_rs(full, dim))
                row["rs_ref_us"] = t * 1e3
                if dim_kind == "0":
                    t = timeit(edb(lambda b_: reshard.all_reduce_start(full, "sum", group, _buf=(b_[2].offset, rb, b_[3].offset), _push=1)))
                    row["ar_edb_us"], row["ar_edb_GBs"] = t * 1e3, 2 * nb * f / t / 1e6
                    t = timeit(lambda: r_ar(full))
                    row["ar_nccl_us"] = t * 1e3
                other = 1 - dim
                if shard_shape[other] % world == 0:
                    t = timeit(edb(lambda b_: reshard.all_to_all_start(shard, dim, other, world, rank, group, _buf=(b_[4].offset, nb // world), _push=1)))
                    row["a2a_edb_us"], row["a2a_edb_GBs"] = t * 1e3, nb / world * f / t / 1e6
                    t = timeit(lambda: r_a2a(shard, dim, other))
                    row["a2a_ref_us"] = t * 1e3
                torch.cuda.synchronize()
                reshard.epoch_barrier(shard, group)
                rt.reset(mark)
                rows_out.append(row)
                if rank == 0 and not quiet:
                    print("BENCH2 " + " ".join(f"{k}={v:.1f}" if isinstance(v, float) else f"{k}={v}"
                                               for k, v in row.items()), flush=True)
    # the barrier itself (its cost is inside every *_edb_us above)
    t = timeit(lambda: reshard.epoch_barrier(shard, group))
    if rank == 0 and not quiet:
        print(f"BENCH2 epoch_barrier_us={t * 1e3:.2f}", flush=True)
    return rows_out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bench", action="store_true")
    ap.add_argument("--bench2", action="store_true", help="only the reshard microbench (config 5)")
    ap.add_argument("--bench2-quick", action="store_true",
                    help="bf16 only, 1 KiB ... 256 MiB (x16 steps): the affordable form at 8 GPUs")
    ap.add_argument("--bench-fused", action="store_true", help="only the fused-kernel microbench")
    ap.add_argument("--heap-gb", type=float, default=8.0)
    ap.add_argument("--ll-bytes", type=int, default=-1,
                    help="override the low-latency protocol threshold (0 = off)")
    args = ap.parse_args()
    rank = int(os.environ["RANK"])
    world = int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rt = runtime.init(rank, world, local, heap_bytes=int(args.heap_gb * (1 << 30)))
    rt.set_option("spin_timeout_ms", 20000)  # fatal (trap) when exceeded
    if args.ll_bytes >= 0:
        rt.set_option("ll_max_bytes", args.ll_bytes)
    group = list(range(world))
    if args.bench2 or args.bench2_quick:
        if args.bench2_quick:
            bench2(rank, world, group, sizes=[1 << k for k in range(10, 29, 4)] + [1 << 28],
                   dtypes=("bfloat16",))
        else:
            bench2(rank, world, group)
        dist.barrier()
        dist.destroy_process_group()
        return
    n = run_cases(rank, world, group)
    n += run_cases(rank, world, group, tag="b")  # second pass: epochs keep counting
    n += run_randn_cases(rank, world, group)
    n += run_p2p(rank, world, group)
    n += run_graph(rank, world, group)
    n += run_graph(rank, world, group, rows=4)
    n += run_epoch(rank, world, group)
    n += run_prefetch(rank, world, group)
    n += run_push_cases(rank, world, group)
    n += run_auto_bundle(rank, world)
    n += run_train_parity(rank, world)
    if world in (2, 4, 8) and os.environ.get("EDB_SKIP_C1") != "1":
        # SURVEY.md config 1 (the reference's examples/torch/gpt_train.py model, fp32) in AUTO-SPMD
        # mode with the plans the reference's solver produced, on real GPUs: outputs, every parameter
        # and every momentum buffer vs vanilla (rtol 1e-4 / atol 1e-5) — with the product's lowering
        # (optimizer on shards, parameter gathers as prefetches, push collectives) and, for the 1-D
        # mesh, also with the reference's communication structure (EDB_LOCALIZE_OPT=0 etc.)
        from tests.test_auto_bundle_cpu import run_c1_bundle
        variants = [(str(world), {})]
        variants.append((str(world), {"EDB_LOCALIZE_OPT": "0", "EDB_AG_PREFETCH": "0",
                                      "EDB_PUSH_COLL": "0"}))
        if world == 4:
            variants.append(("2x2", {}))
        for tag, env in variants:
            saved = {k: os.environ.get(k) for k in env}
            os.environ.update(env)
            try:
                ok, msg, hist = run_c1_bundle(rank, world, reshard, True, "cuda", steps=3, tag=tag)
            finally:
                for k, v in saved.items():
                    if v is None:
                        os.environ.pop(k, None)
                    else:
                        os.environ[k] = v
            assert ok, f"config-1 bundle mesh {tag} on GPUs ({env}): {msg}"
            if rank == 0:
                print(f"AUTO_BUNDLE_C1_OK mesh={tag} env={env} {hist}", flush=True)
            n += 1
    if world >= 4 and world % 2 == 0:
        # 2-D mesh: groups along each mesh dim (ranks in mesh-coordinate order)
        mesh = np.arange(world).reshape(2, world // 2)
        coord = tuple(int(c) for c in np.argwhere(mesh == rank)[0])
        for mdim in (0, 1):
            grp = O.submesh_ranks(mesh, mdim, coord)
            me = grp.index(rank)
            xs = inputs_for(f"mesh{mdim}", (4 * len(grp), 6), "float32", world)
            sub = [xs[r] for r in grp]
            got = reshard.all_gather_start(to_dev(xs[rank], "float32"), 1, grp)
            check_equal(got, O.all_gather(sub, 1)[me], f"2d mesh ag dim{mdim}")
            got = reshard.reduce_scatter_start(to_dev(xs[rank], "float32"), "sum", 0, grp)
            check_equal(got, O.reduce_scatter(sub, "sum", 0)[me], f"2d mesh rs dim{mdim}")
            n += 2
    torch.cuda.synchronize()
    errs = rt.error_flags()
    assert not any(errs), f"spin-wait timeouts recorded: {errs}"
    dist.barrier()
    if rank == 0:
        print(f"MGPU_OK world={world} checks={n} launches={rt.launch_count()}", flush=True)
    if args.bench or args.bench_fused:
        bench_fused(rank, world, group)
    if args.bench:
        bench(rank, world, group)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
