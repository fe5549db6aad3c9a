"""Host logic of the epoch-mode parameter prefetch (lowering.prefetch_param_gathers), on CPU with
a fake symmetric runtime: whatever the byte budgets make of the schedule, every byte of every
parameter shard must be gathered exactly once per step, by nodes that precede the parameter's first
use, and the step must carry its two epoch barriers around the optimizer.  (A missing range would be
stale weights on the GPU, silently.)"""
import os

import pytest
import torch

from tests.test_dp_cpu import make_opt, train_step


class Deep(torch.nn.Module):
    def __init__(self, d=256, layers=4):
        super().__init__()
        self.inp = torch.nn.Linear(d, d)
        self.blocks = torch.nn.ModuleList(
            torch.nn.Sequential(torch.nn.LayerNorm(d), torch.nn.Linear(d, 4 * d), torch.nn.GELU(),
                                torch.nn.Linear(4 * d, d)) for _ in range(layers))

    def forward(self, x):
        x = self.inp(x)
        for b in self.blocks:
            x = x + b(x)
        return x


@pytest.mark.parametrize("gbps,my_index", [("300", 1), ("0.001", 0), ("100000", None)])
def test_every_shard_byte_is_prefetched_once_before_its_first_use(gbps, my_index, monkeypatch):
    monkeypatch.setenv("EDB_PF_GBPS", gbps)
    from easydist_b200 import lowering
    from easydist_b200.api import _flat_inputs
    from easydist_b200.compile import GraphIO, trace_train_step
    from tests import gloo_ops
    torch.manual_seed(0)
    model = Deep().bfloat16()
    opt = make_opt("sgd", model.parameters())
    x = torch.randn(64, 256).bfloat16()
    params, buffers, named_states, gm, module, o = trace_train_step(train_step, (x, model, opt), {},
                                                                   "fake")
    io = GraphIO(gm, params, buffers, named_states)
    ranks, n = [0, 1, 2, 3], 4
    _, shard_info = lowering.transform_fsdp(gm, io, ranks, 1, True, gloo_ops, bucket_numel=2048)
    with torch.no_grad():
        params = {k: v.detach() for k, v in params.items()}
        for ph, name in zip(io.param_ph, io.param_names):
            if ph.name in shard_info:
                params[name] = torch.chunk(params[name].flatten(), n)[1].contiguous()
        flat_states, spec = torch.utils._pytree.tree_flatten(named_states)
        for i, ph in enumerate(io.state_ph):
            if ph.name in shard_info and isinstance(flat_states[i], torch.Tensor):
                flat_states[i] = torch.chunk(flat_states[i].detach().flatten(), n)[1].contiguous()
        named_states = torch.utils._pytree.tree_unflatten(flat_states, spec)
        lowering.propagate_local_meta(gm, [t.detach() if isinstance(t, torch.Tensor) else t for t in
                                           _flat_inputs(params, buffers, named_states, (x, model, opt), {})])
    rt = gloo_ops.FakeSymmRuntime()
    rehomed, nf = lowering.fuse_collective_gemms(gm, io, rt, ranks, gloo_ops, my_index=my_index)
    assert nf["ag_pf"] == len(rehomed) > 0 and nf["ag_mm"] == 0, nf
    nodes = list(gm.graph.nodes)
    order = {nd: i for i, nd in enumerate(nodes)}
    # first use and buffers of every prefetched parameter
    first_use, bufs = {}, {}
    for nd in nodes:
        if nd.op == "call_function" and nd.target is gloo_ops.gathered:
            ph = nd.args[0]
            first_use[ph] = min(first_use.get(ph, 1 << 60), order[nd])
            bufs[ph] = nd.kwargs["_buf"]
    assert len(first_use) == len(rehomed)
    # all prefetch work items with the position of the node that issues them
    issued = []
    for nd in nodes:
        if nd.op != "call_function":
            continue
        if nd.target is gloo_ops.ag_prefetch:
            issued += [(order[nd], it) for it in nd.kwargs["_items"]]
        elif "edb_pf" in nd.meta:
            assert len(nd.meta["edb_pf"]["items"]) <= 4
            issued += [(order[nd], it) for it in nd.meta["edb_pf"]["items"]]
    for ph, (shard_off, full_off) in bufs.items():
        nbytes = ph.meta["val"].numel() * ph.meta["val"].element_size()
        covered = []
        for pos, (src, dst, take, dstride, sstride) in issued:
            if full_off <= dst < full_off + nbytes:
                assert pos < first_use[ph], f"{ph.name}: prefetched after its first use"
                assert dstride == nbytes and take > 0 and take % 16 == 0
                if my_index is None:
                    assert sstride == 0 and src - shard_off == dst - full_off
                else:  # in place: the shard lives in slot my_index of the gathered buffer
                    assert sstride == nbytes and src == dst
                    assert shard_off == full_off + my_index * nbytes
                covered.append((dst - full_off, dst - full_off + take))
        covered.sort()
        assert covered and covered[0][0] == 0 and covered[-1][1] == nbytes, (ph.name, covered)
        for (a0, a1), (b0, b1) in zip(covered, covered[1:]):
            assert a1 == b0, f"{ph.name}: gap or overlap in the prefetched ranges {covered}"
    # the two rendezvous: one behind the last peer access and in front of the first parameter update,
    # one at the very end
    barriers = [order[nd] for nd in nodes if nd.op == "call_function"
                and nd.target is gloo_ops.epoch_barrier]
    assert len(barriers) == 2, barriers
    last_peer = max(pos for pos, _ in issued)
    pushes = [order[nd] for nd in nodes if nd.op == "call_function" and nd.target is gloo_ops.mm_push]
    # (momentum buffers are updated earlier — nobody reads those remotely; parameters are what peers read)
    first_update = min(order[nd] for nd in nodes if nd.op == "call_function"
                       and nd.target == torch.ops.aten.copy_.default and nd.args[0] in io.param_ph)
    assert max([last_peer] + pushes) < barriers[0] < first_update
    assert nodes[barriers[1]].next.op == "output"


def test_static_buffers_mark_push_collectives_and_the_step_ends_with_a_barrier(monkeypatch):
    """lowering.assign_static_buffers(push=True): every remaining collective node of the zero3 graph
    gets dedicated symmetric buffers and `_push=1`; an all-reduce's receive buffer follows the
    one-shot / two-shot rule of edb_all_reduce_push; ensure_end_barrier is idempotent."""
    from easydist_b200 import lowering
    from easydist_b200.api import _flat_inputs
    from easydist_b200.compile import GraphIO, trace_train_step
    from tests import gloo_ops
    torch.manual_seed(0)
    model = Deep(layers=2).bfloat16()
    opt = make_opt("sgd", model.parameters())
    x = torch.randn(64, 256).bfloat16()
    params, buffers, named_states, gm, module, o = trace_train_step(train_step, (x, model, opt), {},
                                                                   "fake")
    io = GraphIO(gm, params, buffers, named_states)
    ranks, n = [0, 1], 2
    _, shard_info = lowering.transform_fsdp(gm, io, ranks, 0, True, gloo_ops, bucket_numel=2048)
    with torch.no_grad():
        params = {k: v.detach() for k, v in params.items()}
        for ph, name in zip(io.param_ph, io.param_names):
            if ph.name in shard_info:
                params[name] = torch.chunk(params[name].flatten(), n)[0].contiguous()
        flat_states, spec = torch.utils._pytree.tree_flatten(named_states)
        for i, ph in enumerate(io.state_ph):
            if ph.name in shard_info and isinstance(flat_states[i], torch.Tensor):
                flat_states[i] = torch.chunk(flat_states[i].detach().flatten(), n)[0].contiguous()
        named_states = torch.utils._pytree.tree_unflatten(flat_states, spec)
        lowering.propagate_local_meta(gm, [t.detach() if isinstance(t, torch.Tensor) else t for t in
                                           _flat_inputs(params, buffers, named_states, (x, model, opt), {})])
    rt = gloo_ops.FakeSymmRuntime()
    total = lowering.assign_static_buffers(gm, rt, gloo_ops, push=True)
    assert total > 0
    comm = [nd for nd in gm.graph.nodes if nd.op == "call_function" and nd.target in gloo_ops.COMM_FUNCS]
    assert comm and all(nd.kwargs.get("_push") == 1 and "_buf" in nd.kwargs for nd in comm)
    for nd in comm:
        if nd.target is gloo_ops.all_reduce_start:
            xv = nd.args[0].meta["val"]
            nb = xv.numel() * xv.element_size()
            rb, ob = gloo_ops.all_reduce_push_sizes(nb, xv.numel(), xv.element_size(), n, 512 * 1024)
            assert nd.kwargs["_buf"][1] == rb and len(nd.kwargs["_buf"]) == 3
            assert rb == (n * nb if nb <= 8 * 512 * 1024 else nb) and ob == nb
    assert lowering.ensure_end_barrier(gm, ranks, gloo_ops) == 1
    assert lowering.ensure_end_barrier(gm, ranks, gloo_ops) == 0
    out = next(nd for nd in gm.graph.nodes if nd.op == "output")
    assert out.prev.target is gloo_ops.epoch_barrier


def _lowered_zero3_graph(n=4, me=1):
    from easydist_b200 import lowering
    from easydist_b200.api import _flat_inputs
    from easydist_b200.compile import GraphIO, trace_train_step
    from tests import gloo_ops
    torch.manual_seed(0)
    model = Deep(layers=2).bfloat16()
    opt = make_opt("sgd", model.parameters())
    x = torch.randn(64, 256).bfloat16()
    params, buffers, named_states, gm, module, o = trace_train_step(train_step, (x, model, opt), {},
                                                                   "fake")
    io = GraphIO(gm, params, buffers, named_states)
    ranks = list(range(n))
    _, shard_info = lowering.transform_fsdp(gm, io, ranks, me, True, gloo_ops, bucket_numel=2048)
    with torch.no_grad():
        params = {k: v.detach() for k, v in params.items()}
        for ph, name in zip(io.param_ph, io.param_names):
            if ph.name in shard_info:
                params[name] = torch.chunk(params[name].flatten(), n)[me].contiguous()
        flat_states, spec = torch.utils._pytree.tree_flatten(named_states)
        for i, ph in enumerate(io.state_ph):
            if ph.name in shard_info and isinstance(flat_states[i], torch.Tensor):
                flat_states[i] = torch.chunk(flat_states[i].detach().flatten(), n)[me].contiguous()
        named_states = torch.utils._pytree.tree_unflatten(flat_states, spec)
        lowering.propagate_local_meta(gm, [t.detach() if isinstance(t, torch.Tensor) else t for t in
                                           _flat_inputs(params, buffers, named_states, (x, model, opt), {})])
    rt = gloo_ops.FakeSymmRuntime()
    lowering.fuse_collective_gemms(gm, io, rt, ranks, gloo_ops, my_index=me)
    lowering.reinplace_optimizer_updates(gm)
    lowering.assign_static_buffers(gm, rt, gloo_ops, push=True)
    lowering.ensure_end_barrier(gm, ranks, gloo_ops)
    lowering.dispatch_compute(gm)
    return gm, ranks


def test_static_epoch_protocol_check_passes_and_catches_planted_races(monkeypatch):
    """lowering.verify_epoch_protocol (the compile-time counterpart of the reference's op_mem_checker,
    compile_auto.py:269-351): the lowered zero3 graph satisfies the contract; a removed barrier, two
    nodes sharing a receive buffer, a dropped prefetch range and a prefetch after the first use are
    each reported."""
    from easydist_b200 import lowering
    from tests import gloo_ops
    gm, ranks = _lowered_zero3_graph()
    rep = lowering.verify_epoch_protocol(gm, gloo_ops, len(ranks))
    assert rep["ok"] and rep["barriers"] == 2 and rep["ranges"] > 4 and rep["items"] > 2, rep

    def fresh():
        return _lowered_zero3_graph()[0]

    # (a) the barrier in front of the optimizer removed
    g = fresh()
    b = next(nd for nd in g.graph.nodes if nd.op == "call_function" and nd.target is gloo_ops.epoch_barrier)
    b.replace_all_uses_with(b.args[0])
    g.graph.erase_node(b)
    probs = lowering.verify_epoch_protocol(g, gloo_ops, len(ranks))["problems"]
    assert any("no epoch barrier" in p for p in probs), probs
    # (b) two push GEMMs write the same receive slots
    g = fresh()
    ps = [nd for nd in g.graph.nodes if nd.op == "call_function" and nd.target is gloo_ops.mm_push]
    ps[1].kwargs = dict(ps[1].kwargs, _buf=ps[0].kwargs["_buf"])
    probs = lowering.verify_epoch_protocol(g, gloo_ops, len(ranks))["problems"]
    assert any("overlap" in p for p in probs), probs
    # (c) a prefetch that lost part of a shard
    g = fresh()
    pf = next(nd for nd in g.graph.nodes if nd.op == "call_function" and nd.target is gloo_ops.ag_prefetch)
    its = list(pf.kwargs["_items"])
    src, dst, take, ds, ss = its[0]
    its[0] = (src, dst, take - 16, ds, ss)
    pf.kwargs = dict(pf.kwargs, _items=its)
    probs = lowering.verify_epoch_protocol(g, gloo_ops, len(ranks))["problems"]
    assert any("shard bytes are prefetched" in p or "gap" in p for p in probs), probs
    # (d) a prefetch issued after the parameter's first use
    g = fresh()
    pf = next(nd for nd in g.graph.nodes if nd.op == "call_function" and nd.target is gloo_ops.ag_prefetch)
    last_g = [nd for nd in g.graph.nodes if nd.op == "call_function" and nd.target is gloo_ops.gathered][-1]
    last_g.append(pf)
    probs = lowering.verify_epoch_protocol(g, gloo_ops, len(ranks))["problems"]
    assert any("after its first use" in p for p in probs), probs
    # (e) the end-of-step barrier removed
    g = fresh()
    out = next(nd for nd in g.graph.nodes if nd.op == "output")
    g.graph.erase_node(out.prev)
    probs = lowering.verify_epoch_protocol(g, gloo_ops, len(ranks))["problems"]
    assert any("does not end with an epoch barrier" in p for p in probs), probs
