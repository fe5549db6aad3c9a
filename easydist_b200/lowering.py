"""Plan -> executable graph: the B200 replacement of the reference's lowering passes.

  sharding_transform(fx_module, opt_strategy, state_io_map)
        drop-in for easydist/torch/passes/sharding.py:852-979 (call site compile_auto.py:569):
        walks the traced graph with the solver's per-node NodeSPMDStrategy, tracks the placement
        of every value (`shard_env`), and wherever producer and consumer placements differ emits
        the reshard steps chosen by the edge planner (insert_comm_node, sharding.py:704-809);
        view/reshape/expand size arguments are rewritten to local shapes (override_args,
        :812-849); user outputs are replicated and state outputs are forced back to the placement
        of their input placeholder + copy_wrapper (:920-949).
  transform_ddp / transform_fsdp
        the data-parallel rewrites of easydist/torch/compile_dp.py:55-198 (modes ddp / zero2 /
        zero3), generalised from "the `_fused_adam` node" to any elementwise optimizer by working
        on the optimizer region of the graph (everything downstream of the final gradients).
  assign_static_buffers / dispatch_compute / propagate_local_meta
        B200-specific finishing passes: symmetric-heap buffers fixed at compile time (so the
        graph is CUDA-graph capturable with zero allocations in the comm path), bf16 `aten.mm` ->
        tcgen05 GEMM dispatch.

The emitted `call_function` targets are the callables of an `ops` namespace with the reference's
names and signatures (default: easydist_b200.reshard -> libedb.so).
"""
import operator
import os
from typing import Dict

import torch
import torch.utils._pytree as pytree
from torch.fx.node import Node

from . import metair as M
from . import planners
from . import reshard as _default_ops
from .device_mesh import get_device_mesh

aten = torch.ops.aten

CREATE_ATEN_OP = [
    aten.empty.memory_format, aten.zeros.default, aten.ones.default, aten.scalar_tensor.default,
    aten.arange.default, aten.arange.start, aten.full.default,
]

# ---- local shapes -----------------------------------------------------------------------------------------


def local_shape(global_shape, mesh, placements):
    """Shape of this rank's shard: torch.chunk (ceil-div) blocks per sharded mesh dim, applied
    outer mesh dim first (DTensor compute_local_shape, used by torch/utils.py:106-136)."""
    shape = list(global_shape)
    coord = mesh.get_coordinate()
    for mdim, p in enumerate(placements):
        if p is not None and p.is_shard():
            d, n = p.dim, mesh.size(mdim)
            full = -(-shape[d] // n)
            lo = min(shape[d], full * coord[mdim])
            hi = min(shape[d], full * (coord[mdim] + 1))
            shape[d] = hi - lo
    return shape


def _torch_placements(strategy):
    from torch.distributed.tensor import Partial, Replicate, Shard
    out = []
    for s in strategy:
        if s.is_shard():
            out.append(Shard(s.dim))
        elif s.is_partial():
            out.append(Partial(s.op))
        else:
            out.append(Replicate())
    return out


def _view_rules(node):
    from torch.distributed.tensor._ops._view_ops import expand, normalize_sizes, view_groups
    if node.target in (aten.view.default, aten._unsafe_view.default, aten.reshape.default):
        return lambda in_shape, shape: view_groups(in_shape, shape)
    if node.target == aten.expand.default:
        return lambda in_shape, sizes: expand(in_shape, normalize_sizes(sizes))
    return None


def override_args(node, invars_strategy, mesh):
    """Rewrite the size argument of view/reshape/expand nodes to the LOCAL output shape under the
    input's placement (sharding.py:812-849)."""
    rules_fn = _view_rules(node)
    if rules_fn is None:
        return
    from torch.distributed.tensor._ops._view_ops import propagate_shape_and_sharding
    global_in_shape = tuple(node.args[0].meta["val"].shape)
    in_spec = _torch_placements(invars_strategy[0])
    rules = rules_fn(global_in_shape, node.args[1])
    _, shard_out = propagate_shape_and_sharding(in_spec, global_in_shape, rules,
                                                tuple(mesh.shape))
    if shard_out is None:
        shard_out = in_spec
    from torch.distributed.tensor import Shard
    out_strategy = [M.S(p.dim) if isinstance(p, Shard) else M.R() for p in shard_out]
    global_out_shape = list(node.meta["val"].shape)
    node.update_arg(1, local_shape(global_out_shape, mesh, out_strategy))


# ---- edge lowering -----------------------------------------------------------------------------------------


def insert_comm_node(gm, node, var_, src_specs, tgt_specs, mesh, ops, planner="GREEDY",
                     copy_innode=None, global_shape_of=None):
    """Emit the reshard steps turning `var_` (placement src_specs) into tgt_specs in front of
    `node` (sharding.py:704-809).  One step = one op on the flat rank group of one mesh dim."""
    p2p_left = None
    if global_shape_of is None and isinstance(var_.meta.get("val"), torch.Tensor):
        global_shape_of = var_.meta["val"].shape  # metas are still global while the pass runs
    if planner == "P2P":
        # single-collective steps first, the rest as one box exchange over the whole mesh
        # (sharding.py:721-723, 795-802)
        steps, reached = planners.plan_immediate(src_specs, tgt_specs)
        if reached != tgt_specs:
            p2p_left = reached
    else:
        steps = planners.PLANNERS[planner](src_specs, tgt_specs)
    coord = mesh.get_coordinate()
    graph = gm.graph
    for mdim, cur, tgt in steps:
        kind = planners.step_kind(cur, tgt)
        if kind is None:
            continue
        n = mesh.size(mdim)
        ranks = mesh.ranks_along(mdim)
        with graph.inserting_before(node):
            if kind == "scatter":
                new = graph.call_function(ops.scatter_wrapper, args=(var_, n, tgt.dim, coord[mdim]))
            elif kind == "all_to_all":
                a = (cur.dim, tgt.dim, n, coord[mdim], ranks)
                s = graph.call_function(ops.all_to_all_start, args=(var_, *a))
                new = graph.call_function(ops.all_to_all_end, args=(s, *a))
            elif kind == "reduce_scatter":
                a = (cur.op, tgt.dim, ranks)
                s = graph.call_function(ops.reduce_scatter_start, args=(var_, *a))
                new = graph.call_function(ops.reduce_scatter_end, args=(s, *a))
            elif kind == "all_gather":
                a = (cur.dim, ranks)
                s = graph.call_function(ops.all_gather_start, args=(var_, *a))
                new = graph.call_function(ops.all_gather_end, args=(s, *a))
            elif kind == "all_reduce":
                a = (cur.op, ranks)
                s = graph.call_function(ops.all_reduce_start, args=(var_, *a))
                new = graph.call_function(ops.all_reduce_end, args=(s, *a))
            else:  # pragma: no cover
                raise AssertionError(kind)
        node.replace_input_with(var_, new)
        var_ = new
    if p2p_left is not None:
        global_shape = [int(d) for d in global_shape_of]
        srcs = planners.partitions_from_spec(p2p_left, global_shape, mesh)
        tgts = planners.partitions_from_spec(tgt_specs, global_shape, mesh)
        ranks = [p.rank for p in srcs]
        me = ranks.index(mesh.get_rank())
        boxes = []
        for it in planners.recv_boxes(srcs, tgts[me]):
            sp = srcs[ranks.index(it.rank)]
            boxes.append((ranks.index(it.rank),
                          [a - b for a, b in zip(it.start, sp.start)],
                          [a - b for a, b in zip(it.start, tgts[me].start)],
                          list(it.shape())))
        with graph.inserting_before(node):
            new = graph.call_function(ops.box_exchange, args=(
                var_, list(tgts[me].shape()), boxes, [list(p.shape()) for p in srcs], ranks))
        node.replace_input_with(var_, new)
        var_ = new
    if copy_innode is not None:
        with graph.inserting_before(node):
            cp = graph.call_function(ops.copy_wrapper, args=(copy_innode, var_))
        node.replace_input_with(var_, cp)
    return gm


def _normalise_plan(opt_strategy):
    """Accept the reference's objects (duck typed) or ours."""
    any_entry = next(iter(opt_strategy.values()), None)
    if any_entry is None or isinstance(any_entry["strategy"], M.NodeSPMDStrategy):
        return opt_strategy
    return M.plan_from_reference(opt_strategy)


def _num_user_returns(gm):
    spec = gm._out_spec
    children = spec.children() if callable(getattr(spec, "children", None)) else spec.children_specs
    return children[-1].num_leaves


def sharding_transform(fx_module: torch.fx.GraphModule, opt_strategy, state_io_map, *,
                       ops=_default_ops, mesh=None, planner="GREEDY"):
    """Drop-in for the reference's sharding_transform (same positional arguments)."""
    mesh = mesh or get_device_mesh("spmd")
    plan = _normalise_plan(opt_strategy)
    shard_env: Dict[str, object] = {}
    replicate = M.replicate_strategy(mesh.ndim)
    n_ret = _num_user_returns(fx_module)
    placeholders = {}
    for node in list(fx_module.graph.nodes):
        if node.op == "placeholder":
            if node.name in plan:
                shard_env[node.name] = plan[node.name]["strategy"].out_strtg_group[0]
            else:
                shard_env[node.name] = replicate
            placeholders[node.name] = node
        elif node.op == "call_function":
            if node.target in CREATE_ATEN_OP:
                shard_env[node.name] = replicate
                continue
            if node.target == operator.getitem:
                shard_env[node.name] = shard_env[node.args[0].name][node.args[1]]
                continue
            invars = [a for a in pytree.tree_flatten(node.args)[0] if isinstance(a, Node)]
            if node.name not in plan:
                raise KeyError(f"no strategy for node {node.name} in the plan")
            strat = plan[node.name]["strategy"]
            in_strats = strat.in_strtg_group
            override_args(node, in_strats, mesh)
            assert len(invars) == len(in_strats), (node.name, len(invars), len(in_strats))
            seen = set()
            for var_, tgt in zip(invars, in_strats):
                if var_ in seen:
                    continue
                seen.add(var_)
                src = shard_env[var_.name]
                if tgt is not None and tgt != src:
                    insert_comm_node(fx_module, node, var_, src, tgt, mesh, ops, planner)
            out = strat.out_strtg_group
            shard_env[node.name] = out[0] if len(out) == 1 else out
        elif node.op == "output":
            outs = list(node.args[0])
            for o in [o for o in outs[len(outs) - n_ret:] if isinstance(o, Node)]:
                src = shard_env[o.name]
                if src is not None and src != replicate:
                    insert_comm_node(fx_module, node, o, src, replicate, mesh, ops, planner)
            for in_node, out_node in state_io_map.items():
                if in_node.name not in shard_env:
                    continue
                o = next((x for x in node.args[0] if isinstance(x, Node) and
                          x.name == out_node.name), None)
                assert o is not None, out_node.name
                src, tgt = shard_env[o.name], shard_env[in_node.name]
                if tgt != src:
                    insert_comm_node(fx_module, node, o, src, tgt, mesh, ops, planner,
                                     copy_innode=placeholders[in_node.name])
    fx_module.graph.lint()
    legalize_views(fx_module, mesh, shard_env)
    fx_module.recompile()
    fx_module._edb_shard_env = shard_env
    return fx_module


def legalize_views(gm, mesh, shard_env):
    """`aten.view` is stride dependent: after a reshard its input may be a non-contiguous local
    tensor and the traced view is no longer legal (the reference hits the same wall: SURVEY.md
    hard part 1; its meta propagation only works under torch 2.11 with the reshape retry of
    oracle/refcompat).  Dry-run the lowered graph on fake LOCAL placeholders and retarget exactly
    the view nodes that fail to `aten.reshape` (same values, copies when it must).  Returns the
    number of nodes changed.  A dry run that cannot complete is an ERROR (views behind the failing
    node would stay unchecked and an illegal one would only surface at run time, on one rank);
    `EDB_LEGALIZE_BEST_EFFORT=1` restores the old log-and-continue behaviour."""
    import os
    from torch._subclasses.fake_tensor import FakeTensorMode
    changed = 0
    env = {}
    cur = None
    try:
        with FakeTensorMode(allow_non_fake_inputs=True):
            for node in gm.graph.nodes:
                if node.op == "placeholder":
                    val = node.meta.get("val")
                    if isinstance(val, torch.Tensor):
                        strat = shard_env.get(node.name)
                        shape = list(val.shape)
                        if isinstance(strat, (M.VarSPMDStrategy, list, tuple)) and all(
                                s is None or hasattr(s, "is_shard") for s in strat):
                            shape = local_shape(shape, mesh, strat)
                        env[node] = torch.empty(shape, dtype=val.dtype, device=val.device)
                    else:
                        env[node] = val
                elif node.op == "call_function":
                    cur = node
                    args, kwargs = pytree.tree_map_only(Node, lambda n: env[n],
                                                        (node.args, node.kwargs))
                    try:
                        env[node] = node.target(*args, **kwargs)
                    except (RuntimeError, ValueError):
                        if node.target not in (aten.view.default, aten._unsafe_view.default):
                            raise
                        node.target = aten.reshape.default
                        env[node] = node.target(*args, **kwargs)
                        changed += 1
                elif node.op == "output":
                    break
                else:
                    return changed
    except Exception as e:  # noqa: BLE001
        if os.environ.get("EDB_LEGALIZE_BEST_EFFORT", "0") == "1":
            import logging
            logging.getLogger(__name__).warning("legalize_views stopped early: %r", e)
            return changed
        raise RuntimeError(
            f"legalize_views: the dry run of the lowered graph failed at node "
            f"{cur.name if cur is not None else '?'} ({getattr(cur, 'target', None)}): {e!r}; views "
            "behind it are unchecked (EDB_LEGALIZE_BEST_EFFORT=1 to continue anyway)") from e
    return changed


# ---- data-parallel rewrites (compile_dp.py:55-198) ---------------------------------------------------------

_ELEMENTWISE_OPT_OPS = None


def _optimizer_elementwise_ops():
    global _ELEMENTWISE_OPT_OPS
    if _ELEMENTWISE_OPT_OPS is None:
        ok = {operator.getitem}
        from .compile import aten_op_names
        for name in aten_op_names("_foreach_"):
            if not name.endswith("_") and "norm" not in name and name != "_foreach_max":
                ok.update(getattr(getattr(aten, name), o) for o in getattr(aten, name).overloads())
        for name in ("_fused_adam", "_fused_adamw", "_fused_sgd", "copy_", "add", "sub", "mul",
                     "div", "addcmul", "addcdiv", "sqrt", "rsqrt", "pow", "neg", "reciprocal",
                     "lerp", "clone", "maximum", "minimum", "_to_copy", "where", "abs", "sign",
                     "zeros_like", "ones_like", "detach", "alias", "lt", "gt", "ge", "le", "eq"):
            if hasattr(aten, name):
                pk = getattr(aten, name)
                ok.update(getattr(pk, o) for o in pk.overloads())
        _ELEMENTWISE_OPT_OPS = ok
    return _ELEMENTWISE_OPT_OPS


def optimizer_region(gm, io):
    """Nodes downstream of the final gradients (the optimizer update), in graph order."""
    grads = [g for g in io.final_grads if isinstance(g, Node)]
    region, stack = set(), list(grads)
    while stack:
        n = stack.pop()
        for u in n.users:
            if u.op != "output" and u not in region:
                region.add(u)
                stack.append(u)
    return [n for n in gm.graph.nodes if n in region]


def transform_ddp(gm, io, ranks, ops=_default_ops, bucket_numel=0):
    """ddp: all-reduce(avg) every final gradient before the optimizer consumes it
    (compile_dp.py:55-79 does this for the gradient list of `_fused_adam`).  Gradients of
    parameters below `bucket_numel` elements share one bucketed all-reduce."""
    ranks = list(ranks)
    if len(ranks) <= 1:
        return gm
    small = {ph for ph in io.param_ph if ph.meta["val"].numel() < bucket_numel}
    if small:
        region = optimizer_region(gm, io)
        if region:
            _bucket_small_grads(gm, io, ranks, small, region, ops)
        else:
            small = set()
    big = [g for ph, g in zip(io.param_ph, io.final_grads) if isinstance(g, Node) and ph not in small]
    for g in dict.fromkeys(big):
        with gm.graph.inserting_after(g):
            s = gm.graph.call_function(ops.all_reduce_start, args=(g, "avg", ranks))
        with gm.graph.inserting_after(s):
            e = gm.graph.call_function(ops.all_reduce_end, args=(s, "avg", ranks))
        g.replace_all_uses_with(e, delete_user_cb=lambda u: u is not s)
    gm.graph.lint()
    gm.recompile()
    return gm


def _bucket_small_grads(gm, io, ranks, small, region, ops):
    """One all-reduce(avg) for all small gradients: cat(flatten(g_i)) -> all_reduce -> views.
    Same rule of thumb as the reference's comm_group pass (passes/comm_optimize.py:223-286 buckets
    all-reduces below 1 MB into one flat buffer); their parameters stay replicated."""
    graph = gm.graph
    grads = [(ph, g) for ph, g in zip(io.param_ph, io.final_grads)
             if ph in small and isinstance(g, Node)]
    if not grads:
        return
    anchor = region[0]
    with graph.inserting_before(anchor):
        flats = [graph.call_function(aten.flatten.using_ints, args=(g,)) for _, g in grads]
        cat = graph.call_function(aten.cat.default, args=(flats, 0))
        s = graph.call_function(ops.all_reduce_start, args=(cat, "avg", list(ranks)))
        e = graph.call_function(ops.all_reduce_end, args=(s, "avg", list(ranks)))
        off = 0
        pieces = []
        for ph, g in grads:
            shape = list(ph.meta["val"].shape)
            numel = ph.meta["val"].numel()
            sl = graph.call_function(aten.slice.Tensor, args=(e, 0, off, off + numel))
            pieces.append(graph.call_function(aten.view.default, args=(sl, shape)))
            off += numel
    own = set(flats)
    for (ph, g), piece in zip(grads, pieces):
        g.replace_all_uses_with(piece, delete_user_cb=lambda u: u not in own)


def transform_fsdp(gm, io, ranks, my_index, shard_param, ops=_default_ops, bucket_numel=0):
    """zero2 (shard_param=False) / zero3 (True), compile_dp.py:82-198: gradients are flattened and
    reduce-scattered(avg), optimizer states (and, for zero3, parameters) live as flat 1/n shards;
    zero3 all-gathers a parameter in front of each forward/backward use, zero2 scatters the
    parameter into the optimizer and all-gathers the updated shard back."""
    ranks = list(ranks)
    n = len(ranks)
    if n <= 1:
        return gm, {}
    graph = gm.graph
    region = optimizer_region(gm, io)
    region_set = set(region)
    allowed = _optimizer_elementwise_ops()
    for node in region:
        if node.op == "call_function" and node.target not in allowed and \
                node.target not in ops.CUSTOM_FUNCS:
            raise NotImplementedError(
                f"zero2/zero3: optimizer op {node.target} is not elementwise over (param, grad, "
                f"state); cannot run it on flat shards")
    shard_info = {}  # placeholder name -> original shape (for pre-sharding the state)
    # parameters below `bucket_numel` elements are not sharded: their gradients travel in ONE
    # bucketed all-reduce and they (and their optimizer state) stay replicated (0 = reference
    # behaviour: everything is sharded tensor by tensor)
    small = {ph for ph in io.param_ph if ph.meta["val"].numel() < bucket_numel}
    if small:
        _bucket_small_grads(gm, io, ranks, small, region, ops)

    def check_divisible(ph):
        numel = ph.meta["val"].numel()
        if numel % n != 0:
            # reduce_scatter_start asserts the same (sharding.py:136-137)
            raise AssertionError(f"{ph.name}: numel {numel} must be a multiple of group_size {n}")

    # (1) gradients: flatten + reduce_scatter(avg) along dim 0
    big_grads = [g for ph, g in zip(io.param_ph, io.final_grads)
                 if isinstance(g, Node) and ph not in small]
    for g in dict.fromkeys(big_grads):
        with graph.inserting_after(g):
            f = graph.call_function(aten.flatten.using_ints, args=(g,))
        with graph.inserting_after(f):
            s = graph.call_function(ops.reduce_scatter_start, args=(f, "avg", 0, ranks))
        with graph.inserting_after(s):
            e = graph.call_function(ops.reduce_scatter_end, args=(s, "avg", 0, ranks))
        g.replace_all_uses_with(e, delete_user_cb=lambda u: u is not f)

    # (2) parameters
    for ph in io.param_ph:
        if ph in small:
            continue
        check_divisible(ph)
        shape = list(ph.meta["val"].shape)
        if shard_param:
            shard_info[ph.name] = shape
            for user in list(ph.users):
                if user in region_set or user.op == "output":
                    continue
                with graph.inserting_before(user):
                    s = graph.call_function(ops.all_gather_start, args=(ph, 0, ranks))
                    e = graph.call_function(ops.all_gather_end, args=(s, 0, ranks))
                    v = graph.call_function(aten.view.default, args=(e, shape))
                user.replace_input_with(ph, v)
        else:
            opt_users = [u for u in ph.users if u in region_set]
            if not opt_users:
                continue
            first = min(opt_users, key=lambda u: region.index(u))
            with graph.inserting_before(first):
                f = graph.call_function(aten.flatten.using_ints, args=(ph,))
                sc = graph.call_function(ops.scatter_wrapper, args=(f, n, 0, my_index))
            for user in opt_users:
                if user.target == aten.copy_.default and user.args[0] is ph:
                    # write-back of the updated shard: gather it into the full parameter
                    new_shard = user.args[1]
                    with graph.inserting_before(user):
                        s = graph.call_function(ops.all_gather_start, args=(new_shard, 0, ranks))
                        e = graph.call_function(ops.all_gather_end, args=(s, 0, ranks))
                        v = graph.call_function(aten.view.default, args=(e, shape))
                    user.update_arg(1, v)
                else:
                    user.replace_input_with(ph, sc)

    # (3) optimizer states with the parameter's numel live as flat shards
    param_numels = {ph.meta["val"].numel() for ph in io.param_ph if ph not in small}
    for ph, is_t in zip(io.state_ph, io.state_is_tensor):
        if not is_t:
            continue
        val = ph.meta.get("val")
        if val is None or val.dim() == 0 or val.numel() not in param_numels:
            continue  # step counters etc. stay replicated
        check_divisible(ph)
        shard_info[ph.name] = list(val.shape)

    graph.lint()
    gm.recompile()
    return gm, shard_info


# ---- finishing passes -----------------------------------------------------------------------------------------


def bucket_small_comm(gm, ops=_default_ops, max_bytes=1 << 20, max_bucket_bytes=32 << 20):
    """Bucket small all-reduces, dim-0 all-gathers and reduce-scatters (any scatter dim) of the
    lowered graph (any parallel mode).

    Auto-SPMD plans reshard many tiny tensors one collective each (SURVEY.md App. B: 16 all-reduces
    of 4 KB and 108 all-gathers of 2 KB per step in the reference's GPT example); the reference
    groups communication below 1 MB into flat buffers in `comm_optimize.comm_group`
    (passes/comm_optimize.py:223-286).  Here, collectives of the same kind / group / dtype (and
    reduce op) whose inputs all exist before the first of their results is read become

        cat(flatten(x_i)) -> ONE collective -> slice / view per tensor

    placed in front of that first reader.  Values are unchanged (all-reduce is elementwise; a dim-0
    all-gather of a flattened concatenation is a [n, total] matrix whose column block i is tensor
    i's gathered rows).  Needs local metas (`propagate_local_meta`).  Returns {kind: buckets}."""
    graph = gm.graph
    order = {nd: i for i, nd in enumerate(graph.nodes)}
    cands = {}
    for st in graph.nodes:
        if st.op != "call_function" or st.target not in (ops.all_reduce_start, ops.all_gather_start,
                                                         ops.reduce_scatter_start):
            continue
        x = st.args[0]
        if not isinstance(x, Node) or len(st.users) != 1 or st.kwargs:
            continue
        end = next(iter(st.users))
        val, out = x.meta.get("val"), st.meta.get("val")
        if not isinstance(val, torch.Tensor) or not isinstance(out, torch.Tensor) or not end.users:
            continue
        if val.numel() == 0 or val.numel() * val.element_size() >= max_bytes:
            continue
        if st.target is ops.all_reduce_start:
            if end.target is not ops.all_reduce_end:
                continue
            key = ("all_reduce", st.args[1], tuple(st.args[2]), val.dtype)
        elif st.target is ops.reduce_scatter_start:
            d = st.args[2]
            if end.target is not ops.reduce_scatter_end or not isinstance(d, int) or val.dim() == 0:
                continue
            d = d + val.dim() if d < 0 else d
            if not 0 <= d < val.dim() or val.shape[d] % len(st.args[3]):
                continue
            key = ("reduce_scatter", st.args[1], tuple(st.args[3]), val.dtype)
        else:
            if end.target is not ops.all_gather_end or st.args[1] != 0 or val.dim() == 0:
                continue
            key = ("all_gather", None, tuple(st.args[2]), val.dtype)
        cands.setdefault(key, []).append((st, end, x, val))

    def first_use(items):
        return min((u for _, end, _, _ in items for u in end.users), key=lambda u: order[u])

    done = {"all_reduce": 0, "all_gather": 0, "reduce_scatter": 0}
    for key, items in cands.items():
        items.sort(key=lambda it: order[it[2]])
        runs, cur, cur_bytes = [], [], 0
        for it in items:
            nbytes = it[3].numel() * it[3].element_size()
            if cur and (order[it[2]] > order[first_use(cur)] or cur_bytes + nbytes > max_bucket_bytes):
                runs.append(cur)
                cur, cur_bytes = [], 0
            cur.append(it)
            cur_bytes += nbytes
        runs.append(cur)
        kind, red, group, _ = key
        n = len(group)
        for run in runs:
            if len(run) < 2:
                continue
            if kind == "reduce_scatter":
                # x_i with its scatter dim in front, as [n, k_i]: row p is what member p keeps.
                # cat over i -> [n, K] -> ONE reduce-scatter along dim 0 -> [1, K] -> column block i
                # back into the shape (and dim order) of the single result
                with graph.inserting_before(first_use(run)):
                    mats, metas = [], []
                    for st, _, x, v in run:
                        d = st.args[2] + v.dim() if st.args[2] < 0 else st.args[2]
                        perm = [d] + [i for i in range(v.dim()) if i != d]
                        y = x if d == 0 else graph.call_function(aten.permute.default, args=(x, perm))
                        mats.append(graph.call_function(aten.reshape.default, args=(y, [n, v.numel() // n])))
                        metas.append((d, perm))
                    cat = graph.call_function(aten.cat.default, args=(mats, 1))
                    s_ = graph.call_function(ops.reduce_scatter_start, args=(cat, red, 0, list(group)))
                    e_ = graph.call_function(ops.reduce_scatter_end, args=(s_, red, 0, list(group)))
                    off = 0
                    for (st, end, x, v), (d, perm) in zip(run, metas):
                        k = v.numel() // n
                        sl = graph.call_function(aten.slice.Tensor, args=(e_, 1, off, off + k))
                        front = [v.shape[d] // n] + [v.shape[i] for i in perm[1:]]
                        piece = graph.call_function(aten.reshape.default, args=(sl, front))
                        if d != 0:
                            inv = [perm.index(i) for i in range(v.dim())]
                            piece = graph.call_function(aten.permute.default, args=(piece, inv))
                            piece = graph.call_function(aten.clone.default, args=(piece,),
                                                        kwargs={"memory_format": torch.contiguous_format})
                        piece.meta = dict(end.meta)
                        end.replace_all_uses_with(piece)
                        off += k
                for st, end, _, _ in run:
                    graph.erase_node(end)
                    graph.erase_node(st)
                done[kind] += 1
                continue
            with graph.inserting_before(first_use(run)):
                flats = [graph.call_function(aten.flatten.using_ints, args=(x,)) for _, _, x, _ in run]
                cat = graph.call_function(aten.cat.default, args=(flats, 0))
                total = sum(v.numel() for *_, v in run)
                if kind == "all_reduce":
                    s_ = graph.call_function(ops.all_reduce_start, args=(cat, red, list(group)))
                    e_ = graph.call_function(ops.all_reduce_end, args=(s_, red, list(group)))
                    src = e_
                else:
                    s_ = graph.call_function(ops.all_gather_start, args=(cat, 0, list(group)))
                    e_ = graph.call_function(ops.all_gather_end, args=(s_, 0, list(group)))
                    src = graph.call_function(aten.view.default, args=(e_, [n, total]))
                off = 0
                for st, end, x, v in run:
                    k = v.numel()
                    if kind == "all_reduce":
                        sl = graph.call_function(aten.slice.Tensor, args=(src, 0, off, off + k))
                        piece = graph.call_function(aten.view.default, args=(sl, list(v.shape)))
                    else:
                        sl = graph.call_function(aten.slice.Tensor, args=(src, 1, off, off + k))
                        piece = graph.call_function(aten.reshape.default,
                                                    args=(sl, [n * v.shape[0]] + list(v.shape[1:])))
                    piece.meta = dict(end.meta)
                    end.replace_all_uses_with(piece)
                    off += k
            for st, end, _, _ in run:
                graph.erase_node(end)
                graph.erase_node(st)
            done[kind] += 1
    if any(done.values()):
        graph.lint()
        gm.recompile()
    return done


def _is_functional_foreach(target):
    schema = getattr(target, "_schema", None)
    return schema is not None and schema.name.startswith("aten::_foreach_") and \
        not schema.name.endswith("_") and "norm" not in schema.name and \
        schema.name not in ("aten::_foreach_max", "aten::_foreach_copy")


def localize_foreach(gm, ops=_default_ops, my_rank=None):
    """Elementwise foreach ops on SHARDS instead of on gathered tensors (auto-SPMD plans).

    The reference only knows a *replicate* strategy for the optimizer's `_foreach_*` ops
    (easydist/torch/preset_propagation.py:113-165) while parameters and optimizer states live
    sharded, so its lowering all-gathers every parameter, gradient and state in front of each
    foreach op and `scatter_wrapper`s + `copy_`s every result back (SURVEY.md fact 5: at mesh (8,)
    the config-1 step carries ~300 all-gathers and 192 local scatters for nothing but this).  An
    elementwise op commutes with sharding:

        scatter(op(all_gather(a_i, d), all_gather(b_i, d), ...), n, d, idx)  ==  op(a_i, b_i, ...)

    bit for bit.  For every list position whose result is only consumed by scatter_wrapper(n, d, idx)
    the inputs are replaced by their shards along d: the source of an all-gather along d (nothing
    moves), an all-to-all for an operand that is sharded along another dimension (1/n of the
    all-gather's traffic), a local slice for a replicated operand.  Positions that do not fit stay
    in a residual foreach node with the gathered inputs.  Returns the number of positions made
    local."""
    graph = gm.graph
    n_local = 0
    if my_rank is None:
        import torch.distributed as dist
        my_rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0

    def ag_source(x):
        """x == all_gather_end(all_gather_start(s, d, group)) -> (s, d, group) else None."""
        if not (isinstance(x, Node) and x.op == "call_function" and x.target is ops.all_gather_end):
            return None
        st = x.args[0]
        if not (isinstance(st, Node) and st.target is ops.all_gather_start):
            return None
        src, d, group = st.args[0], st.args[1], list(st.args[2])
        if isinstance(src, Node) and src.op == "call_function" and src.target is ops.all_gather_end:
            return None  # nested (N-D mesh) shardings are left alone
        return src, d, group

    for F in list(graph.nodes):
        if F.op != "call_function" or not _is_functional_foreach(F.target):
            continue
        list_pos = [k for k, a in enumerate(F.args)
                    if isinstance(a, (list, tuple)) and len(a) > 0 and all(isinstance(x, Node) for x in a)]
        if not list_pos:
            continue
        L = len(F.args[list_pos[0]])
        if any(len(F.args[k]) != L for k in list_pos):
            continue
        outs = {}
        bad = False
        for u in F.users:
            if u.target is not operator.getitem or u.args[1] in outs:
                bad = True
                break
            outs[u.args[1]] = u
        if bad:
            continue
        local = {}  # position -> (n, d, idx, group or None)
        for i in range(L):
            gi = outs.get(i)
            if gi is None or not gi.users:
                continue
            us = list(gi.users)
            if not all(u.op == "call_function" and u.target is ops.scatter_wrapper and u.args[0] is gi
                       and not any(w.op == "call_function" and w.target is ops.scatter_wrapper
                                   for w in u.users) for u in us):
                continue
            sig = {(u.args[1], u.args[2], u.args[3]) for u in us}
            if len(sig) != 1:
                continue
            n, d, idx = sig.pop()
            group = None
            ok = True
            for k in list_pos:
                src = ag_source(F.args[k][i])
                if src is None:
                    continue
                _, _, g = src
                if len(g) != n or my_rank not in g or g.index(my_rank) != idx or \
                        (group is not None and g != group):
                    ok = False
                    break
                group = g
            if ok:
                local[i] = (n, d, idx, group)
        if not local:
            continue
        with graph.inserting_before(F):
            new_lists = {k: [] for k in list_pos}
            for i in sorted(local):
                n, d, idx, group = local[i]
                for k in list_pos:
                    x = F.args[k][i]
                    src = ag_source(x)
                    xv = x.meta.get("val")
                    dd = d + xv.dim() if (d < 0 and isinstance(xv, torch.Tensor)) else d
                    if src is not None and (src[1] == d or src[1] == dd):
                        new_lists[k].append(src[0])                       # already the shard
                    elif src is not None:
                        s_, sd, g = src                                   # sharded along another dim
                        a2a = graph.call_function(ops.all_to_all_start, args=(s_, sd, d, n, idx, g))
                        new_lists[k].append(graph.call_function(
                            ops.all_to_all_end, args=(a2a, sd, d, n, idx, g)))
                    else:                                                 # replicated: my slice
                        new_lists[k].append(graph.call_function(ops.scatter_wrapper, args=(x, n, d, idx)))
            idxs = sorted(local)

            def sub_args(keep, lists):
                out = []
                for k, a in enumerate(F.args):
                    if k in lists:
                        out.append(lists[k])
                    elif isinstance(a, (list, tuple)) and len(a) == L:
                        out.append([a[i] for i in keep])                  # per-element scalars
                    else:
                        out.append(a)
                return tuple(out)

            F_loc = graph.call_function(F.target, args=sub_args(idxs, new_lists), kwargs=dict(F.kwargs))
            rest = [i for i in range(L) if i not in local]
            F_rest = None
            if rest:
                rest_lists = {k: [F.args[k][i] for i in rest] for k in list_pos}
                F_rest = graph.call_function(F.target, args=sub_args(rest, rest_lists),
                                             kwargs=dict(F.kwargs))
        with graph.inserting_after(F_rest if F_rest is not None else F_loc):
            for j, i in enumerate(idxs):
                gi = outs[i]
                new = graph.call_function(operator.getitem, args=(F_loc, j))
                for u in list(gi.users):                                  # the scatter_wrappers
                    new.meta = dict(u.meta)
                    u.replace_all_uses_with(new)
                    graph.erase_node(u)
                graph.erase_node(gi)
            for j, i in enumerate(rest):
                gi = outs.get(i)
                if gi is None:
                    continue
                new = graph.call_function(operator.getitem, args=(F_rest, j))
                new.meta = dict(gi.meta)
                gi.replace_all_uses_with(new)
                graph.erase_node(gi)
        graph.erase_node(F)
        n_local += len(idxs)
    if n_local:
        # all-gathers that only fed the gathered form of those positions are dead now
        for nd in reversed(list(graph.nodes)):
            if nd.op == "call_function" and nd.target in (ops.all_gather_end, ops.all_gather_start) \
                    and not nd.users:
                graph.erase_node(nd)
        graph.lint()
        gm.recompile()
    return n_local


def propagate_local_meta(gm, flat_inputs):
    """Re-run shape propagation on the lowered graph with LOCAL placeholder values so that every
    node's meta['val'] is the per-rank tensor (the reference recomputes metas node by node with
    create_meta_from_node, sharding.py:953-977)."""
    from torch._subclasses.fake_tensor import FakeTensorMode
    from torch.fx.passes.fake_tensor_prop import FakeTensorProp
    mode = FakeTensorMode(allow_non_fake_inputs=True)
    fake_inputs = [mode.from_tensor(x) if isinstance(x, torch.Tensor) else x for x in flat_inputs]
    FakeTensorProp(gm, mode).propagate_dont_convert_inputs(*fake_inputs)
    return gm


def _nbytes(val):
    return val.numel() * val.element_size()


def assign_static_buffers(gm, rt, ops=_default_ops, push=False):
    """Give every communication node fixed symmetric-heap buffers (`_buf` kwarg) sized from the
    local metas: no allocation, no address change on the comm path => CUDA-graph capturable and
    zero-copy outputs.  Returns the number of bytes reserved.

    push=True (the graph ends with an epoch barrier, see insert_epoch_barriers): the nodes are
    marked `_push=1` — with buffers dedicated to a node and a group barrier between two steps the
    collectives need no handshake (edb_*_push in edb.h): data straight into the consumers' buffers
    plus one flag per peer."""
    total = 0
    oneshot = rt.get_option("allreduce_oneshot_bytes")
    for node in gm.graph.nodes:
        if node.op != "call_function" or node.target not in ops.COMM_FUNCS:
            continue
        x = node.args[0].meta["val"]
        if node.target is ops.all_gather_start:
            need = [_nbytes(node.meta["val"])]
        elif node.target is ops.all_reduce_start:
            if push:
                grp = node.args[2]
                need = list(ops.all_reduce_push_sizes(_nbytes(x), x.numel(), x.element_size(),
                                                      len(grp), oneshot))
            else:
                need = [_nbytes(x)] * (2 if _nbytes(x) > oneshot else 1)
        else:
            need = [_nbytes(x)]
        if need[0] == 0:
            continue
        bufs = [rt.alloc(b) for b in need]
        total += sum(need)
        kw = dict(node.kwargs)
        kw["_buf"] = (bufs[0].offset, need[0]) + tuple(b.offset for b in bufs[1:])
        if push:
            kw["_push"] = 1
        node.kwargs = kw
    gm.recompile()
    return total


def fuse_cross_entropy(gm):
    """Rewrite the cross-entropy tail of a traced train step onto edb_loss.cu:

        [_to_copy(fp32)] -> _log_softmax(dim=-1) -> nll_loss_forward          ==> loss.cross_entropy_fwd
        nll_loss_backward -> _log_softmax_backward_data -> [_to_copy(lp)]     ==> loss.cross_entropy_bwd

    Only the exact chain F.cross_entropy(logits.float(), target) traces to is matched (2-D logits,
    weight=None, reduction mean/sum, log-softmax saved for nothing but its own backward).
    Returns the number of chains rewritten."""
    import operator
    from . import loss
    graph = gm.graph
    n = 0
    for ls in [x for x in graph.nodes if x.op == "call_function" and x.target == aten._log_softmax.default]:
        x32, dim, half_to_float = ls.args
        if half_to_float or not isinstance(x32, Node):
            continue
        users = list(ls.users)
        fwd = [u for u in users if u.target == aten.nll_loss_forward.default and u.args[0] is ls]
        bwd = [u for u in users if u.target == aten.nll_loss_backward.default and u.args[1] is ls]
        lsb = [u for u in users if u.target == aten._log_softmax_backward_data.default and u.args[1] is ls]
        if len(users) != 3 or len(fwd) != 1 or len(bwd) != 1 or len(lsb) != 1:
            continue
        fwd, bwd, lsb = fwd[0], bwd[0], lsb[0]
        if len(fwd.args) != 5 or len(bwd.args) != 7 or fwd.kwargs or bwd.kwargs:
            continue
        _, tgt, weight, red, ign = fwd.args
        gout, _, tgt_b, weight_b, red_b, ign_b, tw = bwd.args
        if weight is not None or weight_b is not None or red not in (1, 2) or red_b != red \
                or ign_b != ign or tgt_b is not tgt:
            continue
        if lsb.args[0] is not bwd or list(bwd.users) != [lsb] or lsb.args[2] != dim:
            continue
        if not (isinstance(tw, Node) and tw.target is operator.getitem and tw.args[0] is fwd
                and tw.args[1] == 1):
            continue
        if any(u.target is not operator.getitem for u in fwd.users):
            continue
        val = ls.meta.get("val")
        if isinstance(val, torch.Tensor) and (val.dim() != 2 or dim not in (1, -1)):
            continue
        if val is None and dim != 1:
            continue
        # optional precision round trip around the fp32 log-softmax
        x, last = x32, lsb
        if x32.op == "call_function" and x32.target == aten._to_copy.default and len(x32.users) == 1 \
                and x32.kwargs.get("dtype") == torch.float32 and len(lsb.users) == 1:
            cast_back = next(iter(lsb.users))
            src_val = x32.args[0].meta.get("val") if isinstance(x32.args[0], Node) else None
            if cast_back.target == aten._to_copy.default and isinstance(src_val, torch.Tensor) \
                    and cast_back.kwargs.get("dtype") == src_val.dtype \
                    and set(cast_back.kwargs) <= {"dtype", "layout", "device"} \
                    and cast_back.kwargs.get("layout", torch.strided) == torch.strided \
                    and set(x32.kwargs) <= {"dtype"}:
                x, last = x32.args[0], cast_back
        with graph.inserting_before(fwd):
            ce = graph.call_function(loss.cross_entropy_fwd, (x, tgt, ign, red))
            outs = [graph.call_function(operator.getitem, (ce, i)) for i in range(3)]
        for u in list(fwd.users):
            outs[u.args[1]].meta = dict(u.meta)
            u.replace_all_uses_with(outs[u.args[1]])
        with graph.inserting_before(last):
            dx = graph.call_function(loss.cross_entropy_bwd,
                                     (gout, x, tgt, outs[2], outs[1], ign, red))
        dx.meta = dict(last.meta)
        last.replace_all_uses_with(dx)
        # erase exactly the replaced chain (no graph-wide DCE: userless comm/in-place nodes must stay)
        dead = [last] if last is not lsb else []
        dead += [lsb, bwd] + list(fwd.users) + [fwd, ls]
        if x32 is not x:
            dead.append(x32)
        for d in dead:
            assert not d.users, (d, list(d.users))
            graph.erase_node(d)
        n += 1
    if n:
        gm.recompile()
    return n


def fuse_optimizer_updates(gm):
    """The re-inplaced update of torch.optim.SGD(momentum, foreach=True),
        _foreach_mul_(bufs, mu); _foreach_add_(bufs, grads[, alpha=a]); _foreach_add_(params, bufs, alpha=-lr)
    (three consecutive foreach nodes), becomes one `optim.sgd_momentum_` node = one multi-tensor kernel pass.
    Returns the number of triples fused."""
    from . import optim
    graph = gm.graph
    n = 0
    for mul in [x for x in graph.nodes if x.op == "call_function" and x.target == aten._foreach_mul_.Scalar]:
        # the next two in-place foreach nodes; nodes in between are allowed as long as they do not
        # touch the tensors being updated (zero2/zero3 graphs flatten gradients there)
        def next_foreach(start):
            skipped = []
            nd = start.next
            while nd.op == "call_function" and nd.target != aten._foreach_add_.List:
                if "_foreach_" in str(nd.target):
                    return None, skipped
                skipped.append(nd)
                nd = nd.next
            return (nd if nd.op == "call_function" else None), skipped

        add1, skip1 = next_foreach(mul)
        add2, skip2 = next_foreach(add1) if add1 is not None else (None, [])
        if add1 is None or add2 is None:
            continue
        touched = {a for a in pytree.tree_flatten((mul.args[0], add2.args[0]))[0] if isinstance(a, Node)}
        if any(isinstance(a, Node) and a in touched
               for nd in skip1 + skip2 for a in pytree.tree_flatten((nd.args, nd.kwargs))[0]):
            continue
        if mul.kwargs or set(add1.kwargs) - {"alpha"} or set(add2.kwargs) - {"alpha"}:
            continue
        if mul.users or add1.users or add2.users or len(mul.args) != 2:
            continue
        bufs, mu = mul.args
        if not isinstance(mu, (int, float)) or len(add1.args) != 2 or len(add2.args) != 2:
            continue
        if list(add1.args[0]) != list(bufs) or list(add2.args[1]) != list(bufs):
            continue
        grads, params = add1.args[1], add2.args[0]
        if not (len(grads) == len(bufs) == len(params)):
            continue
        if set(params) & set(bufs) or set(grads) & set(bufs) or set(grads) & set(params):
            continue
        ga, nlr = add1.kwargs.get("alpha", 1), add2.kwargs.get("alpha", 1)
        if not isinstance(ga, (int, float)) or not isinstance(nlr, (int, float)):
            continue
        with graph.inserting_before(add2):
            graph.call_function(optim.sgd_momentum_, (list(params), list(grads), list(bufs), mu, ga, nlr))
        for d in (add2, add1, mul):
            graph.erase_node(d)
        n += 1
    if n:
        gm.recompile()
    return n


def fuse_gemm_epilogues(gm):
    """Elementwise neighbours of the native GEMMs move into their epilogues (edb_gemm_epi_bf16):

        add.Tensor(res, gemm.addmm(bias, a, b) | gemm.mm(a, b))   ==>  gemm.mm_add(a, b, res, bias)
        gelu_backward(gemm.mm(a, b), pre, approximate='tanh')     ==>  gemm.mm_gelu_bwd(a, b, pre)

    when the GEMM result has no other reader and the second operand is a bf16 matrix of the
    result's shape (2-D, or a view of one: the traced Linear works on [tokens, features]).  The
    reference runs these as separate ATen kernels (a14: op-by-op FX execution)."""
    from . import gemm
    graph = gm.graph
    n = 0
    bf16 = torch.bfloat16

    def val(nd):
        return nd.meta.get("val") if isinstance(nd, Node) else None

    def gemm_behind(nd):
        """nd == gemm.mm/addmm(...), or a shape-only view of it with a single reader chain."""
        chain = []
        while isinstance(nd, Node) and nd.op == "call_function" and \
                nd.target in (aten.view.default, aten._unsafe_view.default) and len(nd.users) == 1:
            chain.append(nd)
            nd = nd.args[0]
        if isinstance(nd, Node) and nd.op == "call_function" and nd.target in (gemm.mm, gemm.addmm) \
                and len(nd.users) == 1:
            return nd, chain
        return None, chain

    for node in list(graph.nodes):
        if node.op != "call_function":
            continue
        if node.target == aten.add.Tensor and len(node.args) == 2 and not node.kwargs:
            for gi, oi in ((1, 0), (0, 1)):
                g, chain = gemm_behind(node.args[gi])
                other = node.args[oi]
                gv, ov, nv = val(g), val(other), val(node)
                if g is None or not isinstance(other, Node) or gv is None or ov is None or nv is None:
                    continue
                if ov.dtype != bf16 or gv.dtype != bf16 or gv.shape[1] % 8 or \
                        tuple(ov.shape) != tuple(nv.shape) or ov.numel() != gv.numel():
                    continue
                if not ov.is_contiguous():
                    continue
                order = {nd: i for i, nd in enumerate(graph.nodes)}
                if order[other] > order[g]:
                    continue  # the residual must exist when the GEMM runs
                with graph.inserting_before(g):
                    res2d = other if ov.dim() == 2 else graph.call_function(
                        aten.view.default, args=(other, list(gv.shape)))
                    if g.target is gemm.addmm:
                        bias, a, b = g.args
                    else:
                        (a, b), bias = g.args, None
                    fused = graph.call_function(gemm.mm_add, args=(a, b, res2d, bias),
                                                kwargs={k: v for k, v in g.kwargs.items() if k == "_pf"})
                    fused.meta = dict(g.meta)
                    out = fused
                    if nv.dim() != 2:
                        out = graph.call_function(aten.view.default, args=(fused, list(nv.shape)))
                        out.meta = dict(node.meta)
                node.replace_all_uses_with(out)
                graph.erase_node(node)
                for c in chain:
                    graph.erase_node(c)
                graph.erase_node(g)
                n += 1
                break
        elif node.target == aten.gelu_backward.default and node.kwargs.get("approximate") == "tanh":
            g, chain = gemm_behind(node.args[0])
            pre = node.args[1]
            gv, pv, nv = val(g), val(pre), val(node)
            if g is None or g.target is not gemm.mm or gv is None or pv is None or nv is None:
                continue
            if pv.dtype != bf16 or gv.dtype != bf16 or gv.shape[1] % 8 or pv.numel() != gv.numel() \
                    or not pv.is_contiguous():
                continue
            order = {nd: i for i, nd in enumerate(graph.nodes)}
            if order[pre] > order[g]:
                continue
            with graph.inserting_before(g):
                pre2d = pre if pv.dim() == 2 else graph.call_function(
                    aten.view.default, args=(pre, list(gv.shape)))
                a, b = g.args
                fused = graph.call_function(gemm.mm_gelu_bwd, args=(a, b, pre2d),
                                            kwargs={k: v for k, v in g.kwargs.items() if k == "_pf"})
                fused.meta = dict(g.meta)
                out = fused
                if nv.dim() != 2:
                    out = graph.call_function(aten.view.default, args=(fused, list(nv.shape)))
                    out.meta = dict(node.meta)
            node.replace_all_uses_with(out)
            graph.erase_node(node)
            for c in chain:
                graph.erase_node(c)
            graph.erase_node(g)
            n += 1
    # gradient accumulation behind a LayerNorm backward: add(getitem(ln_bwd, 0), other) -> _add=other
    from . import norm
    order = {nd: i for i, nd in enumerate(graph.nodes)}
    for node in list(graph.nodes):
        if node.op != "call_function" or node.target != aten.add.Tensor or len(node.args) != 2 \
                or node.kwargs:
            continue
        for gi, oi in ((0, 1), (1, 0)):
            g, other = node.args[gi], node.args[oi]
            if not (isinstance(g, Node) and g.op == "call_function" and g.target is operator.getitem
                    and g.args[1] == 0 and len(g.users) == 1 and isinstance(other, Node)):
                continue
            ln = g.args[0]
            if not (isinstance(ln, Node) and ln.target is norm.native_layer_norm_backward
                    and "_add" not in ln.kwargs):
                continue
            lv, ov = val(g), val(other)
            if lv is None or ov is None or tuple(lv.shape) != tuple(ov.shape) or lv.dtype != ov.dtype \
                    or order[other] > order[ln]:
                continue
            ln.kwargs = dict(ln.kwargs, _add=other)
            node.replace_all_uses_with(g)
            graph.erase_node(node)
            n += 1
            break
    if n:
        graph.lint()
        gm.recompile()
    return n


def dispatch_compute(gm):
    """Route bf16 `aten.mm` / `aten.addmm` nodes to the tcgen05 GEMM (sharded-op kernel dispatch)."""
    import os
    from . import gemm, norm
    native_ln = os.environ.get("EDB_NATIVE_LN", "1") == "1"
    n = 0
    if os.environ.get("EDB_NATIVE_CE", "1") == "1":
        n += fuse_cross_entropy(gm)
    if os.environ.get("EDB_NATIVE_OPT", "1") == "1":
        n += fuse_optimizer_updates(gm)
    for node in gm.graph.nodes:
        if node.op != "call_function":
            continue
        if not native_ln:
            pass
        elif node.target == aten.native_layer_norm.default:
            node.target = norm.native_layer_norm
            n += 1
            continue
        elif node.target == aten.native_layer_norm_backward.default:
            node.target = norm.native_layer_norm_backward
            n += 1
            continue
        if native_ln and node.target == aten.sum.dim_IntList:
            node.target = norm.sum_dim_intlist
            n += 1
            continue
        val = node.meta.get("val")
        if not isinstance(val, torch.Tensor) or val.dtype != torch.bfloat16:
            continue
        if node.target == aten.mm.default:
            node.target = gemm.mm
            if "edb_pf" in node.meta:
                node.kwargs = {"_pf": node.meta["edb_pf"]}
            n += 1
        elif node.target == aten.addmm.default and not node.kwargs:
            node.target = gemm.addmm
            if "edb_pf" in node.meta:
                node.kwargs = {"_pf": node.meta["edb_pf"]}
            n += 1
    gm.recompile()
    if os.environ.get("EDB_FUSE_EPILOGUE", "1") == "1":
        n += fuse_gemm_epilogues(gm)
    return n


def prefetch_param_gathers(gm, io, rt, ranks, ops=_default_ops, my_index=None):
    """Epoch mode: every dim-0 all-gather of a parameter shard (zero3: compile_dp.py:136-150 puts
    one in front of each use) becomes a PREFETCH.

    Between the barrier behind the optimizer and the barrier in front of the next one, parameter
    shards never change, so a parameter is gathered ONCE per step into a persistent symmetric
    buffer and every use reads that buffer (`ops.gathered`, a view).  The copies ride on the bf16
    GEMMs that run earlier in the step: `edb_gemm_pf_bf16` gives a GEMM kernel a few extra CTAs
    that pull the peers' shards of an upcoming layer over NVLink while the other CTAs compute, so
    the all-gather of layer i+1 overlaps the tensor-core work of layer i and neither waits
    (the reference issues a blocking NCCL all-gather in front of every use, sharding.py:105-119).
    Packing is earliest-first under a per-GEMM byte budget (its FLOPs at ~900 TFLOP/s times
    EDB_PF_GBPS, default 300 GB/s of NVLink pull); whatever is needed before the first GEMM
    (embeddings, first layer) goes into one stand-alone `ops.ag_prefetch` at the top of the graph.

    Layout: with `my_index` given, a rank's shard LIVES in its own slot of the gathered buffer
    (shard home = full + my_index * shard_bytes; the optimizer updates it there), so the own range
    is never copied and only the n-1 remote ranges travel.

    Returns ({placeholder name: SymmBuffer home of the shard}, number of parameters handled)."""
    import os
    from collections import deque
    graph = gm.graph
    n = len(ranks)
    order = {nd: i for i, nd in enumerate(graph.nodes)}
    uses = {}
    dim1_ok = os.environ.get("EDB_AG_PREFETCH_DIM1", "1") == "1"
    for ag_s in [x for x in graph.nodes if x.op == "call_function" and x.target is ops.all_gather_start]:
        # all_gather(t(W), 1) == t(all_gather(W, 0)): auto-SPMD plans gather the transposed weight
        # of a Linear right in front of its GEMM (and t(t(W)) in front of the data-gradient GEMM)
        ph, n_t = ag_s.args[0], 0
        while isinstance(ph, Node) and ph.op == "call_function" and ph.target == aten.t.default and \
                isinstance(ph.args[0], Node):
            ph, n_t = ph.args[0], n_t + 1
        transposed = bool(n_t % 2)
        if not (isinstance(ph, Node) and ph.op == "placeholder" and ph in io.param_ph):
            continue
        val = ph.meta.get("val")
        if not isinstance(val, torch.Tensor) or (val.numel() * val.element_size()) % 16 or val.numel() == 0:
            continue
        if n_t and val.dim() != 2:
            continue
        d = ag_s.args[1]
        if not isinstance(d, int):
            continue
        d = d + val.dim() if d < 0 else d
        wdim = 1 - d if transposed else d      # the gather dim in W's own coordinates
        if wdim == 1 and not (val.dim() == 2 and dim1_ok):
            continue   # weights the plan shards along dim 1: see the rewrite below
        if wdim not in (0, 1) or list(ag_s.args[2]) != list(ranks) \
                or ag_s.kwargs or len(ag_s.users) != 1 or not val.is_contiguous():
            continue
        ag_e = next(iter(ag_s.users))
        if ag_e.target is not ops.all_gather_end:
            continue
        uses.setdefault(ph, []).append((ag_s, ag_e, transposed, wdim))
    # one sharding dim per parameter (anything else is not a plain shard gather: leave it alone)
    uses = {ph: lst for ph, lst in uses.items() if len({u[3] for u in lst}) == 1}
    if not uses:
        return {}, 0
    rehomed, bufs = {}, {}
    for ph in uses:
        nbytes = _nbytes(ph.meta["val"])
        full = rt.alloc(nbytes * n, align=1024)
        if my_index is None:
            shard = rt.alloc(nbytes, align=1024)
        else:
            shard = full.sub(int(my_index) * nbytes, nbytes)
        rehomed[ph.name] = shard
        bufs[ph] = (shard, full, nbytes)
    gathered_nodes = {}
    for ph, lst in uses.items():
        shard, full, nbytes = bufs[ph]
        pv = ph.meta["val"]
        for ag_s, ag_e, transposed, wdim in lst:
            with graph.inserting_before(ag_s):
                g = graph.call_function(ops.gathered, args=(ph, list(ranks)),
                                        kwargs={"_buf": (shard.offset, full.offset)})
                res = g
                if wdim == 1:
                    # shards [R, C/n] of a weight sharded along dim 1: the buffer holds them one
                    # after the other ([n, R, C/n]); the dim-1 concatenation is one local strided
                    # copy instead of a collective in front of the use
                    r_, c_ = pv.shape
                    res = graph.call_function(aten.view.default, args=(g, [n, r_, c_]))
                    res = graph.call_function(aten.permute.default, args=(res, [1, 0, 2]))
                    res = graph.call_function(aten.reshape.default, args=(res, [r_, n * c_]))
                elif pv.dim() > 1:  # flat concat of dim-0 shards == the dim-0 all-gather, reshaped
                    res = graph.call_function(aten.view.default,
                                              args=(g, [n * pv.shape[0]] + list(pv.shape[1:])))
                if transposed:
                    res = graph.call_function(aten.t.default, args=(res,))
            res.meta = dict(ag_e.meta)
            ag_e.replace_all_uses_with(res)
            graph.erase_node(ag_e)
            graph.erase_node(ag_s)
            gathered_nodes.setdefault(ph, []).append(g)
    for nd in reversed(list(graph.nodes)):  # t(W) / t(t(W)) nodes whose only reader was the all-gather
        if nd.op == "call_function" and nd.target == aten.t.default and not nd.users:
            graph.erase_node(nd)
    # ---- schedule ----------------------------------------------------------------------------
    order = {nd: i for i, nd in enumerate(graph.nodes)}
    first_use = {ph: min(order[g] for g in gathered_nodes[ph]) for ph in uses}
    carriers = []
    for nd in graph.nodes:
        if nd.op != "call_function" or nd.target not in (aten.mm.default, aten.addmm.default):
            continue
        v = nd.meta.get("val")
        a = nd.args[-2].meta.get("val") if isinstance(nd.args[-2], Node) else None
        if isinstance(v, torch.Tensor) and v.dtype == torch.bfloat16 and v.dim() == 2 and \
                isinstance(a, torch.Tensor) and a.dim() == 2:
            carriers.append((nd, 2.0 * v.shape[0] * v.shape[1] * a.shape[1]))
    gbps = float(os.environ.get("EDB_PF_GBPS", "300"))
    BLK = 16384
    need = sorted(uses, key=lambda ph: first_use[ph])
    start_of_carriers = order[carriers[0][0]] if carriers else float("inf")
    initial = [ph for ph in need if first_use[ph] < start_of_carriers]
    queue = deque([ph, 0] for ph in need if ph not in initial)
    late = {}  # ph -> items that found no carrier in time (stand-alone prefetch at the use)
    deps = {ph: [] for ph in uses}

    def item(ph, done, take):
        shard, full, nbytes = bufs[ph]
        if my_index is None:
            return (shard.offset + done, full.offset + done, take, nbytes, 0)
        return (full.offset + done, full.offset + done, take, nbytes, nbytes)  # in place

    for nd, flops in carriers:
        budget = flops / 9e14 * gbps * 1e9 / max(1, n - 1) * 1.0  # bytes per member range
        items = []
        while queue and len(items) < 4:
            ph, done = queue[0]
            if order[nd] >= first_use[ph]:
                # too late for this carrier: the rest is gathered right in front of the use
                late.setdefault(ph, []).append(item(ph, done, bufs[ph][2] - done))
                queue.popleft()
                continue
            left = bufs[ph][2] - done
            take = left if left <= budget else max(BLK, int(budget) // BLK * BLK)
            take = min(take, left)
            items.append(item(ph, done, take))
            deps[ph].append(nd)
            budget -= take
            if take == left:
                queue.popleft()
            else:
                queue[0][1] = done + take
            if budget < BLK:
                break
        if items:
            nd.meta["edb_pf"] = {"group": list(ranks), "items": items}
    for ph, done in queue:
        late.setdefault(ph, []).append(item(ph, done, bufs[ph][2] - done))
    if initial:
        first_node = next(nd for nd in graph.nodes if nd.op != "placeholder")
        with graph.inserting_before(first_node):
            graph.call_function(ops.ag_prefetch, args=(initial[0], list(ranks)),
                                kwargs={"_items": [item(ph, 0, bufs[ph][2]) for ph in initial]})
    for ph, items in late.items():
        g0 = min(gathered_nodes[ph], key=lambda g: order[g])
        with graph.inserting_before(g0):
            graph.call_function(ops.ag_prefetch, args=(ph, list(ranks)), kwargs={"_items": items})
    for ph, lst in gathered_nodes.items():
        for g in lst:
            g.args = (ph, list(ranks)) + tuple(dict.fromkeys(d for d in deps[ph] if order[d] < order[g]))
    graph.lint()
    gm.recompile()
    return rehomed, len(uses)


def insert_epoch_barriers(gm, ranks, ops=_default_ops):
    """The two rendezvous of an epoch-protocol step (see edb.h, edb_epoch_barrier):
      * behind the LAST node that touches peer memory (all-gather prefetches read the peers'
        parameter shards, push GEMMs write the peers' receive slots) unless a barrier already sits
        behind it (the one in front of `rs_finish`): nobody may overwrite a shard that a slower
        peer is still reading, and the optimizer — traced after the whole backward pass — is the
        first to do so;
      * at the very end: the updated shards are final and the receive slots free, the next step
        may start."""
    graph = gm.graph
    order = {nd: i for i, nd in enumerate(graph.nodes)}
    peer_touch = tuple(getattr(ops, k) for k in ("ag_mm", "mm_push", "ag_prefetch") if hasattr(ops, k))
    fused_nodes = [nd for nd in graph.nodes if nd.op == "call_function"
                   and (nd.target in peer_touch or "edb_pf" in nd.meta)]
    if not fused_nodes:
        return 0
    n_new = 0
    last_fused = max(fused_nodes, key=lambda nd: order[nd])
    barriers = [nd for nd in graph.nodes if nd.op == "call_function"
                and nd.target is ops.epoch_barrier]
    if not any(order[b_] > order[last_fused] for b_ in barriers):
        anchor = last_fused
        while anchor.next.op == "call_function" and anchor.next.target is operator.getitem \
                and anchor.next.args[0] is last_fused:
            anchor = anchor.next
        with graph.inserting_after(anchor):
            graph.call_function(ops.epoch_barrier, args=(anchor, list(ranks)))
        n_new += 1
    return n_new + ensure_end_barrier(gm, ranks, ops)


def ensure_end_barrier(gm, ranks, ops=_default_ops):
    """One epoch barrier as the last node of the step (idempotent)."""
    graph = gm.graph
    out_node = next(nd for nd in graph.nodes if nd.op == "output")
    prev = out_node.prev
    if prev.op == "call_function" and prev.target is ops.epoch_barrier:
        return 0
    some = next((nd for nd in reversed(list(graph.nodes)) if nd.op == "call_function"
                 and isinstance(nd.meta.get("val"), torch.Tensor)), None)
    if some is None:
        some = next(nd for nd in graph.nodes if nd.op == "placeholder")
    with graph.inserting_before(out_node):
        graph.call_function(ops.epoch_barrier, args=(some, list(ranks)))
    gm.recompile()
    return 1


def fuse_collective_gemms(gm, io, rt, ranks, ops=_default_ops, my_index=None):
    """Peephole fusion of reshard edges into the adjacent GEMM (B200 runtime only):

      all_gather(param shard) -> view -> t -> mm/addmm        ==>  ops.ag_mm   (AG + GEMM, one kernel)
      mm -> flatten -> reduce_scatter(avg, dim 0)              ==>  ops.mm_push (GEMM pushes its rows
                                                                   to their owners) + ops.rs_finish

    Epoch protocol: no handshake inside the fused kernels; ONE group barrier in front of the
    optimizer (all gradient tiles have landed in their owners' slots, nobody still reads the old
    parameter shards) and ONE behind it (the new shards are final, the slots are free again).
    Returns ({placeholder name: SymmBuffer} for parameter shards that must live in the symmetric
    heap (peers read them directly), {"ag_mm", "ag_pf", "mm_rs": number of rewrites}); "mm_rs"
    counts the GEMM + reduce-scatter pairs turned into pushes."""
    import os
    graph = gm.graph
    n = len(ranks)
    if n <= 1:
        return {}, {"ag_mm": 0, "ag_pf": 0, "mm_rs": 0}
    order = {nd: i for i, nd in enumerate(graph.nodes)}
    rehomed = {}
    n_ag = n_rs = 0
    bf16 = torch.bfloat16
    n_pf = 0
    if os.environ.get("EDB_AG_PREFETCH", "1") == "1":
        # all parameter gathers as prefetches riding on earlier GEMMs (no AG left to fuse below)
        rehomed, n_pf = prefetch_param_gathers(gm, io, rt, ranks, ops, my_index=my_index)
        order = {nd: i for i, nd in enumerate(graph.nodes)}

    def val(nd):
        return nd.meta.get("val") if isinstance(nd, Node) else None

    # ---- all-gather + GEMM ---------------------------------------------------------------
    for ag_s in [x for x in graph.nodes if x.op == "call_function" and x.target is ops.all_gather_start]:
        ph = ag_s.args[0]
        if not (isinstance(ph, Node) and ph.op == "placeholder" and ph in io.param_ph):
            continue
        if ag_s.args[1] != 0 or len(ag_s.users) != 1:
            continue
        ag_e = next(iter(ag_s.users))
        if ag_e.target is not ops.all_gather_end or len(ag_e.users) != 1:
            continue
        v = next(iter(ag_e.users))
        if v.target != aten.view.default or len(v.args[1]) != 2 or len(v.users) != 1:
            continue
        n_out, k_in = (int(d) for d in v.args[1])
        t = next(iter(v.users))
        if t.target != aten.t.default or not t.users:
            continue
        first = min(t.users, key=lambda u: order[u])
        if first.target == aten.addmm.default and first.args[2] is t and not first.kwargs:
            bias, x = first.args[0], first.args[1]
        elif first.target == aten.mm.default and first.args[1] is t:
            bias, x = None, first.args[0]
        else:
            continue
        xv, pv = val(x), val(ph)
        if xv is None or pv is None or xv.dtype != bf16 or pv.dtype != bf16 or xv.dim() != 2:
            continue
        if n_out % n or n_out % 128 or (n_out // n) % 8 or k_in % 8 or xv.shape[1] != k_in:
            continue
        if bias is not None and (val(bias) is None or val(bias).dim() != 1 or n_out % 8):
            continue
        shard = rehomed.get(ph.name) or rt.alloc(n_out // n * k_in * 2, align=1024)
        full = rt.alloc(n_out * k_in * 2, align=1024)
        rehomed[ph.name] = shard
        with graph.inserting_before(first):
            fused = graph.call_function(ops.ag_mm, args=(x, ph, list(ranks), n_out, k_in, bias),
                                        kwargs={"_buf": (shard.offset, full.offset), "_epoch": 1})
            out = graph.call_function(operator.getitem, args=(fused, 0))
            wfull = graph.call_function(operator.getitem, args=(fused, 1))
            t_new = graph.call_function(aten.t.default, args=(wfull,))
        first.replace_all_uses_with(out)
        graph.erase_node(first)
        t.replace_all_uses_with(t_new)
        for dead in (t, v, ag_e, ag_s):
            graph.erase_node(dead)
        n_ag += 1

    # ---- GEMM + reduce-scatter -------------------------------------------------------------
    # the GEMM only pushes its tiles to the owners; one rs_finish node in front of the first
    # consumer reduces every weight gradient's slots in a single kernel
    pushed = []  # (token node, recv buffer, shard numel, rs_end node)
    for rs_s in [x for x in graph.nodes if x.op == "call_function" and x.target is ops.reduce_scatter_start]:
        f = rs_s.args[0]
        if rs_s.args[1] != "avg" or rs_s.args[2] != 0 or rs_s.kwargs:
            continue
        if not (isinstance(f, Node) and f.target == aten.flatten.using_ints and len(f.users) == 1):
            continue
        g = f.args[0]
        if not (isinstance(g, Node) and len(g.users) == 1):
            continue
        # the weight gradient of a Linear reaches the optimizer through a chain of aten.t nodes
        # (t(t(mm(dy^T, x))) in torch 2.11); an odd chain means (A.B)^T = B^T.A^T
        t_chain = []
        mm_node = g
        while mm_node.target == aten.t.default and isinstance(mm_node.args[0], Node) and \
                len(mm_node.args[0].users) == 1:
            t_chain.append(mm_node)
            mm_node = mm_node.args[0]
        transposed = t_chain[0] if len(t_chain) % 2 == 1 else None
        if mm_node.target != aten.mm.default:
            continue
        a0, b0 = mm_node.args
        av, bv = val(a0), val(b0)
        if av is None or bv is None or av.dtype != bf16 or bv.dtype != bf16:
            continue
        M, N = (bv.shape[1], av.shape[0]) if transposed is not None else (av.shape[0], bv.shape[1])
        if M % n or (M // n) % 128 or N % 8:
            continue
        if len(rs_s.users) != 1:
            continue
        rs_e = next(iter(rs_s.users))
        recv = rt.alloc(M * N * 2, align=1024)
        with graph.inserting_before(rs_s):
            if transposed is not None:
                a = graph.call_function(aten.t.default, args=(b0,))
                b = graph.call_function(aten.t.default, args=(a0,))
                for nd, src in ((a, bv), (b, av)):
                    nd.meta["val"] = src.t()
            else:
                a, b = a0, b0
            tok = graph.call_function(ops.mm_push, args=(a, b, list(ranks)),
                                      kwargs={"_buf": (recv.offset,)})
        pushed.append((tok, recv, M // n * N, rs_e))
        # rs_e stays until rs_finish replaces it below; its producers go now
        rs_e.args = (tok,) + tuple(rs_e.args[1:])
        for dead in [rs_s, f] + t_chain + [mm_node]:
            graph.erase_node(dead)
        n_rs += 1
    if pushed:
        order = {nd: i for i, nd in enumerate(graph.nodes)}

        def first_use_of(items):
            return min((u for *_, rs_e in items for u in rs_e.users), key=lambda u: order[u])

        # one rs_finish per run of pushes that all precede the run's first consumer (a single one
        # for a train step whose gradients are only read by the optimizer)
        groups, cur = [], []
        for it in pushed:
            if cur and order[it[0]] > order[first_use_of(cur)]:
                groups.append(cur)
                cur = []
            cur.append(it)
        groups.append(cur)
        for items in groups:
            with graph.inserting_before(first_use_of(items)):
                fin_kw = {"_bufs": [(it[1].offset,) for it in items],
                          "_numels": [it[2] for it in items], "_scale": 1.0 / n}
                toks = [it[0] for it in items]
                # every member's tiles must have landed before anybody reduces its slots
                toks[0] = graph.call_function(ops.epoch_barrier, args=(toks[0], list(ranks)))
                fin = graph.call_function(ops.rs_finish, args=(toks, list(ranks)), kwargs=fin_kw)
                for i, (tok, recv, numel, rs_e) in enumerate(items):
                    gi = graph.call_function(operator.getitem, args=(fin, i))
                    gi.meta = dict(rs_e.meta)
                    rs_e.replace_all_uses_with(gi)
                    graph.erase_node(rs_e)

    # peers read parameter shards in place: keep the optimizer from overwriting them too early
    insert_epoch_barriers(gm, ranks, ops)
    graph.lint()
    gm.recompile()
    return rehomed, {"ag_mm": n_ag, "ag_pf": n_pf, "mm_rs": n_rs}


def verify_epoch_protocol(gm, ops, n):
    """Static race check of a lowered graph against the contract of the epoch protocol (edb.h,
    DESIGN.md §3.1) — the B200-native counterpart of the reference's debug-time `op_mem_checker`
    (an interval-tree ownership check per node, compile_auto.py:269-351), done once at compile time
    because here the hazards are decided by graph structure, not by run-time addresses:

      1. symmetric ranges that peers write without a handshake (gathered parameter buffers, receive
         slots of push GEMMs, static buffers of push collectives) are pairwise disjoint and each is
         written by exactly one node per step;
      2. every byte of every gathered parameter is prefetched exactly once, by nodes that precede its
         first use; no prefetch item points outside a gathered buffer;
      3. a group barrier separates the last node that reads peers' parameter shards from the first
         in-place update of such a parameter; every `rs_finish` has a barrier between its
         last push and itself;
      4. the step ends with a barrier.

    Returns {"ok", "problems": [...], "ranges", "items", "barriers"}; never raises."""
    problems = []
    nodes = list(gm.graph.nodes)
    order = {nd: i for i, nd in enumerate(nodes)}

    def nbytes(nd):
        v = nd.meta.get("val") if isinstance(nd, Node) else None
        return v.numel() * v.element_size() if isinstance(v, torch.Tensor) else None

    has = lambda k: getattr(ops, k, None)
    ranges = []      # (lo, hi, what)
    gathered = {}    # ph -> (full_off, shard_bytes, first_use_pos)
    items = []       # (pos, src, dst, take, dstride, sstride, node name)
    pushes, finishes, barriers = [], [], []
    for nd in nodes:
        if nd.op != "call_function":
            continue
        t = nd.target
        pf = nd.kwargs.get("_pf") or nd.meta.get("edb_pf")
        if pf:
            items += [(order[nd],) + tuple(it) + (nd.name,) for it in pf["items"]]
        if has("ag_prefetch") and t is ops.ag_prefetch:
            items += [(order[nd],) + tuple(it) + (nd.name,) for it in nd.kwargs.get("_items", [])]
        elif has("gathered") and t is ops.gathered:
            ph = nd.args[0]
            nb = nbytes(ph)
            if nb is None:
                problems.append(f"{nd.name}: shard size unknown")
                continue
            shard_off, full_off = nd.kwargs["_buf"]
            prev = gathered.get(ph)
            if prev is None:
                gathered[ph] = (full_off, nb, order[nd])
                ranges.append((full_off, full_off + n * nb, f"gathered({ph.name})"))
                if not (full_off <= shard_off and shard_off + nb <= full_off + n * nb):
                    ranges.append((shard_off, shard_off + nb, f"shard({ph.name})"))
            elif prev[0] != full_off:
                problems.append(f"{nd.name}: parameter {ph.name} has two gathered buffers")
        elif has("mm_push") and t is ops.mm_push:
            a, b = nd.args[0].meta.get("val"), nd.args[1].meta.get("val")
            pushes.append(nd)
            if a is not None and b is not None:
                lo = nd.kwargs["_buf"][0]
                ranges.append((lo, lo + a.shape[0] * b.shape[1] * 2, f"recv({nd.name})"))
        elif has("rs_finish") and t is ops.rs_finish:
            finishes.append(nd)
        elif has("epoch_barrier") and t is ops.epoch_barrier:
            barriers.append(order[nd])
        elif t in ops.COMM_FUNCS and nd.kwargs.get("_push"):
            buf = nd.kwargs.get("_buf")
            if not buf:
                problems.append(f"{nd.name}: push collective without static buffers")
                continue
            ranges.append((buf[0], buf[0] + buf[1], f"{nd.name}[0]"))
            xb = nbytes(nd.args[0])
            for k, off in enumerate(buf[2:]):
                ranges.append((off, off + (xb or 1), f"{nd.name}[{k + 1}]"))
    # 1. disjoint ranges
    ranges.sort()
    for (a0, a1, wa), (b0, b1, wb) in zip(ranges, ranges[1:]):
        if b0 < a1:
            problems.append(f"symmetric ranges overlap: {wa} [{a0},{a1}) and {wb} [{b0},{b1})")
    # 2. prefetch coverage
    by_buf = sorted((full, nb, ph) for ph, (full, nb, _) in gathered.items())
    cover = {ph: [] for ph in gathered}
    for pos, src, dst, take, dstride, sstride, name in items:
        owner = next((ph for full, nb, ph in by_buf if full <= dst and dst + take <= full + nb), None)
        if owner is None:
            problems.append(f"{name}: prefetch item dst={dst} (+{take}) is outside every gathered buffer")
            continue
        full, nb, first = gathered[owner]
        if dstride != nb:
            problems.append(f"{name}: item for {owner.name} has member stride {dstride} != shard {nb}")
        if pos >= first:
            problems.append(f"{name}: prefetch of {owner.name} is issued after its first use")
        cover[owner].append((dst - full, dst - full + take))
    for ph, segs in cover.items():
        nb = gathered[ph][1]
        segs.sort()
        at = 0
        for lo, hi in segs:
            if lo != at:
                problems.append(f"{ph.name}: prefetched ranges {'overlap' if lo < at else 'leave a gap'} "
                                f"at byte {min(lo, at)}")
                break
            at = hi
        else:
            if at != nb:
                problems.append(f"{ph.name}: only {at} of {nb} shard bytes are prefetched")
    # 3. barriers around the optimizer
    if gathered:
        peer_read = set(gathered)

        def writes_param(nd):
            if nd.op != "call_function":
                return False
            name = str(getattr(nd.target, "_schema", None) and nd.target._schema.name or
                       getattr(nd.target, "__name__", ""))
            if nd.target == aten.copy_.default:
                return nd.args[0] in peer_read
            if name.startswith("aten::_foreach_") and name.endswith("_") or name == "sgd_momentum_":
                first = nd.args[0] if nd.args else []
                return isinstance(first, (list, tuple)) and any(x in peer_read for x in first)
            return False

        upd = [order[nd] for nd in nodes if writes_param(nd)]
        last_read = max([pos for pos, *_ in items], default=-1)
        if upd and not any(last_read < b < min(upd) for b in barriers):
            problems.append("no epoch barrier between the last prefetch of peers' parameter shards "
                            f"(node {last_read}) and the first in-place parameter update (node {min(upd)})")
    for fin in finishes:
        toks = [t_ for t_ in fin.args[0] if isinstance(t_, Node)]
        srcs = []
        for t_ in toks:
            while t_.op == "call_function" and has("epoch_barrier") and t_.target is ops.epoch_barrier:
                t_ = t_.args[0]
            srcs.append(t_)
        last_push = max((order[t_] for t_ in srcs), default=-1)
        if not any(last_push < b < order[fin] for b in barriers):
            problems.append(f"{fin.name}: no epoch barrier between its last push and the reduction")
    unfinished = [p_.name for p_ in pushes if not any(
        u.target is ops.rs_finish or (has("epoch_barrier") and u.target is ops.epoch_barrier)
        for u in p_.users)]
    if unfinished:
        problems.append(f"push GEMMs without rs_finish: {unfinished[:4]}")
    # 4. end of step
    if ranges or items:
        out = next((nd for nd in nodes if nd.op == "output"), None)
        if out is None or not (out.prev.op == "call_function" and has("epoch_barrier")
                               and out.prev.target is ops.epoch_barrier):
            problems.append("the step does not end with an epoch barrier")
    return {"ok": not problems, "problems": problems, "ranges": len(ranges), "items": len(items),
            "barriers": len(barriers)}


def reinplace_optimizer_updates(gm):
    """Undo the functionalisation of optimizer updates where it is safe.

    Tracing rewrites `_foreach_op_(xs, ...)` as `ys = _foreach_op(xs, ...); xs[i].copy_(ys[i])`
    (compile.py DECOMPOSITION_TABLE; reference: decomp_utils.py:60-131) so that the graph is
    functional while plans are made.  At run time every such pair costs a full extra pass over
    params/momenta (2 x 292 D2D copies per GPT-2-medium step).  When each output of the functional
    op is only used to overwrite the very tensor it was computed from, the pair is replaced by the
    in-place ATen op and the copies disappear."""
    graph = gm.graph
    n_fixed = 0
    order = {n: i for i, n in enumerate(graph.nodes)}
    for node in list(graph.nodes):
        if node.op != "call_function" or not hasattr(node.target, "_schema"):
            continue
        name = node.target._schema.name  # e.g. aten::_foreach_mul
        if not name.startswith("aten::_foreach_") or name.endswith("_"):
            continue
        inplace_packet = getattr(aten, name.split("::")[1] + "_", None)
        overload = node.target._overloadname
        if inplace_packet is None or not hasattr(inplace_packet, overload):
            continue
        self_list = node.args[0]
        if not isinstance(self_list, (list, tuple)) or not all(isinstance(x, Node) for x in self_list):
            continue
        getitems = {}
        ok = True
        for u in node.users:
            if u.target != operator.getitem or u.args[1] in getitems:
                ok = False
                break
            getitems[u.args[1]] = u
        if not ok or len(getitems) != len(self_list):
            continue
        copies = {}
        for i, gi in getitems.items():
            users = list(gi.users)
            if len(users) != 1 or users[0].target != aten.copy_.default or \
                    users[0].args[0] is not self_list[i] or users[0].args[1] is not gi:
                ok = False
                break
            copies[i] = users[0]
            # nobody else may read the old value of self_list[i] after the op
            for other in self_list[i].users:
                if other is node or other is users[0] or other.op == "output":
                    continue
                if order[other] > order[node]:
                    ok = False
                    break
            if not ok:
                break
        if not ok or len(set(self_list)) != len(self_list):
            continue
        node.target = getattr(inplace_packet, overload)
        for i, cp in copies.items():
            cp.replace_all_uses_with(self_list[i])
            graph.erase_node(cp)
            graph.erase_node(getitems[i])
        n_fixed += 1
    n_fixed += _reinplace_fused_optimizers(gm, order)
    if n_fixed:
        graph.lint()
        gm.recompile()
    return n_fixed


def _reinplace_fused_optimizers(gm, order):
    """Same for the fused optimizers (`_fused_adam`, `_fused_adamw`, `_fused_sgd`: what
    torch.optim(..., fused=True) calls and what the reference's DP rewrites are written around,
    compile_dp.py:55-198).  Tracing turned `_fused_x_(params, grads, states...)` into the functional
    op plus one copy_ per written tensor (compile.py `_fused_multi_output`); when every output is
    only used for that copy the in-place op comes back and 3 copies per parameter disappear."""
    graph = gm.graph
    table = {}
    for name, n_lists, skip in (("_fused_adam", 5, (1,)), ("_fused_adamw", 5, (1,)),
                                ("_fused_sgd", 3, (1,))):
        if hasattr(aten, name) and hasattr(aten, name + "_"):
            table[getattr(aten, name).default] = (getattr(aten, name + "_").default, n_lists, skip)
    n_fixed = 0
    for node in list(graph.nodes):
        if node.op != "call_function" or node.target not in table:
            continue
        inplace, n_lists, skip = table[node.target]
        lists = list(node.args[:n_lists])
        if any(not isinstance(lst, (list, tuple)) for lst in lists):
            continue
        outer = {}
        ok = all(u.target == operator.getitem for u in node.users)
        for u in node.users:
            if ok:
                outer[u.args[1]] = u
        dead, redirect = [], []
        for k, lst in enumerate(lists):
            if not ok:
                break
            if k in skip or not lst:
                # an output list nobody copies back must be unused altogether
                if k in outer and outer[k].users:
                    ok = False
                continue
            if k not in outer:
                ok = False
                break
            inner = {}
            for u in outer[k].users:
                if u.target != operator.getitem or u.args[1] in inner:
                    ok = False
                    break
                inner[u.args[1]] = u
            if not ok or len(inner) != len(lst) or len(set(lst)) != len(lst):
                ok = False
                break
            for i, orig in enumerate(lst):
                users = list(inner[i].users)
                if not isinstance(orig, Node) or len(users) != 1 or \
                        users[0].target != aten.copy_.default or users[0].args[0] is not orig or \
                        users[0].args[1] is not inner[i]:
                    ok = False
                    break
                for other in orig.users:
                    if other is node or other is users[0] or other.op == "output":
                        continue
                    if order[other] > order[node]:
                        ok = False
                        break
                if not ok:
                    break
                redirect.append((users[0], orig))
                dead.append(inner[i])
            dead.append(outer[k])
        if not ok:
            continue
        node.target = inplace
        for cp, orig in redirect:
            cp.replace_all_uses_with(orig)
            graph.erase_node(cp)
        for d in dead:
            graph.erase_node(d)
        for k, u in list(outer.items()):
            if not u.users and u not in dead:
                graph.erase_node(u)
        n_fixed += 1
    return n_fixed


def count_nodes(gm, ops=_default_ops):
    hist = {}
    for node in gm.graph.nodes:
        if node.op == "call_function":
            name = getattr(node.target, "__name__", str(node.target))
            fused = getattr(ops, "FUSED_FUNCS", [])
            if node.target in ops.CUSTOM_FUNCS or node.target in fused or \
                    "gemm" in getattr(node.target, "__module__", ""):
                hist[name] = hist.get(name, 0) + 1
    return hist
