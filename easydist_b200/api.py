"""`easydist_compile` for the B200 backend + registration behind the reference's own decorator.

Two ways in, both keeping the reference's user-facing contract (easydist/torch/api.py:227-256):

  * standalone:  `from easydist_b200 import easydist_compile` — same decorator signature
    (`parallel_mode`, `tracing_mode`, `cuda_graph`, `compile_only`, ...); modes
    "ddp" / "zero2" / "zero3" (compile_dp.py) need no solver and run anywhere; mode "auto" needs a
    plan: from the reference's solver when it is importable, or a recorded plan (`plan=` kwarg).
  * behind the reference:  `register()` plugs the backend into the reference through its
    `register_parallel_method` hook (api.py:39-50, dispatch :136-140) as modes "b200_ddp",
    "b200_zero2", "b200_zero3", and rebinds `compile_auto.sharding_transform` (the name imported
    at compile_auto.py:46-49, called at :569) so `parallel_mode="auto"` lowers through this
    backend while annotation + ILP stay the reference's.

CUDA graphs: as in the reference (`cuda_graph=True` default, api.py:180-224) the whole step is
captured after one eager warm-up and replayed with static input buffers; every kernel on the path
(libedb collectives included) is capture-safe.
"""
import logging
from functools import update_wrapper
from typing import Any

import os

import torch
import torch.utils._pytree as pytree

from . import lowering
from . import reshard as _default_ops
from .compile import EDCompiledFunc, GraphIO, trace_train_step
from .device_mesh import get_device_mesh

logger = logging.getLogger(__name__)

DP_MODES = ("ddp", "zero2", "zero3")
PARALLEL_EXTENTION = {}


def register_parallel_method(parallel_mode: str, compiler_func=None):
    """Same plugin hook as the reference (api.py:39-50)."""

    def wrapper(fn):
        PARALLEL_EXTENTION[parallel_mode] = fn
        return fn

    return wrapper if compiler_func is None else wrapper(compiler_func)


def _dp_group(mesh):
    """Ranks of the data-parallel group: the mesh dim named 'dp' (compile_dp.py:57, 312-315) or,
    for a 1-D mesh, its only dim."""
    if "dp" in mesh.dim_names:
        d = mesh.dim_names.index("dp")
    else:
        assert mesh.ndim == 1, "data-parallel modes need a mesh dim named 'dp'"
        d = 0
    return mesh.ranks_along(d), mesh.get_coordinate()[d]


def _flat_inputs(params, buffers, named_states, args, kwargs):
    return pytree.tree_flatten((params, buffers, named_states, args, kwargs))[0]


def _single_group(gm, ops, ranks):
    """True when every collective of the graph runs on the group `ranks`."""
    want = list(ranks)
    for nd in gm.graph.nodes:
        if nd.op == "call_function" and nd.target in ops.COMM_FUNCS:
            grp = nd.args[5] if nd.target is ops.all_to_all_start else \
                (nd.args[3] if nd.target is ops.reduce_scatter_start else nd.args[2])
            if list(grp) != want:
                return False
    return True


class _ParamIO:
    """The slice of GraphIO the prefetch pass needs (auto path: placeholders by position)."""

    def __init__(self, param_ph, param_names):
        self.param_ph, self.param_names = list(param_ph), list(param_names)


def _finish(gm, params, buffers, named_states, args, kwargs, ops, native, io=None, ranks=None,
            fuse=True, fuse_rt=None, my_index=None, auto_io=None):
    """Local metas -> (fusions) -> static symmetric buffers -> GEMM dispatch."""
    flat = _flat_inputs(params, buffers, named_states, args, kwargs)
    lowering.propagate_local_meta(gm, flat)
    info = {}
    if io is None and os.environ.get("EDB_LOCALIZE_OPT", "1" if native else "0") == "1":
        # auto-SPMD plans: optimizer foreach ops on shards instead of on gathered tensors (changes
        # the communication structure the reference's lowering produces, so the reference-structure
        # tests run without it; the product path has it on)
        info["localized_foreach"] = lowering.localize_foreach(gm, ops, my_rank=get_device_mesh().rank)
        lowering.propagate_local_meta(gm, flat)
    # auto-SPMD plan on a 1-D mesh: gathers of parameter shards become prefetches (below)
    auto_pf = (native or fuse_rt is not None) and fuse and auto_io is not None and ranks is not None \
        and len(ranks) > 1 and os.environ.get("EDB_AG_PREFETCH", "1") == "1"
    bucket = os.environ.get("EDB_BUCKET_COMM", "0") == "1"
    if bucket and not auto_pf:
        # opt-in: changes the communication structure the reference's lowering would produce
        info["bucketed"] = lowering.bucket_small_comm(gm, ops)
        lowering.propagate_local_meta(gm, flat)
    if (native or fuse_rt is not None) and fuse and io is not None and ranks is not None \
            and len(ranks) > 1:
        if fuse_rt is None:
            from .runtime import get_runtime
            fuse_rt = get_runtime()
        rt = fuse_rt
        rehomed, nf = lowering.fuse_collective_gemms(gm, io, rt, ranks, ops, my_index=my_index)
        info["fused"] = nf
        # parameter shards read by peers must live at their symmetric offsets
        name_of = {ph.name: io.param_names[i] for i, ph in enumerate(io.param_ph)}
        for ph_name, buf in rehomed.items():
            pname = name_of[ph_name]
            t = params[pname]
            home = buf.tensor(t.dtype, t.shape)
            home.copy_(t)
            params[pname] = home
        lowering.propagate_local_meta(gm, _flat_inputs(params, buffers, named_states, args,
                                                       kwargs))
    elif auto_pf:
        # gathers of parameter shards become prefetches that ride on the step's GEMMs, one gather
        # per parameter per step (epoch protocol)
        if fuse_rt is None:
            from .runtime import get_runtime
            fuse_rt = get_runtime()
        rt = fuse_rt
        rehomed, n_pf = lowering.prefetch_param_gathers(gm, auto_io, rt, ranks, ops, my_index=my_index)
        if rehomed:
            lowering.insert_epoch_barriers(gm, ranks, ops)
            name_of = dict(zip([ph.name for ph in auto_io.param_ph], auto_io.param_names))
            for ph_name, buf in rehomed.items():
                t = params[name_of[ph_name]]
                home = buf.tensor(t.dtype, t.shape)
                home.copy_(t)
                params[name_of[ph_name]] = home
            lowering.propagate_local_meta(gm, _flat_inputs(params, buffers, named_states, args, kwargs))
        info["fused"] = {"ag_mm": 0, "ag_pf": n_pf, "mm_rs": 0}
        if bucket:
            # ... and only what is still a collective after that is bucketed (a prefetched parameter
            # needs no collective at all: bucketing its gather first would keep one)
            info["bucketed"] = lowering.bucket_small_comm(gm, ops)
            lowering.propagate_local_meta(gm, _flat_inputs(params, buffers, named_states, args, kwargs))
    info["comm_nodes"] = lowering.count_nodes(gm, ops)
    info["reinplaced_updates"] = lowering.reinplace_optimizer_updates(gm)
    if native:
        from .runtime import get_runtime
        # push-protocol collectives need ONE group for the end-of-step barrier: a 1-D mesh / the dp
        # group.  (N-D meshes keep the flag protocol: a barrier per mesh dim would not cover the
        # buffers of the other dims' collectives.)
        push = ranks is not None and len(ranks) > 1 \
            and os.environ.get("EDB_PUSH_COLL", "1") == "1" and hasattr(ops, "epoch_barrier") \
            and _single_group(gm, ops, ranks)
        info["symm_bytes"] = lowering.assign_static_buffers(gm, get_runtime(), ops, push=push)
        if push and any(nd.kwargs.get("_push") for nd in gm.graph.nodes if nd.op == "call_function"):
            lowering.ensure_end_barrier(gm, ranks, ops)
            info["push_collectives"] = True
        info["gemm_nodes"] = lowering.dispatch_compute(gm)
        if ranks is not None and len(ranks) > 1 and (push or info.get("fused")):
            # static race check of the lowered graph against the epoch-protocol contract (diagnostic:
            # problems are logged and reported in `info`; EDB_VERIFY_STRICT=1 makes them fatal)
            try:
                rep = lowering.verify_epoch_protocol(gm, ops, len(ranks))
            except Exception as e:  # noqa: BLE001 — the checker must never break a compilation
                rep = {"ok": None, "problems": [f"checker failed: {e!r}"]}
            info["epoch_check"] = {"ok": rep["ok"], "problems": rep["problems"][:5],
                                   "ranges": rep.get("ranges"), "items": rep.get("items")}
            if rep["problems"]:
                logger.error("epoch-protocol check: %s", rep["problems"][:5])
                if os.environ.get("EDB_VERIFY_STRICT", "0") == "1":
                    raise RuntimeError(f"epoch-protocol check failed: {rep['problems'][:5]}")
    gm.graph.lint()
    gm.recompile()
    return info


def _compile_dp(func, parallel_mode, tracing_mode, args, kwargs, *, ops=_default_ops,
                native=True, fuse=True, bucket_numel=None, fuse_rt=None):
    """ddp / zero2 / zero3 (reference: _compile_dp, compile_dp.py:201-381)."""
    mode = parallel_mode.replace("b200_", "")
    assert mode in DP_MODES, parallel_mode
    ranks, my_index = _dp_group(get_device_mesh())
    n = len(ranks)
    if bucket_numel is None:
        bucket_numel = 65536 if native else 0

    def trace_and_rewrite(a, kw, warm_up=True):
        params, buffers, named_states, gm, module, opt = trace_train_step(func, a, kw, tracing_mode,
                                                                          warm_up=warm_up)
        io = GraphIO(gm, params, buffers, named_states)
        shard_info = {}
        if n > 1:
            if mode == "ddp":
                lowering.transform_ddp(gm, io, ranks, ops, bucket_numel=bucket_numel)
            else:
                _, shard_info = lowering.transform_fsdp(gm, io, ranks, my_index,
                                                        shard_param=(mode == "zero3"), ops=ops,
                                                        bucket_numel=bucket_numel)
        return params, buffers, named_states, gm, io, shard_info

    params, buffers, named_states, gm, io, shard_info = trace_and_rewrite(args, kwargs)
    # pre-shard parameters (zero3) and optimizer states (zero2/zero3): flat 1/n shards
    # (compile_dp.py:330-343)
    with torch.no_grad():
        params = {k: v.detach() for k, v in params.items()}
        if shard_info:
            ph_names = {ph.name: i for i, ph in enumerate(io.param_ph)}
            for ph_name, idx in ph_names.items():
                if ph_name in shard_info:
                    name = io.param_names[idx]
                    params[name] = ops.scatter_wrapper(params[name].flatten(), n, 0, my_index)
            flat_states, spec = pytree.tree_flatten(named_states)
            for i, ph in enumerate(io.state_ph):
                if ph.name in shard_info and isinstance(flat_states[i], torch.Tensor):
                    flat_states[i] = ops.scatter_wrapper(flat_states[i].detach().flatten(), n, 0,
                                                         my_index)
            named_states = pytree.tree_unflatten(flat_states, spec)
    info = _finish(gm, params, buffers, named_states, args, kwargs, ops, native, io=io,
                   ranks=ranks, fuse=fuse, fuse_rt=fuse_rt, my_index=my_index)
    info.update(mode=mode, dp_size=n)
    if native and n > 1:
        # nobody enters the first step (peer waits have a fatal timeout) before everybody has
        # finished compiling and re-homing its parameter shards into the symmetric heap
        from .runtime import get_runtime
        get_runtime().host_barrier()

    def mono_compiler(compiled, a, kw):
        """Same rewrite for another input shape, lowered against the live (sharded) state.  The
        collective/GEMM fusion is left out: it re-homes parameter shards, and the first graph's
        kernels already address the current homes."""
        _, _, _, gm2, io2, _ = trace_and_rewrite(a, kw, warm_up=False)
        p, b, st = compiled.get_state()
        _finish(gm2, p, b, st, a, kw, ops, native, io=io2, ranks=ranks, fuse=False)
        return gm2

    return EDCompiledFunc(gm, params, buffers, named_states, info=info, mono_compiler=mono_compiler)


def _lower_auto(gm, plan, state_io_map, params, buffers, named_states, args, kwargs, *, ops, native,
                planner, mesh, fuse_rt=None):
    """Shared tail of the auto path: lower with the plan, shard state and inputs locally, finish."""
    n_p, n_b = len(params), len(buffers)
    flat_states, spec = pytree.tree_flatten(named_states)
    placeholders = [n for n in gm.graph.nodes if n.op == "placeholder"]
    param_ph = placeholders[:n_p]
    buffer_ph = placeholders[n_p:n_p + n_b]
    state_ph = placeholders[n_p + n_b:n_p + n_b + len(flat_states)]
    input_phs = placeholders[n_p + n_b + len(flat_states):]
    plan = lowering._normalise_plan(plan)
    lowering.sharding_transform(gm, plan, state_io_map, ops=ops, mesh=mesh, planner=planner)
    env = gm._edb_shard_env

    def shard_local(t, ph):
        strat = env.get(ph.name)
        if not isinstance(t, torch.Tensor) or strat is None:
            return t
        coord = mesh.get_coordinate()
        for mdim, s in enumerate(strat):
            if s.is_shard():
                t = ops.scatter_wrapper(t, mesh.size(mdim), s.dim, coord[mdim])
        return t

    with torch.no_grad():
        params = {k: shard_local(v.detach(), ph) for (k, v), ph in zip(params.items(), param_ph)}
        buffers = {k: shard_local(v.detach(), ph) for (k, v), ph in zip(buffers.items(),
                                                                       buffer_ph)}
        flat_states = [shard_local(s.detach() if isinstance(s, torch.Tensor) else s, ph)
                       for s, ph in zip(flat_states, state_ph)]
        named_states = pytree.tree_unflatten(flat_states, spec)

    def input_transform(a, kw):
        flat, spec_in = pytree.tree_flatten((a, kw))
        flat = [shard_local(x.detach() if isinstance(x, torch.Tensor) else x, ph)
                for x, ph in zip(flat, input_phs)]
        return pytree.tree_unflatten(flat, spec_in)

    largs, lkwargs = input_transform(args, kwargs)
    auto_io, ranks1d, my_index = None, None, None
    if mesh.ndim == 1:
        auto_io = _ParamIO(param_ph, list(params.keys()))
        ranks1d, my_index = mesh.ranks_along(0), mesh.get_coordinate()[0]
    info = _finish(gm, params, buffers, named_states, largs, lkwargs, ops, native, auto_io=auto_io,
                   ranks=ranks1d, my_index=my_index, fuse_rt=fuse_rt)
    info.update(mode="auto", mesh=mesh.shape)
    if native:
        from .runtime import get_runtime, is_initialized
        if is_initialized():
            get_runtime().host_barrier()
    return EDCompiledFunc(gm, params, buffers, named_states, input_transform=input_transform,
                          info=info)


def _compile_auto(func, tracing_mode, args, kwargs, *, plan=None, ops=_default_ops, native=True,
                  planner="GREEDY", bundle=None):
    """Auto-SPMD with a given plan: {node_name: {'strategy': NodeSPMDStrategy}} in the vocabulary
    of easydist_b200.metair (or the reference's own objects), keyed by the node names of the
    traced graph.  The plan is what the reference's AutoFlow solver emits
    (compile_auto.py:93-186); producing it stays the reference's job.  `bundle` = JSON text from
    graph_io.dump_bundle (graph + plan recorded where the reference runs)."""
    mesh = get_device_mesh("spmd")
    if bundle is not None:
        return compile_from_bundle(bundle, args, kwargs, ops=ops, native=native, planner=planner)
    if plan is None:
        raise NotImplementedError(
            "parallel_mode='auto' needs a sharding plan: use easydist_b200.api.register() to run "
            "behind the reference's solver, or pass plan=<plan> / bundle=<recorded graph+plan>")
    params, buffers, named_states, gm, module, opt = trace_train_step(func, args, kwargs,
                                                                      tracing_mode)
    io = GraphIO(gm, params, buffers, named_states)
    return _lower_auto(gm, plan, io.state_io_map(), params, buffers, named_states, args, kwargs,
                       ops=ops, native=native, planner=planner, mesh=mesh)


def compile_from_bundle(bundle_text, args, kwargs, *, ops=_default_ops, native=True,
                        planner="GREEDY", fuse_rt=None):
    """Lower and run a graph + plan recorded by graph_io.dump_bundle (e.g. solved by the
    reference on another machine).  `args` must contain the nn.Module and Optimizer the graph was
    traced with (their parameters/optimizer state provide the initial values)."""
    from . import graph_io
    from .compile import find_module_and_optimizer, warm_up_optimizer
    mesh = get_device_mesh("spmd")
    module, opt = find_module_and_optimizer(args, kwargs)
    device = next(module.parameters()).device
    gm, plan, state_io, _ = graph_io.load_bundle(bundle_text, device=device.type)
    params = dict(module.named_parameters())
    buffers = dict(module.named_buffers())
    named_states = warm_up_optimizer(module, opt)
    flat = [x.detach() if isinstance(x, torch.Tensor) else None
            for x in _flat_inputs(params, buffers, named_states, args, kwargs)]
    lowering.propagate_local_meta(gm, flat)  # global metas (nothing is sharded yet)
    class _Named:  # hashable stand-in for the MetaNode/MetaVar keys of the reference's map
        def __init__(self, name):
            self.name = name

    io_map = {_Named(a): _Named(b) for a, b in state_io}
    return _lower_auto(gm, plan, io_map, params, buffers, named_states, args, kwargs, ops=ops,
                       native=native, planner=planner, mesh=mesh, fuse_rt=fuse_rt)


LAST_AUTO_SOURCE = [None]  # "solved" | "cache": where the last b200_auto compilation got its plan


def _plan_cache_key(args, kwargs, mesh):
    """Stable across processes (unlike input_signature, which names modules by id): tensor shapes
    and dtypes, the printed architecture of every module, class + hyper-parameters of every
    optimizer, scalars, and the mesh shape."""
    import hashlib
    leaves, spec = pytree.tree_flatten((args, kwargs))
    parts = [repr(spec), repr(tuple(mesh.shape))]
    for x in leaves:
        if isinstance(x, torch.Tensor):
            parts.append(f"T{tuple(x.shape)}:{x.dtype}")
        elif isinstance(x, torch.nn.Module):
            parts.append(repr(x) + "|" + ",".join(f"{n}{tuple(p.shape)}{p.dtype}"
                                                  for n, p in x.named_parameters()))
        elif isinstance(x, torch.optim.Optimizer):
            parts.append(type(x).__qualname__ + repr([{k: v for k, v in g.items() if k != "params"}
                                                      for g in x.param_groups]))
        else:
            parts.append(repr(x))
    return hashlib.sha256("|".join(parts).encode("utf-8")).hexdigest()[:32]


def input_signature(args, kwargs):
    """Key of a compiled graph: shapes and dtypes of the tensor inputs, repr of everything else
    (scalars; modules and optimizers by identity) — the information the reference's
    get_input_signature hashes (torch/utils.py:210-213: repr of the inputs moved to `meta`)."""
    import hashlib
    leaves, spec = pytree.tree_flatten((args, kwargs))
    parts = [repr(spec)]
    for x in leaves:
        if isinstance(x, torch.Tensor):
            parts.append(f"T{tuple(x.shape)}:{x.dtype}")
        elif isinstance(x, (torch.nn.Module, torch.optim.Optimizer)):
            # the object itself stands for its architecture / hyper-parameters: repr() of a large
            # module costs milliseconds and this runs on every call
            parts.append(f"{type(x).__qualname__}@{id(x):x}")
        else:
            parts.append(repr(x))
    return hashlib.sha256("|".join(parts).encode("utf-8")).hexdigest()


class CompiledFuncWrapper:
    """Dispatch + CUDA-graph capture/replay (reference: api.py:53-224): one compilation, one
    lowered graph per input signature (`enable_mono_graph`), one CUDA graph per signature sharing
    a memory pool."""

    def __init__(self, func, parallel_mode="auto", tracing_mode="fake", cuda_graph=True,
                 enable_mono_graph=False, compile_only=False, compile_kwargs=None):
        update_wrapper(self, func)
        self.original_func = func
        self.compiled_func = None
        self.parallel_mode = parallel_mode
        self.tracing_mode = tracing_mode
        self.enable_cuda_graph = cuda_graph
        self.enable_mono_graph = enable_mono_graph
        self.compile_only = compile_only
        self.compile_kwargs = compile_kwargs or {}
        self.all_input_signature = []
        self.graph_list = {}
        self.cuda_graph_space = {}
        self.graph_pool = None

    def _compile(self, args, kwargs):
        mode = self.parallel_mode
        if mode == "auto":
            return _compile_auto(self.original_func, self.tracing_mode, args, kwargs,
                                 **self.compile_kwargs)
        if mode in DP_MODES:
            return _compile_dp(self.original_func, mode, self.tracing_mode, args, kwargs,
                               **self.compile_kwargs)
        if mode in PARALLEL_EXTENTION:
            return PARALLEL_EXTENTION[mode](self.original_func, mode, self.tracing_mode, args,
                                            kwargs)
        raise NotImplementedError()

    def register_input_signature(self, *args, **kwargs):
        sig = input_signature(args, kwargs)
        if sig not in self.all_input_signature:
            self.all_input_signature.append(sig)
            if self.enable_cuda_graph:
                self.cuda_graph_space[sig] = {"cuda_graph": None, "cuda_graph_input": None,
                                              "cuda_graph_output": None}
        return sig

    def _run(self, sig, args, kwargs):
        if sig not in self.graph_list:
            if not self.enable_mono_graph:
                # same message as the reference (api.py:157-159)
                raise RuntimeError(
                    "Input mismatch. If you are sure that different inputs do not change the graph, "
                    "you can try turning on the enable_mono_graph option.")
            self.graph_list[sig] = self.compiled_func.compile_mono_graph(*args, **kwargs)
            logger.info(f"[Compile API] compile mono graph for {sig}")
        return self.compiled_func.run_with_graph(self.graph_list[sig], *args, **kwargs)

    def __call__(self, *args: Any, **kwargs: Any) -> Any:
        sig = self.register_input_signature(*args, **kwargs)
        if self.compiled_func is None:
            self.compiled_func = self._compile(args, kwargs)
            self.graph_list[sig] = self.compiled_func.graph
        if self.compile_only:
            return self.compiled_func
        if not self.enable_cuda_graph:
            return self._run(sig, args, kwargs)
        space = self.cuda_graph_space[sig]
        flat, spec = pytree.tree_flatten([args, kwargs])
        if space["cuda_graph"] is None:
            space["cuda_graph_input"] = [torch.empty_like(x).copy_(x) if isinstance(x, torch.Tensor)
                                         else x for x in flat]
            sargs, skwargs = pytree.tree_unflatten(space["cuda_graph_input"], spec)
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                space["cuda_graph_output"] = self._run(sig, sargs, skwargs)  # eager warm-up
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            space["cuda_graph"] = torch.cuda.CUDAGraph()
            with torch.cuda.graph(space["cuda_graph"], self.graph_pool):
                space["cuda_graph_output"] = self._run(sig, sargs, skwargs)
            if self.graph_pool is None:
                self.graph_pool = space["cuda_graph"].pool()
        else:
            for dst, src in zip(space["cuda_graph_input"], flat):
                if isinstance(dst, torch.Tensor):
                    dst.copy_(src, non_blocking=True)
        from .compile import _check_health
        _check_health()  # replay launches nothing of ours on the host: check the error record here
        space["cuda_graph"].replay()
        return space["cuda_graph_output"]


def easydist_compile(func=None, parallel_mode="auto", tracing_mode="fake", cuda_graph=True,
                     enable_mono_graph=False, use_hint=False, liveness_only_input=False,
                     max_solver_time=float("inf"), compile_only=False, **compile_kwargs):
    """Same decorator surface as the reference's easydist_compile (api.py:227-256)."""
    if parallel_mode not in ("auto",) + DP_MODES and parallel_mode not in PARALLEL_EXTENTION:
        raise NotImplementedError(
            "please use [auto, ddp, zero2, zero3] for `parallel_mode` or register your parallel "
            "extention")

    def wrap(f):
        return CompiledFuncWrapper(f, parallel_mode, tracing_mode, cuda_graph, enable_mono_graph,
                                   compile_only, compile_kwargs)

    return wrap(func) if func else wrap


def register(reference_api=None, reference_compile_auto=None, **compile_kwargs):
    """Plug this backend into an importable reference (`easydist.torch`).  `compile_kwargs` are
    forwarded to `_compile_dp` (tests run the plugged modes over gloo with `ops=`, `native=False`)."""
    import easydist.torch.api as ref_api
    import easydist.torch.compile_auto as ref_auto
    reference_api = reference_api or ref_api
    reference_compile_auto = reference_compile_auto or ref_auto

    def dp_entry(original_func, parallel_mode, tracing_mode, args, kwargs):
        # the reference's device mesh is the source of truth when this backend is a plugin
        from easydist.torch.device_mesh import get_device_mesh as ref_mesh
        from .device_mesh import set_device_mesh
        set_device_mesh(ref_mesh(), rank=torch.distributed.get_rank())
        return _compile_dp(original_func, parallel_mode, tracing_mode, args, kwargs, **compile_kwargs)

    for mode in DP_MODES:
        reference_api.register_parallel_method(f"b200_{mode}", dp_entry)

    def sharding_transform(fx_module, opt_strategy, state_io_map):
        from easydist.torch.device_mesh import get_device_mesh as ref_mesh
        from .device_mesh import set_device_mesh
        mesh = set_device_mesh(ref_mesh("spmd"), rank=torch.distributed.get_rank())
        ops_ = compile_kwargs.get("ops", _default_ops)
        gm = lowering.sharding_transform(fx_module, opt_strategy, state_io_map, mesh=mesh, ops=ops_)
        if os.environ.get("EDB_LOCALIZE_OPT", "0") == "1":
            # opt-in under Hook B (it changes the communication structure the reference's own
            # lowering would produce): the optimizer's foreach ops on shards; the rewritten graph
            # still only uses the ten reshard callables, so the reference's executor runs it as is
            lowering.localize_foreach(gm, ops_, my_rank=mesh.rank)
        return gm

    reference_compile_auto.sharding_transform = sharding_transform

    # ---- Hook C: the reference's front end, this backend's lowering AND executor ---------------
    class _PlanCaptured(Exception):
        pass

    def auto_entry(original_func, parallel_mode, tracing_mode, args, kwargs):
        """parallel_mode="b200_auto": run the reference's own `_compile_auto` (tracing, sharding
        annotation, MetaIR, AutoFlow ILP on rank 0, plan broadcast — compile_auto.py:456-546) and
        stop it exactly where it would lower (`sharding_transform`, :569): the traced graph and the
        solver's plan are captured and handed to this backend, which lowers them
        (`lowering.sharding_transform` + the product passes), pre-shards the state locally and
        returns ITS `EDCompiledFunc` — so the reference's per-step `distribute_tensor` of every input
        (compile_auto.py:737-745), its op-by-op executor and its NCCL lowering are all out of the
        loop, while `@easydist_compile` and the solver stay the reference's.  Graphs with
        `aten.embedding` need the reference's `fix_embedding(recover=True)` post-pass and are not
        covered."""
        from easydist.torch.device_mesh import get_device_mesh as ref_mesh
        from . import graph_io
        from .device_mesh import set_device_mesh
        mesh = set_device_mesh(ref_mesh("spmd"), rank=torch.distributed.get_rank())
        kw = {k: v for k, v in compile_kwargs.items() if k in ("ops", "native", "planner", "fuse_rt")}
        # plan cache (SURVEY f2; the reference caches the solver's output per input signature,
        # compile_auto.py:97-106,181-184): here the whole captured bundle — traced graph + plan — is
        # cached, so a hit skips tracing, annotation, the ILP and the RPC plan broadcast.  Rank 0
        # decides and ships the text, so the cache directory need not be shared.
        cache_dir = os.environ.get("EDB_PLAN_CACHE_DIR", "")
        cache_file = None
        if cache_dir:
            cache_file = os.path.join(cache_dir, f"b200_auto_{_plan_cache_key(args, kwargs, mesh)}.json.gz")
            import gzip
            box = [None]
            if torch.distributed.get_rank() == 0 and os.path.exists(cache_file):
                with gzip.open(cache_file, "rt") as f:
                    box[0] = f.read()
            if torch.distributed.get_world_size() > 1:
                torch.distributed.broadcast_object_list(box, src=0)
            if box[0] is not None:
                LAST_AUTO_SOURCE[0] = "cache"
                return compile_from_bundle(box[0], args, kwargs, **kw)
        captured = {}
        saved = reference_compile_auto.sharding_transform

        def capture(fx_module, opt_strategy, state_io_map):
            captured["bundle"] = graph_io.dump_bundle(
                fx_module, opt_strategy, [(a.name, b.name) for a, b in state_io_map.items()])
            raise _PlanCaptured()

        reference_compile_auto.sharding_transform = capture
        try:
            reference_compile_auto._compile_auto(original_func, tracing_mode, None, "b200_auto", args,
                                                 kwargs)
            raise RuntimeError("b200_auto: the reference's _compile_auto returned without lowering")
        except _PlanCaptured:
            pass
        finally:
            reference_compile_auto.sharding_transform = saved
        LAST_AUTO_SOURCE[0] = "solved"
        if cache_file is not None and torch.distributed.get_rank() == 0:
            import gzip
            os.makedirs(cache_dir, exist_ok=True)
            tmp = cache_file + f".tmp{os.getpid()}"
            with gzip.open(tmp, "wt") as f:
                f.write(captured["bundle"])
            os.replace(tmp, cache_file)
        return compile_from_bundle(captured["bundle"], args, kwargs, **kw)

    reference_api.register_parallel_method("b200_auto", auto_entry)
    return reference_api
