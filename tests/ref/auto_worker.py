"""Reference-in-the-loop parity worker (CPU container only; needs /root/reference).

Runs the UNMODIFIED reference's auto path (annotation -> MetaIR -> AutoFlow ILP) on 2 gloo ranks
twice on the same model, inputs and plan:
   A. with the reference's own lowering + NCCL/gloo functional collectives (sharding.py), and
   B. with `compile_auto.sharding_transform` rebound to easydist_b200.lowering.sharding_transform
      (the drop-in hook of INTEGRATION.md §3), comm callables bound to tests/gloo_ops.py because
      the product ops need a GPU,
and compares both with vanilla PyTorch step by step (outputs, params, optimizer state), i.e. the
reference's own comparator tests/test_torch/test_spmd.py:54-113.  Optionally records the plan and
the traced graph as a fixture for the GPU box (tests/golden/auto_plan_*.pt).
"""
import copy
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


class Foo(torch.nn.Module):
    def __init__(self, d=64):
        super().__init__()
        self.norm = torch.nn.LayerNorm(d)
        self.linear = torch.nn.Linear(d, d)

    def forward(self, x):
        return self.linear(self.norm(x)).relu()


def train_step(input, model, opt):
    out = model(input)
    loss = out.mean()
    loss.backward()
    opt.step()
    opt.zero_grad()
    return out


def _comm_hist(gm):
    hist = {}
    for n in gm.graph.nodes:
        if n.op == "call_function":
            nm = getattr(n.target, "__name__", str(n.target))
            if "inner" in nm:
                nm = "box_exchange"  # the reference's do_p2p_comm_wrapper closure
            if any(k in nm for k in ("all_", "reduce_scatter", "scatter_wrapper", "copy_wrapper",
                                     "box_exchange")):
                hist[nm] = hist.get(nm, 0) + 1
    return hist


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    mesh_shape = tuple(int(v) for v in os.environ.get("EDB_TEST_MESH", str(world)).split("x"))
    record = os.environ.get("EDB_RECORD", "")
    record_parity = os.environ.get("EDB_RECORD_PARITY", "")
    planner = os.environ.get("EDB_PLANNER", "GREEDY")
    # recording large plans: rank 0 does the sharding discovery + ILP alone while the others wait
    torch.set_num_threads(int(os.environ.get("EDB_THREADS_RANK0" if rank == 0 else "EDB_THREADS", "1")))
    dist.init_process_group("gloo")
    from oracle import refcompat
    refcompat.install()
    from easydist import easydist_setup
    from easydist.torch.api import easydist_compile
    from easydist.torch.device_mesh import set_device_mesh
    import easydist.torch.compile_auto as ref_auto
    from torch.distributed.device_mesh import DeviceMesh
    easydist_setup(backend="torch", device="cpu", allow_tf32=False)
    import easydist.config as mdconfig
    mdconfig.experimental_sharding_transform = planner  # config.py:115-117
    names = [f"spmd{i}" for i in range(len(mesh_shape))]
    tmesh = DeviceMesh("cpu", torch.arange(world).reshape(mesh_shape), mesh_dim_names=names)
    set_device_mesh(tmesh)

    from easydist_b200 import lowering
    from easydist_b200.device_mesh import set_device_mesh as edb_set_mesh
    from tests import gloo_ops
    my_mesh = edb_set_mesh(torch.arange(world).reshape(mesh_shape).numpy(), names, rank=rank)
    gloo_ops.init_groups(my_mesh.mesh)

    torch.manual_seed(42)
    g = torch.Generator().manual_seed(7)
    if os.environ.get("EDB_MODEL", "foo") == "gpt":
        # the reference's own test model: TEST_GPT of tests/test_torch/test_utils.py:55-68
        # (EDB_GPT="depth,dim,heads,batch,seq" scales it up, e.g. "4,1024,32,4,128" = SURVEY.md
        # config 1, the reference's examples/torch/gpt_train.py)
        from benchmark.torch.model.gpt import GPT
        depth, dim, heads, gb, gs = (int(v) for v in os.environ.get("EDB_GPT", "2,64,4,4,32").split(","))
        model0 = GPT(depth=depth, dim=dim, num_heads=heads)
        batches = [torch.randn(gb, gs, dim, generator=g) for _ in range(int(os.environ.get("EDB_STEPS", "2")))]
        model_tag = f"GPT(depth={depth}, dim={dim}, num_heads={heads})"
        batch_shape = [gb, gs, dim]
    else:
        model0 = Foo()
        batches = [torch.randn(16, 64, generator=g) for _ in range(3)]
        model_tag, batch_shape = "Foo(64)", [16, 64]

    def run(variant):
        model = copy.deepcopy(model0)
        opt = torch.optim.SGD(model.parameters(), lr=0.1, momentum=0.9, foreach=True)
        saved = {}
        if variant == "B":
            orig = ref_auto.sharding_transform

            def mine(fx_module, opt_strategy, state_io_map):
                if (record or record_parity) and rank == 0:
                    from easydist_b200 import graph_io
                    saved["plan"] = graph_io.dump_bundle(
                        fx_module, opt_strategy,
                        [(a.name, b.name) for a, b in state_io_map.items()],
                        extra={"mesh": list(mesh_shape), "model": model_tag, "seed": 42,
                               "batch_seed": 7, "batch": batch_shape, "planner": planner})
                if os.environ.get("EDB_SAMEPLAN") == "1":
                    # the reference's lowering of the VERY SAME plan (the ILP may return another
                    # equal-cost plan on a second solve, so run A alone does not isolate the lowering)
                    import torch.fx as fx
                    g2 = fx.GraphModule(fx_module, copy.deepcopy(fx_module.graph))
                    for n_old, n_new in zip(fx_module.graph.nodes, g2.graph.nodes):
                        n_new.meta = dict(n_old.meta)
                    ref_gm = orig(g2, opt_strategy, state_io_map)
                    saved["hist_ref_same_plan"] = _comm_hist(ref_gm)
                return lowering.sharding_transform(fx_module, opt_strategy, state_io_map,
                                                   ops=gloo_ops, mesh=my_mesh, planner=planner)
            ref_auto.sharding_transform = mine
        try:
            step = easydist_compile(train_step, "auto", "fake", cuda_graph=False)
            outs = [step(b, model, opt).detach().clone() for b in batches]
        finally:
            if variant == "B":
                ref_auto.sharding_transform = orig
        cf = step.compiled_func
        return outs, cf, _comm_hist(cf.graph), saved

    # vanilla
    vmodel = copy.deepcopy(model0)
    vopt = torch.optim.SGD(vmodel.parameters(), lr=0.1, momentum=0.9, foreach=True)
    vouts = [train_step(b, vmodel, vopt).detach().clone() for b in batches]

    only_b = os.environ.get("EDB_ONLY_B") == "1"  # recording large plans: skip the pure-reference run
    outs_b, cf_b, hist_b, saved = run("B")
    outs_a, cf_a, hist_a = (outs_b, cf_b, hist_b) if only_b else run("A")[:3]

    def full(cf, name, like):
        """Reassemble a (possibly sharded) parameter for comparison: all_gather along every dim
        whose local size differs from the global one."""
        p = cf.named_parameters()[name]
        p = p.to_local() if hasattr(p, "to_local") else p
        for d in range(like.dim()):
            if p.shape[d] != like.shape[d]:
                parts = [torch.empty_like(p) for _ in range(world)]
                dist.all_gather(parts, p.contiguous())
                p = torch.cat(parts, dim=d)
                # de-duplicate when the mesh shards this dim on a sub-group only
                if p.shape[d] != like.shape[d]:
                    p = p.narrow(d, 0, like.shape[d])
        return p

    ok = True
    msgs = []
    for i in range(len(batches)):
        for tag, o in (("A", outs_a[i]), ("B", outs_b[i])):
            if not torch.allclose(o, vouts[i], rtol=1e-4, atol=1e-5):
                ok = False
                msgs.append(f"step {i} output {tag} vs vanilla: {(o - vouts[i]).abs().max()}")
        if not torch.equal(outs_a[i], outs_b[i]):
            d = (outs_a[i] - outs_b[i]).abs().max().item()
            if d > 1e-6:
                ok = False
                msgs.append(f"step {i} A vs B differ by {d}")
    if len(mesh_shape) == 1:
        for name, p_ref in vmodel.named_parameters():
            for tag, cf in (("A", cf_a), ("B", cf_b)):
                p = full(cf, name, p_ref)
                if p.shape != p_ref.shape or not torch.allclose(p, p_ref.detach(), rtol=1e-4,
                                                                atol=1e-5):
                    ok = False
                    msgs.append(f"param {name} {tag} differs")
    if rank == 0:
        same = saved.get("hist_ref_same_plan")
        print(f"AUTO_PARITY ok={ok} hist_ref={hist_a} hist_b200={hist_b} {msgs}"
              + (f" hist_ref_same_plan={same} same_plan_equal={same == hist_b}" if same else ""),
              flush=True)
        if record and "plan" in saved:
            with open(record, "w") as f:
                f.write(saved["plan"])
        if record_parity:
            # what tests/test_ref_parity.py compares this backend's lowering of the same plan with,
            # where the reference is not importable: its comm structure and (a strided sample of)
            # the outputs of the reference's own lowering
            import gzip
            import json
            sample = lambda o: [float(str(v)) for v in
                                o.flatten()[::max(1, o.numel() // 256)].numpy()]
            with gzip.open(record_parity, "wt") as f:
                json.dump({"bundle": json.loads(saved["plan"]), "hist_ref_same_plan": same,
                           "ref_outputs": [sample(o) for o in outs_a]}, f, separators=(",", ":"))
    dist.barrier()
    dist.destroy_process_group()
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
