"""Parity with the reference's own lowering.

test_dropin_lowering_equals_reference_lowering needs nothing outside the repository: the unmodified
reference traced, annotated and solved each case; the plan, the comm structure of the reference's
own lowering of that plan and the outputs of its own run are stored in
tests/golden/ref_lowering_*.json.gz (tests/ref/auto_worker.py with EDB_SAMEPLAN=1 and
EDB_RECORD_PARITY).  Here easydist_b200.lowering.sharding_transform lowers the same plan over gloo and
is compared with those results and with vanilla PyTorch.

test_plugin_hook_through_the_reference_decorator drives this backend through the reference's own
decorator, so it runs only where the reference source is installed (EASYDIST_REFERENCE)."""
import copy
import gzip
import json
import os
import sys

import pytest
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests._procs import run_torchrun, run_world  # noqa: E402
GOLDEN = os.path.join(ROOT, "tests", "golden")


def _replay_worker(rank, world, mesh, planner, model, port, q):
    os.environ["OMP_NUM_THREADS"] = "1"
    torch.set_num_threads(1)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank,
                            world_size=world)
    import numpy as np
    from easydist_b200 import api
    from easydist_b200.device_mesh import set_device_mesh
    from easydist_b200.workloads import EmbeddingGPT
    from tests import gloo_ops
    from tests.ref.auto_worker import Foo, _comm_hist, train_step
    mesh_shape = tuple(int(v) for v in mesh.split("x"))
    set_device_mesh(np.arange(world).reshape(mesh_shape),
                    [f"spmd{i}" for i in range(len(mesh_shape))], rank=rank)
    gloo_ops.init_groups(np.arange(world).reshape(mesh_shape))
    with gzip.open(os.path.join(GOLDEN, f"ref_lowering_{model}_mesh{mesh}_{planner}.json.gz"),
                   "rt") as f:
        rec = json.load(f)
    # the recording's model, seeds and batches (tests/ref/auto_worker.py); EmbeddingGPT(2, 64, 4) is
    # the reference's GPT test model with the same parameters under the same seed
    torch.manual_seed(42)
    g = torch.Generator().manual_seed(7)
    if model == "gpt":
        model0 = EmbeddingGPT(2, 64, 4)
        batches = [torch.randn(4, 32, 64, generator=g) for _ in range(2)]
    else:
        model0 = Foo()
        batches = [torch.randn(16, 64, generator=g) for _ in range(3)]
    vmodel = copy.deepcopy(model0)
    vopt = torch.optim.SGD(vmodel.parameters(), lr=0.1, momentum=0.9, foreach=True)
    opt = torch.optim.SGD(model0.parameters(), lr=0.1, momentum=0.9, foreach=True)
    compiled = api.compile_from_bundle(json.dumps(rec["bundle"]), (batches[0], model0, opt), {},
                                       ops=gloo_ops, native=False, planner=planner)
    msgs = []
    for i, b in enumerate(batches):
        out = compiled(b, model0, opt).detach()
        want = train_step(b, vmodel, vopt).detach()
        if out.shape != want.shape or not torch.allclose(out, want, rtol=1e-4, atol=1e-5):
            msgs.append(f"step {i}: output vs vanilla {(out - want).abs().max()}")
        got = out.flatten()[::max(1, out.numel() // 256)]
        ref = torch.tensor(rec["ref_outputs"][i])
        if got.shape != ref.shape or (got - ref).abs().max().item() > 1e-6:
            msgs.append(f"step {i}: output vs the reference's lowering {(got - ref).abs().max()}")
    if len(mesh_shape) == 1:
        for name, p_ref in vmodel.named_parameters():
            p = compiled.named_parameters()[name]
            for d in range(p_ref.dim()):
                if p.shape[d] != p_ref.shape[d]:
                    parts = [torch.empty_like(p) for _ in range(world)]
                    dist.all_gather(parts, p.contiguous())
                    p = torch.cat(parts, dim=d).narrow(d, 0, p_ref.shape[d])
            if p.shape != p_ref.shape or not torch.allclose(p, p_ref.detach(), rtol=1e-4, atol=1e-5):
                msgs.append(f"param {name} differs from vanilla")
    all_msgs = [None] * world
    dist.all_gather_object(all_msgs, msgs)
    if rank == 0:
        q.put(([m for ms in all_msgs for m in ms], _comm_hist(compiled.graph),
               rec["hist_ref_same_plan"]))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("mesh,nproc,planner,model", [
    ("2", 2, "GREEDY", "foo"), ("2x2", 4, "GREEDY", "foo"),
    ("2x2", 4, "REPLICATE", "foo"), ("2x2", 4, "P2P", "foo"),
    ("2", 2, "GREEDY", "gpt"),   # the reference's GPT test model: views, expand, bmm
])
def test_dropin_lowering_equals_reference_lowering(mesh, nproc, planner, model):
    msgs, hist, hist_ref = run_world(
        _replay_worker, nproc, lambda r, port, q: (r, nproc, mesh, planner, model, port, q),
        timeout=280)
    assert not msgs, msgs
    # same communication structure as the reference's lowering of the very same plan
    assert hist == hist_ref, (hist, hist_ref)


@pytest.mark.refonly
@pytest.mark.parametrize("mode", ["b200_ddp", "b200_zero3", "auto", "b200_auto", "auto+localize",
                                  "b200_auto+gpt"])
def test_plugin_hook_through_the_reference_decorator(mode):
    """Hook A of INTEGRATION.md: `easydist_b200.api.register()` adds the modes to the reference's
    registry (`register_parallel_method`, api.py:39-50); the REFERENCE's own `easydist_compile`
    decorator and CompiledFuncWrapper then drive this backend's compiled object (`.graph`,
    `.run_with_graph`, state accessors); "auto" = Hook B, the `sharding_transform` name rebound by
    the same call; "b200_auto" = Hook C: the reference's tracing + annotation + ILP produce the plan,
    this backend lowers AND executes it (its own EDCompiledFunc, no per-step distribute_tensor) —
    tests/ref/plugin_worker.py."""
    from oracle import refcompat
    if not refcompat.available():
        pytest.skip("needs the reference source tree (set EASYDIST_REFERENCE)")
    env = dict(os.environ, OMP_NUM_THREADS="1", EDB_PLUGIN_MODE=mode)
    if mode == "auto+localize":
        # Hook B with the optimizer localized: the REFERENCE's executor runs the rewritten graph
        env.update(EDB_PLUGIN_MODE="auto", EDB_LOCALIZE_OPT="1")
    cached = mode == "b200_auto"
    if mode == "b200_auto+gpt":
        # Hook C on the reference's GPT test model, with the product structure of the auto path
        # (optimizer on shards, parameter gathers rewritten to prefetched-buffer reads) executed by
        # this backend's EDCompiledFunc
        mode = "b200_auto"
        env.update(EDB_PLUGIN_MODE="b200_auto", EDB_PLUGIN_MODEL="gpt", EDB_LOCALIZE_OPT="1",
                   EDB_TEST_AUTO_PF="1")
    elif mode == "b200_auto":
        import tempfile
        env["EDB_PLAN_CACHE_DIR"] = tempfile.mkdtemp(prefix="edb_plan_cache_")
    rc, out, err = run_torchrun(os.path.join(ROOT, "tests", "ref", "plugin_worker.py"), 2, env,
                                timeout=280, cwd=ROOT, python=sys.executable)
    line = next((l for l in out.splitlines() if l.startswith("PLUGIN_PARITY")), "")
    assert rc == 0 and "ok=True" in line, out[-2000:] + err[-3000:]
    if mode.startswith("b200_"):
        # the object the reference's wrapper drives is THIS backend's executor
        assert "compiled=easydist_b200.compile.EDCompiledFunc" in line, line
    if env.get("EDB_TEST_AUTO_PF") == "1":
        assert "'ag_pf': 0" not in line and "'ag_pf'" in line, line   # the prefetch rewrite applied
    if cached:
        # ... and a second compilation took graph + plan from the plan cache (SURVEY f2)
        assert "plan_source=['solved', 'cache']" in line, line
