"""Host-side logic of the data-parallel path with world_size 2 on CPU (gloo): tracing front-end,
transform_ddp / transform_fsdp (compile_dp.py:55-198 equivalents), executor — against vanilla
single-process PyTorch on the concatenated batch, the reference's own comparator
(tests/test_torch/test_spmd.py:97-113, rtol=1e-4 atol=1e-5)."""
import os
import sys

import pytest
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests._procs import run_world  # noqa: E402


class Foo(torch.nn.Module):
    """LayerNorm + Linear, the `Foo` model of tests/test_torch/test_spmd.py:31-40 (scaled down)."""

    def __init__(self, d=32):
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
    return loss


def train_step_clipped(input, model, opt):
    out = model(input)
    loss = out.mean()
    loss.backward()
    torch.nn.utils.clip_grad_norm_(model.parameters(), 0.05)
    opt.step()
    opt.zero_grad()
    return loss


def make_opt(kind, params):
    if kind == "sgd":
        return torch.optim.SGD(params, lr=0.1, momentum=0.9, foreach=True)
    if kind == "sgd_plain":
        return torch.optim.SGD(params, lr=0.1, foreach=True)
    if kind == "adam_fused":
        return torch.optim.Adam(params, lr=1e-2, fused=True)
    if kind == "adamw_fused":
        return torch.optim.AdamW(params, lr=1e-2, weight_decay=0.05, fused=True)
    return torch.optim.Adam(params, lr=1e-2, foreach=True)


class Wide(torch.nn.Module):
    """Linear layers wide enough (256 rows per rank at world 2) for the AG+GEMM / GEMM+RS fusion
    patterns to apply."""

    def __init__(self, d=256):
        super().__init__()
        self.norm = torch.nn.LayerNorm(d)
        self.fc1 = torch.nn.Linear(d, 2 * d)
        self.fc2 = torch.nn.Linear(2 * d, d)

    def forward(self, x):
        return self.fc2(torch.nn.functional.gelu(self.fc1(self.norm(x))))


def _fusion_worker(rank, world, port, q, case="epoch", d=256):
    os.environ["OMP_NUM_THREADS"] = "1"
    os.environ["EDB_AG_PREFETCH"] = "0" if case == "no_prefetch" else "1"
    torch.set_num_threads(1)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank,
                            world_size=world)
    from easydist_b200 import api
    from easydist_b200.device_mesh import set_device_mesh
    from tests import gloo_ops
    set_device_mesh(list(range(world)), ["dp"], rank=rank)
    torch.manual_seed(0)
    model = Wide(d).bfloat16()
    ref_model = Wide(d).bfloat16()
    ref_model.load_state_dict(model.state_dict())
    opt = make_opt("sgd", model.parameters())
    ref_opt = make_opt("sgd", ref_model.parameters())
    g = torch.Generator().manual_seed(5)
    batches = [torch.randn(world * 8, d, generator=g).bfloat16() for _ in range(3)]
    compiled = api._compile_dp(train_step, "zero3", "fake", (batches[0][rank * 8:(rank + 1) * 8],
                                                            model, opt), {}, ops=gloo_ops,
                               native=False, bucket_numel=2048, fuse=True,
                               fuse_rt=gloo_ops.FakeSymmRuntime())
    ok, msg = True, ""
    for b in batches:
        loss = compiled(b[rank * 8:(rank + 1) * 8], model, opt)
        ref_loss = train_step(b, ref_model, ref_opt)
        loss_all = loss.detach().float().clone()
        dist.all_reduce(loss_all)
        loss_all /= world
        if not torch.allclose(loss_all, ref_loss.detach().float(), rtol=3e-2, atol=1e-3):
            ok, msg = False, f"loss {loss_all} vs {ref_loss}"
    info = dict(compiled.info)
    info["barriers_run"] = gloo_ops._EPOCHS["barriers"]
    nodes = list(compiled.graph.graph.nodes)
    info["order"] = [n.target.__name__ for n in nodes if n.op == "call_function" and
                     n.target in (gloo_ops.epoch_barrier, gloo_ops.rs_finish, gloo_ops.mm_push,
                                  gloo_ops.ag_mm) or getattr(n.target, "__name__", "") == "sgd_momentum_"]
    info["carried"] = sum(1 for n in nodes if "edb_pf" in n.meta)
    if rank == 0:
        q.put((ok, msg, info))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("case,world,d", [("epoch", 2, 256), ("epoch", 4, 512),
                                          ("no_prefetch", 2, 256), ("no_prefetch", 4, 512)])
def test_fusion_rewrite_on_cpu(case, world, d):
    """The AG+GEMM / GEMM+RS peephole (lowering.fuse_collective_gemms) rewrites the zero3 graph of
    a 2-layer MLP: both weight gradients' reduce-scatters become push-only GEMMs + one rs_finish in
    front of the optimizer, and both weights' all-gathers become prefetches (no_prefetch: fuse into
    their forward GEMMs, ag_mm); training still matches vanilla."""
    ok, msg, info = run_world(_fusion_worker, world,
                              lambda r, port, q: (r, world, port, q, case, d), timeout=180)
    assert ok, msg
    want_fused = {"ag_mm": 0, "ag_pf": 2, "mm_rs": 2} if case == "epoch" else \
        {"ag_mm": 2, "ag_pf": 0, "mm_rs": 2}
    assert info["fused"] == want_fused, info
    assert info["comm_nodes"].get("reduce_scatter_start", 0) == 0, info
    # epoch protocol: flag-free fused kernels, exactly two barriers per step — one between the
    # last push and the reduction of the slots (in front of the optimizer), one at the very end
    assert info["comm_nodes"].get("mm_push") == 2 and info["comm_nodes"].get("rs_finish") == 1, info
    assert info["comm_nodes"].get("epoch_barrier") == 2, info
    assert info["barriers_run"] == 2 * 3, info  # 3 steps
    order = info["order"]
    if case == "epoch":
        # parameter gathers are prefetches: fc1's (needed before the first GEMM) stand-alone at the
        # top, fc2's riding on the fc1 GEMM up to that (tiny) GEMM's byte budget and the remainder
        # stand-alone in front of the use; every use reads the gathered buffer
        assert info["comm_nodes"].get("ag_prefetch") == 2 and "ag_mm" not in info["comm_nodes"], info
        assert info["comm_nodes"].get("gathered", 0) >= 2, info
        assert info["carried"] == 1, info
        assert order.index("rs_finish") == order.index("epoch_barrier") + 1, order
        assert max(i for i, k in enumerate(order) if k == "mm_push") < order.index("epoch_barrier"), order
        assert order[-1] == "epoch_barrier", order
    else:
        assert info["comm_nodes"].get("ag_mm") == 2, info
        assert order == ["ag_mm", "ag_mm", "mm_push", "mm_push", "epoch_barrier", "rs_finish",
                         "epoch_barrier"], order


def _run_case(rank, world, mode, opt_kind, bucket=0, generic_bucket="0", clip=False):
    """One DP case inside an initialised 2-rank gloo job -> (ok, message, comm histogram)."""
    step_fn = train_step_clipped if clip else train_step
    os.environ["EDB_BUCKET_COMM"] = generic_bucket
    from easydist_b200 import api, lowering
    from easydist_b200.device_mesh import set_device_mesh
    from tests import gloo_ops
    set_device_mesh([list(range(world))][0], ["dp"], rank=rank)
    torch.manual_seed(0)
    model = Foo()
    ref_model = Foo()
    ref_model.load_state_dict(model.state_dict())
    opt = make_opt(opt_kind, model.parameters())
    ref_opt = make_opt(opt_kind, ref_model.parameters())
    g = torch.Generator().manual_seed(123)
    batches = [torch.randn(world * 4, 32, generator=g) for _ in range(3)]
    compiled = api._compile_dp(step_fn, mode, "fake", (batches[0][rank * 4:(rank + 1) * 4], model,
                                                      opt), {}, ops=gloo_ops, native=False,
                               bucket_numel=bucket)
    # the optimizer rewrite of the native path (on CPU the fused node takes its ATen branch): the
    # sharded update of every mode must still match vanilla
    n_opt = lowering.fuse_optimizer_updates(compiled.graph)
    # zero2 updates parameter shards out of place (the new shards are all-gathered): no triple
    assert n_opt == (1 if opt_kind == "sgd" and mode != "zero2" else 0), (mode, opt_kind, n_opt)
    ok = True
    msg = ""
    for b in batches:
        loss = compiled(b[rank * 4:(rank + 1) * 4], model, opt)
        ref_loss = step_fn(b, ref_model, ref_opt)
        # local loss is the mean over the local micro-batch; the global mean is their average
        loss_all = loss.detach().clone()
        dist.all_reduce(loss_all)
        loss_all /= world
        if not torch.allclose(loss_all, ref_loss.detach(), rtol=1e-4, atol=1e-5):
            ok, msg = False, f"loss {loss_all} vs {ref_loss}"
    params = compiled.named_parameters()
    for name, p_ref in ref_model.named_parameters():
        p = params[name]
        if mode == "zero3" and p.shape != p_ref.shape:
            parts = [torch.empty_like(p) for _ in range(world)]
            dist.all_gather(parts, p.contiguous())
            p = torch.cat(parts).view(p_ref.shape)
        if not torch.allclose(p, p_ref.detach(), rtol=1e-4, atol=1e-5):
            ok, msg = False, f"param {name} differs: {(p - p_ref).abs().max()}"
    return ok, msg, dict(compiled.info["comm_nodes"])


# every case of this file that runs the Foo MLP through a DP mode; executed once, in ONE 2-rank
# gloo job (process start-up dominates these tests), looked up by the test functions below
CASES = {}
for _mode, _opt, _bucket in [("ddp", "sgd", 0), ("ddp", "sgd_plain", 0), ("zero2", "sgd", 0),
                             ("zero3", "sgd", 0), ("zero3", "sgd_plain", 0), ("zero2", "sgd_plain", 0),
                             ("zero3", "sgd", 100), ("zero2", "sgd", 100), ("ddp", "sgd", 100)]:
    CASES[f"vanilla-{_mode}-{_opt}-{_bucket}"] = dict(mode=_mode, opt_kind=_opt, bucket=_bucket)
for _mode in ("ddp", "zero3"):
    CASES[f"generic-bucket-{_mode}"] = dict(mode=_mode, opt_kind="sgd", generic_bucket="1")
for _mode, _opt in [("ddp", "adamw_fused"), ("zero2", "adamw_fused"), ("zero3", "adam_fused"),
                    ("zero3", "adamw_fused")]:
    CASES[f"fused-{_mode}-{_opt}"] = dict(mode=_mode, opt_kind=_opt)
CASES["clip-ddp"] = dict(mode="ddp", opt_kind="sgd", clip=True)


def _batch_worker(rank, world, port, q):
    os.environ["OMP_NUM_THREADS"] = "1"
    torch.set_num_threads(1)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank,
                            world_size=world)
    results = {}
    for name, case in CASES.items():
        try:
            results[name] = _run_case(rank, world, **case)
        except Exception as e:  # noqa: BLE001 — reported per case
            import traceback
            results[name] = (False, f"{type(e).__name__}: {e}\n{traceback.format_exc()[-1500:]}", {})
        dist.barrier()
    if rank == 0:
        q.put(results)
    dist.barrier()
    dist.destroy_process_group()


@pytest.fixture(scope="module")
def dp_results():
    return run_world(_batch_worker, 2, lambda r, port, q: (r, 2, port, q), timeout=600)


@pytest.mark.parametrize("mode,opt_kind,bucket", [("ddp", "sgd", 0), ("ddp", "sgd_plain", 0),
                                                  ("zero2", "sgd", 0), ("zero3", "sgd", 0),
                                                  ("zero3", "sgd_plain", 0), ("zero2", "sgd_plain", 0),
                                                  ("zero3", "sgd", 100), ("zero2", "sgd", 100),
                                                  ("ddp", "sgd", 100)])
def test_dp_modes_match_vanilla(dp_results, mode, opt_kind, bucket):
    ok, msg, hist = dp_results[f"vanilla-{mode}-{opt_kind}-{bucket}"]
    assert ok, msg
    if mode == "ddp" and bucket == 0:
        assert hist.get("all_reduce_start", 0) == 4      # one per parameter
    if mode == "ddp" and bucket:
        assert hist.get("all_reduce_start", 0) == 2      # the weight + one bucket
    if mode in ("zero2", "zero3") and bucket == 0:
        assert hist.get("reduce_scatter_start", 0) == 4
        assert hist.get("all_gather_start", 0) >= 4
    if bucket and mode != "ddp":
        # only the 32x32 weight is sharded; the three small tensors share one all-reduce
        assert hist.get("reduce_scatter_start", 0) == 1 and hist.get("all_reduce_start", 0) == 1


@pytest.mark.parametrize("mode", ["ddp", "zero3"])
def test_generic_comm_bucketing_in_dp_graphs(dp_results, mode):
    """EDB_BUCKET_COMM=1 (lowering.bucket_small_comm) on the tensor-by-tensor DP graphs: the four
    per-parameter collectives of each kind collapse into buckets and training still matches vanilla."""
    ok, msg, hist = dp_results[f"generic-bucket-{mode}"]
    assert ok, msg
    if mode == "ddp":
        assert hist.get("all_reduce_start", 0) == 1, hist   # 4 gradients, one bucket
    else:
        assert hist.get("all_gather_start", 0) < 4, hist     # parameter shards gathered together


@pytest.mark.parametrize("mode,opt_kind", [("ddp", "adamw_fused"), ("zero2", "adamw_fused"),
                                           ("zero3", "adam_fused"), ("zero3", "adamw_fused")])
def test_fused_adam_in_dp_modes(dp_results, mode, opt_kind):
    """torch.optim.Adam/AdamW(fused=True) — the `_fused_adam` node the reference's DP rewrites are
    written around (compile_dp.py:55-198) — through ddp / zero2 / zero3; in ddp / zero3 the traced
    functional op + copies are re-inplaced to `_fused_adam_`.  AdamW also pins that compiling does not
    touch the parameters: the warm-up step that materialises the optimizer state runs without weight
    decay and the parameter values are restored (the reference's warm-up decays them once)."""
    ok, msg, _ = dp_results[f"fused-{mode}-{opt_kind}"]
    assert ok, msg


def test_ddp_with_gradient_clipping_clips_the_averaged_gradients(dp_results):
    """clip_grad_norm_ between backward and the optimizer: the norm must be taken over the
    all-reduced gradients (what eager DDP does), i.e. every reader of a gradient is rewired to the
    collective's result, not only the optimizer."""
    ok, msg, _ = dp_results["clip-ddp"]
    assert ok, msg
