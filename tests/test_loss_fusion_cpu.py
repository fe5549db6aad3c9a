"""lowering.fuse_cross_entropy: the cross-entropy tail of the traced GPT-2 step is rewritten to
loss.cross_entropy_fwd / cross_entropy_bwd and training still matches the eager model.  (On CPU the
two callables take their ATen branch — the kernel itself is checked by tests/test_gpu_single.py.)"""
import pytest
import torch

from easydist_b200 import api, lowering, loss, workloads
from easydist_b200.device_mesh import set_device_mesh
from tests import gloo_ops

aten = torch.ops.aten


def _targets(gm):
    return [n.target for n in gm.graph.nodes if n.op == "call_function"]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_cross_entropy_chain_is_rewritten_and_matches_eager(dtype):
    set_device_mesh([0], ["dp"], rank=0)
    cfg = workloads.GPT2_CONFIGS["gpt2-tiny"]
    torch.manual_seed(0)
    model = workloads.GPT2(cfg).to(dtype)
    ref = workloads.GPT2(cfg).to(dtype)
    ref.load_state_dict(model.state_dict())
    opt = torch.optim.SGD(model.parameters(), lr=0.05, momentum=0.9)
    ref_opt = torch.optim.SGD(ref.parameters(), lr=0.05, momentum=0.9)
    tok, tgt = workloads.synthetic_tokens(cfg, 2, 32, 0)
    tgt[0, :5] = -100  # ignored positions
    compiled = api._compile_dp(workloads.gpt2_train_step, "ddp", "fake", (tok, tgt, model, opt), {},
                               ops=gloo_ops, native=False)
    gm = compiled.graph
    before = _targets(gm)
    assert aten._log_softmax.default in before and aten.nll_loss_backward.default in before
    assert lowering.fuse_cross_entropy(gm) == 1
    gm.graph.lint()
    after = _targets(gm)
    for t in (aten._log_softmax.default, aten.nll_loss_forward.default, aten.nll_loss_backward.default,
              aten._log_softmax_backward_data.default):
        assert t not in after
    assert after.count(loss.cross_entropy_fwd) == 1 and after.count(loss.cross_entropy_bwd) == 1
    if dtype == torch.bfloat16:  # the fp32 round trip of the logits is gone with the chain
        assert after.count(aten._to_copy.default) == before.count(aten._to_copy.default) - 2
    assert lowering.fuse_cross_entropy(gm) == 0  # idempotent
    for _ in range(3):
        l = compiled(tok, tgt, model, opt)
        l_ref = workloads.gpt2_train_step(tok, tgt, ref, ref_opt)
        assert torch.allclose(l, l_ref.detach(), rtol=1e-5, atol=1e-6), (l, l_ref)
    got = compiled.named_parameters()
    # fp32: same ATen math; bf16: the gradient is rounded to bf16 once in both paths, but from
    # x - lse instead of the stored log-softmax, so single-ulp differences are possible
    rtol, atol = (1e-4, 1e-6) if dtype == torch.float32 else (2e-2, 1e-3)
    for name, p in ref.named_parameters():
        assert torch.allclose(got[name].float(), p.detach().float(), rtol=rtol, atol=atol), name


def test_other_uses_of_log_softmax_block_the_rewrite():
    """A log-softmax whose value is also returned is not a pure cross-entropy chain."""
    set_device_mesh([0], ["dp"], rank=0)

    class M(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.l = torch.nn.Linear(8, 16)

        def forward(self, x):
            return self.l(x)

    def step(x, t, model, opt):
        ls = torch.log_softmax(model(x), -1)
        out = torch.nn.functional.nll_loss(ls, t)
        out.backward()
        opt.step()
        opt.zero_grad(True)
        return out, ls.detach()

    torch.manual_seed(0)
    m = M()
    opt = torch.optim.SGD(m.parameters(), lr=0.1)
    x, t = torch.randn(4, 8), torch.randint(0, 16, (4,))
    compiled = api._compile_dp(step, "ddp", "fake", (x, t, m, opt), {}, ops=gloo_ops, native=False)
    assert lowering.fuse_cross_entropy(compiled.graph) == 0


@pytest.mark.parametrize("opt_kw,expect", [(dict(momentum=0.9), 1), (dict(momentum=0.9, dampening=0.1), 1),
                                           (dict(momentum=0.9, nesterov=True), 0), (dict(), 0)])
def test_sgd_momentum_triple_is_fused_and_matches_unfused(opt_kw, expect):
    """lowering.fuse_optimizer_updates: the three re-inplaced foreach nodes of SGD(momentum) become
    one optim.sgd_momentum_ node; other optimizer flavours are left alone; the step computes the very
    same values as the unfused graph (and as eager SGD; with dampening the traced graph differs from
    eager's first step by construction — the state is warmed up before tracing, as in the reference)."""
    from easydist_b200 import optim
    set_device_mesh([0], ["dp"], rank=0)
    cfg = workloads.GPT2_CONFIGS["gpt2-tiny"]
    tok, tgt = workloads.synthetic_tokens(cfg, 2, 32, 0)

    def build():
        torch.manual_seed(0)
        model = workloads.GPT2(cfg)
        opt = torch.optim.SGD(model.parameters(), lr=0.05, foreach=True, **opt_kw)
        return model, opt

    model, opt = build()
    plain_model, plain_opt = build()
    ref, ref_opt = build()
    compiled = api._compile_dp(workloads.gpt2_train_step, "ddp", "fake", (tok, tgt, model, opt), {},
                               ops=gloo_ops, native=False)
    plain = api._compile_dp(workloads.gpt2_train_step, "ddp", "fake", (tok, tgt, plain_model, plain_opt),
                            {}, ops=gloo_ops, native=False)
    gm = compiled.graph
    assert lowering.fuse_optimizer_updates(gm) == expect
    gm.graph.lint()
    after = _targets(gm)
    assert after.count(optim.sgd_momentum_) == expect
    if expect:
        assert aten._foreach_mul_.Scalar not in after and aten._foreach_add_.List not in after
        gm.graph.eliminate_dead_code()  # the userless update node must survive DCE
        gm.recompile()
        assert _targets(gm).count(optim.sgd_momentum_) == 1
    for _ in range(3):
        l = compiled(tok, tgt, model, opt)
        l_plain = plain(tok, tgt, plain_model, plain_opt)
        l_ref = workloads.gpt2_train_step(tok, tgt, ref, ref_opt)
        assert torch.equal(l, l_plain)
        if "dampening" not in opt_kw:
            assert torch.allclose(l, l_ref.detach(), rtol=1e-5, atol=1e-6), (l, l_ref)
    got, want = compiled.named_parameters(), plain.named_parameters()
    for name in want:
        assert torch.equal(got[name], want[name]), name
