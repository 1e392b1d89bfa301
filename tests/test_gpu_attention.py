"""Attention core (public cuda_ops entry points) vs the fp32 reference: the un-fused pair (batched tcgen05 GEMMs +
softmax kernels) and every fused kernel ops/attention_plan.py can choose, each checked to be the one that runs."""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from vit_10b_fsdp_example_b200.ops import attention_plan as ap  # noqa: E402

pytestmark = pytest.mark.gpu

FWD_FAMILY = {ap.ONESHOT: "attn_fwd_sm100_kernel", ap.LONG: "attn_fwd_long_sm100_kernel",
              ap.PERSIST: "attn_fwd_persist_sm100_kernel", ap.UNFUSED: "softmax_fwd_kernel"}
BWD_FAMILY = {ap.ONESHOT: "attn_bwd_sm100_kernel", ap.PERSIST: "attn_bwd_persist_sm100_kernel"}

# (B, N, H, hd) and what the plan runs there (fwd_lse / fwd / bwd)
FUSED_SHAPES = [
    (1, 256, 2, 64),    # oneshot / oneshot / oneshot, keys padded to 256
    (3, 196, 3, 64),    # ViT-L/16 tokens: masked key columns
    (4, 64, 2, 64),     # keys padded to 128
    (2, 64, 2, 128),
    (2, 128, 2, 128),
    (3, 100, 2, 160),   # oneshot / unfused / masked persist
    (2, 130, 2, 160),   # masked persist / masked persist / oneshot (N % 4 == 2)
    (3, 196, 3, 160),   # masked persist / masked persist / masked persist
    (2, 256, 4, 160),   # ViT-10B tokens: persist everywhere, masks compiled out
    (40, 256, 8, 160),  # more work items (640) than SMs: every persistent CTA runs several pipelined items
    (1, 320, 2, 64),    # long / unfused / oneshot
    (2, 576, 2, 128),
    (1, 1024, 2, 64),   # the longest sequence the fused backward takes
    (1, 576, 2, 160),   # 336 px tokens: long / unfused / persist
]


def _close(got, ref, rel=3e-2):
    """Per-element relative + absolute bound (tests/helpers.py), not a max-normalised one."""
    from helpers import assert_close_elementwise

    assert_close_elementwise(got, ref, rtol=rel, atol_rel=rel)


def _families(fn, table):
    """Run fn under torch.profiler; return its result and which kernel families of `table` it launched."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    return res, {fam for fam in table.values() if any(fam in n for n in names)}


def test_shapes_cover_every_kernel_the_plan_returns():
    fields = ("fwd_lse", "fwd", "bwd")
    possible = {(f, getattr(ap.plan(N, hd), f)) for hd in (64, 128, 160) for N in range(2, 1101) for f in fields}
    tested = {(f, getattr(ap.plan(N, hd), f)) for _, N, _, hd in FUSED_SHAPES for f in fields}
    assert possible - {(f, None) for f in fields} <= tested


@pytest.mark.parametrize("B,N,H,hd", [(2, 256, 4, 160), (3, 196, 3, 64), (1, 576, 2, 160)])
def test_attention_fwd_bwd(B, N, H, hd):
    from vit_10b_fsdp_example_b200.ops import cuda_ops as co, torch_ops as to

    D = H * hd
    qkv = (torch.randn(B * N, 3 * D, device="cuda") * 0.5).to(torch.bfloat16)
    out, p = co.attention_fwd(qkv, B, N, H, hd)
    outr, pr = to.attention_fwd(qkv.float(), B, N, H, hd)
    _close(p.view(B, H, N, -1)[..., :N], pr)
    _close(out, outr)
    dout = (torch.randn(B * N, D, device="cuda")).to(torch.bfloat16)
    dqkv, cs = co.attention_bwd(dout, qkv, p, B, N, H, hd, want_colsum=True)
    dqkvr, csr = to.attention_bwd(dout.float(), qkv.float(), pr, B, N, H, hd, want_colsum=True)
    _close(dqkv, dqkvr)
    _close(cs, csr, rel=5e-2)


@pytest.mark.parametrize("B,N,H,hd", FUSED_SHAPES)
def test_attention_forward_runs_the_planned_kernel(B, N, H, hd):
    """Both forwards (with and without the row log-sum-exp) run the kernel the plan names and match the reference."""
    from vit_10b_fsdp_example_b200.ops import cuda_ops as co, torch_ops as to

    plan = ap.plan(N, hd)
    D = H * hd
    qkv = (torch.randn(B * N, 3 * D, device="cuda") * 0.7).to(torch.bfloat16)
    outr, _ = to.attention_fwd(qkv.float(), B, N, H, hd)
    _, lser = to.attention_fwd_lse(qkv.float(), B, N, H, hd)
    (out, p), fams = _families(lambda: co.attention_fwd(qkv, B, N, H, hd, need_p=False), FWD_FAMILY)
    assert fams == {FWD_FAMILY[plan.fwd]}
    assert (p is None) == (plan.fwd != ap.UNFUSED)
    _close(out, outr)
    (out2, lse), fams = _families(lambda: co.attention_fwd_lse(qkv, B, N, H, hd), FWD_FAMILY)
    assert fams == {FWD_FAMILY[plan.fwd_lse]}
    _close(out2, outr)
    assert (lse - lser).abs().max().item() < 2e-2
    if plan.fwd == plan.fwd_lse:  # the same kernel with and without the lse output
        assert torch.equal(out2, out)


@pytest.mark.parametrize("B,N,H,hd", FUSED_SHAPES)
def test_attention_backward_runs_the_planned_kernel(B, N, H, hd):
    """The fused backward (delta kernel + dK/dV role + dQ role) runs the kernel the plan names and matches the
    reference; the persistent kernels produce the qkv bias gradient themselves, in the same launch."""
    from vit_10b_fsdp_example_b200.ops import cuda_ops as co, torch_ops as to

    plan = ap.plan(N, hd)
    D = H * hd
    qkv = (torch.randn(B * N, 3 * D, device="cuda") * 0.7).to(torch.bfloat16)
    dout = torch.randn(B * N, D, device="cuda").to(torch.bfloat16)
    out, lse = co.attention_fwd_lse(qkv, B, N, H, hd)
    outr, lser = to.attention_fwd_lse(qkv.float(), B, N, H, hd)
    n0 = co.launch_count()
    (dqkv, cs), fams = _families(lambda: co.attention_bwd_lse(dout, qkv, out, lse, B, N, H, hd, want_colsum=True),
                                 BWD_FAMILY)
    assert fams == {BWD_FAMILY[plan.bwd]}
    if plan.bwd == ap.PERSIST:
        assert co.launch_count() - n0 == 1, "bias-gradient column sums must come out of the backward kernels themselves"
    dqkvr, csr = to.attention_bwd_lse(dout.float(), qkv.float(), outr, lser, B, N, H, hd, want_colsum=True)
    for name, sl in (("dq", slice(0, D)), ("dk", slice(D, 2 * D)), ("dv", slice(2 * D, 3 * D))):
        got, ref = dqkv[:, sl].float(), dqkvr[:, sl].float()
        err = (got - ref).abs().max().item() / (ref.abs().max().item() + 1e-6)
        assert err < 3e-2, f"{name}: rel err {err}"
    sums = dqkv.float().sum(dim=0)  # sums of the bf16 values that were stored
    assert (cs - sums).abs().max().item() <= 2e-3 * sums.abs().max().item() + 1e-3, "qkv bias gradient"
    if B * N < 1024:  # summed over many more rows, per-column bf16 noise can outgrow this bound; the check above holds
        _close(cs, csr, rel=5e-2)


@pytest.mark.parametrize("B,N,H,hd", [(1, 320, 2, 64), (1, 576, 2, 160), (2, 576, 2, 128)])
def test_fused_attention_long_sequence(B, N, H, hd):
    """Two-pass long-sequence forward + the fused backward at N > 256 (336 px config) vs the fp32 reference."""
    from vit_10b_fsdp_example_b200.ops import cuda_ops as co, torch_ops as to

    D = H * hd
    qkv = (torch.randn(B * N, 3 * D, device="cuda") * 0.7).to(torch.bfloat16)
    dout = torch.randn(B * N, D, device="cuda").to(torch.bfloat16)
    out, lse = co.attention_fwd_lse(qkv, B, N, H, hd)
    outr, lser = to.attention_fwd_lse(qkv.float(), B, N, H, hd)
    _close(out, outr)
    assert (lse - lser).abs().max().item() < 2e-2
    dqkv = co.attention_bwd_lse(dout, qkv, out, lse, B, N, H, hd)
    dqkvr = to.attention_bwd_lse(dout.float(), qkv.float(), outr, lser, B, N, H, hd)
    for name, sl in (("dq", slice(0, D)), ("dk", slice(D, 2 * D)), ("dv", slice(2 * D, 3 * D))):
        got, ref = dqkv[:, sl].float(), dqkvr[:, sl].float()
        err = (got - ref).abs().max().item() / (ref.abs().max().item() + 1e-6)
        assert err < 3e-2, f"{name}: rel err {err}"

