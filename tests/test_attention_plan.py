"""The attention kernel selection (ops/attention_plan.py) over a grid of shapes, stated as a table independent of the
implementation.  CPU only: the plan module imports neither torch's CUDA side nor the extension."""
import pytest

from vit_10b_fsdp_example_b200.ops import attention_plan as ap

HEAD_DIMS = (32, 64, 80, 128, 160, 256)
SEQ_LENS = range(2, 1101)  # every even and odd N, across the 128 / 256 / 1024 boundaries


def expected(N, hd):
    """(fwd_lse, fwd, bwd) for one shape: the table in the module docstring, row by row."""
    ok = hd in (64, 128, 160) and N % 2 == 0
    if not ok or N > 1024:
        return None, "unfused", None
    if hd <= 128:
        if N <= 256:
            return "oneshot", "oneshot", "oneshot"
        return "long", "unfused", "oneshot"
    bwd = "persist" if N % 4 == 0 else "oneshot"
    if N <= 128:
        return "oneshot", "unfused", bwd
    if N <= 256:
        return "persist", "persist", bwd
    return "long", "unfused", bwd


@pytest.mark.parametrize("hd", HEAD_DIMS)
def test_plan_matches_the_table(hd):
    for N in SEQ_LENS:
        p = ap.plan(N, hd)
        assert (p.fwd_lse, p.fwd, p.bwd) == expected(N, hd), (N, hd)


def test_plan_shapes_the_models_run():
    """ViT-L/16 (N 196, hd 64), ViT-10B (N 256, hd 160), its 336 px variant (N 576) and a 112 px one (N 64)."""
    assert ap.plan(196, 64) == ap.AttentionPlan(ap.ONESHOT, ap.ONESHOT, ap.ONESHOT)
    assert ap.plan(256, 160) == ap.AttentionPlan(ap.PERSIST, ap.PERSIST, ap.PERSIST)
    assert ap.plan(576, 160) == ap.AttentionPlan(ap.LONG, ap.UNFUSED, ap.PERSIST)
    assert ap.plan(64, 160) == ap.AttentionPlan(ap.ONESHOT, ap.UNFUSED, ap.PERSIST)


def test_a_fused_forward_always_comes_with_a_fused_backward():
    for hd in HEAD_DIMS:
        for N in SEQ_LENS:
            p = ap.plan(N, hd)
            assert (p.fwd_lse is None) == (p.bwd is None), (N, hd)


def test_plan_is_frozen():
    with pytest.raises(AttributeError):
        ap.plan(256, 160).fwd = ap.UNFUSED
