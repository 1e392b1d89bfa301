"""Which attention kernels run for a sequence length N and a head dim hd.

``plan(N, hd)`` is the whole policy; ``cuda_ops`` dispatches on its fields and nothing else.  It needs no GPU and
no extension, so the CPU suite states it (tests/test_attention_plan.py).  Let "ok" mean hd in {64, 128, 160} and
N even:

  shape                           fwd_lse (saved block)  fwd (checkpointed block, eval)  bwd (from the lse)
  ok, hd <= 128, N <= 256         oneshot                oneshot                         oneshot
  ok, hd <= 128, 256 < N <= 1024  long                   unfused                         oneshot
  ok, hd = 160, N <= 128          oneshot                unfused                         persist (oneshot if N % 4 == 2)
  ok, hd = 160, 128 < N <= 256    persist                persist                         persist (oneshot if N % 4 == 2)
  ok, hd = 160, 256 < N <= 1024   long                   unfused                         persist (oneshot if N % 4 == 2)
  not ok, or N > 1024             None                   unfused                         None

fwd_lse is None: the model keeps (or re-materialises) P and runs the un-fused backward (``cuda_ops.use_flash`` is
false).  Attention dropout is outside this table: with it on, every shape runs the un-fused forward and backward,
which materialise P and regenerate the dropout mask.

Kernels (csrc/):  oneshot = attn_fwd_sm100 (forward, N <= 256) / attn_bwd_sm100 (backward, N <= 1024);
long = attn_fwd_long_sm100; persist = attn_fwd_persist_sm100 / attn_bwd_persist_sm100, instantiated for hd = 160
only (they need N % 4 == 0 in backward to bulk-copy per-row statistics in 16-byte units); unfused = batched GEMMs
around softmax_fwd.

Why, measured on a B200 (profiles/r2_attention.md):
  * hd <= 128: two CTAs of the one-shot kernels fit an SM; the persistent kernels lose there (hd = 64: 254 vs
    159 us).  ViT-L (B128 N196 H16 hd64): fused 159 + 387 us vs un-fused 279 + 500 + 204 us.
  * hd = 160: one CTA per SM (200 KB of shared memory); the persistent kernels win (ViT-10B, B128 N256 H32:
    forward 311 vs 763 us one-shot, 664 us un-fused; backward 1352 vs 1814 us one-shot).  The one-shot forward
    loses to the un-fused one there, so at N <= 128 it runs only where it feeds the fused backward.
  * N > 256 (336 px, B56 N576 H32 hd160): the forward that feeds the backward is the long kernel (1584 us), the
    P-less forward stays un-fused (1424 us); the pair also saves 1.2 GB of P per block.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

ONESHOT, LONG, PERSIST, UNFUSED = "oneshot", "long", "persist", "unfused"

MAX_FUSED_N = 1024  # the one-shot backward keeps the dK/dV role's column statistics in shared memory


@dataclass(frozen=True)
class AttentionPlan:
    fwd_lse: Optional[str]  # forward that keeps the row log-sum-exp (ONESHOT / LONG / PERSIST), None: keep P instead
    fwd: str                # forward without it (ONESHOT / PERSIST / UNFUSED)
    bwd: Optional[str]      # backward from the log-sum-exp (ONESHOT / PERSIST), None when fwd_lse is None


def plan(N: int, hd: int) -> AttentionPlan:
    if hd not in (64, 128, 160) or N % 2 != 0 or N > MAX_FUSED_N:
        return AttentionPlan(None, UNFUSED, None)
    if hd <= 128:
        if N <= 256:
            return AttentionPlan(ONESHOT, ONESHOT, ONESHOT)
        return AttentionPlan(LONG, UNFUSED, ONESHOT)
    bwd = PERSIST if N % 4 == 0 else ONESHOT
    if N <= 128:
        return AttentionPlan(ONESHOT, UNFUSED, bwd)
    if N <= 256:
        return AttentionPlan(PERSIST, PERSIST, bwd)
    return AttentionPlan(LONG, UNFUSED, bwd)
