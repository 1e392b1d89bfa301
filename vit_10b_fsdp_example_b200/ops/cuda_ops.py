"""sm_100a implementation of the functional op set (same contract as ``torch_ops``).

Every function launches hand-written kernels from ``_C.so``:
  * GEMMs: persistent 2-CTA tcgen05 kernel with TMEM accumulators and fused epilogues
    (bias / GELU / dGELU / residual / pre-activation side output / bias-gradient column sums);
    forward (NT), dgrad (NN) and wgrad (TN) run on the same kernel via K-major / MN-major descriptors.
  * attention core: fused tcgen05 forward (keeps the row log-sum-exp) + fused backward kernels that read q/k/v in
    place from the packed qkv buffer through 4-D TMA tensor maps; scores never reach HBM.  The un-fused path (batched
    tcgen05 GEMMs + softmax / softmax-backward kernels with materialised P) serves attention dropout and the shapes
    the fused kernels do not cover.  Which kernel runs for a shape is decided in one place: ``attention_plan.plan``.
  * LayerNorm fwd/bwd, cross-entropy, im2col, column sums, sum of squares, fused AdamW.

What each group replaces in the reference (all of it reached through timm / torch_xla there):
  linear_fwd / dgrad / wgrad      nn.Linear in timm Attention.qkv / proj, Mlp.fc1 / fc2, the head (run_vit_training.py:134-141,153)
  attention_fwd / attention_bwd   timm Attention's softmax(q k^T * hd^-0.5) v with materialised scores (:134)
  ln_fwd / ln_bwd                 nn.LayerNorm in timm Block (eps 1e-5) and the final norm (:151, eps 1e-6)
  patch_im2col + linear_fwd       timm PatchEmbed conv k = s = P plus the pos_embed add (:124-129,156)
  cross_entropy                   nn.CrossEntropyLoss (:229,262) and the eval argmax/eq (:312-313)
  adamw_* / sumsq / clip_coef     torch.optim.AdamW (:237,278) and FSDP.clip_grad_norm_ (:270)

bf16 activations / weights, fp32 accumulation and statistics.  There is no PyTorch fallback here: if the
extension is missing this module fails to import on purpose.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import attention_plan, native
from .attention_plan import LONG, ONESHOT, PERSIST

NAME = "sm100"


class _CountingModule:
    """Proxy over the native module that counts kernel launches (every entry point launches exactly one
    hand-written kernel); ``launch_count()`` feeds the ``gpu_launches`` field of bench.py."""

    def __init__(self, mod):
        object.__setattr__(self, "_mod", mod)
        object.__setattr__(self, "count", 0)

    def __getattr__(self, name):
        fn = getattr(self._mod, name)
        if not callable(fn):
            return fn

        def wrapped(*a, **k):
            object.__setattr__(self, "count", self.count + 1)
            return fn(*a, **k)

        object.__setattr__(self, name, wrapped)
        return wrapped


_C = _CountingModule(native.load())


def launch_count() -> int:
    return _C.count

ACT_NONE, ACT_GELU, ACT_DGELU = 0, 1, 2
# GELU / dGELU are fused into the GEMM epilogue only when the reduction is deep enough to hide the math
# (ViT-10B: K = 5120 fused; ViT-L: K = 1024 -> plain GEMM + stand-alone elementwise kernel, measured 1.5x faster)
import os as _os

FUSE_ACT_MIN_K = int(_os.environ.get("B200_FUSE_ACT_MIN_K", "2048"))

# SM carve-out for compute kernels while a communication kernel runs next to them (0 = all SMs).
_max_ctas = 0


def set_compute_max_ctas(n: int) -> None:
    global _max_ctas
    _max_ctas = int(n)


def _ld(t: torch.Tensor) -> int:
    assert t.dim() == 2 and t.stride(1) == 1, "expected a row-major 2-D (possibly strided) matrix"
    return t.stride(0)


def _pad8(n: int) -> int:
    return (n + 7) // 8 * 8


def _tma_rows(t: torch.Tensor) -> torch.Tensor:
    """TMA needs 16-byte row strides and base.  Matrices whose width is not a multiple of 8 (e.g. a classifier
    with an odd class count) are copied into a zero-padded buffer and used through a strided view."""
    if t.stride(1) == 1 and t.stride(0) % 8 == 0 and t.data_ptr() % 16 == 0:
        return t
    rows, cols = t.shape
    buf = torch.zeros(rows, _pad8(cols), dtype=t.dtype, device=t.device)
    buf[:, :cols].copy_(t)
    return buf[:, :cols]


def _bias_ok(b: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    """The epilogue reads bias in 16-byte vectors: pad odd-length biases so the tail read stays in bounds."""
    if b is None or b.numel() % 8 == 0:
        return b
    buf = torch.zeros(_pad8(b.numel()), dtype=b.dtype, device=b.device)
    buf[: b.numel()].copy_(b)
    return buf


def gemm_raw(a, lda, major_a, b, ldb, major_b, d, ldd, M, N, K, *, bias=None, residual=None, ld_res=0,
             res_row_mod=0, aux_in=None, ld_aux=0, aux_out=None, ld_aux_out=0, colsum=None, colsum_bi_stride=0,
             act=ACT_NONE, batch=(), block_n=0, max_ctas=None, ag=()):
    _C.gemm(a, lda, major_a, b, ldb, major_b, d, ldd, M, N, K, bias, residual, ld_res, res_row_mod, aux_in, ld_aux,
            aux_out, ld_aux_out, colsum, colsum_bi_stride, act, list(batch), block_n,
            _max_ctas if max_ctas is None else max_ctas, list(ag))


# ------------------------------------------------------------------------------------------------
# LayerNorm
# ------------------------------------------------------------------------------------------------
def ln_fwd(x, w, b, eps: float):
    rows = x.shape[0]
    y = torch.empty_like(x)
    mean = torch.empty(rows, dtype=torch.float32, device=x.device)
    rstd = torch.empty(rows, dtype=torch.float32, device=x.device)
    _C.layernorm_fwd(x, w, b, y, mean, rstd, eps)
    return y, mean, rstd


def ln_bwd(dy, x, w, mean, rstd, dres=None, want_dxsum: bool = False):
    D = x.shape[1]
    dx = torch.empty_like(x)
    acc = torch.zeros(3 if want_dxsum else 2, D, dtype=torch.float32, device=x.device)
    _C.layernorm_bwd(dy, x, w, mean, rstd, dres, dx, acc[0], acc[1], acc[2] if want_dxsum else None)
    return dx, acc[0], acc[1], (acc[2] if want_dxsum else None)


# ------------------------------------------------------------------------------------------------
# Linear
# ------------------------------------------------------------------------------------------------
def linear_fwd(x, w, bias=None, act: Optional[str] = None, residual=None, res_row_mod: int = 0,
               want_preact: bool = False, ag=None):
    """ag: optional all-gather fusion spec (see Sm100Backend.ag_fuse_spec): the kernel itself pulls the peers'
    shards of `w` over NVLink while it computes."""
    M, K = x.shape
    N = w.shape[0]
    if act == "gelu" and K < FUSE_ACT_MIN_K and N % 8 == 0 and ag is None:
        # short K: the activation math would not fit under a tile's MMA time -> plain GEMM + memory-bound GELU
        pre = linear_fwd(x, w, bias, residual=None)
        y = torch.empty_like(pre)
        _C.gelu_fwd(pre, y)
        if residual is not None:
            y += residual
        return (y, pre) if want_preact else y
    x, w = _tma_rows(x), _tma_rows(w)
    ldy = _pad8(N)
    y = torch.empty(M, ldy, dtype=x.dtype, device=x.device)
    pre = torch.empty(M, ldy, dtype=x.dtype, device=x.device) if want_preact else None
    gemm_raw(x, _ld(x), 0, w, _ld(w), 0, y, ldy, M, N, K, bias=_bias_ok(bias), residual=residual,
             ld_res=_ld(residual) if residual is not None else 0, res_row_mod=res_row_mod, aux_out=pre,
             ld_aux_out=ldy, act=ACT_GELU if act == "gelu" else ACT_NONE, ag=ag or ())
    if ldy != N:
        y = y[:, :N].contiguous()
        pre = pre[:, :N].contiguous() if pre is not None else None
    return (y, pre) if want_preact else y


def linear_dgrad(dy, w, dgelu_preact=None, want_colsum: bool = False):
    M, N = dy.shape
    K = w.shape[1]
    if dgelu_preact is not None and N < FUSE_ACT_MIN_K and K % 8 == 0:
        dx = linear_dgrad(dy, w)
        _C.dgelu_mul(dx, dgelu_preact, dx)
        if want_colsum:
            return dx, colsum(dx)
        return dx
    dy, w = _tma_rows(dy), _tma_rows(w)
    dx = torch.empty(M, K, dtype=dy.dtype, device=dy.device)
    cs = torch.zeros(K, dtype=torch.float32, device=dy.device) if want_colsum else None
    gemm_raw(dy, _ld(dy), 0, w, _ld(w), 1, dx, K, M, K, N, aux_in=dgelu_preact,
             ld_aux=_ld(dgelu_preact) if dgelu_preact is not None else 0,
             act=ACT_DGELU if dgelu_preact is not None else ACT_NONE, colsum=cs)
    return (dx, cs) if want_colsum else dx


def linear_wgrad(dy, x, out=None, block_n: int = 0):
    T, N = dy.shape
    K = x.shape[1]
    dy, x = _tma_rows(dy), _tma_rows(x)
    if out is None:
        out = torch.empty(N, K, dtype=dy.dtype, device=dy.device)
    gemm_raw(dy, _ld(dy), 1, x, _ld(x), 1, out, _ld(out), N, K, T, block_n=block_n)
    return out


def gelu_fwd(u):
    g = torch.empty_like(u)
    _C.gelu_fwd(u, g)
    return g


def dgelu_mul(dg, u):
    du = torch.empty_like(dg)
    _C.dgelu_mul(dg.contiguous(), u, du)
    return du


def colsum(x):
    out = torch.zeros(x.shape[1], dtype=torch.float32, device=x.device)
    _C.colsum(x, out)
    return out


# ------------------------------------------------------------------------------------------------
# Attention core
# ------------------------------------------------------------------------------------------------
def dropout(x, p: float, key: int):
    """Philox-keyed dropout kernel (csrc/elementwise.cu): the mask is a function of (key, position), never stored."""
    xc = x.contiguous()
    assert xc.numel() % 8 == 0, "dropout kernel works on whole 16-byte vectors"
    y = torch.empty_like(xc)
    _C.dropout(xc, y, float(p), int(key) & 0x7FFFFFFFFFFFFFFF)
    return y


def mean_pool(xn, B: int, N: int):
    pooled = torch.empty(B, xn.shape[1], dtype=xn.dtype, device=xn.device)
    _C.meanpool_fwd(xn, pooled, B, N)
    return pooled


def mean_pool_bwd(dpooled, B: int, N: int):
    dxn = torch.empty(B * N, dpooled.shape[1], dtype=dpooled.dtype, device=dpooled.device)
    _C.meanpool_bwd(dpooled.contiguous(), dxn, B, N)
    return dxn


def attention_fwd(qkv, B: int, N: int, H: int, hd: int, drop=None, need_p: bool = True):
    """Returns (out [B*N, D], P).  P = softmax probabilities [B*H, N, ldp] for the backward, or None when a fused
    kernel ran (scores never reach HBM then); need_p=True always takes the un-fused path.
    drop = (p, key): attention dropout.  The probabilities are materialised (un-fused path), the dropped copy that
    feeds P V comes from the Philox dropout kernel; the returned P is the un-dropped one (backward regenerates the mask)."""
    D = H * hd
    out = torch.empty(B * N, D, dtype=qkv.dtype, device=qkv.device)
    kernel = None if (need_p or drop is not None) else attention_plan.plan(N, hd).fwd
    if kernel == PERSIST:
        _C.attention_fwd_persist(qkv, out, None, B, N, H, hd)
        return out, None
    if kernel == ONESHOT:
        _C.attention_fwd(qkv, out, None, B, N, H, hd)
        return out, None
    p = attention_probs(qkv, B, N, H, hd)
    pv = p if drop is None else dropout(p, drop[0], drop[1])
    ldp, ld3 = p.shape[2], qkv.stride(0)
    # O = P V  (V is MN-major: head-dim contiguous, keys strided)
    gemm_raw(pv, ldp, 0, qkv[:, 2 * D:], ld3, 1, out, D, N, hd, N,
             batch=(H, B, N * ldp, H * N * ldp, hd, N * ld3, hd, N * D))
    return out, p


def use_flash(N: int, hd: int) -> bool:
    """Model-level policy: run the attention core through the fused forward (log-sum-exp) + fused backward pair?"""
    return attention_plan.plan(N, hd).fwd_lse is not None


def attention_fwd_lse(qkv, B: int, N: int, H: int, hd: int):
    kernel = attention_plan.plan(N, hd).fwd_lse
    out = torch.empty(B * N, H * hd, dtype=qkv.dtype, device=qkv.device)
    lse = torch.empty(B * H, N, dtype=torch.float32, device=qkv.device)
    if kernel == PERSIST:
        _C.attention_fwd_persist(qkv, out, lse, B, N, H, hd)
    elif kernel == ONESHOT:
        _C.attention_fwd(qkv, out, lse, B, N, H, hd)
    elif kernel == LONG:
        _C.attention_fwd_long(qkv, out, lse, B, N, H, hd)
    else:
        raise ValueError(f"no fused attention forward for N={N}, hd={hd}")
    return out, lse


def attention_bwd_lse(dout, qkv, out, lse, B: int, N: int, H: int, hd: int, want_colsum: bool = False):
    kernel = attention_plan.plan(N, hd).bwd
    if kernel not in (ONESHOT, PERSIST):
        raise ValueError(f"no fused attention backward for N={N}, hd={hd}")
    persist = kernel == PERSIST
    dqkv = torch.empty(B * N, 3 * H * hd, dtype=qkv.dtype, device=qkv.device)
    # scratch: rowsum(dO o O); the persistent kernels get a second plane holding lse * log2(e)
    delta = torch.empty(2 if persist else 1, B * H, N, dtype=torch.float32, device=qkv.device)
    # the persistent kernels reduce the qkv bias gradient (column sums of dq | dk | dv) from their epilogue tiles
    cs = torch.zeros(3 * H * hd, dtype=torch.float32, device=qkv.device) if (want_colsum and persist) else None
    _C.attention_bwd(qkv, dout, out, lse, delta, dqkv, cs, B, N, H, hd, persist)
    if want_colsum and cs is None:
        cs = colsum(dqkv)
    return (dqkv, cs) if want_colsum else dqkv


def attention_probs(qkv, B: int, N: int, H: int, hd: int):
    """P = softmax(Q K^T / sqrt(hd)) alone: re-materialised in backward for blocks that kept only qkv."""
    D = H * hd
    ldp = _pad8(N)
    p = torch.empty(B * H, N, ldp, dtype=qkv.dtype, device=qkv.device)
    if ldp != N:
        p[:, :, N:].zero_()
    ld3 = qkv.stride(0)
    gemm_raw(qkv[:, :D], ld3, 0, qkv[:, D:2 * D], ld3, 0, p, ldp, N, N, hd,
             batch=(H, B, hd, N * ld3, hd, N * ld3, N * ldp, H * N * ldp))
    _C.softmax_fwd(p, B * H * N, N, ldp, hd ** -0.5)
    return p


def attention_bwd(dout, qkv, p, B: int, N: int, H: int, hd: int, want_colsum: bool = False, drop=None):
    """drop = (p, key) of the forward: the dropped probabilities (for dV) and the mask on dP are regenerated."""
    D = H * hd
    ldp = p.shape[2]
    ld3 = qkv.stride(0)
    q, k, v = qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:]
    dqkv = torch.empty(B * N, 3 * D, dtype=qkv.dtype, device=qkv.device)
    dq, dk, dv = dqkv[:, :D], dqkv[:, D:2 * D], dqkv[:, 2 * D:]
    cs = torch.zeros(3 * D, dtype=torch.float32, device=qkv.device) if want_colsum else None
    ldo = dout.stride(0)
    bp = (N * ldp, H * N * ldp)      # batch strides of P-shaped buffers
    bq = (hd, N * ld3)               # ... of q/k/v inside qkv
    bo = (hd, N * ldo)
    bd = (hd, N * 3 * D)             # ... of dq/dk/dv inside dqkv
    # dV = P^T dO   (with attention dropout: the dropped P that fed the forward P V)
    pv = p if drop is None else dropout(p, drop[0], drop[1])
    gemm_raw(pv, ldp, 1, dout, ldo, 1, dv, 3 * D, N, hd, N, batch=(H, B, *bp, *bo, *bd),
             colsum=cs[2 * D:] if want_colsum else None, colsum_bi_stride=hd)
    del pv
    # dP = dO V^T
    dp = torch.empty_like(p)
    if ldp != N:
        dp[:, :, N:].zero_()
    gemm_raw(dout, ldo, 0, v, ld3, 0, dp, ldp, N, N, hd, batch=(H, B, *bo, *bq, *bp))
    if drop is not None:
        _C.dropout(dp, dp, float(drop[0]), int(drop[1]) & 0x7FFFFFFFFFFFFFFF)  # same key and shape -> same mask
    # dS = scale * P * (dP - rowsum(dP * P))   (in place)
    _C.softmax_bwd(dp, p, B * H * N, N, ldp, hd ** -0.5)
    # dQ = dS K ; dK = dS^T Q
    gemm_raw(dp, ldp, 0, k, ld3, 1, dq, 3 * D, N, hd, N, batch=(H, B, *bp, *bq, *bd),
             colsum=cs[:D] if want_colsum else None, colsum_bi_stride=hd)
    gemm_raw(dp, ldp, 1, q, ld3, 1, dk, 3 * D, N, hd, N, batch=(H, B, *bp, *bq, *bd),
             colsum=cs[D:2 * D] if want_colsum else None, colsum_bi_stride=hd)
    return (dqkv, cs) if want_colsum else dqkv


# ------------------------------------------------------------------------------------------------
# Patch embedding, loss
# ------------------------------------------------------------------------------------------------
def patch_im2col(images, P: int, kpad: int, dtype):
    B, _, S, _ = images.shape
    G = S // P
    cols = torch.empty(B * G * G, kpad, dtype=dtype, device=images.device)
    _C.im2col(images.contiguous(), cols, P)
    return cols


def cross_entropy(logits, target, want_grad: bool = True):
    loss = torch.zeros(1, dtype=torch.float32, device=logits.device)
    correct = torch.zeros(1, dtype=torch.int32, device=logits.device)
    dlogits = torch.empty_like(logits) if want_grad else None
    _C.cross_entropy(logits, target, dlogits, loss, correct)
    return loss[0], dlogits, correct[0]


# ------------------------------------------------------------------------------------------------
# Optimizer pieces
# ------------------------------------------------------------------------------------------------
def sumsq(x, out):
    _C.sumsq(x, out)


def clip_coef(sumsq_t, max_norm: float):
    coef = torch.empty(1, dtype=torch.float32, device=sumsq_t.device)
    norm = torch.empty(1, dtype=torch.float32, device=sumsq_t.device)
    _C.clip_coef(sumsq_t, max_norm, coef, norm)
    return coef, norm


def adamw_fp32(w, m, v, grad, clip, lr, beta1, beta2, eps, wd, step: int):
    _C.adamw_fp32(w, m, v, grad, clip, lr, beta1, beta2, eps, wd, step)


def adamw_split(hi, lo, m, v, grad, clip, lr, beta1, beta2, eps, wd, step: int, hyper=None):
    """hyper: optional device tensor [lr, step] that overrides the host scalars (CUDA-graph replay)."""
    _C.adamw_split(hi, lo, m, v, grad, clip, lr, beta1, beta2, eps, wd, step, hyper)


def split_fp32(w, hi, lo):
    _C.split_fp32(w, hi, lo)


def merge_fp32(hi, lo, w):
    _C.merge_fp32(hi, lo, w)
