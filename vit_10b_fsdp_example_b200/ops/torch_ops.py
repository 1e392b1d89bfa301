"""Reference implementation of the functional op set in plain PyTorch.

This is (a) the CPU / gloo test backend, (b) the fp32 numerical oracle every sm_100a kernel is tested
against, and (c) the semantics contract for ``cuda_ops``.  Every function here has a same-named,
same-signature twin in ``cuda_ops`` that runs the hand-written kernels.

All matrices are 2-D ``[tokens, features]``; the model code does its own reshapes.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn.functional as F

NAME = "torch"


def _f32(t: torch.Tensor) -> torch.Tensor:
    return t if t.dtype == torch.float32 else t.float()


# ------------------------------------------------------------------------------------------------
# LayerNorm (timm Block.norm1 / norm2, final norm) -- reference run_vit_training.py:134-141,151
# ------------------------------------------------------------------------------------------------
def ln_fwd(x, w, b, eps: float):
    xf = _f32(x)
    mean = xf.mean(dim=-1)
    var = xf.var(dim=-1, unbiased=False)
    rstd = torch.rsqrt(var + eps)
    y = (xf - mean[:, None]) * rstd[:, None] * _f32(w) + _f32(b)
    return y.to(x.dtype), mean, rstd


def ln_bwd(dy, x, w, mean, rstd, dres=None, want_dxsum: bool = False):
    """Returns dx (= dres + LN backward), dw fp32, db fp32, colsum(dx) fp32 or None."""
    dyf, xf, wf = _f32(dy), _f32(x), _f32(w)
    xhat = (xf - mean[:, None]) * rstd[:, None]
    g = dyf * wf
    s1 = g.mean(dim=-1, keepdim=True)
    s2 = (g * xhat).mean(dim=-1, keepdim=True)
    dx = rstd[:, None] * (g - s1 - xhat * s2)
    if dres is not None:
        dx = dx + _f32(dres)
    dw = (dyf * xhat).sum(dim=0)
    db = dyf.sum(dim=0)
    dx = dx.to(x.dtype)
    dxsum = _f32(dx).sum(dim=0) if want_dxsum else None
    return dx, dw, db, dxsum


# ------------------------------------------------------------------------------------------------
# Linear layers (timm Attention.qkv / proj, Mlp.fc1 / fc2, head) and their backward
# ------------------------------------------------------------------------------------------------
def gelu(x):
    return F.gelu(x)  # exact erf form, like timm's nn.GELU


def gelu_fwd(u):
    return F.gelu(_f32(u)).to(u.dtype)


def dgelu_mul(dg, u):
    """du = dg * gelu'(u)  (exact erf GELU)."""
    return (_f32(dg) * dgelu(u)).to(dg.dtype)


def dgelu(u):
    uf = _f32(u)
    cdf = 0.5 * (1.0 + torch.erf(uf * (1.0 / math.sqrt(2.0))))
    pdf = torch.exp(-0.5 * uf * uf) * (1.0 / math.sqrt(2.0 * math.pi))
    return cdf + uf * pdf


def linear_fwd(x, w, bias=None, act: Optional[str] = None, residual=None, res_row_mod: int = 0,
               want_preact: bool = False, ag=None):
    """y = act(x @ w.T + bias) + residual.  residual rows may be broadcast with period res_row_mod."""
    y = _f32(x) @ _f32(w).t()
    if bias is not None:
        y = y + _f32(bias)
    pre = y.to(x.dtype) if want_preact else None
    if act == "gelu":
        y = gelu(y)
    elif act is not None:
        raise ValueError(act)
    if residual is not None:
        r = _f32(residual)
        if res_row_mod:
            reps = y.shape[0] // res_row_mod
            r = r[:res_row_mod].repeat(reps, 1)
        y = y + r
    y = y.to(x.dtype)
    return (y, pre) if want_preact else y


def linear_dgrad(dy, w, dgelu_preact=None, want_colsum: bool = False):
    """dx = dy @ w  (optionally  * gelu'(preact)); colsum(dx) is the bias grad of the layer below."""
    dx = _f32(dy) @ _f32(w)
    if dgelu_preact is not None:
        dx = dx * dgelu(dgelu_preact)
    dx = dx.to(dy.dtype)
    cs = _f32(dx).sum(dim=0) if want_colsum else None
    return (dx, cs) if want_colsum else dx


def linear_wgrad(dy, x, out=None):
    """dw[N, K] = dy[T, N].T @ x[T, K]"""
    dw = _f32(dy).t() @ _f32(x)
    if out is not None:
        out.copy_(dw)
        return out
    return dw.to(dy.dtype)


def colsum(x):
    return _f32(x).sum(dim=0)


# ------------------------------------------------------------------------------------------------
# Attention core (timm Attention: softmax(q k^T * hd^-0.5) v, no mask) -- run_vit_training.py:134
# qkv is the packed [T, 3*D] projection; head h of q lives at columns [h*hd, (h+1)*hd).
# ------------------------------------------------------------------------------------------------
def dropout(x, p: float, key: int):
    """y = x * keep / (1 - p); keep is a pure function of (key, position), so the checkpoint recompute and the
    backward pass regenerate it instead of storing it (reference: nn.Dropout inside timm Block / after pos_embed,
    run_vit_training.py:129,138-139)."""
    gen = torch.Generator(device=x.device)
    gen.manual_seed(int(key) & 0x7FFFFFFFFFFFFFFF)
    keep = torch.rand(x.shape, generator=gen, device=x.device) >= p
    return (x.float() * keep * (1.0 / (1.0 - p))).to(x.dtype)


def mean_pool(xn, B: int, N: int):
    """[B*N, D] -> [B, D]: mean over the tokens of an image (run_vit_training.py:161)."""
    return xn.view(B, N, -1).mean(dim=1, dtype=torch.float32).to(xn.dtype)


def mean_pool_bwd(dpooled, B: int, N: int):
    """d(mean over tokens): every token row of image b receives dpooled[b] / N."""
    D = dpooled.shape[1]
    return (dpooled.float() / N).to(dpooled.dtype)[:, None, :].expand(B, N, D).reshape(B * N, D)


def attention_fwd(qkv, B: int, N: int, H: int, hd: int, drop=None, need_p: bool = True):
    """drop = (p, key): attention dropout on the probabilities (timm Attention.attn_drop)."""
    D = H * hd
    q, k, v = _f32(qkv).view(B, N, 3, H, hd).permute(2, 0, 3, 1, 4)  # [B, H, N, hd]
    s = (q @ k.transpose(-1, -2)) * (hd ** -0.5)
    p = torch.softmax(s, dim=-1).to(qkv.dtype)
    pd = p if drop is None else dropout(p, drop[0], drop[1])
    o = (_f32(pd) @ v).permute(0, 2, 1, 3).reshape(B * N, D).to(qkv.dtype)
    return o, p


# Flash-style pair: the forward keeps only the log-sum-exp of every score row, the backward rebuilds P from it
# (csrc/attention_bwd_sm100.cu on the GPU).  Off by default; tests flip FLASH_ATTENTION to exercise the model path.
FLASH_ATTENTION = False


def use_flash(N: int, hd: int) -> bool:
    return FLASH_ATTENTION


def attention_fwd_lse(qkv, B: int, N: int, H: int, hd: int):
    D = H * hd
    q, k, v = _f32(qkv).view(B, N, 3, H, hd).permute(2, 0, 3, 1, 4)
    s = (q @ k.transpose(-1, -2)) * (hd ** -0.5)
    lse = torch.logsumexp(s, dim=-1)  # [B, H, N]
    o = (torch.exp(s - lse[..., None]) @ v).permute(0, 2, 1, 3).reshape(B * N, D).to(qkv.dtype)
    return o, lse.reshape(B * H, N).contiguous()


def attention_bwd_lse(dout, qkv, out, lse, B: int, N: int, H: int, hd: int, want_colsum: bool = False):
    D = H * hd
    q, k, v = _f32(qkv).view(B, N, 3, H, hd).permute(2, 0, 3, 1, 4)
    do = _f32(dout).view(B, N, H, hd).permute(0, 2, 1, 3)
    o = _f32(out).view(B, N, H, hd).permute(0, 2, 1, 3)
    p = torch.exp((q @ k.transpose(-1, -2)) * (hd ** -0.5) - lse.view(B, H, N, 1))
    delta = (do * o).sum(dim=-1, keepdim=True)
    dv = p.transpose(-1, -2) @ do
    ds = (hd ** -0.5) * p * (do @ v.transpose(-1, -2) - delta)
    dq = ds @ k
    dk = ds.transpose(-1, -2) @ q
    dqkv = torch.stack([dq, dk, dv], dim=0).permute(1, 3, 0, 2, 4).reshape(B * N, 3 * D).to(qkv.dtype)
    cs = _f32(dqkv).sum(dim=0) if want_colsum else None
    return (dqkv, cs) if want_colsum else dqkv


def attention_probs(qkv, B: int, N: int, H: int, hd: int):
    """P alone (re-materialised in backward when only qkv was kept)."""
    q, k, _ = _f32(qkv).view(B, N, 3, H, hd).permute(2, 0, 3, 1, 4)
    return torch.softmax((q @ k.transpose(-1, -2)) * (hd ** -0.5), dim=-1).to(qkv.dtype)


def attention_bwd(dout, qkv, p, B: int, N: int, H: int, hd: int, want_colsum: bool = False, drop=None):
    D = H * hd
    q, k, v = _f32(qkv).view(B, N, 3, H, hd).permute(2, 0, 3, 1, 4)
    do = _f32(dout).view(B, N, H, hd).permute(0, 2, 1, 3)  # [B, H, N, hd]
    pf = _f32(p)
    pdrop = pf if drop is None else dropout(p, drop[0], drop[1]).float()
    dv = pdrop.transpose(-1, -2) @ do
    dp = (do @ v.transpose(-1, -2)).to(qkv.dtype)
    if drop is not None:
        dp = dropout(dp, drop[0], drop[1])  # same key, same shape -> same mask
    dp = dp.float()
    ds = (hd ** -0.5) * pf * (dp - (dp * pf).sum(dim=-1, keepdim=True))
    ds = ds.to(qkv.dtype).float()
    dq = ds @ k
    dk = ds.transpose(-1, -2) @ q
    dqkv = torch.stack([dq, dk, dv], dim=0).permute(1, 3, 0, 2, 4).reshape(B * N, 3 * D).to(qkv.dtype)
    cs = _f32(dqkv).sum(dim=0) if want_colsum else None
    return (dqkv, cs) if want_colsum else dqkv


# ------------------------------------------------------------------------------------------------
# Patch embedding (timm PatchEmbed = Conv2d(k=s=P)) as im2col + GEMM -- run_vit_training.py:124,156
# ------------------------------------------------------------------------------------------------
def patch_im2col(images, P: int, kpad: int, dtype):
    B, C, S, _ = images.shape
    G = S // P
    cols = images.view(B, C, G, P, G, P).permute(0, 2, 4, 1, 3, 5).reshape(B * G * G, C * P * P)
    out = torch.zeros(B * G * G, kpad, dtype=dtype, device=images.device)
    out[:, : C * P * P] = cols.to(dtype)
    return out


# ------------------------------------------------------------------------------------------------
# Loss (torch.nn.CrossEntropyLoss, mean) -- run_vit_training.py:229,262 ; eval argmax -- :312-313
# ------------------------------------------------------------------------------------------------
def cross_entropy(logits, target, want_grad: bool = True):
    lf = _f32(logits)
    lse = torch.logsumexp(lf, dim=-1)
    picked = lf.gather(1, target.view(-1, 1)).squeeze(1)
    loss = (lse - picked).mean()
    dlogits = None
    if want_grad:
        prob = torch.exp(lf - lse[:, None])
        prob[torch.arange(lf.shape[0], device=lf.device), target] -= 1.0
        dlogits = (prob / lf.shape[0]).to(logits.dtype)
    correct = (lf.argmax(dim=-1) == target).sum()
    return loss, dlogits, correct


# ------------------------------------------------------------------------------------------------
# Optimizer pieces (torch.optim.AdamW + clip_grad_norm_) -- run_vit_training.py:237,270,278
# ------------------------------------------------------------------------------------------------
def sumsq(x, out):
    out += _f32(x).pow(2).sum()


def clip_coef(sumsq_t, max_norm: float):
    norm = torch.sqrt(sumsq_t)
    return torch.clamp(max_norm / (norm + 1e-6), max=1.0), norm


def adamw_fp32(w, m, v, grad, clip, lr, beta1, beta2, eps, wd, step: int):
    g = _f32(grad)
    if clip is not None:
        g = g * clip
    m.mul_(beta1).add_(g, alpha=1.0 - beta1)
    v.mul_(beta2).addcmul_(g, g, value=1.0 - beta2)
    bc1 = 1.0 - beta1 ** step
    bc2 = 1.0 - beta2 ** step
    w.mul_(1.0 - lr * wd)
    denom = (v / bc2).sqrt_().add_(eps)
    w.addcdiv_(m / bc1, denom, value=-lr)


# Split fp32 master representation: fp32 bits == (hi_bf16_bits << 16) + lo_int16, hi = nearest bf16
# (ties round up in the bit pattern so that lo always fits a signed 16-bit integer).
def split_fp32(w, hi, lo):
    bits = w.contiguous().view(torch.int32)
    rounded = bits + 0x8000  # round-half-up keeps lo within int16 for every input (ties included)
    h = rounded >> 16
    hi.copy_((h << 16).view(torch.float32).to(torch.bfloat16))
    lo.copy_((bits - (h << 16)).to(torch.int16))


def merge_fp32(hi, lo, w):
    bits = (hi.view(torch.int16).to(torch.int32) << 16) + lo.to(torch.int32)
    w.copy_(bits.view(torch.float32))


def adamw_split(hi, lo, m, v, grad, clip, lr, beta1, beta2, eps, wd, step: int, hyper=None):
    w = torch.empty(hi.shape, dtype=torch.float32, device=hi.device)
    merge_fp32(hi, lo, w)
    adamw_fp32(w, m, v, grad, clip, lr, beta1, beta2, eps, wd, step)
    split_fp32(w, hi, lo)
