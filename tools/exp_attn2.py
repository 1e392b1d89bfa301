"""Attention variants at the headline shapes: un-fused (batched GEMMs + softmax kernels), one-shot fused, long,
persistent fused (hd = 160); forward and backward.  Every variant is launched through its own extension entry point,
whatever ops/attention_plan.py would choose.  CUDA-event timing, inputs >> L2 (qkv is 1 GB at the ViT-10B shape).

    python tools/exp_attn2.py [--shapes 10b,l,336] [--json gpurun_out/attn_times.json]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vit_10b_fsdp_example_b200.ops import cuda_ops as co  # noqa: E402

SHAPES = {"10b": (128, 256, 32, 160), "l": (128, 196, 16, 64), "336": (56, 576, 32, 160)}


def timeit(fn, n=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(n):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / n * 1e3


def guarded(name, fn, res):
    try:
        res[name] = round(timeit(fn), 1)
    except Exception as ex:  # a trapping kernel poisons the context: report and stop
        res[name] = f"FAILED: {type(ex).__name__}: {str(ex)[:120]}"
        raise


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="10b,l")
    ap.add_argument("--json", default="")
    ap.add_argument("--skip", default="", help="comma list of variants to skip")
    args = ap.parse_args()
    skip = set(args.skip.split(",")) if args.skip else set()
    allres = {}
    for key in args.shapes.split(","):
        B, N, H, hd = SHAPES[key]
        D = H * hd
        qkv = (torch.randn(B * N, 3 * D, device="cuda") * 0.5).to(torch.bfloat16)
        dout = torch.randn(B * N, D, device="cuda").to(torch.bfloat16)
        res = {"shape": [B, N, H, hd]}
        flops_fwd = 4.0 * B * H * N * N * hd
        try:
            out = torch.empty(B * N, D, dtype=qkv.dtype, device="cuda")
            lse = torch.empty(B * H, N, device="cuda")
            guarded("fwd_unfused_us", lambda: co.attention_fwd(qkv, B, N, H, hd, need_p=True), res)
            if N <= 256:
                guarded("fwd_oneshot_us", lambda: co._C.attention_fwd(qkv, out, lse, B, N, H, hd), res)
                if "persist_fwd" not in skip and hd == 160 and N > 128:
                    o2, l2 = torch.empty_like(out), torch.empty_like(lse)
                    guarded("fwd_persist_us", lambda: co._C.attention_fwd_persist(qkv, o2, l2, B, N, H, hd), res)
                    res["fwd_persist_max_err_vs_oneshot"] = float((o2.float() - out.float()).abs().max())
            else:
                guarded("fwd_long_us", lambda: co._C.attention_fwd_long(qkv, out, lse, B, N, H, hd), res)
            _, p = co.attention_fwd(qkv, B, N, H, hd, need_p=True)
            guarded("bwd_unfused_us", lambda: co.attention_bwd(dout, qkv, p, B, N, H, hd, want_colsum=True), res)
            guarded("probs_remat_us", lambda: co.attention_probs(qkv, B, N, H, hd), res)
            del p

            def bwd(persist):  # delta kernel + dK/dV + dQ kernels + qkv bias gradient, as attention_bwd_lse runs them
                dqkv = torch.empty(B * N, 3 * D, dtype=qkv.dtype, device="cuda")
                delta = torch.empty(2 if persist else 1, B * H, N, device="cuda")
                cs = torch.zeros(3 * D, device="cuda") if persist else None
                co._C.attention_bwd(qkv, dout, out, lse, delta, dqkv, cs, B, N, H, hd, persist)
                return dqkv, (cs if persist else co.colsum(dqkv))

            guarded("bwd_oneshot_us", lambda: bwd(False), res)
            if "persist_bwd" not in skip and hd == 160 and N % 4 == 0:
                ref = bwd(False)[0]
                guarded("bwd_persist_us", lambda: bwd(True), res)
                res["bwd_persist_max_err_vs_oneshot"] = float((bwd(True)[0].float() - ref.float()).abs().max())
        except Exception as ex:
            res["error"] = f"{type(ex).__name__}: {str(ex)[:200]}"
            allres[key] = res
            print(json.dumps({key: res}), flush=True)
            break
        res["fwd_gflop"] = flops_fwd / 1e9
        allres[key] = res
        print(json.dumps({key: res}), flush=True)
        del qkv, dout
        torch.cuda.empty_cache()
    if args.json:
        json.dump(allres, open(args.json, "w"), indent=1)


if __name__ == "__main__":
    main()
