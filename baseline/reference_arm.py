"""`bench.py --impl reference`: the UNMODIFIED reference script on stock PyTorch (see baseline/README.md)."""
from __future__ import annotations

import json
import os
import sys
import time

from oracle import reference

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = reference.REF_DIR
SHIMS = os.path.join(HERE, "shims")


def _ensure_ref():
    if reference.is_staged():
        return None
    return ("oracle/_ref is missing: build with VIT_REFERENCE_DIR set to a checkout of the original example to "
            "stage its script there")


def run(args, MODELS, ClockSampler, time_steps):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))

    def bail(msg):
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": msg[:300]}), flush=True)

    err = _ensure_ref()
    if err:
        return bail(err)
    torch.cuda.set_device(local_rank)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29533")
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))

    sys.path.insert(0, SHIMS)
    sys.path.insert(0, REF_DIR)  # the reference's own `utils` must win over this repo's top-level utils.py
    for m in ("utils",):
        sys.modules.pop(m, None)
    import run_vit_training as ref  # noqa: E402  (unmodified reference file)
    import utils as ref_utils  # noqa: E402
    import torch_xla.core.xla_model as xm  # noqa: E402  (shim)

    from vit_10b_fsdp_example_b200.config import parse_args  # flag-compatible argparse (same 29 flags/defaults)

    image, patch, dim, heads, blocks, mlp, desc = MODELS[args.model]
    reduced = bool(args.num_blocks)
    if reduced:
        blocks = args.num_blocks
    global_batch = args.local_batch * world
    cfg = parse_args(["--fake_data", "--image_size", str(image), "--patch_size", str(patch), "--embed_dim", str(dim),
                      "--num_heads", str(heads), "--num_blocks", str(blocks), "--mlp_ratio", str(mlp),
                      "--batch_size", str(global_batch)] + (["--no_grad_ckpt"] if args.no_grad_ckpt else []))
    device = xm.xla_device()
    try:
        t0 = time.time()
        model = ref.build_fsdp_vit_model(cfg, device)              # reference :228
        loss_fn = torch.nn.CrossEntropyLoss()                       # :229
        parameters = list(model.parameters())                       # :233
        optimizer = torch.optim.AdamW(parameters, lr=cfg.lr, weight_decay=cfg.weight_decay)  # :237
        lr_scheduler = ref_utils.get_warmup_cosine_scheduler(       # :238-240
            optimizer, warmup_iteration=cfg.warmup_steps, max_iteration=1281167 // global_batch * cfg.num_epochs)
        model.train()
        t_init = time.time() - t0
        B = args.local_batch
        host_images = torch.zeros(B, 3, image, image).pin_memory()
        host_target = torch.zeros(B, dtype=torch.long).pin_memory()
        dev_images, dev_target = host_images.to(device), host_target.to(device)
        last = [0.0]

        def train_step(data, target):
            # body of the reference training loop, run_vit_training.py:261-280
            output = model(data)
            loss = loss_fn(output, target)
            loss.backward()
            if not cfg.run_without_fsdp:
                if cfg.clip_grad_norm > 0:
                    model.clip_grad_norm_(cfg.clip_grad_norm)
            optimizer.step()
            lr_scheduler.step()
            optimizer.zero_grad(set_to_none=True)
            return loss

        def step_e2e():
            loss = train_step(host_images.to(device, non_blocking=True), host_target.to(device, non_blocking=True))
            last[0] = float(loss.item())

        def step_dev():
            train_step(dev_images, dev_target)

        for _ in range(max(args.warmup, 3)):
            step_e2e()
        sampler = ClockSampler(local_rank) if rank == 0 else None
        if sampler:
            sampler.start()
        e2e_ms = None if args.no_e2e else time_steps(torch, dist, world, step_e2e, args.steps)
        dev_ms = time_steps(torch, dist, world, step_dev, args.steps)
        clocks = sampler.stop() if sampler else {}
    except torch.OutOfMemoryError as e:
        bail(f"CUDA out of memory running the stock PyTorch FSDP reference at local batch {args.local_batch} on "
             f"{world} GPU(s): {str(e)[:120]}")
        dist.destroy_process_group()
        return
    if rank == 0:
        h2d = host_images.numel() * 4 + host_target.numel() * 8
        rec = {
            "metric": "ViT-10B images/sec (device-timed, max over ranks)" if args.model == "vit10b" and not reduced
            else f"{args.model} images/sec (device-timed, max over ranks)",
            "value": global_batch / (dev_ms * 1e-3), "unit": "images/sec", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": dev_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic (--fake_data zeros, random-init weights)",
            "impl": "reference",
            "config": {"model": desc + (f" [REDUCED to {blocks} blocks]" if reduced else ""),
                       "global_batch": global_batch, "local_batch": B, "seq_len": (image // patch) ** 2,
                       "parallelism": f"fsdp{world} (unmodified reference script; torch_xla/timm provided by stock-PyTorch "
                                      f"shims: torch FSDP bf16 MixedPrecision + NCCL + cuBLAS + SDPA, act-ckpt)"},
            "clocks": {"sm_mhz": clocks.get("sm_mhz"), "sm_max_mhz": clocks.get("sm_max_mhz"),
                       "reasons": clocks.get("reasons", []), "samples": clocks.get("samples", 0)},
            "gpu_launches": 0, "peak_mem_gb": torch.cuda.max_memory_allocated() / 1e9, "init_s": t_init,
            "loss": last[0],
        }
        if e2e_ms is not None:
            rec["e2e"] = {"value": global_batch / (e2e_ms * 1e-3), "unit": "images/sec", "ms_per_step": e2e_ms,
                          "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4}
        print(json.dumps(rec), flush=True)
    dist.barrier()
    dist.destroy_process_group()
