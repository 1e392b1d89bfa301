#!/usr/bin/env python
"""Headline benchmark: ViT-10B FSDP training throughput (images/sec) on N B200 GPUs of one node.

    python bench.py                                   # 1 GPU, 5 timed steps, 3 warm-ups
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus 8 --steps 5 --warmup 3
    python bench.py --impl reference ...              # the UNMODIFIED reference script on stock PyTorch
    python bench.py --dump-outputs DIR ...            # also write what the last timed step computed to DIR/*.npy

The timed step is the body of the reference's training loop (run_vit_training.py:259-280): forward + loss, backward,
clip_grad_norm_ on the full gradient, optimizer.step, lr_scheduler.step, zero_grad.

Protocol (BASELINE.md): ViT-10B (embed 5120, 32 heads, 32 blocks, MLP 4x, patch 14, 224 px), bf16 compute,
`--fake_data` zeros, random-init weights, FSDP ZeRO-3 + activation checkpointing + grad clipping + AdamW +
warmup-cosine -- the full training step of the reference.  Weak scaling: 128 images per GPU (= the
reference's global batch 1024 on 8 GPUs).  Step time comes from CUDA events on the device, max over ranks.

Two timed regions of K steps each:
  * e2e   : every step copies that step's batch from pinned host memory to the device and reads the loss back;
  * value : kernel-only (device-resident batch, no host read-back).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MODELS = {
    # name: (image, patch, dim, heads, blocks, mlp_ratio, description)
    "vit10b": (224, 14, 5120, 32, 32, 4.0, "ViT-10B (embed_dim=5120, 32 heads, 32 blocks, mlp_ratio 4.0, patch 14, 224px)"),
    "vit10b_336": (336, 14, 5120, 32, 32, 4.0, "ViT-10B at 336px / patch 14 (576 tokens)"),
    "vitl": (224, 16, 1024, 16, 24, 4.0, "ViT-Large (embed_dim=1024, 16 heads, 24 blocks, patch 16, 224px)"),
    "vitb": (224, 16, 768, 12, 12, 4.0, "ViT-Base (debug)"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", type=str, default="vit10b", choices=sorted(MODELS))
    ap.add_argument("--local_batch", type=int, default=128)
    ap.add_argument("--num_blocks", type=int, default=0, help="debug: override depth (marks the result as reduced)")
    ap.add_argument("--backend", type=str, default="sm100", choices=["sm100", "nccl"])
    ap.add_argument("--no_grad_ckpt", action="store_true")
    ap.add_argument("--ckpt_keep_blocks", type=int, default=-1,
                    help="blocks that keep lean activations instead of being recomputed; -1 = what free HBM allows "
                         "(decided after the first warm-up step), 0 = checkpoint every block like the reference")
    ap.add_argument("--no_full_ckpt_probe", action="store_true",
                    help="skip the extra (untimed-region) measurement with every block recomputed")
    ap.add_argument("--no_e2e", action="store_true")
    ap.add_argument("--cuda_graph", type=int, default=-1,
                    help="1/0: replay the training step as one CUDA graph; -1 = auto (on for launch-bound models)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float32): its "
                         "loss and gradient norm, and a fixed sample of the parameters and AdamW first moments it "
                         "left behind")
    return ap.parse_args()


class ClockSampler:
    """Samples SM clocks / throttle reasons of one GPU with nvidia-smi while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        clocks, reasons, maxc, power = [], set(), None, []
        try:
            for line in open(self.path):
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 8:
                    continue
                try:
                    clocks.append(float(parts[0]))
                    maxc = float(parts[1])
                    power.append(float(parts[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                     parts[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if clocks:
            clocks.sort()
            out.update(sm_mhz=clocks[len(clocks) // 2], sm_max_mhz=maxc, reasons=sorted(reasons), samples=len(clocks),
                       power_w_max=max(power) if power else None)
        return out


def _maybe_relaunch(args) -> bool:
    """`python bench.py --gpus N` without torchrun: re-launch ourselves under torch.distributed.run."""
    if args.gpus > 1 and "RANK" not in os.environ:
        import socket

        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    return False


def _time_steps(torch, dist, world, step_fn, steps):
    """K steps bracketed by barrier + synchronize, timed with CUDA events; returns max-over-ranks ms/step."""
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step_fn()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1) / steps], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


DUMP_SAMPLE = 1 << 20  # sampled values per array over all ranks (4 MB of float32)


def _dump_outputs(torch, dist, world, rank, model, last, out_dir):
    """Writes what the last training step computed as float32 .npy files: the loss and gradient norm it returned,
    and the parameters / AdamW first moments it left behind, sampled at indices drawn from a fixed seed so that two
    builds run with the same arguments can be compared value by value."""
    import numpy as np

    per_unit = max(1, DUMP_SAMPLE // (world * len(model.all_units)))
    gen = torch.Generator().manual_seed(0)
    params, moments = [], []
    for u in model.all_units:
        n = u.layout.shard_numel
        idx = torch.randint(n, (min(n, per_unit),), generator=gen).to(model.device)
        w = torch.empty(idx.numel(), dtype=torch.float32, device=model.device)
        # the fp32 master lives split in bf16 hi + int16 lo halves: merge only the sampled entries
        model.ops.merge_fp32(u.hi.index_select(0, idx), u.lo.index_select(0, idx), w)
        params.append(w)
        moments.append(u.exp_avg.index_select(0, idx))
    out = {"loss": last["loss"], "grad_norm": last["grad_norm"], "params_sample": torch.cat(params),
           "exp_avg_sample": torch.cat(moments)}
    if world > 1:
        for k in ("params_sample", "exp_avg_sample"):
            parts = [torch.empty_like(out[k]) for _ in range(world)]
            dist.all_gather(parts, out[k])
            out[k] = torch.cat(parts)
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        for k, v in out.items():
            np.save(os.path.join(out_dir, k + ".npy"), v.detach().float().reshape(-1).cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist

    from vit_10b_fsdp_example_b200.config import ViTConfig
    from vit_10b_fsdp_example_b200.ops import cuda_ops
    from vit_10b_fsdp_example_b200.parallel import FSDPViT, ShardedAdamW
    from vit_10b_fsdp_example_b200.utils import get_warmup_cosine_scheduler

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)

    image, patch, dim, heads, blocks, mlp, desc = MODELS[args.model]
    reduced = False
    if args.num_blocks:
        blocks, reduced = args.num_blocks, True
    vcfg = ViTConfig(image_size=image, patch_size=patch, embed_dim=dim, num_heads=heads, num_blocks=blocks,
                     mlp_ratio=mlp, num_classes=1000)
    t_init = time.time()
    model = FSDPViT(vcfg, world=world, rank=rank, device=device, dtype=torch.bfloat16,
                    reshard_after_forward=True, flatten_parameters=False, grad_ckpt=not args.no_grad_ckpt,
                    backend="sm100" if args.backend == "sm100" else "torchdist", seed=0, init_device="cuda",
                    ckpt_keep_blocks=args.ckpt_keep_blocks)
    opt = ShardedAdamW(model, lr=1e-3, weight_decay=0.1)
    global_batch = args.local_batch * world
    sched = get_warmup_cosine_scheduler(opt, warmup_iteration=10000, max_iteration=(1281167 // global_batch) * 300)
    torch.cuda.synchronize()
    t_init = time.time() - t_init

    B = args.local_batch
    host_images = torch.zeros(B, 3, image, image).pin_memory()   # --fake_data: zeros, label 0
    host_target = torch.zeros(B, dtype=torch.long).pin_memory()
    dev_images = host_images.to(device)
    dev_target = host_target.to(device)
    h2d_bytes = host_images.numel() * host_images.element_size() + host_target.numel() * host_target.element_size()
    last_loss = [0.0]
    last = {}  # device tensors returned by the latest step (kept without a host sync)

    use_graph = args.cuda_graph == 1 or (args.cuda_graph == -1 and dim < 2048)
    graphed = None
    if use_graph:
        from vit_10b_fsdp_example_b200.parallel import GraphedTrainStep

        graphed = GraphedTrainStep(model, opt, clip_grad_norm=1.0, warmup=2)

    def train_step(images, target):
        if graphed is not None:
            loss = graphed(images, target)
            norm = graphed.grad_norm
        else:
            loss = model.forward_backward(images, target)
            norm = model.clip_grad_norm_(1.0)
            opt.step()
        sched.step()
        opt.zero_grad(set_to_none=True)
        last.update(loss=loss, grad_norm=norm)
        return loss

    def step_e2e():
        images = host_images.to(device, non_blocking=True)
        target = host_target.to(device, non_blocking=True)
        loss = train_step(images, target)
        last_loss[0] = float(loss.item())  # device -> host read of the step's result (4 bytes)

    def step_dev():
        train_step(dev_images, dev_target)

    for _ in range(max(args.warmup, 3) + (2 if use_graph else 0)):
        step_e2e()  # with --cuda_graph the first calls are eager warm-up + capture
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    e2e_ms = None
    if not args.no_e2e:
        e2e_ms = _time_steps(torch, dist, world, step_e2e, args.steps)
    n0 = cuda_ops.launch_count()
    dev_ms = _time_steps(torch, dist, world, step_dev, args.steps)
    launches = cuda_ops.launch_count() - n0
    if graphed is not None:  # kernels replayed from the graph never pass through the Python wrappers
        launches = graphed.launches_per_step * args.steps
    clocks = sampler.stop() if sampler else {}
    peak_gb = torch.cuda.max_memory_allocated() / 1e9
    if args.dump_outputs:  # before the probes below take further optimizer steps
        _dump_outputs(torch, dist, world, rank, model, last, args.dump_outputs)
    exposed = None
    if graphed is None:
        # Secondary metric of BASELINE.json: exposed communication per step, probed outside the timed region.
        # A rank that is ahead of its peers also waits for *them* inside these events (GPUs under a power cap run at
        # different clocks), so the rank with the smallest stall is the critical path: its number is the exposed
        # communication; the largest one mostly measures how unequal the GPUs are.
        probe_steps = 2
        with model.exposed_comm_probe() as pr:
            for _ in range(probe_steps):
                step_dev()
        lo = torch.tensor([pr["ms"] / probe_steps], dtype=torch.float64, device=device)
        hi = lo.clone()
        if world > 1:
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
            dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        exposed = {"critical_path_rank_ms": float(lo.item()), "max_over_ranks_ms": float(hi.item()),
                   "waits_per_step": pr["waits"] // probe_steps}
    kept = max(0, model.keep_blocks)
    full_ckpt_ms = None
    if kept > 0 and graphed is None and not args.no_full_ckpt_probe:
        # same activation policy as the reference (every block recomputed), timed like the headline (CUDA events, max
        # over ranks, up to 10 steps after 2 untimed ones).  This is the equal-work point for scaling comparisons: the
        # headline's kept-block count changes with N (more GPUs -> more free HBM -> fewer recomputed blocks).
        model.keep_blocks = 0
        for _ in range(2):
            step_dev()
        full_ckpt_steps = min(args.steps, 10)  # the GPUs are at their power-capped steady state by now
        full_ckpt_ms = _time_steps(torch, dist, world, step_dev, full_ckpt_steps)
        model.keep_blocks = kept

    if rank == 0:
        recomputed = 0.0 if args.no_grad_ckpt else (blocks - kept) / max(1, blocks)
        flops = vcfg.flops_per_image(grad_ckpt=False) * (1.0 + recomputed / 3.0) * B
        rec = {
            "metric": "ViT-10B images/sec (device-timed, max over ranks)" if args.model == "vit10b" and not reduced
            else f"{args.model} images/sec (device-timed, max over ranks)",
            "value": global_batch / (dev_ms * 1e-3), "unit": "images/sec", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": dev_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic (--fake_data zeros, random-init weights)",
            "impl": "ours",
            "config": {"model": desc + (f" [REDUCED to {blocks} blocks]" if reduced else ""),
                       "global_batch": global_batch, "local_batch": B, "seq_len": vcfg.num_patches,
                       "parallelism": f"fsdp{world} (ZeRO-3, per-block units, activation checkpointing"
                                      f"{' off' if args.no_grad_ckpt else ''}, backend {model.backend.name})",
                       "activation_ckpt": ("off" if args.no_grad_ckpt else
                                           f"memory-aware: {kept} of {blocks} blocks keep a lean activation set "
                                           f"(no GEMM recompute; of those {model.keep_extras} also keep P / LN "
                                           f"outputs / gelu(u)), {blocks - kept} are recomputed in backward"),
                       "optimizer": "AdamW + clip_grad_norm 1.0 + warmup-cosine, every step",
                       "cuda_graph": bool(use_graph),
                       "l2": "no explicit flush: each step streams ~20 GB of bf16 weights plus activations (>> 126 MB L2)",
                       "params": vcfg.total_numel()},
            "clocks": {"sm_mhz": clocks.get("sm_mhz"), "sm_max_mhz": clocks.get("sm_max_mhz"),
                       "reasons": clocks.get("reasons", []), "samples": clocks.get("samples", 0),
                       "power_w_max": clocks.get("power_w_max")},
            "gpu_launches": launches,
            "exposed_comm_ms_per_step": exposed,
            "model_tflops_per_gpu": flops / (dev_ms * 1e-3) / 1e12,
            "peak_mem_gb": peak_gb, "init_s": t_init, "loss": last_loss[0],
        }
        if full_ckpt_ms is not None:
            rec["full_recompute"] = {"value": global_batch / (full_ckpt_ms * 1e-3), "ms_per_step": full_ckpt_ms,
                                     "steps": min(args.steps, 10),
                                     "note": "same step with --ckpt_keep_blocks 0 (every block recomputed, the "
                                             "reference's policy); equal work per GPU at every N"}
        if e2e_ms is not None:
            rec["e2e"] = {"value": global_batch / (e2e_ms * 1e-3), "unit": "images/sec", "ms_per_step": e2e_ms,
                          "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4}
        print(json.dumps(rec), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_reference(args):
    try:
        from baseline import reference_arm
    except Exception as e:  # pragma: no cover
        print(json.dumps({"impl": "reference", "unavailable": f"reference arm not importable: {e!r}"[:300]}))
        return
    reference_arm.run(args, MODELS, ClockSampler, _time_steps)


def main():
    args = parse()
    _maybe_relaunch(args)
    if args.impl == "reference":
        try:
            run_reference(args)
        except SystemExit:
            raise
        except BaseException as e:  # the reference arm must always exit 0 with one JSON line
            if int(os.environ.get("RANK", 0)) == 0:
                print(json.dumps({"impl": "reference", "unavailable": f"{type(e).__name__}: {str(e)[:240]}"}))
        return
    run_ours(args)


if __name__ == "__main__":
    main()
