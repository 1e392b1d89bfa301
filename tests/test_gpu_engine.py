"""End-to-end engine on the GPU (sm_100a kernels, bf16) vs the fp32 PyTorch reference ops on the same data."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _run(device, dtype, steps, cfg_kw, init_from=None):
    from vit_10b_fsdp_example_b200.config import ViTConfig
    from vit_10b_fsdp_example_b200.parallel import FSDPViT, ShardedAdamW

    cfg = ViTConfig(**cfg_kw)
    model = FSDPViT(cfg, device=device, dtype=dtype, seed=1)
    opt = ShardedAdamW(model, lr=1e-3, weight_decay=0.1)
    g = torch.Generator().manual_seed(0)
    images = torch.randn(8, 3, cfg.image_size, cfg.image_size, generator=g)
    target = torch.randint(0, cfg.num_classes, (8,), generator=g)
    losses, norms = [], []
    for _ in range(steps):
        loss = model.forward_backward(images.to(device), target.to(device))
        norm = model.clip_grad_norm_(1.0)
        opt.step()
        losses.append(loss.item())
        norms.append(norm.item())
    return losses, norms, model


@pytest.mark.parametrize("cfg_kw", [
    dict(image_size=112, patch_size=14, embed_dim=320, num_heads=2, num_blocks=2, mlp_ratio=4.0, num_classes=100),
    dict(image_size=224, patch_size=16, embed_dim=256, num_heads=4, num_blocks=2, mlp_ratio=4.0, num_classes=1000),
])
def test_training_matches_fp32_reference(cfg_kw):
    ref_losses, ref_norms, _ = _run(torch.device("cpu"), torch.float32, 4, cfg_kw)
    losses, norms, model = _run(torch.device("cuda"), torch.bfloat16, 4, cfg_kw)
    assert model.ops.NAME == "sm100"
    for a, b in zip(losses, ref_losses):
        assert abs(a - b) < 0.05 * abs(b) + 0.02, (losses, ref_losses)
    for a, b in zip(norms, ref_norms):
        assert abs(a - b) < 0.1 * abs(b) + 0.02, (norms, ref_norms)
    assert losses[-1] < losses[0]


def test_eval_forward_and_state_dict_roundtrip():
    from vit_10b_fsdp_example_b200.parallel import FSDPViT
    from vit_10b_fsdp_example_b200.config import ViTConfig

    cfg = ViTConfig(image_size=112, patch_size=14, embed_dim=320, num_heads=2, num_blocks=2, mlp_ratio=4.0,
                    num_classes=100)
    dev = torch.device("cuda")
    m = FSDPViT(cfg, device=dev, dtype=torch.bfloat16, seed=2)
    x = torch.randn(4, 3, 112, 112, device=dev)
    logits = m.eval()(x)
    assert logits.shape == (4, 100) and torch.isfinite(logits.float()).all()
    sd = m.state_dict()
    m2 = FSDPViT(cfg, device=dev, dtype=torch.bfloat16, seed=3)
    m2.load_state_dict(sd)
    assert torch.equal(m2.eval()(x), logits)
    # the split (bf16 hi, int16 lo) master representation is exact
    ref = FSDPViT(cfg, device=torch.device("cpu"), dtype=torch.float32, seed=2).state_dict()
    for k in sd:
        assert torch.equal(sd[k], ref[k]), k


def test_smoke_entry():
    import __graft_entry__ as ge

    ge.smoke()


def test_cuda_graph_step_matches_eager():
    """The whole training step replayed as one CUDA graph must follow the eager trajectory (lr schedule included)."""
    from vit_10b_fsdp_example_b200.config import ViTConfig
    from vit_10b_fsdp_example_b200.parallel import FSDPViT, GraphedTrainStep, ShardedAdamW
    from vit_10b_fsdp_example_b200.utils import get_warmup_cosine_scheduler

    cfg = ViTConfig(image_size=112, patch_size=14, embed_dim=320, num_heads=2, num_blocks=2, mlp_ratio=4.0,
                    num_classes=96)
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(0)
    images = [torch.randn(8, 3, 112, 112, generator=g).to(dev) for _ in range(3)]
    targets = [torch.randint(0, 96, (8,), generator=g).to(dev) for _ in range(3)]
    results = {}
    for mode in ("eager", "graph"):
        model = FSDPViT(cfg, device=dev, dtype=torch.bfloat16, seed=4)
        opt = ShardedAdamW(model, lr=2e-3, weight_decay=0.1)
        sched = get_warmup_cosine_scheduler(opt, 3, 50)
        step = GraphedTrainStep(model, opt, clip_grad_norm=1.0, warmup=2) if mode == "graph" else None
        losses = []
        for i in range(9):
            x, y = images[i % 3], targets[i % 3]
            if step is not None:
                loss = step(x, y)
            else:
                loss = model.forward_backward(x, y)
                model.clip_grad_norm_(1.0)
                opt.step()
            sched.step()
            losses.append(loss.item())
        results[mode] = (losses, model.state_dict(), opt.state[model.all_units[0].name]["step"])
        if step is not None:
            assert step.graph is not None and step.launches_per_step > 0
    (le, sde, ste), (lg, sdg, stg) = results["eager"], results["graph"]
    assert ste == stg == 9
    for a, b in zip(le, lg):
        assert abs(a - b) < 2e-2 * abs(a) + 1e-3, (le, lg)
    # parameters agree up to atomics-order noise amplified by Adam's sign-like early updates (lr 2e-3, 9 steps)
    for k in sde:
        assert (sde[k] - sdg[k]).abs().mean().item() < 2e-3, k
        assert (sde[k] - sdg[k]).abs().max().item() < 4e-2, k


def _full_grads(model):
    return {u.name: u.shard_grad.float().clone() for u in model.all_units}


@pytest.mark.gpu
@pytest.mark.parametrize("heads,dim", [(2, 320), (4, 256)])
def test_lean_blocks_vs_recompute(heads, dim):
    from vit_10b_fsdp_example_b200.config import ViTConfig
    from vit_10b_fsdp_example_b200.parallel import FSDPViT

    cfg = ViTConfig(image_size=112, patch_size=14, embed_dim=dim, num_heads=heads, num_blocks=3, mlp_ratio=4.0,
                    num_classes=96)
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(0)
    x = torch.randn(8, 3, 112, 112, generator=g).to(dev)
    y = torch.randint(0, 96, (8,), generator=g).to(dev)
    grads, losses = [], []
    for keep in (0, 2, 3):
        model = FSDPViT(cfg, device=dev, dtype=torch.bfloat16, seed=4, ckpt_keep_blocks=keep)
        losses.append(model.forward_backward(x, y).item())
        grads.append(_full_grads(model))
    assert abs(losses[0] - losses[1]) < 1e-3 and abs(losses[0] - losses[2]) < 1e-3
    for other in grads[1:]:
        for k in grads[0]:
            a, b = grads[0][k], other[k]
            assert (a - b).norm().item() <= 2e-2 * a.norm().item() + 1e-6, k
    auto = FSDPViT(cfg, device=dev, dtype=torch.bfloat16, seed=4, ckpt_keep_blocks=-1)
    auto.forward_backward(x, y)
    assert auto.keep_blocks == -1
    auto.forward_backward(x, y)
    assert 0 <= auto.keep_blocks <= 3


@pytest.mark.gpu
@pytest.mark.parametrize("heads,dim,img", [(4, 256, 112), (2, 256, 224), (2, 320, 224), (2, 320, 336)])
def test_fused_attention_pair_matches_unfused_in_the_engine(heads, dim, img, monkeypatch):
    """Same model, same data: gradients with the flash-style attention pair (lse + fused backward kernels) must
    match the un-fused path (GEMMs + softmax kernels, forced by replacing the plan) to bf16 noise.  Covers N = 64 / 256 / 576 (the 336 px
    long-sequence kernels), hd = 64 / 128 / 160."""
    from vit_10b_fsdp_example_b200.config import ViTConfig
    from vit_10b_fsdp_example_b200.ops import attention_plan as ap
    from vit_10b_fsdp_example_b200.parallel import FSDPViT

    cfg = ViTConfig(image_size=img, patch_size=14, embed_dim=dim, num_heads=heads, num_blocks=2, mlp_ratio=4.0,
                    num_classes=96)
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(0)
    x = torch.randn(4, 3, img, img, generator=g).to(dev)
    y = torch.randint(0, 96, (4,), generator=g).to(dev)
    res = []
    default_plan = ap.plan
    assert default_plan(cfg.num_patches, cfg.head_dim).fwd_lse is not None
    unfused = ap.AttentionPlan(None, ap.UNFUSED, None)
    for flash in (False, True):
        monkeypatch.setattr(ap, "plan", default_plan if flash else (lambda N, hd: unfused))
        for keep in (0, 2):
            model = FSDPViT(cfg, device=dev, dtype=torch.bfloat16, seed=4, ckpt_keep_blocks=keep)
            loss = model.forward_backward(x, y).item()
            res.append((loss, _full_grads(model)))
    for loss, grads in res[1:]:
        assert abs(loss - res[0][0]) < 2e-3
        for k in grads:
            a, b = res[0][1][k], grads[k]
            assert (a - b).norm().item() <= 3e-2 * a.norm().item() + 1e-6, k


@pytest.mark.gpu
def test_dropout_kernel_path():
    """--pos_dropout / --att_dropout / --mlp_dropout on the CUDA engine: Philox dropout kernels, no eager fallback.
    (a) keep fraction and scaling, (b) same key -> same mask (recompute consistency), (c) a checkpointed and a
    non-checkpointed model give the same gradients (the recompute regenerates the masks), (d) training still learns."""
    from vit_10b_fsdp_example_b200.config import ViTConfig
    from vit_10b_fsdp_example_b200.ops import cuda_ops as co
    from vit_10b_fsdp_example_b200.parallel import FSDPViT, ShardedAdamW

    dev = torch.device("cuda")
    x = torch.ones(1 << 20, device=dev, dtype=torch.bfloat16)
    n0 = co.launch_count()
    y1, y2, y3 = co.dropout(x, 0.25, 12345), co.dropout(x, 0.25, 12345), co.dropout(x, 0.25, 12346)
    assert co.launch_count() - n0 == 3
    keep = (y1 != 0).float().mean().item()
    assert abs(keep - 0.75) < 5e-3, keep
    assert torch.equal(y1, y2) and not torch.equal(y1, y3)
    assert abs(y1.float().max().item() - 1.0 / 0.75) < 1e-2
    cfg = ViTConfig(image_size=112, patch_size=14, embed_dim=256, num_heads=4, num_blocks=2, mlp_ratio=4.0,
                    num_classes=96, pos_dropout=0.1, att_dropout=0.1, mlp_dropout=0.1)
    g = torch.Generator().manual_seed(0)
    xi = torch.randn(8, 3, 112, 112, generator=g).to(dev)
    yi = torch.randint(0, 96, (8,), generator=g).to(dev)
    grads = []
    for ckpt, keepb in ((True, 0), (False, 0), (True, 2)):
        model = FSDPViT(cfg, device=dev, dtype=torch.bfloat16, seed=4, grad_ckpt=ckpt, ckpt_keep_blocks=keepb)
        model.forward_backward(xi, yi)
        grads.append(_full_grads(model))
    for other in grads[1:]:
        for k in grads[0]:
            a, b = grads[0][k], other[k]
            assert (a - b).norm().item() <= 2e-2 * a.norm().item() + 1e-6, k
    model = FSDPViT(cfg, device=dev, dtype=torch.bfloat16, seed=4)
    opt = ShardedAdamW(model, lr=1e-3, weight_decay=0.0)
    losses = []
    for _ in range(8):
        losses.append(model.forward_backward(xi, yi).item())
        model.clip_grad_norm_(1.0)
        opt.step()
    assert losses[-1] < losses[0], losses
    model.eval()
    a, b = model(xi), model(xi)  # inference: dropout off -> deterministic
    assert torch.equal(a, b)


@pytest.mark.gpu
def test_mean_pool_kernels():
    from vit_10b_fsdp_example_b200.ops import cuda_ops as co, torch_ops as to

    B, N, D = 6, 196, 1024
    xn = torch.randn(B * N, D, device="cuda").to(torch.bfloat16)
    got, ref = co.mean_pool(xn, B, N).float(), to.mean_pool(xn.float(), B, N)
    assert (got - ref).abs().max().item() <= 4e-3 * ref.abs().max().item() + 1e-3
    dp = torch.randn(B, D, device="cuda").to(torch.bfloat16)
    got, ref = co.mean_pool_bwd(dp, B, N).float(), to.mean_pool_bwd(dp.float(), B, N)
    assert got.shape == ref.shape
    assert (got - ref).abs().max().item() <= 8e-3 * ref.abs().max().item() + 1e-6
