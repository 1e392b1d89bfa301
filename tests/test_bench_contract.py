"""bench.py's contract with the driver, as far as a CPU box can check it: flags and defaults, the clock / throttle
sampler, the keys of the JSON line, and the reference arm's 'always one JSON line, exit 0' rule."""
import json
import os
import stat
import subprocess
import sys
import time

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_flags_and_defaults(monkeypatch):
    import bench

    monkeypatch.setattr(sys, "argv", ["bench.py"])
    a = bench.parse()
    assert a.gpus == 1 and a.impl == "ours" and a.model == "vit10b" and a.local_batch == 128
    assert a.warmup >= 3 and 1 <= a.steps <= 20          # no flags: one GPU, finishes within minutes
    monkeypatch.setattr(sys, "argv", ["bench.py", "--gpus", "8", "--steps", "20", "--warmup", "5", "--impl", "reference"])
    a = bench.parse()
    assert (a.gpus, a.steps, a.warmup, a.impl) == (8, 20, 5, "reference")
    assert a.dump_outputs is None
    monkeypatch.setattr(sys, "argv", ["bench.py", "--dump-outputs", "out"])
    assert bench.parse().dump_outputs == "out"
    img, patch, dim, heads, blocks, ratio, _ = bench.MODELS["vit10b"]
    assert (img, patch, dim, heads, blocks, ratio) == (224, 14, 5120, 32, 32, 4.0)   # BASELINE.json's headline config


def test_clock_sampler_parses_nvidia_smi_rows(tmp_path, monkeypatch):
    import bench

    fake = tmp_path / "nvidia-smi"
    fake.write_text("#!/bin/bash\n"
                    "echo '1305, 1965, 931.20, 0x0000000000000004, Not Active, Not Active, Not Active, Active'\n"
                    "echo '1290, 1965, 955.00, 0x0000000000000004, Not Active, Not Active, Not Active, Active'\n"
                    "echo '1335, 1965, 940.10, 0x0000000000000000, Not Active, Not Active, Not Active, Not Active'\n"
                    "echo '[N/A], broken row'\n"
                    "sleep 30\n")
    fake.chmod(fake.stat().st_mode | stat.S_IEXEC)
    monkeypatch.setenv("PATH", f"{tmp_path}:{os.environ['PATH']}")
    s = bench.ClockSampler(0)
    s.start()
    time.sleep(0.5)
    out = s.stop()
    assert out["samples"] == 3 and out["sm_mhz"] == 1305.0 and out["sm_max_mhz"] == 1965.0
    assert out["reasons"] == ["sw_power_cap"] and out["power_w_max"] == 955.0


def test_json_line_has_every_key_the_driver_reads():
    src = open(os.path.join(ROOT, "bench.py")).read()
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "model", "global_batch", "seq_len", "parallelism", "l2",
                "clocks", "sm_mhz", "sm_max_mhz", "reasons", "e2e", "h2d_bytes_per_step", "d2h_bytes_per_step",
                "gpu_launches", "impl"):
        assert f'"{key}"' in src, key
    ref = open(os.path.join(ROOT, "baseline", "reference_arm.py")).read()
    for key in ("metric", "value", "n_gpus", "ms_per_step", "e2e", "clocks", "impl", "unavailable"):
        assert f'"{key}"' in ref, key


def test_reference_arm_always_prints_one_json_line_and_exits_zero():
    """On this GPU-less box the reference cannot run: the arm must still exit 0 with {"impl": "reference",
    "unavailable": ...} (the driver's rule for an arm that cannot be measured)."""
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "1"], cwd=ROOT,
                       capture_output=True, text=True, timeout=300, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    rec = json.loads(lines[0])
    assert rec["impl"] == "reference" and "unavailable" in rec


def _load_dump(d):
    import numpy as np

    names = sorted(os.listdir(d))
    assert names == ["exp_avg_sample.npy", "grad_norm.npy", "loss.npy", "params_sample.npy"], names
    out = {n[:-4]: np.load(os.path.join(d, n)) for n in names}
    assert all(a.dtype == np.float32 for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    return out


def test_dump_outputs_writes_the_step_results_and_a_fixed_sample(tmp_path):
    """--dump-outputs on a tiny bf16 model (CPU ops): the step's loss and norm as returned, and the same parameter /
    moment sample on every call."""
    import numpy as np
    import torch

    import bench
    from helpers import tiny_cfg
    from vit_10b_fsdp_example_b200.parallel import FSDPViT, ShardedAdamW

    model = FSDPViT(tiny_cfg(), world=1, rank=0, dtype=torch.bfloat16, seed=0)
    opt = ShardedAdamW(model, lr=1e-3, weight_decay=0.1)
    loss = model.forward_backward(torch.zeros(2, 3, 32, 32), torch.zeros(2, dtype=torch.long))
    norm = model.clip_grad_norm_(1.0)
    opt.step()
    for d in ("a", "b"):
        bench._dump_outputs(torch, None, 1, 0, model, {"loss": loss, "grad_norm": norm}, str(tmp_path / d))
    a, b = _load_dump(tmp_path / "a"), _load_dump(tmp_path / "b")
    assert float(a["loss"][0]) == float(loss) and float(a["grad_norm"][0]) == float(norm.reshape(-1)[0])
    per_unit = bench.DUMP_SAMPLE // len(model.all_units)
    n = sum(min(per_unit, u.layout.shard_numel) for u in model.all_units)
    assert a["params_sample"].shape == a["exp_avg_sample"].shape == (n,)
    master = np.concatenate([model.master_fp32(u).numpy() for u in model.all_units])
    assert np.isin(a["params_sample"], master).all()
    for k in a:
        np.testing.assert_array_equal(a[k], b[k])


@pytest.mark.gpu
def test_bench_dump_outputs_repeat_from_run_to_run(tmp_path):
    """Two runs of the benchmark with the same arguments compute the same thing: their dumps agree."""
    import numpy as np

    dumps = []
    for d in ("a", "b"):
        r = subprocess.run([sys.executable, "bench.py", "--model", "vitb", "--num_blocks", "2", "--local_batch", "16",
                            "--steps", "2", "--warmup", "1", "--cuda_graph", "0", "--no_full_ckpt_probe",
                            "--dump-outputs", str(tmp_path / d)], cwd=ROOT, capture_output=True, text=True,
                           timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        dumps.append(_load_dump(tmp_path / d))
    a, b = dumps
    assert np.isfinite(a["loss"]).all() and a["grad_norm"][0] > 0
    # fp32 atomics (LayerNorm / bias gradients, the loss) sum in a different order from run to run and bf16 rounding
    # carries the last-bit differences into almost every value: two ViT-10B runs on a B200 (1000 W limit) differed by
    # 0.24% in relative L2 in the AdamW moments.  A wrong sample or different inputs differ by ~100%.
    for k in a:
        x, y = a[k].astype(np.float64), b[k].astype(np.float64)
        assert np.linalg.norm(y - x) <= 1e-2 * np.linalg.norm(x) + 1e-6, (k, x[:4], y[:4])
