"""Training throughput of the text-conditioned bedroom network (config/text/diffusion_bedrooms_instancond_lat32_v_bert.yaml)
through the drop-in `train_on_batch`, one JSON line per batch size in bench.py's style.

Two arms run in the same process on the same synthetic batch, alternating iteration by iteration after warm-up and
timed with device events:
  native    ds_train_step (forward + hand-written backward, cross-attention included) + NativeAdam
  autograd  native_backward = False: torch autograd over networks/functional.py + torch.optim.Adam
The text condition is a stand-in for BERT's last hidden states, [B, L, 768] (L = 32 as in `bench.py --config text`);
fc_text_f trains in both arms.  Random-init weights, loss_separate + loss_iou, gradient clip 10.

    python scripts/bench_train_text.py --batch 128,1024 --steps 20 --warmup 5
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _config(stats_path):
    import yaml
    with open(os.path.join(ROOT, "config", "text/diffusion_bedrooms_instancond_lat32_v_bert.yaml")) as f:
        cfg = yaml.safe_load(f.read().replace("\r", ""))
    cfg["network"]["diffusion_kwargs"]["train_stats_file"] = stats_path
    cfg["training"]["max_grad_norm"] = 10
    return cfg


def _batch(B, L, gen, dev):
    N, class_dim = 12, 22
    cls = torch.randint(0, class_dim, (B, N), generator=gen)
    sp = dict(translations=torch.rand(B, N, 3, generator=gen) * 2 - 1, sizes=torch.rand(B, N, 3, generator=gen) * 2 - 1,
              angles=torch.nn.functional.normalize(torch.randn(B, N, 2, generator=gen), dim=-1),
              class_labels=torch.nn.functional.one_hot(cls, class_dim).float() * 2 - 1,
              objfeats_32=torch.rand(B, N, 32, generator=gen) * 2 - 1, room_layout=torch.zeros(B, 1, 64, 64),
              description=torch.randn(B, L, 768, generator=gen))
    return {k: v.to(dev) for k, v in sp.items()}


def _gpu(index):
    """name and power limit of the card, read now (the numbers depend on both)"""
    out = {"name": torch.cuda.get_device_name(index), "power_limit_w": None, "max_sm_clock_mhz": None}
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        p, c = [v.strip() for v in r.stdout.strip().split(",")[:2]]
        out["power_limit_w"], out["max_sm_clock_mhz"] = float(p), float(c)
    except Exception as e:      # the measurement stands without it; say why it is missing
        out["error"] = repr(e)
    return out


def run(B, L, steps, warmup, prec, dev, stats_path):
    from scene_synthesis.networks import build_network, optimizer_factory
    from diffuscene_b200.optim import NativeAdam
    cfg = _config(stats_path)
    torch.manual_seed(0)
    net_n, train_on_batch, _ = build_network(0, 23, cfg, None, device=dev, precision=prec)
    net_a, _, _ = build_network(0, 23, cfg, None, device=dev, precision=prec)
    net_a.load_state_dict(net_n.state_dict())
    net_a.native_backward = False
    opt_n = optimizer_factory(cfg["training"], net_n.parameters())
    assert isinstance(opt_n, NativeAdam)
    opt_a = torch.optim.Adam(net_a.parameters(), lr=cfg["training"]["lr"], weight_decay=0.0)
    sp = _batch(B, L, torch.Generator().manual_seed(1), dev)
    arms = {"native": (net_n, opt_n), "autograd": (net_a, opt_a)}
    for _ in range(warmup):
        for net, opt in arms.values():
            train_on_batch(net, opt, sp, cfg)
    torch.cuda.synchronize(dev)
    assert net_n._native_grads_ready and not net_a._native_grads_ready, "an arm did not take its path"
    ms = {k: 0.0 for k in arms}
    loss = {}
    launches = 0
    for i in range(steps):
        for k, (net, opt) in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = net_n.engine(commit=False).launch_count()
            e0.record()
            loss[k] = train_on_batch(net, opt, sp, cfg)
            e1.record()
            torch.cuda.synchronize(dev)
            ms[k] += e0.elapsed_time(e1)
            if k == "native":
                launches = net_n.engine(commit=False).launch_count() - l0
    phases = net_n.engine(commit=False).train_phase_ms()
    assert all(v == v for v in loss.values()), loss
    per = {k: v / steps for k, v in ms.items()}
    return {
        "metric": "text-conditioned training scenes/sec (optimizer iterations x batch / s), native arm",
        "value": B / (per["native"] / 1000.0), "unit": "scenes/s", "n_gpus": 1, "steps": steps, "warmup": warmup,
        "higher_is_better": True, "dtype": prec, "data": "synthetic",
        "config": {"workload": "train_on_batch, text bedroom N=12 d=62 (config/text/diffusion_bedrooms_instancond_lat32_v_bert.yaml), "
                               "BERT stand-in hidden states [B, %d, 768] -> fc_text_f, Adam, loss_separate + loss_iou, "
                               "clip 10, random-init weights" % L,
                   "name": "train_text", "scenes_per_gpu": B, "text_tokens": L},
        "arms": {k: {"ms_per_step": per[k], "scenes_per_s": B / (per[k] / 1000.0), "last_loss": loss[k]} for k in arms},
        "speedup_native_vs_autograd": per["autograd"] / per["native"],
        "timing": "device events per iteration, arms alternating after %d warm-up iterations each" % warmup,
        "engine_launches_per_step": int(launches), "phases_ms": phases, "gpu": _gpu(dev.index or 0),
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--batch", default="128,1024", help="scenes per iteration, comma-separated")
    ap.add_argument("--L", type=int, default=32, help="text tokens per scene")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--precision", default="bf16", choices=("bf16", "fp32"))
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 1:
        ap.error("--steps and --warmup must be at least 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_text.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    from tests.cases import STATS
    fd, stats = tempfile.mkstemp(prefix="ds_b200_text_stats_", suffix=".json")
    try:
        with os.fdopen(fd, "w") as f:
            json.dump(STATS, f)
        for B in [int(b) for b in a.batch.split(",")]:
            print(json.dumps(run(B, a.L, a.steps, a.warmup, a.precision, dev, stats)), flush=True)
    finally:
        os.remove(stats)


if __name__ == "__main__":
    main()
