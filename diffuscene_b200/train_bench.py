"""`bench.py --config train`: BASELINE configs[4] -- data-parallel training of the unconditional living-room network
(N = 21 objects, d = 65), global batch 8192 over the ranks (1024 scenes per GPU at 8 GPUs), Adam (weight decay 0),
loss_separate + loss_iou, gradient clip 10, gradient all-reduce over NCCL.

One "step" = one optimizer iteration through the drop-in `train_on_batch`: native forward + backward
(ds_train_step), flat-buffer all-reduce, device-side gradient norm, fused Adam.  `value` = scenes per second of the
whole job; `e2e` = the same with the batch coming from pinned host memory every iteration and the loss read back.
"""
from __future__ import annotations

import json
import os
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F_TRAIN_MFLOP = 3 * 1455.7        # SURVEY 8d: training ~ 3 x forward FLOPs per scene per iteration (living N = 21)
GLOBAL_BATCH = 8192


def _config():
    """The training config; its `train_stats_file` is a private temporary file (a fixed name under a shared /tmp may
    belong to another user), read once when the network is built: remove it after build_network()."""
    import yaml
    cfg = yaml.safe_load(open(os.path.join(ROOT, "config", "uncond/diffusion_livingrooms_instancond_lat32_v.yaml")).read().replace("\r", ""))
    from tests.cases import STATS
    fd, tmp_stats = tempfile.mkstemp(prefix="ds_b200_train_stats_", suffix=".json")
    with os.fdopen(fd, "w") as f:
        json.dump(STATS, f)
    cfg["network"]["diffusion_kwargs"]["train_stats_file"] = tmp_stats
    cfg["network"]["diffusion_kwargs"]["loss_iou"] = True
    cfg["training"]["max_grad_norm"] = 10
    cfg["training"]["optimizer"] = "Adam"
    return cfg


def _batch(B, N, class_dim, gen):
    cls = torch.randint(0, class_dim, (B, N), generator=gen)
    return dict(translations=torch.rand(B, N, 3, generator=gen) * 2 - 1, sizes=torch.rand(B, N, 3, generator=gen) * 2 - 1,
                angles=torch.nn.functional.normalize(torch.randn(B, N, 2, generator=gen), dim=-1),
                class_labels=torch.nn.functional.one_hot(cls, class_dim).float() * 2 - 1,
                objfeats_32=torch.rand(B, N, 32, generator=gen) * 2 - 1, room_layout=torch.zeros(B, 1, 64, 64))


def run_reference_train(args):
    """CPU arm: the reference's own train_on_batch (oracle/_ref, unmodified) on the host cores, B = 128 per iteration."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import build_ref
    torch.set_num_threads(min(os.cpu_count() or 1, 32))
    kind = "port"
    B, N = 128, 21
    gen = torch.Generator().manual_seed(0)
    if "scene_synthesis" not in sys.modules and build_ref.activate():
        import contextlib
        import io
        from scene_synthesis.networks import build_network, optimizer_factory       # the vendored reference
        cfg = _config()
        with contextlib.redirect_stdout(io.StringIO()):
            net, train_on_batch, _ = build_network(0, 26, cfg, None, "cpu")
        os.remove(cfg["network"]["diffusion_kwargs"]["train_stats_file"])
        opt = optimizer_factory(cfg["training"], net.parameters())
        kind = "reference"
        sp = _batch(B, N, 25, gen)

        def one():
            with contextlib.redirect_stdout(io.StringIO()):
                return train_on_batch(net, opt, sp, cfg)
    else:
        raise SystemExit(json.dumps({"impl": "reference", "unavailable": "oracle/_ref did not travel; the oracle has no training loop"}))
    ts = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        one()
        if i >= args.warmup:
            ts.append(time.perf_counter() - t0)
    sec = sum(ts) / len(ts)
    v = B / sec
    print(json.dumps({
        "impl": "reference", "metric": "training scenes/sec (optimizer iterations x batch / s)", "value": v, "unit": "scenes/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * sec, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "DDP training uncond living room N=21 d=65 (BASELINE configs[4]), Adam, loss_separate + loss_iou, clip 10",
                   "name": "train"},
        "cpu_baseline": {"value": v, "unit": "scenes/s", "cores": torch.get_num_threads(), "kind": kind,
                         "sample": "reference train_on_batch, %d scenes per iteration, fp32 torch CPU" % B},
        "e2e": {"value": v, "unit": "scenes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def run_train_bench(args):
    if args.impl == "reference":
        return run_reference_train(args)
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sys.path.insert(0, ROOT)
    from bench import ClockSampler, dump_outputs, measured_peaks
    from scene_synthesis.networks import build_network, optimizer_factory
    cfg = _config()
    prec = args.precision or "bf16"
    B = args.batch or (GLOBAL_BATCH // world if args.scaling == "strong" else 1024)
    N = 21
    torch.manual_seed(0)
    net, train_on_batch, _ = build_network(0, 26, cfg, None, device=dev, precision=prec)
    os.remove(cfg["network"]["diffusion_kwargs"]["train_stats_file"])
    opt = optimizer_factory(cfg["training"], net.parameters())
    gen = torch.Generator().manual_seed(1 + rank)
    host = {k: v.pin_memory() for k, v in _batch(B, N, 25, gen).items()}
    resident = {k: v.to(dev) for k, v in host.items()}

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def step_resident(i):
        return train_on_batch(net, opt, resident, cfg)

    def step_e2e(i):
        sp = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        return train_on_batch(net, opt, sp, cfg)          # returns the loss as a Python float (device -> host read)

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = net.engine(commit=False).launch_count()
        e0.record()
        for i in range(steps):
            last = fn(warmup + i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), net.engine(commit=False).launch_count() - l0, last

    clocks = ClockSampler(local)
    clocks.start()
    try:
        ms, launches, last = timed(step_resident, args.steps, args.warmup)
    finally:                        # the sampler is a child process: never leave it polling after a failed step
        clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": torch.tensor([last], dtype=torch.float64)})
    phases = net.engine(commit=False).train_phase_ms()
    n_e2e = max(1, min(args.steps, 3))
    ms_e2e, _, _ = timed(step_e2e, n_e2e, 1)
    # share of the gradient all-reduce: time the same collective alone
    ar_ms = 0.0
    if world > 1:
        from diffuscene_b200.parallel import allreduce_flat
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            allreduce_flat(net._flat_grads)
        e1.record()
        torch.cuda.synchronize(dev)
        ar_ms = e0.elapsed_time(e1) / 5
    if rank == 0:
        total = B * world
        value = total * args.steps / (ms / 1000.0)
        ms_per_step = ms / args.steps
        peak_tf, _, which = measured_peaks()
        ach = B * F_TRAIN_MFLOP * 1e6 / (ms_per_step * 1e-3) / 1e12
        assert last == last, "loss is NaN"
        print(json.dumps({
            "metric": "training scenes/sec (optimizer iterations x global batch / s)", "value": value, "unit": "scenes/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": prec, "data": "synthetic",
            "config": {"workload": "DDP training uncond living room N=21 d=65 (BASELINE configs[4]), Adam, loss_separate + "
                                   "loss_iou, clip 10, %d scenes/GPU, random-init weights" % B, "name": "train",
                       "scenes_per_gpu": B, "global_batch": total, "parallelism": "data-parallel x%d (%s scaling)" % (world, args.scaling),
                       "l2": "activations kept for the backward pass (%.1f GB) exceed the 126 MB L2; no explicit flush"
                             % (190 * B * N * 512 * (2 if prec == "bf16" else 4) / 1e9)},
            "gpu_launches": int(launches), "clocks": clk, "last_loss": last,
            "phases_ms": phases, "allreduce_ms": ar_ms, "allreduce_share": ar_ms / ms_per_step if ms_per_step else None,
            "e2e": {"value": total * n_e2e / (ms_e2e / 1000.0), "unit": "scenes/s",
                    "h2d_bytes_per_step": int(sum(v.numel() * 4 for v in host.values())), "d2h_bytes_per_step": 4},
            "roofline": {"bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                         "traffic": None, "peak_source": which + " bf16 sustained",
                         "launch": "one optimizer iteration over %d scenes; algorithmic 3 x 1455.7 MFLOP/scene" % B}}))
    if world > 1:
        dist.destroy_process_group()
