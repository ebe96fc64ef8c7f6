#!/usr/bin/env python
"""Benchmark of the DiffuScene denoising hot path on B200 (contract: see the task statement / DESIGN.md 5).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME] [--scaling weak|strong]
                    [--dump-outputs DIR]

One "step" = one full T-step ancestral DDPM sample of the per-GPU batch: T denoiser forwards + T posterior updates,
nothing skipped, per-step noise from the in-kernel Philox generator.  `value` = scenes/s with inputs resident in
HBM; `e2e` = the same through the public sampling API with host (pinned) x_T / condition in and the host result out.
Multi-GPU: scenes shard over ranks, no data-path collective (sampling is embarrassingly parallel); `--scaling weak`
keeps the per-GPU batch, `--scaling strong` splits the config's batch over the ranks; max-over-ranks timing.

Configs (BASELINE.json `configs`, SURVEY 8d):
  bed_d97   (default) configs[1]: uncond bedroom N=12, BASELINE's synthetic d=97, T=1000, 4096 scenes, bf16
  bed_d62   the same network at the reference's real bedroom layout d=62
  liv_d105  configs[2]: living / dining N=21, synthetic d=105, T=1000, 2048 scenes, bf16
  liv_d65   ... at the reference's real layout d=65
  text      configs[3]: text-conditioned bedroom (cross-attention on a [B, 32, 512] prefix), T=1000, 1024 scenes
  T100_fp32 configs[0]: bedroom d=97, T=100, 128 scenes, fp32 parity mode (the reference's CPU-runnable case)
  lat1 / lat16  the reference generation script's mode (batch 1) and batch 16: us per diffusion step against the
            weight-read HBM floor (SURVEY 8d "single-scene latency mode")
  train     configs[4]: data-parallel training, living N=21 (see --config train; scenes/s per optimizer iteration)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

_BED = dict(dim=512, dim_mults=[1, 1, 1, 1], channels=62, objectness_dim=0, class_dim=22, angle_dim=2,
            objfeat_dim=32, context_dim=0, instanclass_dim=128, seperate_all=True)
_D97 = dict(channels=97, class_dim=23, angle_dim=4, objfeat_dim=64)
# name -> (net_kwargs, N objects, d, T, scenes (the config's batch), precision, MFLOP / scene / step (SURVEY 8d), label)
CONFIGS = {
    "bed_d97": (dict(_BED, **_D97), 12, 97, 1000, 4096, "bf16", 871.2, "uncond bedroom N=12 d=97 (BASELINE configs[1])"),
    "bed_d62": (dict(_BED), 12, 62, 1000, 4096, "bf16", 870.3, "uncond bedroom N=12 d=62 (configs[1], reference's real layout)"),
    "liv_d105": (dict(_BED, channels=105, class_dim=31, angle_dim=4, objfeat_dim=64), 21, 105, 1000, 2048, "bf16", 1457.4,
                 "uncond living/dining N=21 d=105 (BASELINE configs[2])"),
    "liv_d65": (dict(_BED, channels=65, class_dim=25), 21, 65, 1000, 2048, "bf16", 1455.7,
                "uncond living/dining N=21 d=65 (configs[2], reference's real layout)"),
    "text": (dict(_BED, text_condition=True, text_dim=512), 12, 62, 1000, 1024, "bf16", 977.4,
             "text-conditioned bedroom N=12 d=62, L=32 prefix tokens (BASELINE configs[3])"),
    "T100_fp32": (dict(_BED, **_D97), 12, 97, 100, 128, "fp32", 871.2, "uncond bedroom N=12 d=97 T=100 fp32 (BASELINE configs[0])"),
    "lat1": (dict(_BED), 12, 62, 1000, 1, "bf16", 870.3, "batch-1 generation (scripts/generate_diffusion.py mode), bedroom d=62"),
    "lat16": (dict(_BED), 12, 62, 1000, 16, "bf16", 870.3, "batch-16 generation, bedroom d=62"),
}
W_BYTES_BF16 = 155.35e6          # weights read once per step per GPU (SURVEY 8d)
TEXT_L = 32
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: write each tensor as <out_dir>/<name>.npy (float64 stays float64, anything else becomes
    float32) so that two builds can be compared output for output.  When the arrays come to more than DUMP_MAX_BYTES
    in all, each keeps a fixed, seeded sample of rows along its first (scene) axis, in ascending order: the same rows
    on every run with the same arguments."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: (v if v.dtype == torch.float64 else v.float()).detach().cpu() for k, v in arrays.items()}
    total = sum(a.numel() * a.element_size() for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_MAX_BYTES and a.dim() > 0:
            keep = max(1, a.shape[0] * DUMP_MAX_BYTES // total)
            a = a[torch.randperm(a.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values]
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation (oracle/_ref, vendored by oracle/build_ref.py) when it travelled to this
# box, else the oracle port.  BASELINE.md 3: B = 128 scenes, K = 5 diffusion steps per bench step, all host cores.
# ---------------------------------------------------------------------------------------------------------------
CPU_B, CPU_K = 128, 5


def _cpu_threads():
    return os.cpu_count() or 1


def _yaml_network(cfg_name):
    """The reference's `config['network']` section for a bench config (shipped YAML + the shape overrides)."""
    import yaml
    kw, N, d, T, _, _, _, _ = CONFIGS[cfg_name]
    fn = {12: "uncond/diffusion_bedrooms_instancond_lat32_v.yaml", 21: "uncond/diffusion_livingrooms_instancond_lat32_v.yaml"}[N]
    if kw.get("text_condition"):
        fn = "text/diffusion_bedrooms_instancond_lat32_v_bert.yaml"
    cfg = yaml.safe_load(open(os.path.join(ROOT, "config", fn)).read().replace("\r", ""))
    net = cfg["network"]
    for k in ("class_dim", "angle_dim", "objfeat_dim"):
        net[k] = kw[k]
        net["net_kwargs"][k] = kw[k]
    net["net_kwargs"]["channels"] = kw["channels"]
    net["point_dim"] = d
    net["sample_num_points"] = N
    net["diffusion_kwargs"]["loss_iou"] = False
    net["diffusion_kwargs"]["time_num"] = CPU_K
    return cfg


class CpuArm:
    """Times K diffusion steps of B scenes on the host cores through network.sample() of the vendored reference
    (kind "reference") or, when oracle/_ref did not travel, through the oracle port (kind "port")."""

    def __init__(self, cfg_name, threads=None):
        self.cfg_name = cfg_name
        kw, self.N, self.d, _, _, _, _, _ = CONFIGS[cfg_name]
        self.text = bool(kw.get("text_condition"))
        torch.set_grad_enabled(False)
        self.threads = threads or _cpu_threads()
        self.cores_available = _cpu_threads()
        torch.set_num_threads(self.threads)
        self.kind = "port"
        self.net = None
        from oracle import build_ref
        if not self.text and "scene_synthesis" not in sys.modules and build_ref.activate():
            # text configs would need the BERT checkpoint (no network): they stay on the port, fed a synthetic prefix
            try:
                import contextlib
                import io
                from scene_synthesis.networks import build_network      # the vendored, unmodified reference
                torch.manual_seed(0)
                with contextlib.redirect_stdout(io.StringIO()):
                    self.net, _, _ = build_network(0, kw["class_dim"] + 1, _yaml_network(cfg_name), None, "cpu")
                self.net.eval()
                self.kind = "reference"
            except Exception as e:       # e.g. torchvision missing on the box
                sys.stderr.write("bench: vendored reference unusable (%r); timing the oracle port\n" % (e,))
                self.net = None
        if self.net is None:
            from diffuscene_b200.weights import NetSpec, seeded_state_dict, unet1d_param_specs
            from oracle import diffusion_ref as D
            self.spec = NetSpec.from_net_kwargs(kw)
            self.sd = seeded_state_dict(unet1d_param_specs(self.spec), seed=0)
            self.sched = D.make_schedule(D.make_betas("linear", 1e-4, 0.02, 1000), "v", "fixedsmall")
            self.D = D

    def tune_threads(self):
        """"All the host threads it can use": torch's CPU kernels at these sizes stop scaling (and oversubscribe) well
        before a large host's core count, so one diffusion step is timed at {all cores, 64, 32, 16} threads and the
        fastest setting is kept; `cores` in the JSON is the thread count actually used."""
        if getattr(self, "_tuned", False) or self.cores_available <= 16:
            return
        global CPU_K
        best, k0 = None, CPU_K
        for n in sorted({self.cores_available, 64, 32, 16}, reverse=True):
            if n > self.cores_available:
                continue
            torch.set_num_threads(n)
            self._one(32, 1)
            dt = self._one(32, 1)
            if best is None or dt < best[0]:
                best = (dt, n)
        self.threads = best[1]
        torch.set_num_threads(self.threads)
        self._tuned = True

    def _one(self, B, K):
        """K denoiser evaluations + posterior updates of B scenes through the same code path as step()."""
        N, d = self.N, self.d
        t0 = time.perf_counter()
        if self.net is not None:
            import contextlib
            import io
            # a K-step schedule would need a rebuilt network; time the denoiser + one reverse step directly instead
            dp = self.net.diffusion
            x = torch.randn(B, N, d)
            cond = self.net.positional_embedding[None].expand(B, -1, -1)
            with contextlib.redirect_stdout(io.StringIO()):
                for _ in range(K):
                    t = torch.zeros(B, dtype=torch.int64)
                    x = dp.diffusion.p_sample(dp._denoise, x, t, cond, None, torch.randn, clip_denoised=True)
        else:
            from oracle.unet1d_ref import unet1d_forward
            ctx = torch.randn(N, 128)[None].expand(B, N, 128).contiguous()
            cross = torch.randn(B, TEXT_L, 512) if self.text else None
            x = torch.randn(B, N, d)
            den = lambda xx, tt: unet1d_forward(self.sd, self.spec, xx, tt, ctx, cross)
            for _ in range(K):
                t = torch.full((B,), 500, dtype=torch.int64)
                x, _ = self.D.p_sample_step(self.sched, den, x, t, torch.randn_like(x), True)
        return time.perf_counter() - t0

    def step(self):
        """One bench step of the CPU arm = K diffusion steps of B scenes; returns seconds per diffusion step."""
        self.tune_threads()
        B, K, N, d = CPU_B, CPU_K, self.N, self.d
        if self.net is not None:
            import contextlib
            import io
            room = torch.zeros(B, 1, 64, 64)
            t0 = time.perf_counter()
            with contextlib.redirect_stdout(io.StringIO()):
                out = self.net.sample(room, N, d, batch_size=B, clip_denoised=True)
            dt = time.perf_counter() - t0
            assert tuple(out.shape) == (B, N, d)
            return dt / K
        from oracle.unet1d_ref import unet1d_forward
        ctx = torch.randn(N, 128)[None].expand(B, N, 128).contiguous()
        cross = torch.randn(B, TEXT_L, 512) if self.text else None
        x = torch.randn(B, N, d)
        den = lambda xx, tt: unet1d_forward(self.sd, self.spec, xx, tt, ctx, cross)
        t0 = time.perf_counter()
        for step in reversed(range(1000 - K, 1000)):
            t = torch.full((B,), step, dtype=torch.int64)
            x, _ = self.D.p_sample_step(self.sched, den, x, t, torch.randn_like(x), True)
        return (time.perf_counter() - t0) / K

    def describe(self, T):
        src = "reference network.sample() (oracle/_ref, unmodified)" if self.kind == "reference" else "oracle port"
        return "%d diffusion steps x %d scenes per bench step through the %s, fp32 torch CPU; scaled linearly to a " \
               "%d-step sample (extrapolated: all steps cost the same)" % (CPU_K, CPU_B, src, T)


def run_reference(args):
    """`--impl reference`: rank 0 times the reference's own CPU implementation of the path on the host cores."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    kw, N, d, T, scenes, _, _, label = CONFIGS[args.config]
    arm = CpuArm(args.config)
    per_step = []
    for i in range(args.warmup + args.steps):
        s = arm.step()
        if i >= args.warmup:
            per_step.append(s)
    sec_per_dstep = sum(per_step) / len(per_step)
    v = CPU_B / (sec_per_dstep * T)
    print(json.dumps({
        "impl": "reference", "metric": "scenes/sec full %d-step DDPM sample" % T, "value": v, "unit": "scenes/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * sec_per_dstep * CPU_K,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "%s, T=%d DDPM sampling" % (label, T), "name": args.config},
        "cpu_baseline": {"value": v, "unit": "scenes/s", "cores": arm.threads, "cores_available": arm.cores_available,
                         "kind": arm.kind, "sample": arm.describe(T), "sec_per_scene_step": sec_per_dstep / CPU_B},
        "e2e": {"value": v, "unit": "scenes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="bed_d97", choices=sorted(CONFIGS) + ["train"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--batch", type=int, default=0, help="scenes per GPU (0: the config's batch; strong scaling divides it)")
    ap.add_argument("--timesteps", type=int, default=0, help="override T (profiling runs)")
    ap.add_argument("--precision", default=None)
    ap.add_argument("--backend", default="auto")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--chunk", type=int, default=0, help="scenes per L2-resident sub-batch (0: whole batch at once)")
    ap.add_argument("--shape", default=None, help="deprecated alias: real62 -> --config bed_d62, synth97 -> bed_d97")
    ap.add_argument("--fuse", type=int, default=None, help="fuse_level override; default: the engine's")
    ap.add_argument("--profile-ops", action="store_true", help="print the per-op device time table to stderr")
    ap.add_argument("--kv-hoist", type=int, default=1, help="text config: 1 = K/V of the text prefix precomputed once "
                    "per scene (default); 0 = recomputed before every diffusion step (what the reference does)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy: the sampled x_0 "
                         "[scenes, N, d] (--config train: the loss)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.shape:
        args.config = {"real62": "bed_d62", "synth97": "bed_d97"}[args.shape]
    if args.config == "train":
        from diffuscene_b200.train_bench import run_train_bench
        return run_train_bench(args)
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    from diffuscene_b200.engine import DenoiserEngine
    from diffuscene_b200.schedule import get_betas, make_tables
    from diffuscene_b200.weights import NetSpec, seeded_state_dict, unet1d_param_specs

    kw, N_OBJ, D_ATTR, T, scenes, prec, F_SCENE, label = CONFIGS[args.config]
    if args.precision:
        prec = args.precision
    if args.timesteps:
        T = args.timesteps
    B = args.batch or (max(1, scenes // world) if args.scaling == "strong" else scenes)
    spec = NetSpec.from_net_kwargs(kw)
    eng = DenoiserEngine(spec, N_OBJ, T, precision=prec, gemm_backend=args.backend, device=local, fuse_level=args.fuse)
    eng.load_state_dict(seeded_state_dict(unet1d_param_specs(spec), seed=0))      # random-init weights
    eng.set_schedule(make_tables(get_betas("linear", 1e-4, 0.02, T), "v", "fixedsmall"))
    g = torch.Generator().manual_seed(1)
    pos_emb = torch.randn(N_OBJ, 128, generator=g).pin_memory()                      # positional_embedding
    x_T_host = torch.randn(B, N_OBJ, D_ATTR, generator=g).pin_memory()
    cross_host = torch.randn(B, TEXT_L, 512, generator=g).pin_memory() if spec.text_condition else None
    eng.set_context(pos_emb.to(dev), shared=True)
    if cross_host is not None:
        eng.set_context_cross(cross_host.to(dev))
    x_T_dev = x_T_host.to(dev)
    cross_dev = None if cross_host is None else cross_host.to(dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def resident_step(i):
        if cross_dev is not None and not args.kv_hoist:
            # the reference projects the text to K/V inside every denoiser call: emulate by re-projecting per step
            for _ in range(T):
                eng.set_context_cross(cross_dev)
            return eng.sample(B, clip_denoised=True, x_init=x_T_dev, seed=100 + i, scene_offset=rank * B, chunk_scenes=args.chunk)
        return eng.sample(B, clip_denoised=True, x_init=x_T_dev, seed=100 + i, scene_offset=rank * B, chunk_scenes=args.chunk)

    def e2e_step(i):
        # public sampling call with host buffers: H2D of this step's x_T and condition(s), D2H of the result
        eng.set_context(pos_emb.to(dev, non_blocking=True), shared=True)
        if cross_host is not None:
            eng.set_context_cross(cross_host.to(dev, non_blocking=True))
        return eng.sample(B, clip_denoised=True, x_init=x_T_host.to(dev, non_blocking=True), seed=100 + i,
                          scene_offset=rank * B, host_output=True, chunk_scenes=args.chunk)

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = eng.launch_count()
        e0.record()
        for i in range(steps):
            out = fn(warmup + i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), eng.launch_count() - l0, out

    clocks = ClockSampler(local)
    clocks.start()
    try:
        ms, launches, out = timed(resident_step, args.steps, args.warmup)
    finally:                        # the sampler is a child process: never leave it polling after a failed step
        clk = clocks.stop()
    assert torch.isfinite(out).all()
    if args.dump_outputs:
        from diffuscene_b200.parallel import gather_scenes
        x0 = gather_scenes(out, B * world)          # a collective: every rank takes part
        if rank == 0:
            dump_outputs(args.dump_outputs, {"x0": x0})
    n_e2e = max(1, min(args.steps, 2))
    ms_e2e = None
    if not args.no_e2e:
        ms_e2e, _, _ = timed(e2e_step, n_e2e, 1)

    if rank == 0:
        total_scenes = B * world
        value = total_scenes * args.steps / (ms / 1000.0)
        ms_per_step = ms / args.steps
        us_per_dstep = ms_per_step * 1000.0 / T
        peak_tf, peak_gbs, which = measured_peaks()
        flops_per_launch = B * F_SCENE * 1e6            # one diffusion step of one GPU's batch
        achieved_tf = flops_per_launch / (us_per_dstep * 1e-6) / 1e12
        # which roof binds this per-GPU batch (SURVEY 8d): tensor pipe above ~50 scenes, weight-read HBM below
        t_tensor = flops_per_launch / (peak_tf * 1e12)
        wbytes = W_BYTES_BF16 * (2 if prec == "fp32" else 1)
        t_hbm = wbytes / (peak_gbs * 1e9)
        hbm_bound = t_hbm > t_tensor
        h2d = int(x_T_host.numel() * 4 + pos_emb.numel() * 4 + (0 if cross_host is None else cross_host.numel() * 4))
        res = {
            "metric": "scenes/sec full %d-step DDPM sample" % T, "value": value, "unit": "scenes/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": prec, "data": "synthetic",
            "config": {"workload": "%s, T=%d DDPM sampling, %d scenes/GPU, random-init weights" % (label, T, B),
                       "name": args.config, "scenes_per_gpu": B, "global_batch": total_scenes,
                       "parallelism": "scene-shard x%d (%s scaling)" % (world, args.scaling),
                       "l2": "per-step working set (activation buffers of %.0f MB each + 63 MB weights) %s the 126 MB L2; "
                             "no explicit flush" % (B * N_OBJ * 512 * 2 / 1e6, "exceeds" if B * N_OBJ * 512 * 2 * 20 > 126e6 else "fits")},
            "denoiser_fwd_us_per_step": us_per_dstep,
            "gpu_launches": int(launches),
            "graph_builds": eng.graph_build_count(),
            "clocks": clk,
        }
        if ms_e2e is not None:
            res["e2e"] = {"value": total_scenes * n_e2e / (ms_e2e / 1000.0), "unit": "scenes/s", "h2d_bytes_per_step": h2d,
                          "d2h_bytes_per_step": int(B * N_OBJ * D_ATTR * 4)}
        if hbm_bound:
            ach = wbytes / (us_per_dstep * 1e-6) / 1e9
            res["roofline"] = {"bound": "hbm", "achieved": ach, "peak": peak_gbs, "unit": "GB/s", "frac": ach / peak_gbs,
                               "traffic": None, "peak_source": which + " HBM copy bandwidth",
                               "launch": "one diffusion step over %d scenes: %.2f MB of weights read once (floor %.1f us)"
                                         % (B, wbytes / 1e6, t_hbm * 1e6)}
        else:
            res["roofline"] = {"bound": "tensor", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                               "frac": achieved_tf / peak_tf, "traffic": None, "peak_source": which + " bf16 sustained",
                               "launch": "one diffusion step (CUDA graph of the step program) over %d scenes; "
                                         "algorithmic %.1f MFLOP/scene/step" % (B, F_SCENE)}
        # dominant kernel: k_gemm_gnt<N>, the channels-on-lanes tcgen05 GEMM that carries the 56 fused conv + GroupNorm
        # + FiLM + SiLU blocks and the epilogue-bound plain GEMMs.  Timed live with CUDA events around each op of one
        # eager pass of the step program (launching stream); DRAM traffic from the committed ncu capture.
        from diffuscene_b200 import capi
        ops = eng.profile_ops(B) if prec == "bf16" else []
        us_by_name = dict(ops)

        def on_gnt(o):      # mirrors gemm_variant() in csrc/engine.cu
            if eng.fuse_level < 2 or N_OBJ not in (12, 21) or o["name"] not in us_by_name:
                return False
            if o["kind"] == 7:
                return True
            k = o["in0"]["k"] + o["in1"]["k"]
            return o["kind"] == 1 and eng.fuse_level >= 3 and o["N"] % 128 == 0 and (k <= 128 or o["N"] % 256 != 0)

        dom = [o for o in capi.plan_export(eng.cfg)["ops"] if on_gnt(o)] if ops else []
        if dom:
            dom_us = sum(us_by_name[o["name"]] for o in dom)
            dom_flop = sum(2.0 * B * N_OBJ * o["N"] * (o["in0"]["k"] + o["in1"]["k"]) for o in dom)
            res["roofline"]["dominant_kernel"] = {
                "name": "k_gemm_gnt<%d> (tcgen05 GEMM, output channels on the TMEM lanes; conv+GroupNorm+FiLM+SiLU "
                        "epilogue, bias-only for the plain launches)" % N_OBJ, "launches_per_step": len(dom),
                "avg_us": dom_us / len(dom), "achieved": dom_flop / (dom_us * 1e-6) / 1e12, "unit": "TFLOP/s",
                "frac": dom_flop / (dom_us * 1e-6) / 1e12 / peak_tf,
                "share_of_step": dom_us / max(1e-9, sum(u for _, u in ops))}
        tpath = os.path.join(ROOT, "profiles", "round2_dram_traffic_%s.json" % args.config)
        if B == scenes and args.fuse is None and os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            res["roofline"]["traffic"] = tj["step_dram_bytes"]
            res["roofline"]["traffic_source"] = "profiles/%s (ncu dram__bytes_read+write, one step)" % os.path.basename(tpath)
            # every instantiation of the kernel that ran in the step (single-CTA and CTA-pair)
            ks = [v for n, v in tj["kernels"].items() if n.startswith("k_gemm_gnt<%d" % N_OBJ)]
            if ks and dom:
                res["roofline"]["dominant_kernel"]["traffic"] = (
                    sum(k["dram_read_bytes"] + k["dram_write_bytes"] for k in ks) / sum(k["launches"] for k in ks))
                res["roofline"]["dominant_kernel"]["ncu_share_of_step"] = sum(k["time_ns"] for k in ks) / tj["step_time_ns"]
        if args.profile_ops:
            tot = sum(u for _, u in ops)
            sys.stderr.write("per-op device time (us), total %.1f\n" % tot)
            for n, u in ops:
                sys.stderr.write("  %-40s %8.1f\n" % (n, u))
        if not args.no_cpu_baseline:
            # bounded sample on the host cores; the same sample gives the parity figure of the benched precision
            arm = CpuArm(args.config)
            arm.step()
            sec = arm.step()
            v = CPU_B / (sec * T)
            res["cpu_baseline"] = {"value": v, "unit": "scenes/s", "cores": arm.threads, "cores_available": arm.cores_available,
                                   "kind": arm.kind, "sample": arm.describe(T), "sec_per_scene_step": sec / CPU_B}
            from oracle.unet1d_ref import unet1d_forward
            sd = seeded_state_dict(unet1d_param_specs(spec), seed=0)
            pb = min(B, 8)
            xs = x_T_host[:pb].clone()
            ts = torch.randint(0, T, (pb,), generator=g)
            cr = None if cross_host is None else cross_host[:pb].clone()
            ref = unet1d_forward(sd, spec, xs, ts, pos_emb[None].expand(pb, N_OBJ, 128).contiguous(), cr)
            if cr is not None:
                eng.set_context_cross(cr.to(dev))
            got = eng.forward(xs.to(dev), ts.to(dev)).cpu()
            if cr is not None:
                eng.set_context_cross(cross_dev)
            res["parity_max_abs"] = float((got - ref).abs().max())
            res["parity_mean_abs"] = float((got - ref).abs().mean())
            b0 = spec.bbox_dim
            res["parity_class_argmax_agreement"] = float(
                (got[..., b0:b0 + spec.class_dim - 1].argmax(-1) == ref[..., b0:b0 + spec.class_dim - 1].argmax(-1)).float().mean())
            res["parity_note"] = "denoiser forward on %d scenes vs the CPU oracle (fp32); %s mode" % (pb, prec)
        print(json.dumps(res))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
