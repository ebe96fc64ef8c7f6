"""Python host wrapper over the C ABI: owns one `ds_handle`, feeds it torch-allocated device memory.

PyTorch is plumbing here (device allocations, streams); every FLOP of the denoiser and of the
diffusion step runs in the CUDA library.  If the library or the GPU is missing, construction raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import capi
from .schedule import DiffusionTables
from .weights import NetSpec

_PREC = {"fp32": capi.DS_PREC_FP32, "bf16": capi.DS_PREC_BF16}
_BACKEND = {"auto": capi.DS_GEMM_AUTO, "simt": capi.DS_GEMM_SIMT, "tcgen05": capi.DS_GEMM_TCGEN05}
LOSS_KEYS = ["loss.bbox", "loss.trans", "loss.size", "loss.angle", "loss.class", "loss.object", "loss.objfeat",
             "loss.liou", "loss.bbox_iou"]


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


class DenoiserEngine:
    """One Unet1D + diffusion schedule on one GPU (reference: DiffusionPoint, diffusion_ddpm.py:721-803)."""

    def __init__(self, spec: NetSpec, num_objects: int, num_timesteps: int, precision: str = "bf16",
                 gemm_backend: str = "auto", device: int = 0, fuse_level: Optional[int] = None):
        if not torch.cuda.is_available():
            raise RuntimeError("diffuscene_b200 needs a CUDA device (B200, sm_100a); there is no CPU path")
        self.lib = capi.load()
        self.spec = spec
        self.num_objects = num_objects
        self.num_timesteps = num_timesteps
        self.precision = precision
        self.device = torch.device("cuda", device)
        if fuse_level is None:      # fused GEMM epilogues exist for the tcgen05 path only
            # 2: conv + GroupNorm GEMMs with the channels on the TMEM lanes where the library supports the shape
            # (N = 12 objects), the row-major fused kernel (level 1) otherwise
            # 3: ... and the epilogue-bound plain GEMMs (to_qkv, to_out) on the same kernel
            # 4: ... and to_out + LayerNorm + residual of the attention wrappers as one kernel (k_gemm_ln)
            # 5: ... and LayerNorm + to_qkv + linear-attention core as one kernel (k_ln_qkv_attn, N = 12)
            fuse_level = 5 if (precision == "bf16" and gemm_backend != "simt") else 0
        self.fuse_level = fuse_level
        self.cfg = capi.make_config(spec, num_objects, num_timesteps, _PREC[precision], _BACKEND[gemm_backend],
                                    device, fuse_level)
        h = C.c_void_p()
        capi.check(self.lib.ds_create(C.byref(self.cfg), C.byref(h)))
        self.h = h
        self.d = spec.point_dim
        self.tables: Optional[DiffusionTables] = None
        self._keep: List[torch.Tensor] = []

    def close(self):
        if getattr(self, "h", None):
            self.lib.ds_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- weights --------------------------------------------------------------------------------
    def expected_weights(self) -> List[tuple]:
        n = self.lib.ds_expected_weight_count(self.h)
        out = []
        for i in range(n):
            name, numel = C.c_char_p(), C.c_int64()
            capi.check(self.lib.ds_expected_weight(self.h, i, C.byref(name), C.byref(numel)))
            out.append((name.value.decode(), numel.value))
        return out

    def load_state_dict(self, sd: Dict[str, torch.Tensor], prefix: str = "diffusion.model."):
        """Load reference-format weights (keys as in the reference checkpoints) and commit them."""
        for name, numel in self.expected_weights():
            key = prefix + name
            if key not in sd:
                raise KeyError("state dict is missing '%s'" % key)
            w = sd[key].detach().to(device="cpu", dtype=torch.float32).contiguous()
            if w.numel() != numel:
                raise ValueError("'%s' has %d elements, expected %d" % (key, w.numel(), numel))
            capi.check(self.lib.ds_load_weight(self.h, name.encode(), C.c_void_p(w.data_ptr()), numel))
        capi.check(self.lib.ds_commit_weights(self.h))

    # ---- schedule / conditioning ----------------------------------------------------------------
    def set_schedule(self, tables: DiffusionTables):
        s = capi.DsSchedule()
        s.T = tables.T
        s.mean_type = capi.MEAN_TYPES[tables.mean_type]
        keep = []
        for f in ("sqrt_ac", "sqrt_1mac", "sqrt_recip_ac", "sqrt_recipm1_ac", "coef1", "coef2", "sigma",
                  "alphas_cumprod", "loss_weight"):
            a = tables[f].detach().to(dtype=torch.float32, device="cpu").contiguous()
            keep.append(a)
            setattr(s, f, C.cast(C.c_void_p(a.data_ptr()), C.POINTER(C.c_float)))
        capi.check(self.lib.ds_set_schedule(self.h, C.byref(s)))
        self.tables = tables

    def set_context(self, context: torch.Tensor, shared: Optional[bool] = None):
        """context: [B, N, cond_dim] or [N, cond_dim] (shared over the batch), fp32."""
        if context.dim() == 2:
            shared, batch = True, 0
        else:
            batch = context.shape[0]
            if shared is None:
                shared = False
            if shared:
                context = context[0]
        ctx = context.detach().to(device=self.device, dtype=torch.float32).contiguous()
        capi.check(self.lib.ds_set_context(self.h, _ptr(ctx), batch, int(bool(shared)), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()

    def set_context_cross(self, cross: Optional[torch.Tensor]):
        if cross is None:
            capi.check(self.lib.ds_set_context_cross(self.h, None, 0, 0, self._stream()))
            return
        c = cross.detach().to(device=self.device, dtype=torch.float32).contiguous()
        capi.check(self.lib.ds_set_context_cross(self.h, _ptr(c), c.shape[0], c.shape[1], self._stream()))
        torch.cuda.current_stream(self.device).synchronize()

    # ---- denoiser -------------------------------------------------------------------------------
    def forward(self, x_t: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
        """Unet1D.forward on device tensors: x_t [B, N, d] fp32, t [B] int64 -> [B, N, d] fp32."""
        assert x_t.is_cuda and x_t.dtype == torch.float32 and t.dtype == torch.int64
        x_t, t = x_t.contiguous(), t.to(self.device).contiguous()
        out = torch.empty_like(x_t)
        capi.check(self.lib.ds_denoise_forward(self.h, _ptr(x_t), _ptr(t), _ptr(out), x_t.shape[0], self._stream()))
        return out

    def forward_host(self, x_t: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
        """Same through HOST buffers (H2D + D2H inside the call)."""
        x_t = x_t.detach().to("cpu", torch.float32).contiguous()
        t = t.detach().to("cpu", torch.int64).contiguous()
        out = torch.empty_like(x_t)
        capi.check(self.lib.ds_denoise_forward_host(self.h, _ptr(x_t), _ptr(t), _ptr(out), x_t.shape[0]))
        return out

    # ---- sampling -------------------------------------------------------------------------------
    def _sample_args(self, batch, clip_denoised, num_steps, ddim, ddim_eta, seed, scene_offset, x_init, noise,
                     partial, partial_noise, traj_freq, traj, use_graph, ddim_times, chunk_scenes=0):
        a = capi.DsSampleArgs()
        a.chunk_scenes = int(chunk_scenes)
        a.batch, a.clip_denoised, a.num_steps = batch, int(clip_denoised), num_steps
        a.ddim, a.ddim_eta, a.seed, a.scene_offset = int(ddim), float(ddim_eta), seed, scene_offset
        a.x_init_dev = None if x_init is None else x_init.data_ptr()
        a.noise_dev = None if noise is None else noise.data_ptr()
        a.partial_dev = None if partial is None else partial.data_ptr()
        a.num_partial = 0 if partial is None else partial.shape[1]
        a.partial_noise_dev = None if partial_noise is None else partial_noise.data_ptr()
        a.traj_freq = traj_freq
        a.traj_dev = None if traj is None else traj.data_ptr()
        a.use_graph = int(use_graph)
        if ddim_times is not None:
            arr = (C.c_int32 * len(ddim_times))(*ddim_times)
            self._keep = [arr]
            a.ddim_times = C.cast(arr, C.POINTER(C.c_int32))
        return a

    def sample(self, batch: int, clip_denoised: bool = True, num_steps: int = 0, ddim: bool = False,
               ddim_eta: float = 0.0, seed: int = 0, scene_offset: int = 0, x_init: Optional[torch.Tensor] = None,
               noise: Optional[torch.Tensor] = None, partial: Optional[torch.Tensor] = None,
               partial_noise: Optional[torch.Tensor] = None, traj_freq: int = 0, use_graph: bool = True,
               ddim_times: Optional[Sequence[int]] = None, host_output: bool = False, chunk_scenes: int = 0):
        """p_sample_loop (diffusion_ddpm.py:355-371) and its trajectory / completion / DDIM variants.

        noise: optional [steps, B, N, d] injected step noise (loop order T-1 .. 0); x_init: optional x_T.
        Returns x_0 [B, N, d] (device, or host when host_output), or (x_0, trajectory) when traj_freq > 0."""
        dev = self.device
        f = lambda z: None if z is None else z.detach().to(device=dev, dtype=torch.float32).contiguous()
        x_init, noise, partial, partial_noise = f(x_init), f(noise), f(partial), f(partial_noise)
        if ddim and ddim_times is None:
            # the reference's grid expression, evaluated by torch itself (fp32 linspace, then .int()):
            # diffusion_ddpm.py:407-408 -- identical truncation when S does not divide T
            S = num_steps if num_steps > 0 else 50
            ddim_times = list(reversed(torch.linspace(-1, self.num_timesteps - 1, steps=S + 1).int().tolist()))
        traj = None
        if traj_freq > 0:
            if ddim:      # snapshots follow the timestep VALUES the loop visits (engine.cu: ts[i] % freq == 0 or i == 0)
                n_snap = sum(1 for i, tt in enumerate(ddim_times[:-1]) if tt % traj_freq == 0 or i == 0)
            else:
                n_snap = self.lib.ds_traj_count(num_steps if num_steps > 0 else self.num_timesteps, traj_freq)
            traj = torch.zeros((n_snap, batch, self.num_objects, self.d), device=dev, dtype=torch.float32)
        a = self._sample_args(batch, clip_denoised, num_steps, ddim, ddim_eta, seed, scene_offset, x_init, noise,
                              partial, partial_noise, traj_freq, traj, use_graph, ddim_times, chunk_scenes)
        torch.cuda.current_stream(dev).synchronize()
        if host_output:
            out = torch.empty((batch, self.num_objects, self.d), dtype=torch.float32).pin_memory()
            capi.check(self.lib.ds_sample_loop_host(self.h, C.byref(a), _ptr(out)))
        else:
            out = torch.empty((batch, self.num_objects, self.d), device=dev, dtype=torch.float32)
            capi.check(self.lib.ds_sample_loop(self.h, C.byref(a), _ptr(out), None))
        return (out, traj) if traj is not None else out

    def p_sample_step(self, x_t: torch.Tensor, t: torch.Tensor, noise: torch.Tensor, clip_denoised: bool):
        x_t, t, noise = x_t.contiguous(), t.to(self.device).contiguous(), noise.to(self.device).contiguous()
        out = torch.empty_like(x_t)
        capi.check(self.lib.ds_p_sample_step(self.h, _ptr(x_t), _ptr(t), _ptr(noise), int(clip_denoised), _ptr(out),
                                             x_t.shape[0], self._stream()))
        return out

    def q_sample(self, x0: torch.Tensor, t: torch.Tensor, noise: torch.Tensor):
        x0, t, noise = x0.contiguous(), t.to(self.device).contiguous(), noise.contiguous()
        out = torch.empty_like(x0)
        capi.check(self.lib.ds_q_sample(self.h, _ptr(x0), _ptr(t), _ptr(noise), _ptr(out), x0.shape[0], self._stream()))
        return out

    def p_losses(self, x0: torch.Tensor, t: torch.Tensor, noise: torch.Tensor, loss_separate: bool, loss_iou: bool,
                 bounds: Optional[Sequence[float]] = None):
        """Forward value of p_losses (diffusion_ddpm.py:520-652): (losses [B], dict of 9 scalar means)."""
        x0, t, noise = x0.contiguous(), t.to(self.device).contiguous(), noise.contiguous()
        B = x0.shape[0]
        losses = torch.empty(B, device=self.device, dtype=torch.float32)
        ld = torch.empty(9, device=self.device, dtype=torch.float32)
        barr = None
        if bounds is not None:
            barr = (C.c_float * 12)(*[float(v) for v in bounds])
        capi.check(self.lib.ds_p_losses(self.h, _ptr(x0), _ptr(t), _ptr(noise), int(loss_separate), int(loss_iou),
                                        barr, _ptr(losses), _ptr(ld), B, self._stream()))
        return losses, {k: ld[i] for i, k in enumerate(LOSS_KEYS)}

    # ---- native training ------------------------------------------------------------------------
    def flat_layout(self, prefix: str = "diffusion.model.") -> Dict[str, tuple]:
        """name -> (offset, numel) of every denoiser parameter inside the flat fp32 parameter / gradient buffers."""
        out, off = {}, 0
        for name, numel in self.expected_weights():
            out[prefix + name] = (off, numel)
            off += numel
        return out

    def train_step(self, flat_params: torch.Tensor, x0: torch.Tensor, t: torch.Tensor, noise: torch.Tensor,
                   context: torch.Tensor, shared: bool, loss_separate: bool, loss_iou: bool,
                   bounds: Optional[Sequence[float]] = None, flat_grads: Optional[torch.Tensor] = None,
                   want_dcontext: bool = True, grad_scale: float = 1.0,
                   context_cross: Optional[torch.Tensor] = None):
        """Forward of p_losses + the native backward pass: (losses [B], loss dict, d(context) or None).
        Gradients of every denoiser parameter land in `flat_grads` (flat_layout order).

        Text-conditioned networks pass `context_cross` [B, L, text_dim] (the input of every cross-attention to_kv);
        the result then has a fourth entry, d(context_cross) (None without flat_grads)."""
        assert flat_params.is_cuda and flat_params.dtype == torch.float32 and flat_params.is_contiguous()
        x0, t, noise = x0.contiguous(), t.to(self.device).contiguous(), noise.contiguous()
        ctx = context.detach().to(self.device, torch.float32).contiguous()
        B = x0.shape[0]
        losses = torch.empty(B, device=self.device, dtype=torch.float32)
        ld = torch.empty(9, device=self.device, dtype=torch.float32)
        dctx = torch.empty_like(ctx) if (want_dcontext and flat_grads is not None) else None
        barr = None if bounds is None else (C.c_float * 12)(*[float(v) for v in bounds])
        cross = dcross = None
        if context_cross is not None:
            cross = context_cross.detach().to(self.device, torch.float32).contiguous()
            dcross = torch.empty_like(cross) if flat_grads is not None else None
            capi.check(self.lib.ds_train_set_context_cross(self.h, _ptr(cross), cross.shape[0], cross.shape[1],
                                                           _ptr(dcross)))
        try:
            capi.check(self.lib.ds_train_step(self.h, _ptr(flat_params), _ptr(x0), _ptr(t), _ptr(noise), _ptr(ctx),
                                              0 if shared else B, int(bool(shared)), int(loss_separate), int(loss_iou),
                                              barr, float(grad_scale), _ptr(losses), _ptr(ld), _ptr(flat_grads),
                                              _ptr(dctx), B, self._stream()))
        finally:
            if cross is not None:      # the handle only borrows the pointers: never leave them behind
                capi.check(self.lib.ds_train_set_context_cross(self.h, None, 0, 0, None))
        out = (losses, {k: ld[i] for i, k in enumerate(LOSS_KEYS)}, dctx)
        return out + (dcross,) if context_cross is not None else out

    def train_set_buckets(self, bounds: Sequence[int], events: Sequence["torch.cuda.Event"]):
        """Gradient buckets for the overlapped all-reduce (see ds_train_set_buckets); `events` are torch.cuda.Event
        objects (recorded once so that their cudaEvent_t exists), kept alive by this object."""
        n = len(events)
        self._bucket_events = list(events)
        arr_b = (C.c_int64 * (n + 1))(*[int(b) for b in bounds]) if n else None
        arr_e = (C.c_void_p * n)(*[C.c_void_p(e.cuda_event) for e in events]) if n else None
        capi.check(self.lib.ds_train_set_buckets(self.h, arr_b, n, arr_e))

    def train_phase_ms(self):
        out = (C.c_float * 6)()
        capi.check(self.lib.ds_train_phase_ms(self.h, out))
        return dict(zip(("pack", "forward", "loss", "backward", "cond_paths", "unpack"), [float(v) for v in out]))

    # ---- debugging ------------------------------------------------------------------------------
    def enable_taps(self, on: bool = True):
        capi.check(self.lib.ds_enable_taps(self.h, int(on)))

    def read_tap(self, name: str, rows: int) -> torch.Tensor:
        cap = 1 << 26
        buf = torch.empty(cap, dtype=torch.float32)
        r, w = C.c_int32(), C.c_int32()
        capi.check(self.lib.ds_read_tap(self.h, name.encode(), _ptr(buf), cap, C.byref(r), C.byref(w)))
        return buf[: r.value * w.value].reshape(r.value, w.value)[:rows].clone()

    def launch_count(self) -> int:
        return int(self.lib.ds_launch_count(self.h))

    def graph_build_count(self) -> int:
        return int(self.lib.ds_graph_build_count(self.h))

    def profile_ops(self, batch: int):
        names = C.create_string_buffer(1 << 16)
        us = (C.c_float * 1024)()
        n = capi.check(self.lib.ds_profile_ops(self.h, batch, names, len(names), us, 1024))
        nm = names.value.decode().strip().split("\n")
        return [(nm[i], us[i]) for i in range(min(n, len(nm)))]
