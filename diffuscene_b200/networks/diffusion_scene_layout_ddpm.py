"""Drop-in model class for the reference's `DiffusionSceneLayout_DDPM`
(scene_synthesis/networks/diffusion_scene_layout_ddpm.py:14-482) backed by the CUDA engine.

Same constructor arguments, same public methods (`get_loss`, `sample`, `generate_layout`,
`generate_layout_progressive`, `complete_scene`, `arrange_scene`, `delete_empty_from_network_samples`,
`delete_empty_boxes`) and the same state-dict key names (`positional_embedding`, `diffusion.model.*`,
`fc_*`), so reference checkpoints load unchanged.  Parameters are fp32 `nn.Parameter`s (the master copy the
optimizer updates); the engine keeps a packed copy that is refreshed lazily when the parameters change.

Sampling, validation loss, every diffusion step and the training step (forward and backward pass of the denoiser,
`ds_train_step`) run in the CUDA library; `native_backward = False` differentiates `functional.DenoiserFn` with
torch autograd instead (the reference path the tests compare against).  Differences from the reference that are deliberate: the per-call `print`s are gone, `sample()` honours
`ddim=True` (the reference ignores it and its DDIM loop is dead code), and emptiness is decided per scene when
batch_size > 1 via `delete_empty_batched` (the reference looks at batch row 0 only).  Like the reference
(`sample()` dispatches on input_boxes / partial_boxes first, :293-299), `complete_scene` / `arrange_scene` accept
`ret_traj` / `ddim` and ignore them.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch
import torch.nn as nn
from torch.nn.utils import clip_grad_norm_

from ..engine import DenoiserEngine
from ..optim import NativeAdam
from ..parallel import allreduce_flat, allreduce_gradients
from ..schedule import get_betas, make_tables
from ..stats_logger import StatsLogger
from ..weights import NetSpec, seeded_tensor, unet1d_param_specs
from .functional import DenoiserFn


class _Tree(nn.Module):
    """Plain container whose children are created on demand from dotted parameter names."""


def _register(root: nn.Module, dotted: str, param: nn.Parameter):
    parts = dotted.split(".")
    mod = root
    for part in parts[:-1]:
        if part not in mod._modules:
            mod.add_module(part, _Tree())
        mod = mod._modules[part]
    mod.register_parameter(parts[-1], param)


class _NativeTrainLoss(torch.autograd.Function):
    """p_losses(...).mean() with the forward AND the backward pass of the denoiser in the CUDA library (ds_train_step).
    The differentiable inputs are the conditioning tensor and, for text networks, `context_cross` (their gradients
    flow on into positional_embedding / the condition MLPs / fc_text_f through ordinary autograd); the denoiser
    parameters receive their gradients as views of the model's flat gradient buffer when backward() runs."""

    @staticmethod
    def forward(ctx, cond, cross, model, x0, t, noise, shared):
        losses, ld, dcond, dcross = model._native_fwd_bwd(x0, t, noise, cond, shared, cross)
        ctx.model, ctx.dcond, ctx.dcross = model, dcond, dcross
        model._last_loss_dict = ld
        return losses.mean()

    @staticmethod
    def backward(ctx, g):
        ctx.model._assign_native_grads(g)
        d, dx = ctx.dcond, ctx.dcross
        dx = dx * g if (dx is not None and ctx.needs_input_grad[1]) else None
        return (None if d is None else d * g), dx, None, None, None, None, None


class DiffusionSceneLayout_DDPM(nn.Module):
    def __init__(self, n_classes, feature_extractor, config, precision: str = "bf16", gemm_backend: str = "auto"):
        super().__init__()
        self.room_mask_condition = config.get("room_mask_condition", True)
        self.text_condition = config.get("text_condition", False)
        self.text_glove_embedding = config.get("text_glove_embedding", False)
        self.text_clip_embedding = config.get("text_clip_embedding", False)
        if self.room_mask_condition:
            raise NotImplementedError("room_mask_condition (floor-plan encoder) is outside the hot path; every "
                                      "shipped config sets it to false")
        if self.text_condition:
            text_embed_dim = config.get("text_embed_dim", 512)
            if self.text_glove_embedding:
                self.fc_text_f = nn.Linear(50, text_embed_dim)
            elif self.text_clip_embedding:
                raise NotImplementedError("CLIP text embedding needs the `clip` package (absent)")
            else:
                # the frozen BERT encoder runs once per scene outside the denoising loop; it is loaded lazily so
                # that synthetic `context_cross` tensors can be used without the HF checkpoint (no network here)
                # The encoder is frozen and is NOT a registered submodule (object.__setattr__): the state dict of
                # this class never carries `bertmodel.*`, whether or not BERT has been loaded; reference
                # checkpoints, which do carry those keys, load through the filter in load_state_dict below.
                self.tokenizer = None
                object.__setattr__(self, "bertmodel", None)
                self.fc_text_f = nn.Linear(768, text_embed_dim)
        if config["net_type"] != "unet1d":
            raise NotImplementedError()

        self.n_classes = n_classes
        self.config = config
        self.objectness_dim = config.get("objectness_dim", 1)
        self.class_dim = config.get("class_dim", 21)
        self.translation_dim = config.get("translation_dim", 3)
        self.size_dim = config.get("size_dim", 3)
        self.angle_dim = config.get("angle_dim", 1)
        self.bbox_dim = self.translation_dim + self.size_dim + self.angle_dim
        self.objfeat_dim = config.get("objfeat_dim", 0)

        self.learnable_embedding = config.get("learnable_embedding", False)
        self.instance_condition = config.get("instance_condition", False)
        self.sample_num_points = config.get("sample_num_points", 12)
        self.instance_emb_dim = config.get("instance_emb_dim", 64)
        if self.learnable_embedding:
            if self.instance_condition:
                self.register_parameter("positional_embedding",
                                        nn.Parameter(torch.randn(self.sample_num_points, self.instance_emb_dim)))
            else:
                self.instance_emb_dim = 0
        else:
            if self.instance_condition:
                self.fc_instance_condition = nn.Sequential(
                    nn.Linear(self.sample_num_points, self.instance_emb_dim, bias=False),
                    nn.LeakyReLU(0.1, inplace=True),
                    nn.Linear(self.instance_emb_dim, self.instance_emb_dim, bias=False))
            else:
                self.instance_emb_dim = 0
        self.room_partial_condition = config.get("room_partial_condition", False)
        self.partial_num_points = config.get("partial_num_points", 0)
        self.partial_emb_dim = config.get("partial_emb_dim", 64)
        if self.room_partial_condition:
            self.fc_partial_condition = nn.Sequential(
                nn.Linear(self.bbox_dim + self.class_dim + self.objectness_dim + self.objfeat_dim,
                          self.partial_emb_dim, bias=False),
                nn.LeakyReLU(0.1, inplace=True),
                nn.Linear(self.partial_emb_dim, self.partial_emb_dim, bias=False))
        else:
            self.partial_emb_dim = 0
        self.room_arrange_condition = config.get("room_arrange_condition", False)
        self.arrange_emb_dim = config.get("arrange_emb_dim", 64)
        if self.room_arrange_condition:
            self.fc_arrange_condition = nn.Sequential(
                nn.Linear(self.size_dim + self.class_dim + self.objectness_dim + self.objfeat_dim,
                          self.arrange_emb_dim, bias=False),
                nn.LeakyReLU(0.1, inplace=True),
                nn.Linear(self.arrange_emb_dim, self.arrange_emb_dim, bias=False))
        else:
            self.arrange_emb_dim = 0

        # ---- denoiser parameters under the reference's names ("diffusion.model.*") ----
        self.spec = NetSpec.from_net_kwargs(config["net_kwargs"])
        self._param_names: List[str] = []
        seed = int(torch.randint(0, 2 ** 31 - 1, (1,)).item())      # follows torch.manual_seed like nn init does
        for name, shape, kind in unet1d_param_specs(self.spec):
            _register(self, name, nn.Parameter(seeded_tensor(name, shape, kind, seed, perturb_norms=False)))
            self._param_names.append(name)

        dk = dict(config["diffusion_kwargs"])
        self.time_num = dk.get("time_num", 1000)
        self.mean_type = dk.get("model_mean_type", "eps")
        self.var_type = dk.get("model_var_type", "fixedsmall")
        self.loss_type = dk.get("loss_type", "mse")
        self.loss_separate = dk.get("loss_separate", False)
        self.loss_iou = dk.get("loss_iou", False)
        if self.loss_type != "mse":
            raise NotImplementedError("loss_type %r (the reference's 'kl' branch is broken: SURVEY A.6.6)" % self.loss_type)
        self.tables = make_tables(get_betas(dk.get("schedule_type", "linear"), dk.get("beta_start", 1e-4),
                                            dk.get("beta_end", 0.02), self.time_num), self.mean_type, self.var_type)
        self.bounds = None
        if self.loss_iou:
            import json
            with open(dk["train_stats_file"], "r") as f:
                st = json.load(f)
            self.bounds = list(st["bounds_translations"]) + list(st["bounds_sizes"])

        self._precision = precision
        self._backend = gemm_backend
        self._engine: Optional[DenoiserEngine] = None
        self._flat = None
        self._flat_layout = None
        self._flat_grads = None
        self._native_grads_ready = False
        self._overlap = None
        self.native_backward = True      # False: differentiate functional.DenoiserFn with torch autograd instead
        self._weights_version = 0
        self._engine_version = -1
        self.register_load_state_dict_post_hook(lambda module, incompatible: module.mark_weights_dirty())

    # ---- checkpoints ----------------------------------------------------------------------------
    FROZEN_PREFIXES = ("bertmodel.", "clip_model.", "feature_extractor.", "fc_room_f.")

    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        """Reference checkpoints of the text configs carry the frozen encoder (`bertmodel.*`: the reference
        registers it as a submodule, diffusion_scene_layout_ddpm.py:47-48); those keys are dropped here -- the
        encoder is loaded from its own pretrained files -- so that `strict=True` keeps checking everything that
        is trained on this path."""
        sd = {k: v for k, v in state_dict.items() if not k.startswith(self.FROZEN_PREFIXES)}
        return super().load_state_dict(sd, strict=strict, **kw)

    # ---- engine management ----------------------------------------------------------------------
    def mark_weights_dirty(self):
        self._weights_version += 1

    def _device(self) -> torch.device:
        return next(self.parameters()).device

    def engine(self, commit: bool = True) -> DenoiserEngine:
        """The CUDA engine of this model; commit=False skips the refresh of the sampling-side packed weights (the
        training step reads the flat parameter buffer directly)."""
        dev = self._device()
        if dev.type != "cuda":
            raise RuntimeError("DiffusionSceneLayout_DDPM runs on a CUDA device only (no CPU fallback); call .to('cuda')")
        if self._engine is None:
            self._engine = DenoiserEngine(self.spec, self.sample_num_points, self.time_num, precision=self._precision,
                                          gemm_backend=self._backend, device=dev.index or 0)
            self._engine.set_schedule(self.tables)
        if commit and self._engine_version != self._weights_version:
            sd = {n: p.detach() for n, p in self.named_parameters() if n.startswith("diffusion.model.")}
            self._engine.load_state_dict(sd)
            self._engine_version = self._weights_version
        return self._engine

    # ---- native training: flat parameter / gradient buffers ---------------------------------------
    def native_training_supported(self) -> bool:
        return self.sample_num_points <= 32 and self._device().type == "cuda"

    def _ensure_flat(self):
        """All denoiser parameters as views into ONE flat fp32 device buffer (ds_expected_weight order), gradients
        likewise: the native training step, the fused Adam and the data-parallel all-reduce work on these two
        contiguous buffers; state_dict / load_state_dict / optimizers keep seeing ordinary nn.Parameters."""
        eng = self.engine(commit=False)
        params = dict(self.named_parameters())
        if self._flat is not None:
            base = self._flat.data_ptr()
            if all(params[n].data_ptr() == base + 4 * off for n, (off, _) in self._flat_layout.items()):
                return eng
        layout = eng.flat_layout()
        total = sum(n for _, n in layout.values())
        dev = self._device()
        flat = torch.empty(total, device=dev, dtype=torch.float32)
        for name, (off, n) in layout.items():
            p = params[name]
            flat[off:off + n].copy_(p.data.reshape(-1))
            p.data = flat[off:off + n].view(p.shape)
            p._ds_flat_owner = self
        self._flat, self._flat_layout = flat, layout
        self._flat_grads = torch.zeros(total, device=dev, dtype=torch.float32)
        self._native_grads_ready = False
        self._overlap = None
        return eng

    def _native_fwd_bwd(self, x0, t, noise, cond, shared, cross=None):
        eng = self._ensure_flat()
        world = torch.distributed.get_world_size() if (torch.distributed.is_available() and torch.distributed.is_initialized()) else 1
        if world > 1 and self._overlap is None:
            from ..parallel import GradOverlap
            self._overlap = GradOverlap(eng, self._flat_grads)
        res = eng.train_step(self._flat, x0, t, noise, cond, shared, self.loss_separate, self.loss_iou, self.bounds,
                             flat_grads=self._flat_grads, grad_scale=1.0 / world, context_cross=cross)
        losses, ld, dcond = res[:3]
        dcross = res[3] if cross is not None else None
        if world > 1:
            # the kernels of the backward pass are only ENQUEUED at this point: the bucket all-reduces go to a side
            # stream, each gated by the event the engine records when that bucket's gradients are final
            self._overlap.launch()
        self._native_grads_ready = False
        return losses, ld, dcond, dcross

    def _assign_native_grads(self, g):
        """Called from the autograd node of the native loss: expose the flat gradient buffer as the .grad of every
        denoiser parameter (views, no copies)."""
        if self._overlap is not None:
            self._overlap.wait()                 # the current stream waits for the bucket all-reduces
        if not (torch.is_tensor(g) and g.numel() == 1 and float(g) == 1.0):
            self._flat_grads.mul_(g)
        params = dict(self.named_parameters())
        for name, (off, n) in self._flat_layout.items():
            p = params[name]
            view = self._flat_grads[off:off + n].view(p.shape)
            if p.grad is None or p.grad.data_ptr() == view.data_ptr():
                p.grad = view
            else:                      # gradient accumulation across several backward() calls
                p.grad = p.grad + view
        self._native_grads_ready = True

    def _denoiser_params(self) -> Dict[str, torch.Tensor]:
        pre = "diffusion.model."
        return {n[len(pre):]: p for n, p in self.named_parameters() if n.startswith(pre)}

    # ---- conditioning (reference :162-221, :234-291) ---------------------------------------------
    def _instance_condition(self, batch, device):
        if not self.instance_condition:
            return None, False
        if self.learnable_embedding:
            return self.positional_embedding, True           # [N, E], identical for every scene
        eye = torch.eye(self.sample_num_points, device=device)
        return self.fc_instance_condition(eye), True

    def _condition(self, batch, device, layout_target=None, partial_boxes=None, input_boxes=None, num_points=None):
        """Returns (condition [B,N,E] or [N,E], shared flag)."""
        inst, shared = self._instance_condition(batch, device)
        cond = inst
        N = num_points or self.sample_num_points
        if self.room_partial_condition:
            if partial_boxes is not None:
                zeros = torch.zeros((batch, N - partial_boxes.shape[1], partial_boxes.shape[2]), device=device)
                partial_input = torch.cat([partial_boxes, zeros], dim=1)
            else:
                mask = torch.cat([torch.ones((batch, self.partial_num_points, 1), device=device),
                                  torch.zeros((batch, N - self.partial_num_points, 1), device=device)], dim=1)
                partial_input = layout_target * mask
            f = self.fc_partial_condition(partial_input)
            cond = torch.cat([cond[None].expand(batch, -1, -1) if cond.dim() == 2 else cond, f], dim=-1)
            shared = False
        if self.room_arrange_condition:
            src = input_boxes if input_boxes is not None else layout_target
            arr = torch.cat([src[:, :, self.translation_dim:self.translation_dim + self.size_dim],
                             src[:, :, self.bbox_dim:]], dim=-1)
            f = self.fc_arrange_condition(arr)
            cond = torch.cat([cond[None].expand(batch, -1, -1) if cond.dim() == 2 else cond, f], dim=-1)
            shared = False
        return cond, shared

    def _text_condition(self, text, device):
        if not self.text_condition:
            return None
        if torch.is_tensor(text):
            if text.dim() == 3 and text.shape[-1] == self.spec.text_dim:
                return text.to(device)                        # already-projected [B, L, text_dim] (synthetic prefix)
            return self.fc_text_f(text.to(device))            # GloVe [B, L, 50] or BERT hidden states [B, L, 768]
        if self.text_glove_embedding:
            raise ValueError("glove text condition expects the desc_emb tensor")
        if self.bertmodel is None:
            from transformers import BertModel, BertTokenizer
            self.tokenizer = BertTokenizer.from_pretrained("bert-base-cased")
            bert = BertModel.from_pretrained("bert-base-cased").to(device).eval()
            for p in bert.parameters():
                p.requires_grad = False
            object.__setattr__(self, "bertmodel", bert)          # frozen, kept out of _modules / state_dict
        tok = self.tokenizer(text, return_tensors="pt", padding=True).to(device)
        with torch.no_grad():
            hid = self.bertmodel(**tok).last_hidden_state
        return self.fc_text_f(hid)

    # ---- training loss (reference :131-226) -------------------------------------------------------
    def _pack_target(self, sample_params):
        parts = [sample_params["translations"], sample_params["sizes"], sample_params["angles"],
                 sample_params["class_labels"]]
        if self.objectness_dim > 0:
            parts.append(sample_params["objectness"])
        if self.objfeat_dim > 0:
            parts.append(sample_params["objfeats_32"] if self.objfeat_dim == 32 else sample_params["objfeats"])
        full = torch.cat(parts, dim=-1).contiguous()
        pd = self.config["point_dim"]
        if pd == full.shape[-1]:
            return full
        if pd == self.bbox_dim:
            return full[..., :self.bbox_dim].contiguous()
        raise NotImplementedError

    def get_loss(self, sample_params, t=None, noise=None):
        """Reference :131-226.  `t` / `noise` (optional) replace the draws of diffusion_ddpm.py:764,767 -- the
        parity tests inject the numbers the reference drew."""
        target = self._pack_target(sample_params).float()
        B, N, _ = target.shape
        device = target.device
        cond, shared = self._condition(B, device, layout_target=target)
        if self.room_arrange_condition:
            target = torch.cat([target[:, :, :self.translation_dim],
                                target[:, :, self.translation_dim + self.size_dim:self.bbox_dim]], dim=-1).contiguous()
        text = sample_params.get("desc_emb") if self.text_glove_embedding else sample_params.get("description")
        if self.text_condition and "context_cross" in sample_params:
            text = sample_params["context_cross"]
        cross = self._text_condition(text, device) if self.text_condition else None
        t = torch.randint(0, self.time_num, (B,), device=device) if t is None else t.to(device)
        noise = torch.randn_like(target) if noise is None else noise.to(device)
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            if self.native_backward and self.native_training_supported():
                c = cond if cond.requires_grad else cond.detach().requires_grad_(True)
                loss = _NativeTrainLoss.apply(c, cross, self, target, t, noise, shared)
                ld = self._last_loss_dict
                if self.room_arrange_condition:
                    ld = {k: ld[k] for k in ("loss.trans", "loss.angle")}
                return loss, ld
            losses, ld = self._p_losses_autograd(target, t, noise, cond, shared, cross)
        else:
            losses, ld = self.p_losses_native(target, t, noise, cond, shared, cross)
        return losses.mean(), ld

    def p_losses_native(self, x0, t, noise, cond, shared, cross=None):
        """Forward value of p_losses entirely in the CUDA library (validation path)."""
        eng = self.engine()
        eng.set_context(cond.detach(), shared=shared)
        if self.text_condition:
            eng.set_context_cross(cross.detach())
        losses, ld = eng.p_losses(x0, t, noise, self.loss_separate, self.loss_iou, self.bounds)
        if self.room_arrange_condition:      # the reference logs only these two for arrangement (diffusion_ddpm.py:560-572)
            ld = {k: ld[k] for k in ("loss.trans", "loss.angle")}
        return losses, ld

    def _p_losses_autograd(self, x0, t, noise, cond, shared, cross):
        """p_losses (diffusion_ddpm.py:520-652) with torch autograd for the backward pass."""
        tb = {k: v.to(x0.device) for k, v in self.tables.tables.items()}
        ex = lambda a: a[t].reshape(-1, 1, 1)
        x_t = ex(tb["sqrt_ac"]) * x0 + ex(tb["sqrt_1mac"]) * noise
        if self.mean_type == "eps":
            target = noise
        elif self.mean_type == "x0":
            target = x0
        else:
            target = ex(tb["sqrt_ac"]) * noise - ex(tb["sqrt_1mac"]) * x0
        if cond.dim() == 2:
            cond = cond[None].expand(x0.shape[0], -1, -1)
        out = DenoiserFn(self._denoiser_params(), self.spec)(x_t, t, cond, cross)
        sq = (target - out) ** 2
        m = lambda a, b: sq[:, :, a:b].mean(dim=(1, 2))
        td, sd, ad, cd = self.translation_dim, self.size_dim, self.angle_dim, self.class_dim
        zero = torch.zeros(x0.shape[0], device=x0.device)
        if self.room_arrange_condition:
            l_tr, l_an = m(0, td), m(td, td + ad)
            losses = (l_tr + l_an) if self.loss_separate else sq.mean(dim=(1, 2))
            return losses * tb["loss_weight"][t], {"loss.trans": l_tr.mean(), "loss.angle": l_an.mean()}
        bb = self.bbox_dim
        l_tr, l_sz, l_an, l_bb, l_cl = m(0, td), m(td, td + sd), m(td + sd, bb), m(0, bb), m(bb, bb + cd)
        l_ob = m(bb + cd - 1, bb + cd) if self.objectness_dim == 0 else m(bb + cd, bb + cd + self.objectness_dim)
        l_of = m(bb + cd + self.objectness_dim, sq.shape[-1]) if self.objfeat_dim > 0 else zero
        if self.loss_separate:
            losses = l_bb + l_cl
            if self.objectness_dim > 0:
                losses = losses + l_ob
            if self.objfeat_dim > 0:
                losses = losses + l_of
        else:
            losses = sq.mean(dim=(1, 2))
        losses = losses * tb["loss_weight"][t]
        l_iou, iou_avg = zero, zero
        if self.loss_iou:
            if self.mean_type == "v":
                xr = ex(tb["sqrt_ac"]) * x_t - ex(tb["sqrt_1mac"]) * out
            elif self.mean_type == "eps":
                xr = ex(tb["sqrt_recip_ac"]) * x_t - ex(tb["sqrt_recipm1_ac"]) * out
            else:
                xr = out
            xr = xr.clamp(-1.0, 1.0)
            valid = (xr[:, :, bb + cd] >= 0).float() if self.objectness_dim > 0 else (xr[:, :, bb + cd - 1] <= 0).float()
            bnd = torch.tensor(self.bounds, device=x0.device, dtype=torch.float32)
            tr = (xr[:, :, :td] + 1) / 2 * (bnd[3:6] - bnd[0:3]) + bnd[0:3]
            sz = (xr[:, :, td:td + sd] + 1) / 2 * (bnd[9:12] - bnd[6:9]) + bnd[6:9]
            lo, hi = tr - sz, tr + sz
            vol = (hi - lo).prod(dim=-1)
            inter = (torch.min(hi[:, :, None], hi[:, None]) - torch.max(lo[:, :, None], lo[:, None])).clamp(min=0).prod(-1)
            union = torch.clamp(vol[:, :, None] + vol[:, None, :] - inter, min=1e-6)
            mask = valid[:, :, None] * valid[:, None, :]
            iou_valid = inter / union * mask
            denom = mask.sum(dim=(1, 2)) + 1e-6
            iou_avg = iou_valid.sum(dim=(1, 2)) / denom
            l_iou = (tb["alphas_cumprod"][t].reshape(-1, 1, 1) * 0.1 * iou_valid).sum(dim=(1, 2)) / denom
            losses = losses + l_iou
        return losses, {"loss.bbox": l_bb.mean(), "loss.trans": l_tr.mean(), "loss.size": l_sz.mean(),
                        "loss.angle": l_an.mean(), "loss.class": l_cl.mean(), "loss.object": l_ob.mean(),
                        "loss.objfeat": l_of.mean(), "loss.liou": l_iou.mean(), "loss.bbox_iou": iou_avg.mean()}

    # ---- sampling (reference :228-347) -----------------------------------------------------------
    @torch.no_grad()
    def sample(self, room_mask, num_points, point_dim, batch_size=1, text=None, partial_boxes=None, input_boxes=None,
               ret_traj=False, ddim=False, clip_denoised=False, freq=40, batch_seeds=None, ddim_steps=50,
               ddim_eta=0.0, noise=None, x_init=None, seed=None, host_output=False, partial_noise=None):
        device = room_mask.device if torch.is_tensor(room_mask) else self._device()
        if num_points != self.sample_num_points:
            raise ValueError("num_points must equal sample_num_points (%d)" % self.sample_num_points)
        cond, shared = self._condition(batch_size, device, partial_boxes=partial_boxes, input_boxes=input_boxes,
                                       num_points=num_points)
        eng = self.engine()
        eng.set_context(cond, shared=shared)
        if self.text_condition:
            eng.set_context_cross(self._text_condition(text, device))
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if batch_seeds is None else int(batch_seeds[0])
        kw = dict(clip_denoised=clip_denoised, seed=seed, noise=noise, x_init=x_init, ddim=bool(ddim),
                  num_steps=ddim_steps if ddim else 0, ddim_eta=ddim_eta, host_output=host_output)
        if input_boxes is not None:
            x = eng.sample(batch_size, **kw)
            td, sd = self.translation_dim, self.size_dim
            ib = input_boxes.to(x.device)
            return torch.cat([x[..., :td], ib[..., td:td + sd], x[..., td:], ib[..., self.bbox_dim:]], dim=-1).contiguous()
        if partial_boxes is not None:
            return eng.sample(batch_size, partial=partial_boxes, partial_noise=partial_noise, **kw)
        if ret_traj:
            x, traj = eng.sample(batch_size, traj_freq=freq, **kw)
            return [None] + list(traj.unbind(0))              # slot 0 stands for x_T (the reference drops it too)
        return eng.sample(batch_size, **kw)

    @torch.no_grad()
    def generate_layout(self, room_mask, num_points, point_dim, batch_size=1, text=None, ret_traj=False, ddim=False,
                        clip_denoised=False, batch_seeds=None, device="cpu", keep_empty=False):
        samples = self.sample(room_mask, num_points, point_dim, batch_size, text=text, ret_traj=ret_traj, ddim=ddim,
                              clip_denoised=clip_denoised, batch_seeds=batch_seeds)
        return self.delete_empty_from_network_samples(samples, device=device, keep_empty=keep_empty)

    @torch.no_grad()
    def generate_layout_progressive(self, room_mask, num_points, point_dim, batch_size=1, text=None, ret_traj=True,
                                    ddim=False, clip_denoised=False, batch_seeds=None, device="cpu", keep_empty=False,
                                    num_step=100):
        traj = self.sample(room_mask, num_points, point_dim, batch_size, text=text, ret_traj=True, ddim=ddim,
                           clip_denoised=clip_denoised, batch_seeds=batch_seeds, freq=num_step)[1:]
        return {num_step * i: self.delete_empty_from_network_samples(s, device=device, keep_empty=keep_empty)
                for i, s in enumerate(traj)}

    @torch.no_grad()
    def complete_scene(self, room_mask, num_points, point_dim, partial_boxes, batch_size=1, ret_traj=False, ddim=False,
                       clip_denoised=False, batch_seeds=None, device="cpu", keep_empty=False):
        samples = self.sample(room_mask, num_points, point_dim, batch_size, partial_boxes=partial_boxes,
                              clip_denoised=clip_denoised, batch_seeds=batch_seeds)
        return self.delete_empty_from_network_samples(samples, device=device, keep_empty=keep_empty)

    @torch.no_grad()
    def arrange_scene(self, room_mask, num_points, point_dim, input_boxes, batch_size=1, ret_traj=False, ddim=False,
                      clip_denoised=False, batch_seeds=None, device="cpu", keep_empty=False):
        samples = self.sample(room_mask, num_points, point_dim, batch_size, input_boxes=input_boxes,
                              clip_denoised=clip_denoised, batch_seeds=batch_seeds)
        return self.delete_empty_from_network_samples(samples, device=device, keep_empty=keep_empty)

    # ---- post-processing (reference :351-454) ----------------------------------------------------
    def _split(self, samples):
        td, sd, bb, cd = self.translation_dim, self.size_dim, self.bbox_dim, self.class_dim
        out = {"translations": samples[:, :, :td], "sizes": samples[:, :, td:td + sd], "angles": samples[:, :, td + sd:bb],
               "class_labels": samples[:, :, bb:bb + cd - 1], "objectness": samples[:, :, bb + cd - 1:bb + cd]}
        if self.objfeat_dim > 0:
            out["objfeats"] = samples[:, :, bb + cd:bb + cd + self.objfeat_dim]
        return out

    @torch.no_grad()
    def delete_empty_from_network_samples(self, samples, device="cpu", keep_empty=False):
        """Reference semantics (diffusion_scene_layout_ddpm.py:351-406): object i is dropped for the WHOLE batch
        when scene 0 marks it empty -- the reference builds `objectness = last class channel >= 0` (:360) and
        tests that bool with `> 0` (:379), i.e. a score of exactly 0.0 counts as empty; class scores are returned
        raw (the `one_hot(argmax)` at :358 is computed and discarded)."""
        parts = self._split(samples)
        keep = torch.ones(samples.shape[1], dtype=torch.bool) if keep_empty else \
            ~(parts["objectness"][0, :, -1] >= 0).cpu()
        idx = keep.nonzero().flatten().to(samples.device)
        keys = ["class_labels", "translations", "sizes", "angles"] + (["objfeats"] if self.objfeat_dim > 0 else [])
        return {k: parts[k].index_select(1, idx).to("cpu") for k in keys}

    @torch.no_grad()
    def delete_empty_batched(self, samples, keep_empty=False):
        """Per-scene variant for batch_size > 1 (the reference decides from batch row 0 only, SURVEY A.6.3): list
        (one dict per scene) of the non-empty objects, plus the integer class argmax (the north star's bit-exact
        gate).  The keep mask and the argmax are computed on the device for the whole batch; ONE device->host copy
        moves the packed result, the per-scene views are cut on the host."""
        B, N, _ = samples.shape
        bb, cd = self.bbox_dim, self.class_dim
        empty = samples[:, :, bb + cd - 1] >= 0
        keep = torch.ones_like(empty) if keep_empty else ~empty
        cls_idx = samples[:, :, bb:bb + cd - 1].argmax(dim=-1)
        packed = torch.cat([samples.float(), keep[..., None].float(), cls_idx[..., None].float()], dim=-1).cpu()
        keep_h = packed[:, :, -2] > 0.5
        idx_h = packed[:, :, -1].long()
        parts = self._split(packed[:, :, :-2])
        out = []
        for b in range(B):
            sel = keep_h[b]
            d = {k: v[b][sel] for k, v in parts.items() if k != "objectness"}
            d["class_index"] = idx_h[b][sel]
            out.append(d)
        return out

    @torch.no_grad()
    def delete_empty_boxes(self, samples_dict, device="cpu", keep_empty=False):
        cl = samples_dict["class_labels"]
        keep = torch.ones(cl.shape[1], dtype=torch.bool) if keep_empty else ~(cl[0, :, -1] > 0).cpu()
        idx = keep.nonzero().flatten().to(cl.device)
        out = {"class_labels": cl[:, :, :self.class_dim - 1].index_select(1, idx).to("cpu")}
        for k in ["translations", "sizes", "angles"] + (["objfeats"] if self.objfeat_dim > 0 else []):
            out[k] = samples_dict[k].index_select(1, idx).to("cpu")
        return out


def train_on_batch(model, optimizer, sample_params, config):
    """Reference diffusion_scene_layout_ddpm.py:456-473 (the 11 per-key `.item()` syncs collapse into one)."""
    optimizer.zero_grad(set_to_none=True)
    loss, loss_dict = model.get_loss(sample_params)
    loss.backward()
    max_norm = config["training"]["max_grad_norm"]
    if getattr(model, "_native_grads_ready", False) and isinstance(optimizer, NativeAdam):
        # native path: gradients live in one flat buffer -> one all-reduce stream, device-side global norm, and the
        # clip coefficient applied inside the fused Adam kernel (no host synchronisation until the log values below)
        # (the flat buffer itself was all-reduced bucket by bucket DURING the backward pass: parallel.GradOverlap)
        allreduce_flat(None if model._overlap is not None else model._flat_grads,
                       [p for p in model.parameters() if p.grad is not None and not hasattr(p, "_ds_flat_owner")])
        grad_norm = optimizer.step_clipped(model, max_norm)
    else:
        allreduce_gradients(model.parameters())       # no-op outside a torch.distributed process group
        grad_norm = clip_grad_norm_(model.parameters(), max_norm)
        optimizer.step()
    model.mark_weights_dirty()
    keys = list(loss_dict.keys())
    vals = torch.stack([loss_dict[k].detach().float() for k in keys] + [grad_norm.detach().float(), loss.detach().float()]).tolist()
    for k, v in zip(keys, vals):
        StatsLogger.instance()[k].value = v
    StatsLogger.instance()["gradnorm"].value = vals[-2]
    StatsLogger.instance()["lr"].value = optimizer.param_groups[0]["lr"]
    return vals[-1]


@torch.no_grad()
def validate_on_batch(model, sample_params, config):
    loss, loss_dict = model.get_loss(sample_params)
    keys = list(loss_dict.keys())
    vals = torch.stack([loss_dict[k].float() for k in keys] + [loss.float()]).tolist()
    for k, v in zip(keys, vals):
        StatsLogger.instance()[k].value = v
    return vals[-1]
