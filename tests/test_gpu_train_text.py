"""GPU: the native training step of the text-conditioned networks (cross-attention backward, ds_train_set_context_cross)
against torch autograd over the CPU oracle: loss, the 9 dict entries, every parameter gradient (all to_kv / to_q /
cross-attention LayerNorm gains included), d(context) and d(context_cross) in fp32 parity mode; bf16 mode against the
same gradients; the drop-in train_on_batch against the autograd path with torch.optim.Adam; changing (B, L) on one
handle, gradient buckets, argument checks; and the text forward for L beyond the old shared-memory limit."""
import copy
import json
import os

import numpy as np
import pytest
import torch

from diffuscene_b200 import capi
from diffuscene_b200.engine import DenoiserEngine
from diffuscene_b200.weights import NetSpec, seeded_state_dict, unet1d_param_specs
from oracle import diffusion_ref as D
from oracle.unet1d_ref import unet1d_forward
from tests.cases import CASES, STATS, make_inputs
from tests.gpu_common import case_tables

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_BED_TEXT = dict(CASES["bed62"]["net_kwargs"], text_condition=True, text_dim=512)
_LIV_TEXT = dict(CASES["liv65"]["net_kwargs"], text_condition=True, text_dim=512)
_BED_CFG = CASES["bed62"]["net_cfg"]
# local cases (tests/cases.py feeds the parameter sets of other test files)
TEXT_CASES = {
    # shipped text bedroom network (N = 12, d = 62), v-prediction with the IoU term, three text lengths
    "bed_L1": dict(seed=41, B=2, N=12, L=1, net_kwargs=_BED_TEXT, net_cfg=_BED_CFG,
                   diffusion_kwargs=CASES["bed62"]["diffusion_kwargs"]),
    "bed_L7": dict(seed=42, B=2, N=12, L=7, net_kwargs=_BED_TEXT, net_cfg=_BED_CFG,
                   diffusion_kwargs=CASES["bed62"]["diffusion_kwargs"]),
    "bed_L77": dict(seed=43, B=3, N=12, L=77, net_kwargs=_BED_TEXT, net_cfg=_BED_CFG,
                    diffusion_kwargs=CASES["bed62"]["diffusion_kwargs"]),
    # living-room shape (N = 21, d = 65), x0-prediction with the IoU term
    "liv_x0": dict(seed=44, B=2, N=21, L=9, net_kwargs=_LIV_TEXT, net_cfg=CASES["liv65"]["net_cfg"],
                   diffusion_kwargs=CASES["liv65"]["diffusion_kwargs"]),
    # per-scene (non-shared) condition
    "bed_scene_ctx": dict(seed=45, B=3, N=12, L=5, net_kwargs=_BED_TEXT, net_cfg=_BED_CFG,
                          diffusion_kwargs=CASES["bed62"]["diffusion_kwargs"], shared_context=False),
}


def _setup(case):
    spec = NetSpec.from_net_kwargs(case["net_kwargs"])
    sd = seeded_state_dict(unet1d_param_specs(spec), seed=case["seed"])
    inp = make_inputs(case, spec)
    shared = case.get("shared_context", True)
    ctx = inp["context"][0] if shared else inp["context"]
    return spec, sd, inp, shared, ctx


def _oracle_grads(case, spec, sd, inp, ctx, cross):
    """autograd through the oracle: (losses, dict, grads by name, d(context), d(context_cross))."""
    dk = case["diffusion_kwargs"]
    sched = D.make_schedule(D.make_betas(dk["schedule_type"], dk["beta_start"], dk["beta_end"], dk["time_num"]),
                            dk["model_mean_type"], dk["model_var_type"])
    cfg = case["net_cfg"]
    ls = D.LossSpec(class_dim=cfg["class_dim"], angle_dim=cfg["angle_dim"], objfeat_dim=cfg["objfeat_dim"],
                    objectness_dim=cfg["objectness_dim"], loss_separate=dk["loss_separate"], loss_iou=dk["loss_iou"],
                    bounds_translations=STATS["bounds_translations"], bounds_sizes=STATS["bounds_sizes"])
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    c = ctx.clone().requires_grad_(True)
    x = cross.clone().requires_grad_(True)
    B, N = case["B"], case["N"]
    cfull = c[None].expand(B, N, -1) if c.dim() == 2 else c
    with torch.enable_grad():
        den = lambda xx, tt: unet1d_forward(sdg, spec, xx, tt, cfull, x)
        losses, ld = D.p_losses(sched, ls, den, inp["x0"], inp["t_loss"], inp["noise_loss"])
        losses.mean().backward()
    return losses.detach(), ld, {k: v.grad for k, v in sdg.items()}, c.grad, x.grad


def _engine(case, spec, prec):
    eng = DenoiserEngine(spec, case["N"], case["diffusion_kwargs"]["time_num"], precision=prec)
    eng.set_schedule(case_tables(case))
    return eng


def _flat(eng, sd):
    layout = eng.flat_layout()
    total = sum(n for _, n in layout.values())
    flat = torch.empty(total, device="cuda")
    for k, (off, n) in layout.items():
        flat[off:off + n] = sd[k].reshape(-1).cuda()
    return layout, flat


def _native_step(eng, case, sd, inp, ctx, shared, cross, grads=None):
    layout, flat = _flat(eng, sd)
    if grads is None:
        grads = torch.full((flat.numel(),), float("nan"), device="cuda")
    dk = case["diffusion_kwargs"]
    bounds = STATS["bounds_translations"] + STATS["bounds_sizes"]
    losses, ld, dctx, dcross = eng.train_step(flat, inp["x0"].cuda(), inp["t_loss"].cuda(), inp["noise_loss"].cuda(),
                                              ctx.cuda(), shared, dk["loss_separate"], dk["loss_iou"], bounds,
                                              flat_grads=grads, context_cross=cross.cuda())
    torch.cuda.synchronize()
    g = {k: grads[off:off + n].reshape(sd[k].shape).cpu() for k, (off, n) in layout.items()}
    return losses.cpu(), {k: float(v) for k, v in ld.items()}, g, dctx.cpu(), dcross.cpu()


def _native(case, spec, sd, inp, ctx, shared, cross, prec):
    eng = _engine(case, spec, prec)
    try:
        return _native_step(eng, case, sd, inp, ctx, shared, cross)
    finally:
        eng.close()


@pytest.mark.parametrize("name", list(TEXT_CASES))
def test_text_gradients_match_oracle_autograd_fp32(name):
    case = TEXT_CASES[name]
    spec, sd, inp, shared, ctx = _setup(case)
    cross = inp["context_cross"]
    ref_losses, ref_ld, ref_g, ref_dc, ref_dx = _oracle_grads(case, spec, sd, inp, ctx, cross)
    losses, ld, g, dc, dx = _native(case, spec, sd, inp, ctx, shared, cross, "fp32")
    np.testing.assert_allclose(losses.numpy(), ref_losses.numpy(), rtol=1e-3, atol=1e-4)
    for k, v in ref_ld.items():
        np.testing.assert_allclose(ld[k], float(v), rtol=1e-3, atol=1e-4, err_msg=k)
    assert set(g) == set(ref_g)
    assert sum(k.endswith("to_kv.weight") for k in g) == 9
    worst = []
    for k in sorted(g):
        a, b = g[k], ref_g[k]
        assert torch.isfinite(a).all(), k
        scale = max(b.abs().max().item(), 1e-6)
        worst.append(((a - b).abs().max().item() / scale, k))
    worst.sort(reverse=True)
    print("worst relative gradient errors:", worst[:5])
    assert worst[0][0] < 2e-3, worst[:8]
    np.testing.assert_allclose(dc.numpy(), ref_dc.numpy(), rtol=2e-3, atol=2e-3 * ref_dc.abs().max().item())
    np.testing.assert_allclose(dx.numpy(), ref_dx.numpy(), rtol=2e-3, atol=2e-3 * ref_dx.abs().max().item())


def test_text_gradients_bf16_mode_close_to_fp32_oracle():
    case = TEXT_CASES["bed_L7"]
    spec, sd, inp, shared, ctx = _setup(case)
    cross = inp["context_cross"]
    _, _, ref_g, _, ref_dx = _oracle_grads(case, spec, sd, inp, ctx, cross)
    _, _, g, _, dx = _native(case, spec, sd, inp, ctx, shared, cross, "bf16")
    cos = []
    for k in sorted(g):
        a, b = g[k].flatten().double(), ref_g[k].flatten().double()
        if b.norm() < 1e-10:
            continue
        cos.append((float(a @ b / (a.norm() * b.norm() + 1e-30)), k))
    cos.sort()
    print("lowest gradient cosines (bf16 mode):", cos[:5])
    assert cos[0][0] > 0.97 and np.mean([c for c, _ in cos]) > 0.995
    a, b = dx.flatten().double(), ref_dx.flatten().double()
    assert float(a @ b / (a.norm() * b.norm())) > 0.99


def yaml_cfg(tmp_path):
    import yaml
    with open(os.path.join(ROOT, "config", "text/diffusion_bedrooms_instancond_lat32_v_bert.yaml")) as f:
        cfg = yaml.safe_load(f)
    stats = tmp_path / "stats.json"
    stats.write_text(json.dumps(STATS))
    cfg["network"]["diffusion_kwargs"]["train_stats_file"] = str(stats)
    cfg["training"]["max_grad_norm"] = 0.05          # small enough that the clip is active
    return cfg


def _text_batch(B, L):
    from tests.cases_class import fake_bert_hidden
    g = torch.Generator().manual_seed(0)
    cls = torch.randint(0, 22, (B, 12), generator=g)
    sp = dict(translations=torch.rand(B, 12, 3, generator=g) * 2 - 1, sizes=torch.rand(B, 12, 3, generator=g) * 2 - 1,
              angles=torch.nn.functional.normalize(torch.randn(B, 12, 2, generator=g), dim=-1),
              class_labels=torch.nn.functional.one_hot(cls, 22).float() * 2 - 1,
              objfeats_32=torch.rand(B, 12, 32, generator=g) * 2 - 1, room_layout=torch.zeros(B, 1, 64, 64))
    texts = ["a bedroom with a double bed", "wardrobe next to the desk", "two nightstands and a lamp",
             "a chair in front of a table"][:B]
    sp["description"] = fake_bert_hidden(texts, L=L)
    return {k: v.cuda() for k, v in sp.items()}


def test_text_train_on_batch_native_matches_torch_adam(tmp_path):
    """Two iterations through the drop-in API with the shipped text config: native step + NativeAdam against the
    autograd functional + torch.optim.Adam (+ clip_grad_norm_, active) on a twin model; fc_text_f trains through
    ordinary autograd from d(context_cross).  During a native iteration the only ATen matmuls are fc_text_f's."""
    from scene_synthesis.networks import build_network, optimizer_factory
    from diffuscene_b200.optim import NativeAdam
    cfg = yaml_cfg(tmp_path)
    torch.manual_seed(3)
    net_a, train_on_batch, _ = build_network(30, 23, cfg, None, device="cuda", precision="fp32")
    net_b, _, _ = build_network(30, 23, cfg, None, device="cuda", precision="fp32")
    net_b.load_state_dict(copy.deepcopy(net_a.state_dict()))
    net_b.native_backward = False
    assert net_a.native_training_supported()
    opt_a = optimizer_factory(cfg["training"], net_a.parameters())
    assert isinstance(opt_a, NativeAdam)
    opt_b = torch.optim.Adam(net_b.parameters(), lr=cfg["training"]["lr"], weight_decay=0.0)
    B, L = 4, 11
    sp = _text_batch(B, L)
    fc0 = net_a.fc_text_f.weight.detach().clone()
    for it in range(2):
        torch.manual_seed(100 + it)
        la = train_on_batch(net_a, opt_a, sp, cfg)
        assert net_a._native_grads_ready
        torch.manual_seed(100 + it)
        lb = train_on_batch(net_b, opt_b, sp, cfg)
        assert abs(la - lb) < 1e-3 * max(1.0, abs(lb)), (it, la, lb)
    sa, sb = net_a.state_dict(), net_b.state_dict()
    worst = max(((sa[k] - sb[k]).abs().max().item(), k) for k in sa)
    print("largest parameter difference after 2 iterations:", worst)
    lr = cfg["training"]["lr"]
    assert worst[0] < 3 * lr, worst
    mean_diff = np.mean([(sa[k] - sb[k]).abs().mean().item() for k in sa])
    assert mean_diff < 0.05 * lr, mean_diff
    fa, fb = sa["fc_text_f.weight"], sb["fc_text_f.weight"]
    assert (fa - fb).abs().max().item() < 3 * lr and (fa - fb).abs().mean().item() < 0.05 * lr
    # fc_text_f trained: its gradient arrived through d(context_cross)
    assert (fa - fc0).abs().max().item() > 0.5 * lr

    from torch.profiler import ProfilerActivity, profile
    matmuls = ("aten::mm", "aten::addmm", "aten::bmm", "aten::baddbmm", "aten::matmul", "aten::linear", "aten::mv",
               "aten::addmv", "aten::einsum")
    with profile(activities=[ProfilerActivity.CPU], record_shapes=True) as prof:
        train_on_batch(net_a, opt_a, sp, cfg)
        torch.cuda.synchronize()
    seen = [(e.name, e.input_shapes) for e in prof.events() if e.name in matmuls]
    print("ATen matmuls in one native text iteration:", seen)
    assert seen, "fc_text_f's projection should appear"
    fc_in = net_a.fc_text_f.in_features
    for name, shapes in seen:
        assert any(fc_in in s for s in shapes if s), (name, shapes)


def _assert_close_runs(a, b, prec):
    """two native runs of the same step: equal up to the order of fp32 atomic sums (and its bf16 rounding)"""
    rel = 1e-5 if prec == "fp32" else 2e-2
    for x, y in zip(a, b):
        if isinstance(x, dict):
            for k in x:
                s = max(y[k].abs().max().item(), 1e-6) if torch.is_tensor(y[k]) else max(abs(y[k]), 1e-6)
                d = (x[k] - y[k]).abs().max().item() if torch.is_tensor(x[k]) else abs(x[k] - y[k])
                assert d <= rel * s + 1e-7, (k, d, s)
        else:
            s = max(y.abs().max().item(), 1e-6)
            assert (x - y).abs().max().item() <= rel * s + 1e-7


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_text_shape_changes_on_one_handle(prec):
    """(B, L) = (2, 7), (3, 40), (2, 7) on one handle give what fresh handles give: the text buffers and plans grow
    and are reused without stale state."""
    base = TEXT_CASES["bed_L7"]
    eng = _engine(base, NetSpec.from_net_kwargs(base["net_kwargs"]), prec)
    try:
        for i, (B, L) in enumerate([(2, 7), (3, 40), (2, 7)]):
            case = dict(base, B=B, L=L, seed=50 + i)
            spec, sd, inp, shared, ctx = _setup(case)
            got = _native_step(eng, case, sd, inp, ctx, shared, inp["context_cross"])
            fresh = _native(case, spec, sd, inp, ctx, shared, inp["context_cross"], prec)
            _assert_close_runs(got, fresh, prec)
    finally:
        eng.close()


def test_text_gradient_buckets():
    """With gradient buckets set, each bucket's event is recorded once its gradients are final (a side stream that
    waits on it copies final values), every event has completed after the step, and the gradients equal the run
    without buckets."""
    case = TEXT_CASES["bed_L7"]
    spec, sd, inp, shared, ctx = _setup(case)
    eng = _engine(case, spec, "fp32")
    try:
        n = sum(k for _, k in eng.flat_layout().values())
        bounds = [0] + [n * i // 6 for i in range(1, 6)] + [n]
        events = [torch.cuda.Event() for _ in range(6)]
        for e in events:
            e.record()
        eng.train_set_buckets(bounds, events)
        grads = torch.full((n,), float("nan"), device="cuda")
        side = torch.cuda.Stream()
        _, flat = _flat(eng, sd)
        dk = case["diffusion_kwargs"]
        b12 = STATS["bounds_translations"] + STATS["bounds_sizes"]
        eng.train_step(flat, inp["x0"].cuda(), inp["t_loss"].cuda(), inp["noise_loss"].cuda(), ctx.cuda(), shared,
                       dk["loss_separate"], dk["loss_iou"], b12, flat_grads=grads, context_cross=inp["context_cross"].cuda())
        copies = []
        with torch.cuda.stream(side):
            for k, e in enumerate(events):
                side.wait_event(e)
                copies.append(grads[bounds[k]:bounds[k + 1]].clone())
        torch.cuda.synchronize()
        assert all(e.query() for e in events)
        for k, c in enumerate(copies):
            assert torch.equal(c, grads[bounds[k]:bounds[k + 1]]), k
        eng.train_set_buckets([], [])
        ref = _native_step(eng, case, sd, inp, ctx, shared, inp["context_cross"])
        s = ref[2]
        layout = eng.flat_layout()
        for k, (off, m) in layout.items():
            a, b = grads[off:off + m].cpu(), s[k].reshape(-1)
            assert (a - b).abs().max().item() <= 1e-5 * max(b.abs().max().item(), 1e-6) + 1e-7, k
    finally:
        eng.close()


def test_text_train_argument_checks():
    case = TEXT_CASES["bed_L7"]
    spec, sd, inp, shared, ctx = _setup(case)
    eng = _engine(case, spec, "fp32")
    try:
        layout, flat = _flat(eng, sd)
        grads = torch.zeros(flat.numel(), device="cuda")
        dk = case["diffusion_kwargs"]
        b12 = STATS["bounds_translations"] + STATS["bounds_sizes"]
        args = (flat, inp["x0"].cuda(), inp["t_loss"].cuda(), inp["noise_loss"].cuda(), ctx.cuda(), shared,
                dk["loss_separate"], dk["loss_iou"], b12)
        with pytest.raises(capi.DsError):                 # text network, no context_cross
            eng.train_step(*args, flat_grads=grads)
        cross = inp["context_cross"].cuda()
        with pytest.raises(capi.DsError):                 # batch mismatch (context_cross for 1 scene, step for 2)
            eng.train_step(*args, flat_grads=grads, context_cross=cross[:1].contiguous())
        for L in (0, 513):
            with pytest.raises(capi.DsError):
                capi.check(eng.lib.ds_train_set_context_cross(eng.h, torch.empty(2, 513, 512, device="cuda").data_ptr(),
                                                              2, L, None))
        out = eng.train_step(*args, flat_grads=grads, context_cross=cross)      # and a valid call still works
        torch.cuda.synchronize()
        assert len(out) == 4 and torch.isfinite(out[3]).all()
    finally:
        eng.close()
    plain = CASES["bed62"]
    eng = _engine(plain, NetSpec.from_net_kwargs(plain["net_kwargs"]), "fp32")
    try:
        with pytest.raises(capi.DsError):                 # no text condition
            capi.check(eng.lib.ds_train_set_context_cross(eng.h, torch.empty(2, 7, 512, device="cuda").data_ptr(),
                                                          2, 7, None))
    finally:
        eng.close()


def test_text_forward_long_context_matches_oracle():
    """L = 300 > 200: ds_set_context_cross streams the tokens (the text context used to need L KB of shared memory)."""
    case = dict(CASES["text62"], B=2, L=300, seed=46)
    spec = NetSpec.from_net_kwargs(case["net_kwargs"])
    sd = seeded_state_dict(unet1d_param_specs(spec), seed=case["seed"])
    inp = make_inputs(case, spec)
    ref = unet1d_forward(sd, spec, inp["x"], inp["t"], inp["context"], inp["context_cross"])
    eng = DenoiserEngine(spec, case["N"], case["diffusion_kwargs"]["time_num"], precision="fp32")
    try:
        eng.load_state_dict(sd)
        eng.set_schedule(case_tables(case))
        eng.set_context(inp["context"][0].cuda(), shared=True)
        eng.set_context_cross(inp["context_cross"].cuda())
        out = eng.forward(inp["x"].cuda(), inp["t"].cuda()).cpu()
    finally:
        eng.close()
    np.testing.assert_allclose(out.numpy(), ref.numpy(), rtol=1e-3, atol=1e-4)
