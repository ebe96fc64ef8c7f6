"""Differentiable (torch autograd) forward of the denoiser: the reference training path.

`train_on_batch` runs the native CUDA training step (ds_train_step: forward and hand-written backward pass) for
every network the library builds, text-conditioned ones included.  This functional form is what a model with
`native_backward = False` differentiates with torch autograd instead, on the same parameters; the tests compare
the native step against it.  Semantics: reference scene_synthesis/networks/denoise_net.py:507-593 in
token-major layout.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F


def _w(p):
    return p.reshape(p.shape[0], -1)


def _ws(w):
    w = _w(w)
    mean = w.mean(dim=1, keepdim=True)
    var = w.var(dim=1, unbiased=False, keepdim=True)
    return (w - mean) * torch.rsqrt(var + 1e-5)


def _ln(x, g):
    mean = x.mean(dim=-1, keepdim=True)
    var = x.var(dim=-1, unbiased=False, keepdim=True)
    return (x - mean) * torch.rsqrt(var + 1e-5) * g.reshape(1, 1, -1)


def _gn(x, gamma, beta, groups=8):
    B, N, C = x.shape
    xg = x.reshape(B, N, groups, C // groups)
    mean = xg.mean(dim=(1, 3), keepdim=True)
    var = xg.var(dim=(1, 3), unbiased=False, keepdim=True)
    return ((xg - mean) * torch.rsqrt(var + 1e-5)).reshape(B, N, C) * gamma + beta


class DenoiserFn:
    """Callable closure over a name -> parameter mapping (names without the 'diffusion.model.' prefix)."""

    def __init__(self, params, spec):
        self.p = params
        self.s = spec

    def block(self, n, x, ss=None):
        p = self.p
        h = F.linear(x, _ws(p[n + ".proj.weight"]), p[n + ".proj.bias"])
        h = _gn(h, p[n + ".norm.weight"], p[n + ".norm.bias"])
        if ss is not None:
            h = h * (ss[0] + 1) + ss[1]
        return F.silu(h)

    def res(self, n, x, cond):
        p = self.p
        e = F.linear(F.silu(cond), p[n + ".mlp.1.weight"], p[n + ".mlp.1.bias"])
        if e.dim() == 2:
            e = e[:, None, :]
        h = self.block(n + ".block2", self.block(n + ".block1", x, e.chunk(2, dim=-1)))
        if (n + ".res_conv.weight") in p:
            return h + F.linear(x, _w(p[n + ".res_conv.weight"]), p[n + ".res_conv.bias"])
        return h + x

    def _heads(self, t):
        B, N, HC = t.shape
        return t.reshape(B, N, 4, HC // 4)

    def linattn(self, n, x):
        p = self.p
        qkv = F.linear(_ln(x, p[n + ".fn.norm.g"]), _w(p[n + ".fn.fn.to_qkv.weight"]))
        q, k, v = (self._heads(t) for t in qkv.chunk(3, dim=-1))
        q = q.softmax(dim=-1) * (32 ** -0.5)
        k = k.softmax(dim=1)
        ctx = torch.einsum("bnhd,bnhe->bhde", k, v)
        o = torch.einsum("bhde,bnhd->bnhe", ctx, q).reshape(x.shape[0], x.shape[1], -1)
        y = F.linear(o, _w(p[n + ".fn.fn.to_out.0.weight"]), p[n + ".fn.fn.to_out.0.bias"])
        return _ln(y, p[n + ".fn.fn.to_out.1.g"]) + x

    def attn(self, n, x):
        p = self.p
        qkv = F.linear(_ln(x, p[n + ".fn.norm.g"]), _w(p[n + ".fn.fn.to_qkv.weight"]))
        q, k, v = (self._heads(t) for t in qkv.chunk(3, dim=-1))
        sim = torch.einsum("bihd,bjhd->bhij", q * (32 ** -0.5), k)
        o = torch.einsum("bhij,bjhd->bihd", sim.softmax(dim=-1), v).reshape(x.shape[0], x.shape[1], -1)
        return F.linear(o, _w(p[n + ".fn.fn.to_out.weight"]), p[n + ".fn.fn.to_out.bias"]) + x

    def xattn(self, n, x, text):
        p = self.p
        q = self._heads(F.linear(_ln(x, p[n + ".fn.norm.g"]), _w(p[n + ".fn.fn.to_q.weight"])))
        kv = F.linear(text, _w(p[n + ".fn.fn.to_kv.weight"]))
        k, v = (t.reshape(t.shape[0], t.shape[1], 4, 32) for t in kv.chunk(2, dim=-1))
        q = q.softmax(dim=-1) * (32 ** -0.5)
        k = k.softmax(dim=1)
        ctx = torch.einsum("blhd,blhe->bhde", k, v)
        o = torch.einsum("bhde,bnhd->bnhe", ctx, q).reshape(x.shape[0], x.shape[1], -1)
        y = F.linear(o, _w(p[n + ".fn.fn.to_out.0.weight"]), p[n + ".fn.fn.to_out.0.bias"])
        return _ln(y, p[n + ".fn.fn.to_out.1.g"]) + x

    def mlp3(self, n, x):
        p = self.p
        h = F.gelu(F.linear(x, _w(p[n + ".0.weight"]), p[n + ".0.bias"]))
        h = F.gelu(F.linear(h, _w(p[n + ".2.weight"]), p[n + ".2.bias"]))
        return F.linear(h, _w(p[n + ".4.weight"]), p[n + ".4.bias"])

    def __call__(self, x, t, context, context_cross=None):
        p, s = self.p, self.s
        b0 = s.bbox_dim
        if s.seperate_all:
            c0 = b0 + s.class_dim
            h = self.mlp3("class_embedf", x[..., b0:c0]) + self.mlp3("bbox_embedf", x[..., :b0])
            if s.objectness_dim > 0:
                h = h + self.mlp3("objectness_embedf", x[..., c0:c0 + s.objectness_dim])
            if s.objfeat_dim > 0:
                o0 = c0 + s.objectness_dim
                h = h + self.mlp3("objfeat_embedf", x[..., o0:o0 + s.objfeat_dim])
        else:
            h = x
        h = F.linear(h, _w(p["init_conv.weight"]), p["init_conv.bias"])
        r = h
        half = s.dim // 2
        freq = torch.exp(torch.arange(half, device=x.device, dtype=torch.float32) * -(math.log(10000) / (half - 1)))
        ang = t.to(torch.float32)[:, None] * freq[None, :]
        e = torch.cat([ang.sin(), ang.cos()], dim=-1)
        e = F.gelu(F.linear(e, p["time_mlp.1.weight"], p["time_mlp.1.bias"]))
        temb = F.linear(e, p["time_mlp.3.weight"], p["time_mlp.3.bias"])
        text = context_cross if s.text_condition else None
        skips = []
        for i in range(s.n_stages):
            d = "downs.%d" % i
            h = self.res(d + ".0", h, context)
            h = self.res(d + ".1", h, temb)
            skips.append(h)
            if text is not None:
                h = self.xattn(d + ".2", h, text)
            h = self.res(d + ".3", h, temb)
            h = self.linattn(d + ".4", h)
            skips.append(h)
            if i == s.n_stages - 1:
                h = F.linear(h, _w(p[d + ".5.weight"]), p[d + ".5.bias"])
        h = self.res("mid_block0", h, context)
        h = self.res("mid_block1", h, temb)
        if text is not None:
            h = self.xattn("mid_attn_cross", h, text)
        h = self.attn("mid_attn", h)
        h = self.res("mid_block2", h, temb)
        for i in range(s.n_stages):
            u = "ups.%d" % i
            h = self.res(u + ".0", h, context)
            h = self.res(u + ".1", torch.cat([h, skips.pop()], dim=-1), temb)
            if text is not None:
                h = self.xattn(u + ".2", h, text)
            h = self.res(u + ".3", torch.cat([h, skips.pop()], dim=-1), temb)
            h = self.linattn(u + ".4", h)
            if i == s.n_stages - 1:
                h = F.linear(h, _w(p[u + ".5.weight"]), p[u + ".5.bias"])
        h = self.res("final_res_block", torch.cat([h, r], dim=-1), temb)
        if s.seperate_all:
            outs = [self.mlp3("bbox_hidden2output", h), self.mlp3("class_hidden2output", h)]
            if s.objectness_dim > 0:
                outs.append(self.mlp3("objectness_hidden2output", h))
            if s.objfeat_dim > 0:
                outs.append(self.mlp3("objfeat_hidden2output", h))
            return torch.cat(outs, dim=-1)
        return F.linear(h, _w(p["final_conv.weight"]), p["final_conv.bias"])
