"""Bring-up aid (run on the GPU box): per-role cycle breakdown of the tcgen05 GEMM kernel for the hot shapes."""
import ctypes as C
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from diffuscene_b200 import capi   # noqa: E402

lib = capi.load()
names = ["prod_wait_empty", "prod_total", "mma_wait_tmem", "mma_wait_full", "mma_total", "epi_wait_tfull", "epi_total", "tiles"]


def gnt_rows(N):
    """stored row -> channel of the channels-on-lanes kernel (tc_gnt_row in kernels.cuh)"""
    r = torch.arange(N)
    l = r & 31
    return (r & ~31) + 8 * (l & 3) + (l >> 2)


def reference(a, w, bias, gamma, beta, r, n_obj):
    y = a.float() @ w.float().t() + bias
    if n_obj:
        M, N = y.shape
        z = y.view(M // n_obj, n_obj, N // 64, 64)
        mean = z.mean(dim=(1, 3), keepdim=True)
        var = z.var(dim=(1, 3), unbiased=False, keepdim=True)
        y = ((z - mean) * torch.rsqrt(var + 1e-5)).view(M, N) * gamma + beta
        y = torch.nn.functional.silu(y)
    if r is not None:
        y = y + r.float()
    return y


def run(M, N, K, n_obj=0, res=False, tag="", gnt=False, check=False, plain_act=None):
    """plain_act (0 none / 1 GELU / 2 SiLU) with gnt=True: the channels-on-lanes kernel as a plain GEMM"""
    g = torch.Generator().manual_seed(0)
    a = torch.randn(M, K, generator=g).to(torch.bfloat16).cuda()
    w = (torch.randn(N, K, generator=g) / K ** 0.5).to(torch.bfloat16).cuda()
    bias = torch.randn(N, generator=g).cuda()
    gamma = (1.0 + 0.2 * torch.randn(N, generator=g)).cuda() if check else torch.ones(N).cuda()
    beta = (0.2 * torch.randn(N, generator=g)).cuda() if check else torch.zeros(N).cuda()
    r = torch.randn(M, N, generator=g).to(torch.bfloat16).cuda() if res else None
    d = torch.zeros(M, N, dtype=torch.bfloat16, device="cuda")
    tr = np.zeros((256, 8), dtype=np.uint64)
    us = C.c_float()
    w_dev = w[gnt_rows(N).cuda()].contiguous() if gnt else w
    plain = plain_act is not None
    rc = lib.ds_test_gemm_trace(a.data_ptr(), w_dev.data_ptr(), bias.data_ptr(), None if r is None else r.data_ptr(),
                                d.data_ptr(), M, N, K, -n_obj if gnt else n_obj, None if plain else gamma.data_ptr(),
                                None if plain else beta.data_ptr(), 20 | ((plain_act or 0) << 8),
                                tr.ctypes.data, C.byref(us))
    if rc:
        print("FAILED", lib.ds_last_error().decode())
        return
    if check:
        if plain:
            ref = a.float() @ w.float().t() + bias
            ref = [lambda z: z, torch.nn.functional.gelu, torch.nn.functional.silu][plain_act](ref)
            ref = ref + r.float() if r is not None else ref
        else:
            ref = reference(a, w, bias, gamma, beta, r, n_obj)
        err = (d.float() - ref).abs()
        bad = (err > 0.05 + 0.02 * ref.abs()).sum().item()
        print("   check %-20s max|err|=%.4f mean|err|=%.5f  out-of-tolerance=%d  %s" % (
            tag, err.max().item(), err.mean().item(), bad, "OK" if bad == 0 else "MISMATCH"))
        if bad:
            idx = (err > 0.05 + 0.02 * ref.abs()).nonzero()[:8]
            for i, j in idx.tolist():
                print("      row %d col %d got %.4f want %.4f" % (i, j, d[i, j].item(), ref[i, j].item()))
    t = tr[:148].astype(np.float64)
    tf = 2.0 * M * N * K / us.value / 1e6
    print("%-28s M=%d N=%d K=%d n_obj=%d res=%d: %.1f us  %.0f TFLOP/s" % (tag, M, N, K, n_obj, res, us.value, tf))
    print("   " + "  ".join("%s=%.0f" % (n, t[:, i].mean()) for i, n in enumerate(names)))


M = 49152
if os.environ.get("PLAIN_ONLY"):      # row-major plain kernel (k_gemm_tc): numeric checks incl. odd tile counts, then timings
    for m_chk in (128 * 5, 128 * 5 - 37, 12 * 1000, 128 * 301):
        run(m_chk, 512, 512, tag="plain 512x512", check=True)
        run(m_chk, 512, 512, res=True, tag="plain+res", check=True)
        run(m_chk, 1024, 512, tag="plain N=1024", check=True)
        run(m_chk, 512, 1024, tag="plain K=1024", check=True)
        run(m_chk, 384, 512, tag="plain N=384 (BN=128)", check=True)
        run(m_chk, 512, 128, tag="plain K=128", check=True)
    run(M, 512, 128, tag="to_out K=128")
    run(M, 1536, 64, tag="enc.l0")
    run(M, 1024, 512, tag="enc.l1")
    run(M, 512, 3072, tag="encoder K=3072")
    run(M, 3072, 512, tag="dec.l0")
    run(M, 512, 1024, tag="plain 512x1024")
    run(M, 512, 512, tag="plain 512x512")
    sys.exit(0)
if os.environ.get("GNT_ONLY"):
    for m_chk in (12 * 16 * 3, 12 * 1000):      # whole tiles / ragged last tile
        run(m_chk, 512, 512, n_obj=12, tag="GN", check=True)
        run(m_chk, 512, 512, n_obj=12, tag="GNT", gnt=True, check=True)
        run(m_chk, 512, 512, n_obj=12, res=True, tag="GNT+res", gnt=True, check=True)
        run(m_chk, 512, 1024, n_obj=12, res=True, tag="GNT+res K=1024", gnt=True, check=True)
    for m_chk in (12 * 16 * 3, 12 * 1000):
        run(m_chk, 512, 128, n_obj=12, tag="T plain K=128", gnt=True, check=True, plain_act=0)
        run(m_chk, 384, 512, n_obj=12, tag="T plain N=384", gnt=True, check=True, plain_act=0)
        run(m_chk, 1536, 64, n_obj=12, tag="T gelu N=1536 K=64", gnt=True, check=True, plain_act=1)
        run(m_chk, 512, 512, n_obj=12, res=True, tag="T silu+res", gnt=True, check=True, plain_act=2)
    run(M, 512, 128, n_obj=12, tag="T to_out K=128", gnt=True, plain_act=0)
    run(M, 384, 512, n_obj=12, tag="T qkv N=384", gnt=True, plain_act=0)
    run(M, 1536, 64, n_obj=12, tag="T enc.l0 gelu", gnt=True, plain_act=1)
    run(M, 1024, 512, n_obj=12, tag="T enc.l1 gelu", gnt=True, plain_act=1)
    run(M, 3072, 512, n_obj=12, tag="T dec.l0 gelu", gnt=True, plain_act=1)
    run(M, 512, 1024, n_obj=12, tag="T res_conv K=1024", gnt=True, plain_act=0)
    run(M, 512, 128, tag="to_out K=128")
    run(M, 384, 512, tag="qkv (BN=128)")
    run(M, 1536, 64, tag="enc.l0")
    run(M, 1024, 512, tag="enc.l1")
    run(M, 3072, 512, tag="dec.l0")
    run(M, 512, 1024, tag="plain 512x1024")
    run(M, 512, 512, n_obj=12, tag="GNT", gnt=True)
    run(M, 512, 512, n_obj=12, res=True, tag="GNT+res", gnt=True)
    run(M, 512, 1024, n_obj=12, res=True, tag="GNT+res K=1024", gnt=True)
    run(M, 512, 512, n_obj=12, tag="GN")
    run(M, 512, 512, n_obj=12, res=True, tag="GN+res")
    sys.exit(0)
run(M, 512, 512, tag="plain 512x512")
run(M, 512, 1024, tag="plain 512x1024")
run(M, 512, 512, res=True, tag="plain+res")
run(M, 3072, 512, tag="dec.l0")
run(M, 1024, 512, tag="enc.l1")
for m_chk in (12 * 16 * 3, 12 * 1000):      # whole tiles / ragged last tile
    run(m_chk, 512, 512, n_obj=12, tag="GN", check=True)
    run(m_chk, 512, 512, n_obj=12, tag="GNT", gnt=True, check=True)
    run(m_chk, 512, 512, n_obj=12, res=True, tag="GNT+res", gnt=True, check=True)
    run(m_chk, 512, 1024, n_obj=12, res=True, tag="GNT+res K=1024", gnt=True, check=True)
run(M, 512, 512, n_obj=12, tag="GNT", gnt=True)
run(M, 512, 512, n_obj=12, res=True, tag="GNT+res", gnt=True)
run(M, 512, 1024, n_obj=12, res=True, tag="GNT+res K=1024", gnt=True)
run(M, 512, 512, n_obj=12, tag="GN")
run(M, 512, 512, n_obj=12, res=True, tag="GN+res")
run(M, 512, 1024, n_obj=12, res=True, tag="GN+res K=1024")
run(M, 384, 512, tag="qkv (BN=128)")
run(M, 512, 128, tag="to_out K=128")
