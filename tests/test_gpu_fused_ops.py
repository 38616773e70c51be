"""GPU tests of the fused ResNet stem (implicit-GEMM forward with BN statistics in the epilogue, implicit weight
gradient), and every epilogue of the cta_group::2 GEMM.

First run on a B200 in round 2 (``scratch/round2_first_call.sh`` → 29 passed) and part of the default ``pytest -m gpu``
run since.  Each compares the kernel with a plain PyTorch fp32 reference of the same op.
"""
import copy

import pytest
import torch
import torch.nn.functional as F

pytestmark = [pytest.mark.gpu]


def _cl(t):
    return t.contiguous(memory_format=torch.channels_last)


def _rel(a, b):
    return (a.float() - b.float()).abs().max().item() / max(b.float().abs().max().item(), 1e-6)


@pytest.mark.parametrize("shape", [(2, 224, 224), (3, 64, 64), (1, 30, 40), (5, 17, 8), (2, 225, 256)])
def test_fused_stem_forward_and_bn_sums(shape):
    from pytorch_ps_mpi_b200.ops import ext
    from pytorch_ps_mpi_b200.ops.stem import _w2d
    n, h, w = shape
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    wt = (torch.randn(64, 3, 7, 7, device=dev) * 0.05).bfloat16()
    x = _cl(torch.randn(n, 3, h, w, device=dev).bfloat16())
    y, sums = ext.cuda().stem_fwd(x, _w2d(wt), True)
    ref = F.conv2d(x.float(), wt.float(), stride=2, padding=3)
    assert y.shape == ref.shape and y.is_contiguous(memory_format=torch.channels_last)
    assert _rel(y, ref) < 2e-2
    yf = y.float()
    want = torch.cat([yf.sum((0, 2, 3)), (yf * yf).sum((0, 2, 3))])
    assert ((sums - want).abs() / (want.abs() + 1.0)).max().item() < 1e-3


@pytest.mark.parametrize("shape", [(8, 224, 224), (2, 64, 64), (1, 30, 40), (3, 17, 8), (2, 33, 256)])
def test_implicit_stem_wgrad(shape):
    from pytorch_ps_mpi_b200.ops.stem import _w2d, stem_wgrad_implicit
    n, h, w = shape
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    x = _cl(torch.randn(n, 3, h, w, device=dev).bfloat16())
    g = _cl(torch.randn(n, 64, (h - 1) // 2 + 1, (w - 1) // 2 + 1, device=dev).bfloat16())
    # fp64 convolution weight gradient, mapped to the [64,176] GEMM layout: no repository kernel in the reference
    ref = _w2d(torch.nn.grad.conv2d_weight(x.double(), (64, 3, 7, 7), g.double(), stride=2, padding=3))
    assert _rel(stem_wgrad_implicit(x, g), ref) < 1e-2


def test_fused_stem_autograd_matches_default_path(monkeypatch):
    from pytorch_ps_mpi_b200.ops import stem as stem_mod
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    wt = (torch.randn(64, 3, 7, 7, device=dev) * 0.05).bfloat16()
    x = _cl(torch.randn(4, 3, 224, 224, device=dev).bfloat16())
    gy = _cl(torch.randn(4, 64, 112, 112, device=dev).bfloat16())
    grads = []
    for fused, implicit in ((False, False), (True, False), (True, True)):
        monkeypatch.setattr(stem_mod, "_IMPLICIT_WGRAD", implicit)       # restored after the test: later tests see the default
        wv = wt.clone().requires_grad_(True)
        y = stem_mod.stem_conv_fused(x, wv)[0] if fused else stem_mod.stem_conv(x, wv)
        y.backward(gy)
        grads.append(wv.grad.float())
    assert _rel(grads[1], grads[0]) < 1e-2 and _rel(grads[2], grads[0]) < 1e-2


@pytest.mark.parametrize("epi", [0, 1, 3, 4])   # 0 auto (TMA store / staged), 1 staged, 3 TMA store, 4 round-1 row-strided stores
@pytest.mark.parametrize("mnk", [(512, 256, 128), (1000, 328, 264), (4096, 3072, 768), (300, 64, 176), (515, 330, 72)])
def test_gemm_epilogue_variants(epi, mnk):
    from pytorch_ps_mpi_b200.ops.linear import bcast_linear
    M, N, K = mnk
    if epi == 3 and N % 8:
        pytest.skip("TMA-store epilogue needs N % 8 == 0")
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    x = (torch.randn(M, K, device=dev) / K ** 0.5).bfloat16()
    w = torch.randn(N, K, device=dev).bfloat16()
    b = torch.randn(N, device=dev)
    ref = torch.relu(x.float() @ w.float().t() + b)
    y = bcast_linear(x, w, b, relu=True, variant=2 | epi << 4)
    assert _rel(y, ref) < 2e-2
