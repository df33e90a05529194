"""Parity of the CUDA depthwise-conv path (through the C ABI) against the oracle.

Cases: the reference's own test grid (test_correctness.py:16-127: batch{1,16} x C{64,192} x
k{3,7,13,31} x res{16,32} x seed{0,42}, its tolerances) plus what the reference never tests:
rectangular 51x5 / 5x51, kernels larger than the map, bf16, ragged sizes.
"""
import os

import numpy as np
import pytest
import torch

from oracle import dwconv as orc
from slak_b200 import ops
from slak_b200.dwconv import DepthWiseConv2dImplicitGEMM

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _rel_linf(a, b):
    return (a.double() - b.double()).abs().max().item() / max(b.double().abs().max().item(), 1e-30)


# ---- the reference's own grid, its own oracle and tolerances -------------------------
@pytest.mark.parametrize("batch_size", [1, 16])
@pytest.mark.parametrize("channels", [64, 192])
@pytest.mark.parametrize("kernel_size", [3, 7, 13, 31])
@pytest.mark.parametrize("resolution", [16, 32])
@pytest.mark.parametrize("seed", [0, 42])
def test_forward_fp32_reference_grid(batch_size, channels, kernel_size, resolution, seed):
    torch.random.manual_seed(seed)
    x = torch.randn(batch_size, channels, resolution, resolution)
    m = DepthWiseConv2dImplicitGEMM(channels, kernel_size)
    y_ref = orc.fwd_torch(x, m.weight.detach())
    y = m.to(DEV)(x.to(DEV))
    assert y.dtype == torch.float
    assert torch.allclose(y.cpu(), y_ref, rtol=1e-5, atol=1e-6), (y.cpu() - y_ref).abs().max()


@pytest.mark.parametrize("batch_size", [1, 16])
@pytest.mark.parametrize("kernel_size", [3, 7, 13])
@pytest.mark.parametrize("seed", [0, 42])
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_forward_half_reference_grid(batch_size, kernel_size, seed, dtype):
    channels, resolution = 64, 16
    torch.random.manual_seed(seed)
    x = torch.randn(batch_size, channels, resolution, resolution).to(dtype)
    m = DepthWiseConv2dImplicitGEMM(channels, kernel_size)
    # oracle: fp32 conv of the rounded operands, then rounded to the output type
    y_ref = orc.fwd_torch(x.float(), orc.round_like(m.weight.detach(), dtype)).to(dtype)
    y = m.to(DEV)(x.to(DEV))
    assert y.dtype == dtype
    tol = dict(rtol=1e-3, atol=1e-6) if dtype == torch.float16 else dict(rtol=8e-3, atol=1e-6)
    assert torch.allclose(y.cpu().float(), y_ref.float(), **tol), (y.cpu().float() - y_ref.float()).abs().max()


@pytest.mark.parametrize("batch_size", [1, 16])
@pytest.mark.parametrize("kernel_size", [3, 7, 13])
@pytest.mark.parametrize("seed", [0, 42])
def test_backward_fp32_reference_grid(batch_size, kernel_size, seed):
    channels, resolution = 64, 16
    torch.random.manual_seed(seed)
    x = torch.randn(batch_size, channels, resolution, resolution)
    m = DepthWiseConv2dImplicitGEMM(channels, kernel_size)
    w = m.weight.detach().clone()
    xr = x.clone().requires_grad_(True)
    wr = w.clone().requires_grad_(True)
    orc.fwd_torch(xr, wr).mean().backward()
    xg = x.to(DEV).requires_grad_(True)
    mg = m.to(DEV)
    mg(xg).mean().backward()
    assert torch.allclose(xg.grad.cpu(), xr.grad, rtol=1e-5, atol=1e-8), (xg.grad.cpu() - xr.grad).abs().max()
    assert mg.weight.grad.dtype == torch.float
    assert torch.allclose(mg.weight.grad.cpu(), wr.grad, rtol=1e-4, atol=1e-6), (mg.weight.grad.cpu() - wr.grad).abs().max()


# ---- SLaK shapes: rectangular, kernel > map, odd channel counts, all three ops ------------
SLAK_CASES = [
    # N, C, H, W, kh, kw
    (3, 5, 56, 56, 51, 5), (3, 5, 56, 56, 5, 51), (3, 5, 56, 56, 5, 5),
    (5, 6, 28, 28, 49, 5), (5, 6, 28, 28, 5, 49), (5, 6, 28, 28, 5, 5),
    (9, 7, 14, 14, 47, 5), (9, 7, 14, 14, 5, 47), (9, 7, 14, 14, 5, 5),
    (11, 9, 7, 7, 13, 5), (11, 9, 7, 7, 5, 13), (11, 9, 7, 7, 5, 5),
    (2, 3, 96, 96, 51, 5), (2, 3, 96, 96, 5, 51),
    (2, 4, 33, 45, 61, 5), (2, 4, 45, 33, 5, 61), (1, 1, 1, 1, 5, 5), (2, 2, 5, 70, 7, 3),
    (2, 3, 20, 20, 51, 51), (1, 2, 40, 24, 9, 11), (2, 2, 130, 130, 5, 51),
]


@pytest.mark.parametrize("case", SLAK_CASES)
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
def test_slak_shapes_fwd_dgrad_wgrad(case, dtype):
    N, C, H, W, kh, kw = case
    g = torch.Generator().manual_seed(1234 + N + kh)
    x = torch.randn(N, C, H, W, generator=g).to(dtype)
    dy = torch.randn(N, C, H, W, generator=g).to(dtype)
    w = (torch.randn(C, 1, kh, kw, generator=g) * 0.02)
    # truth: float64 conv of the operands as the kernel sees them (weights rounded to dtype)
    wq = orc.round_like(w, dtype)
    y64 = orc.fwd_torch(x.double(), wq.double())
    dx64, dw64 = orc.grads_torch(x.double(), wq.double(), dy.double())
    xg, dyg, wg = x.to(DEV), dy.to(DEV), w.to(DEV)
    y = ops.dwconv2d_forward(xg, wg).cpu()
    dx = ops.dwconv2d_backward_data(dyg, wg).cpu()
    dw = ops.dwconv2d_backward_filter(dyg, xg, wg).cpu()
    assert y.dtype == dtype and dx.dtype == dtype and dw.dtype == torch.float32
    out_eps = {torch.float32: 1e-5, torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}[dtype]
    assert _rel_linf(y, y64) <= 1e-5 + out_eps, _rel_linf(y, y64)
    assert _rel_linf(dx, dx64) <= 1e-5 + out_eps, _rel_linf(dx, dx64)
    assert _rel_linf(dw, dw64) <= 1e-4, _rel_linf(dw, dw64)   # fp32 result for every dtype


def test_small_case_against_c_oracle_and_reference_host_code():
    g = torch.Generator().manual_seed(7)
    x = torch.randn(2, 3, 12, 10, generator=g)
    dy = torch.randn(2, 3, 12, 10, generator=g)
    w = torch.randn(3, 1, 7, 5, generator=g)
    y = ops.dwconv2d_forward(x.to(DEV), w.to(DEV)).cpu().numpy()
    dx = ops.dwconv2d_backward_data(dy.to(DEV), w.to(DEV)).cpu().numpy()
    dw = ops.dwconv2d_backward_filter(dy.to(DEV), x.to(DEV), w.to(DEV)).cpu().numpy()
    np.testing.assert_allclose(y, orc.fwd_c(x.numpy(), w.numpy()), rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(dx, orc.bwd_data_c(dy.numpy(), w.numpy()), rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(dw, orc.bwd_filter_c(dy.numpy(), x.numpy(), w.shape), rtol=1e-5, atol=1e-4)
    ref = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_host_dwconv.npz"))["small.fwd"]
    np.testing.assert_allclose(y, ref, rtol=1e-5, atol=1e-5)             # the reference's host code (oracle/gen_golden.py)


def test_full_size_linearity_and_adjointness():
    """BASELINE config-2 stage-1 size (128x96x56x56, 51x5, bf16): size-independent properties.
    <conv(x), dy> == <x, dgrad(dy)> == <w, wgrad(dy, x)> and conv(a*x) == a*conv(x)."""
    torch.manual_seed(0)
    N, C, H, W = 128, 96, 56, 56
    x = torch.randn(N, C, H, W, device=DEV).bfloat16()
    dy = torch.randn(N, C, H, W, device=DEV).bfloat16()
    w = (torch.randn(C, 1, 51, 5, device=DEV) * 0.02)
    y = ops.dwconv2d_forward(x, w)
    dx = ops.dwconv2d_backward_data(dy, w)
    dw = ops.dwconv2d_backward_filter(dy, x, w)
    wq = w.bfloat16().double()
    a = (y.double() * dy.double()).sum().item()       # y rounded to bf16: ~2^-9 relative noise, averaged
    b = (x.double() * dx.double()).sum().item()
    c = (wq * dw.double()).sum().item()
    scale = (y.double().abs() * dy.double().abs()).sum().item()
    assert abs(a - c) / scale < 1e-4 and abs(b - c) / scale < 1e-4, (a, b, c, scale)
    y2 = ops.dwconv2d_forward((x * 2).contiguous(), w)
    assert torch.equal(y2, y * 2)                      # power-of-two scaling is exact in bf16
    # determinism of wgrad (fixed reduction order, no atomics)
    dw2 = ops.dwconv2d_backward_filter(dy, x, w)
    assert torch.equal(dw, dw2)


def test_error_behaviour():
    x = torch.randn(1, 4, 8, 8, device=DEV)
    m = DepthWiseConv2dImplicitGEMM(4, 3).to(DEV)
    with pytest.raises(TypeError):
        m(x.double())
    with pytest.raises(RuntimeError):
        ops.dwconv2d_forward(x.cpu(), m.weight.detach())
    with pytest.raises(RuntimeError):
        ops.dwconv2d_forward(x.permute(0, 1, 3, 2), m.weight.detach())
    with pytest.raises(ValueError):
        DepthWiseConv2dImplicitGEMM(4, 4)


def test_single_conv_entry_points_route_bf16_slak_shapes_to_tensor_cores():
    """The six frontend symbols (frontend.h:3-10) reach the tcgen05 kernels for bf16 K x 5 / 5 x K / 5 x 5 on every
    SLaK-T stage geometry; fp32 (exact path), fp16, square kernels and planes above 62 x 62 stay on the CUDA cores."""
    from slak_b200 import _lib
    lib = _lib.load()
    BF, F32, F16 = _lib.SLAK_BF16, _lib.SLAK_F32, _lib.SLAK_F16
    for C, hw, K in ((96, 56, 51), (192, 28, 49), (384, 14, 47), (768, 7, 13)):
        for kh, kw in ((K, 5), (5, K), (5, 5)):
            assert lib.slak_dwconv2d_uses_tc(128, C, hw, hw, kh, kw, BF, F32) == 1
            assert lib.slak_dwconv2d_uses_tc(128, C, hw, hw, kh, kw, F32, F32) == 0
            assert lib.slak_dwconv2d_uses_tc(128, C, hw, hw, kh, kw, F16, F32) == 0
    assert lib.slak_dwconv2d_uses_tc(32, 128, 96, 96, 51, 5, BF, F32) == 0
    assert lib.slak_dwconv2d_uses_tc(32, 128, 32, 32, 31, 31, BF, F32) == 0
    # the module surface under bf16: forward + backward through the tensor-core route against the oracle
    torch.manual_seed(0)
    m = DepthWiseConv2dImplicitGEMM(96, (51, 5)).to(DEV)
    x = torch.randn(8, 96, 56, 56, device=DEV).bfloat16().requires_grad_(True)
    y = m(x)
    dy = torch.randn_like(y)
    y.backward(dy)
    wq = orc.round_like(m.weight.detach().cpu(), torch.bfloat16).double()
    y64 = orc.fwd_torch(x.detach().cpu().double(), wq)
    dx64, dw64 = orc.grads_torch(x.detach().cpu().double(), wq, dy.cpu().double())
    assert _rel_linf(y.detach().cpu(), y64) <= 2.0 ** -8 + 1e-5
    assert _rel_linf(x.grad.cpu(), dx64) <= 2.0 ** -8 + 1e-5
    assert m.weight.grad.dtype == torch.float32 and _rel_linf(m.weight.grad.cpu(), dw64) <= 1e-4
