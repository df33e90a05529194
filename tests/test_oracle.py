"""The oracle against (a) the reference's own host code (its outputs stored in
tests/golden/ref_host_dwconv.npz by oracle/gen_golden.py), (b) the torch statement the
reference's test uses, (c) committed golden vectors.  CPU only."""
import os

import numpy as np
import pytest
import torch

from oracle import dwconv as orc

CASES = [(2, 3, 9, 8, 7, 3), (1, 2, 16, 16, 13, 13), (2, 2, 14, 14, 47, 5), (1, 3, 7, 7, 5, 13), (1, 1, 1, 1, 3, 3)]
HOST = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_host_dwconv.npz"))


@pytest.mark.parametrize("case", CASES)
def test_c_restatement_equals_torch_float64(case):
    N, C, H, W, R, S = case
    g = torch.Generator().manual_seed(sum(case))
    x = torch.randn(N, C, H, W, generator=g)
    dy = torch.randn(N, C, H, W, generator=g)
    w = torch.randn(C, 1, R, S, generator=g)
    y64 = orc.fwd_torch(x.double(), w.double())
    dx64, dw64 = orc.grads_torch(x.double(), w.double(), dy.double())
    np.testing.assert_allclose(orc.fwd_c(x.numpy(), w.numpy()), y64.float().numpy(), rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(orc.bwd_data_c(dy.numpy(), w.numpy()), dx64.float().numpy(), rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(orc.bwd_filter_c(dy.numpy(), x.numpy(), w.shape), dw64.float().numpy(), rtol=1e-6, atol=1e-5)


@pytest.mark.parametrize("case", CASES)
def test_c_restatement_equals_reference_host_code(case):
    N, C, H, W, R, S = case
    g = torch.Generator().manual_seed(sum(case) + 1)
    x = torch.randn(N, C, H, W, generator=g).numpy()
    dy = torch.randn(N, C, H, W, generator=g).numpy()
    w = torch.randn(C, 1, R, S, generator=g).numpy()
    k = "_".join(map(str, case))
    # the reference accumulates in fp32, the restatement in double
    np.testing.assert_allclose(orc.fwd_c(x, w), HOST[k + ".fwd"], rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(orc.bwd_data_c(dy, w), HOST[k + ".bwd_data"], rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(orc.bwd_filter_c(dy, x, w.shape), HOST[k + ".bwd_filter"], rtol=1e-4, atol=1e-3)


def test_integer_valued_exact_equality_like_cutlass_testbed():
    """cutlass/test/unit/convolution/device/testbed.h:254-277,438 checks exact equality on
    integer-valued fills in +-8: sums stay exact in fp32, so all three must agree bit for bit."""
    g = torch.Generator().manual_seed(3)
    x = torch.randint(-8, 9, (3, 7, 16, 16), generator=g).float()
    w = torch.randint(-8, 9, (7, 1, 15, 5), generator=g).float()
    y_t = orc.fwd_torch(x, w).numpy()
    assert np.array_equal(orc.fwd_c(x.numpy(), w.numpy()), y_t)
    assert np.array_equal(HOST["int.fwd"].astype(np.float32), y_t)


def test_config1_plumbing_case():
    """BASELINE.json configs[0]: single 51x5 depthwise fwd, 1x96x56x56 fp32 on CPU nn.Conv2d."""
    torch.manual_seed(0)
    x = torch.randn(1, 96, 56, 56)
    w = torch.randn(96, 1, 51, 5) * 0.02
    m = torch.nn.Conv2d(96, 96, (51, 5), padding=(25, 2), groups=96, bias=False)
    with torch.no_grad():
        m.weight.copy_(w)
        y = m(x)
    assert torch.allclose(y, orc.fwd_torch(x, w), rtol=1e-5, atol=1e-6)
    sub = orc.fwd_c(x[:, :2].numpy(), w[:2].numpy())
    np.testing.assert_allclose(sub, y[:, :2].numpy(), rtol=1e-4, atol=1e-5)
