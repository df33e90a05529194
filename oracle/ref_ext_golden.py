"""Stored outputs of the reference's own CUDA operator (the MegEngine-CUTLASS example-19 extension built for sm_100a
by oracle/build_ref_ext.py) for tests/test_ref_ext_gpu.py.  TEST INFRASTRUCTURE.

The inputs come from seeded CPU generators, so a test rebuilds them bit for bit anywhere; for every output the file
keeps its largest magnitude and mean magnitude over the whole tensor and its values at a fixed, seeded sample of
positions.  Regenerate on a GPU machine where oracle/_ref/ext is built:

    python oracle/ref_ext_golden.py tests/golden/ref_ext_ops.npz
"""
from __future__ import annotations

import os
import sys
import zlib

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
EXT_DIR = os.path.join(HERE, "_ref", "ext")

# the reference's own test grid (test_correctness.py:16-35) plus the SLaK geometries it never tests: (N, C, HW, kh, kw)
FP32_CASES = [(1, 64, 16, 3, 3), (16, 64, 32, 7, 7), (16, 192, 16, 13, 13), (1, 192, 32, 31, 31),
              (4, 96, 56, 51, 5), (4, 96, 56, 5, 51), (4, 96, 56, 5, 5), (8, 192, 28, 49, 5), (8, 384, 14, 5, 47),
              (16, 768, 7, 13, 5)]
# the four SLaK stages: (N, C, HW, K) with the K x 5, 5 x K and 5 x 5 branches
BF16_CASES = [(4, 96, 56, 51), (8, 192, 28, 49), (8, 384, 14, 47), (16, 768, 7, 13)]
SAMPLES = 512


def key(case) -> str:
    return "_".join(str(v) for v in case)


def fp32_inputs(case):
    """x, dy, w of one fp32 case, CPU fp32."""
    N, C, HW, kh, kw = case
    g = torch.Generator().manual_seed(kh * 100 + kw + N)
    x = torch.randn(N, C, HW, HW, generator=g)
    dy = torch.randn(N, C, HW, HW, generator=g)
    w = torch.randn(C, 1, kh, kw, generator=g) * 0.05
    return x, dy, w


def bf16_inputs(case):
    """x (bf16) and the three branch weights (fp32) of one stage case, CPU."""
    N, C, HW, KL = case
    g = torch.Generator().manual_seed(KL)
    x = torch.randn(N, C, HW, HW, generator=g).bfloat16()
    ws = [torch.randn(C, 1, *k, generator=g) * 0.05 for k in ((KL, 5), (5, KL), (5, 5))]
    return x, ws


def sample_index(numel: int, name: str) -> torch.Tensor:
    """The fixed positions (flat, int64, CPU) at which the output `name` of `numel` elements is stored."""
    if numel <= SAMPLES:
        return torch.arange(numel)
    g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
    return torch.randint(numel, (SAMPLES,), generator=g)


def _store(out: dict, name: str, t: torch.Tensor) -> None:
    flat = t.detach().double().flatten().cpu()
    out[name + ".amax"] = np.float64(flat.abs().max())
    out[name + ".amean"] = np.float64(flat.abs().mean())
    out[name + ".val"] = flat[sample_index(flat.numel(), name)].float().numpy()


def generate(path: str) -> None:
    if EXT_DIR not in sys.path:
        sys.path.insert(0, EXT_DIR)
    import _depthwise_conv2d_implicit_gemm_C as ext
    dev = "cuda"
    out = {}
    for case in FP32_CASES:
        x, dy, w = (t.to(dev) for t in fp32_inputs(case))
        k = "fp32_" + key(case)
        _store(out, k + ".fwd", ext.forward_fp32(x, w))
        _store(out, k + ".dgrad", ext.backward_data_fp32(dy, w))
        _store(out, k + ".wgrad", ext.backward_filter_fp32(dy, x, w))
    for case in BF16_CASES:
        x, ws = bf16_inputs(case)
        x = x.to(dev)
        for i, w in enumerate(ws):     # fp32 on bf16-representable operands
            _store(out, f"bf16_{key(case)}.y{i}", ext.forward_fp32(x.float(), w.to(dev).bfloat16().float()))
    torch.cuda.synchronize()
    out["gpu"] = np.array(torch.cuda.get_device_name(0))
    np.savez_compressed(path, **out)


if __name__ == "__main__":
    generate(sys.argv[1])
    print(sys.argv[1], os.path.getsize(sys.argv[1]))
