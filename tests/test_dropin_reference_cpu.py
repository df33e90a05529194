"""INTEGRATION.md section 1 on the host side: slak_b200/dropin stands in for the CUTLASS example directory the
reference's models/SLaK.py, sparse_core.py and depthwise_conv2d_implicit_gemm.py import.  What those reference files
built and called with the drop-in in place is stored in tests/golden/ref_dropin.npz (oracle/gen_golden.py dropin);
these tests check the drop-in and this library against it.  Nothing is executed on a GPU."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "ref_dropin.npz")

SCRIPT = textwrap.dedent("""
    import sys, types
    import numpy as np
    root, golden = sys.argv[1], np.load(sys.argv[2])
    # the drop-in directory in place of the CUTLASS example directory (models/SLaK.py:9-10)
    sys.path[:0] = [root, root + "/slak_b200/dropin"]
    import torch
    import depthwise_conv2d_implicit_gemm as op
    assert op.__file__.startswith(root + "/slak_b200/dropin"), op.__file__
    from slak_b200.dwconv import DepthWiseConv2dImplicitGEMM
    assert op.DepthWiseConv2dImplicitGEMM is DepthWiseConv2dImplicitGEMM
    from slak_b200 import slak
    slak.use_sync_bn = False
    ours = slak.SLaK_tiny(kernel_size=[51, 49, 47, 13, 5], Decom=True, bn=True, width_factor=0.25)
    convs = [m for m in ours.modules() if isinstance(m, DepthWiseConv2dImplicitGEMM)]
    # the reference model built on the drop-in holds as many of them: 18 Blocks x 3 branches
    assert len(convs) == int(golden["tiny.dwconv_modules"]) == 54 and all(isinstance(m, torch.nn.Conv2d) for m in convs)
    sd = ours.state_dict()
    assert list(sd.keys()) == list(golden["tiny.keys"])
    assert [",".join(map(str, v.shape)) for v in sd.values()] == list(golden["tiny.shapes"])
    assert [str(v.dtype) for v in sd.values()] == list(golden["tiny.dtypes"])
    # reference checkpoints load unchanged: a state_dict with the reference's keys, shapes and dtypes
    g = torch.Generator().manual_seed(0)
    ref_sd = {}
    for k, s, d in zip(golden["tiny.keys"], golden["tiny.shapes"], golden["tiny.dtypes"]):
        shape = [int(v) for v in s.split(",") if v]
        dt = getattr(torch, d.split(".")[1])
        ref_sd[k] = torch.randn(shape, generator=g).to(dt) if dt.is_floating_point else torch.zeros(shape, dtype=dt)
    ours.load_state_dict(ref_sd)
    assert all(torch.equal(ours.state_dict()[k], v) for k, v in ref_sd.items())
    # the mask engine picks the tensors the reference's sparse_core.Masking picked on its model (--only-L: the LoRAs)
    from slak_b200 import sparse_core
    opt = torch.optim.SGD(ours.parameters(), lr=0.1, momentum=0.9)
    args = types.SimpleNamespace(device="cpu", fix=False, update_frequency=100, only_L=True, sparse_init="uniform",
                                 sparsity=0.4, distributed=False)
    mask = sparse_core.Masking(opt, train_loader=None, prune_rate_decay=sparse_core.CosineDecay(0.3, 100),
                               prune_rate=0.3, prune_mode="magnitude", growth_mode="random", redistribution_mode="none",
                               args=args)
    mask.add_module(ours)
    assert sorted(mask.masks) == sorted(golden["tiny.mask_names"]) and len(mask.masks) == 36
    # without a CUDA device the operator refuses instead of computing on the CPU
    try:
        convs[0](torch.zeros(1, convs[0].in_channels, 8, 8))
    except RuntimeError as e:
        assert "CUDA" in str(e)
    else:
        raise AssertionError("CPU tensor accepted")
    print("DROPIN_OK")
""")


@pytest.mark.timeout(600)
def test_reference_model_and_mask_engine_run_on_the_dropin_module():
    r = subprocess.run([sys.executable, "-c", SCRIPT, ROOT, GOLDEN], capture_output=True, text=True, timeout=580, cwd=ROOT)
    assert r.returncode == 0 and "DROPIN_OK" in r.stdout, (r.stdout[-1500:], r.stderr[-3000:])


SCRIPT_C = textwrap.dedent("""
    import sys
    import numpy as np
    root, golden = sys.argv[1], np.load(sys.argv[2])
    # only the native module is replaced: a directory holding just our _depthwise_conv2d_implicit_gemm_C stand-in
    import os, shutil, tempfile
    tmp = tempfile.mkdtemp()
    shutil.copy(root + "/slak_b200/dropin/_depthwise_conv2d_implicit_gemm_C.py", tmp)
    sys.path[:0] = [root, tmp]
    import torch
    import _depthwise_conv2d_implicit_gemm_C as native
    shutil.rmtree(tmp)
    # every native function the reference's depthwise_conv2d_implicit_gemm.py calls (frontend.h:3-10)
    names = list(golden["op.native_calls"])
    assert len(names) == 6, names
    for name in names:
        fn = getattr(native, name)
        dt = torch.float16 if name.endswith("fp16") else torch.float32
        args = {"forward": 2, "backward_data": 2, "backward_filter": 3}[name.rsplit("_", 1)[0]]
        ins = [torch.zeros(1, 8, 16, 16, dtype=dt)] * (args - 1) + [torch.zeros(8, 1, 13, 5, dtype=dt)]
        try:
            fn(*ins)
        except RuntimeError as e:
            assert "CUDA" in str(e), (name, str(e))
        else:
            raise AssertionError(name + ": CPU tensor accepted")
    print("DROPIN_C_OK")
""")


@pytest.mark.timeout(300)
def test_reference_python_module_runs_on_the_native_standin():
    r = subprocess.run([sys.executable, "-c", SCRIPT_C, ROOT, GOLDEN], capture_output=True, text=True, timeout=280,
                       cwd=ROOT)
    assert r.returncode == 0 and "DROPIN_C_OK" in r.stdout, (r.stdout[-1500:], r.stderr[-3000:])


def test_kernel_merge_and_bn_folding_equal_the_reference():
    """get_equivalent_kernel_bias / merge_kernel (models/SLaK.py:49-58,102-122) against the reference's results on the
    same non-trivial statistics and affine parameters."""
    sys.path.insert(0, ROOT)
    from slak_b200 import slak
    golden = np.load(GOLDEN)
    for K, small in ((13, 5), (7, 3), (9, None)):
        tag = f"merge_{K}_{small}."
        kw = dict(in_channels=6, out_channels=6, kernel_size=K, stride=1, groups=6, small_kernel=small,
                  small_kernel_merged=False, Decom=False, bn=True)
        ours = slak.ReparamLargeKernelConv(**kw)
        sd0 = {k[len(tag) + 4:]: torch.from_numpy(golden[k]) for k in golden.files if k.startswith(tag + "sd0.")}
        assert list(ours.state_dict().keys()) == list(sd0.keys())
        ours.load_state_dict(sd0)
        k1, b1 = ours.get_equivalent_kernel_bias()
        assert torch.equal(k1, torch.from_numpy(golden[tag + "kernel"])), (K, small)
        assert torch.equal(b1, torch.from_numpy(golden[tag + "bias"])), (K, small)
        ours.merge_kernel()
        sd1 = {k[len(tag) + 4:]: golden[k] for k in golden.files if k.startswith(tag + "sd1.")}
        assert list(ours.state_dict().keys()) == list(sd1.keys()) == ["lkb_reparam.weight", "lkb_reparam.bias"]
        for k, v in ours.state_dict().items():
            assert torch.equal(v, torch.from_numpy(sd1[k])), (K, small, k)
