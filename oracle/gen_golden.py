"""Generate tests/golden/*.npz by IMPORTING THE REFERENCE (models/SLaK.py, sparse_core.py,
funcs.py under /root/reference, unmodified) in the authoring container.  The reference cannot
travel to the GPU box, so the vectors are committed.  Run:  python oracle/gen_golden.py
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("SLAK_REFERENCE", "/root/reference")
OUT = os.path.join(ROOT, "tests", "golden")


def import_reference():
    sys.path.insert(0, REF)
    sys.path.insert(0, os.path.join(HERE, "ref_shims"))   # shims shadow timm and the CUDA-only op module
    import models.SLaK as ref_slak        # noqa
    import sparse_core as ref_sparse      # noqa
    import funcs as ref_funcs             # noqa
    ref_slak.use_sync_bn = True           # nn.SyncBatchNorm works on CPU without a process group
    return ref_slak, ref_sparse, ref_funcs


def sd_numpy(module, prefix=""):
    return {prefix + k: v.detach().cpu().numpy().copy() for k, v in module.state_dict().items()}


def gen_block(ref_slak):
    """One Block (Decom, bn) forward + backward in train mode, and forward in eval mode."""
    for tag, dim, ks, hw in [("k13", 8, (13, 5), 14), ("k51", 6, (51, 5), 20)]:
        torch.manual_seed(11)
        blk = ref_slak.Block(dim=dim, drop_path=0.0, layer_scale_init_value=0.5, kernel_size=ks, Decom=True, bn=True)
        for p in blk.parameters():
            if p.dim() > 1:
                torch.nn.init.normal_(p, std=0.2)
        for m in blk.modules():
            if isinstance(m, torch.nn.modules.batchnorm._BatchNorm):
                torch.nn.init.uniform_(m.weight, 0.5, 1.5)
                torch.nn.init.uniform_(m.bias, -0.5, 0.5)
        x = torch.randn(3, dim, hw, hw, requires_grad=True)
        cot = torch.randn(3, dim, hw, hw)
        out = {"x": x.detach().numpy(), "cot": cot.numpy()}
        out.update(sd_numpy(blk, "sd0."))           # parameters + running stats BEFORE the step
        blk.train()
        y = blk(x)
        (y * cot).sum().backward()
        out["y_train"] = y.detach().numpy()
        out["dx"] = x.grad.numpy()
        for n, p in blk.named_parameters():
            out["grad." + n] = p.grad.numpy()
        out.update(sd_numpy(blk, "sd1."))           # running stats AFTER one training forward
        blk.eval()
        with torch.no_grad():
            out["y_eval"] = blk(x.detach()).numpy()
        np.savez_compressed(os.path.join(OUT, f"ref_block_{tag}.npz"), **out)


def gen_model(ref_slak):
    """A narrow SLaK (reference class, reference init) end to end, eval and train mode."""
    torch.manual_seed(5)
    depths, dims = [1, 1, 2, 1], [8, 12, 16, 24]
    net = ref_slak.SLaK(depths=depths, dims=dims, num_classes=10, drop_path_rate=0.0, layer_scale_init_value=1.0,
                        kernel_size=[17, 15, 13, 7, 5], width_factor=1.0, Decom=True, bn=True)
    x = torch.randn(2, 3, 64, 64)
    out = {"x": x.numpy(), "depths": np.array(depths), "dims": np.array(dims)}
    out.update(sd_numpy(net, "sd."))
    net.eval()
    with torch.no_grad():
        out["logits_eval"] = net(x).numpy()
    net.train()
    out["logits_train"] = net(x).detach().numpy()
    np.savez_compressed(os.path.join(OUT, "ref_slak_narrow.npz"), **out)


# (file tag, init, only_L, prune mode, growth mode); the first four are the SLaK defaults (funcs.py:107-114,170-175)
MASKING_VARIANTS = [
    ("uniform_all", "uniform", False, "magnitude", "random"),
    ("uniform_onlyL", "uniform", True, "magnitude", "random"),
    ("ERK_all", "ERK", False, "magnitude", "random"),
    ("ERK_onlyL", "ERK", True, "magnitude", "random"),
    # the other modes of sparse_core.py:141-261 / funcs.py that slak_b200 mirrors
    ("snip_all", "snip", False, "magnitude", "random"),
    ("uniform_all_gradient", "uniform", False, "magnitude", "gradient"),
    ("uniform_all_momentum", "uniform", False, "magnitude", "momentum"),
    # prune_mode "SET" cannot be pinned: the reference's magnitude_and_negativity_prune reads a Masking attribute
    # that does not exist (funcs.py:150 `name2prune_rate`) and raises at the first prune round
]


def gen_masking(ref_slak, ref_sparse, only=None):
    """sparse_core.Masking on CPU: init (uniform / ERK / snip), per-step apply_mask, and three prune-and-grow
    rounds per variant, CPU RNG seeded like main.py:232.  `only`: write just the variants whose tag is listed."""
    torch.Tensor.cuda = lambda self, *a, **k: self      # funcs.py:174 calls .cuda() on the CPU draw
    for tag, init, only_l, prune_mode, growth_mode in MASKING_VARIANTS:
        if only is not None and tag not in only:
            continue
        torch.manual_seed(0)
        np.random.seed(0)
        net = torch.nn.Sequential()
        net.add_module("stages", torch.nn.Sequential(
            ref_slak.Block(dim=8, kernel_size=(13, 5), Decom=True, bn=True, layer_scale_init_value=1.0),
            ref_slak.Block(dim=8, kernel_size=(9, 5), Decom=True, bn=True, layer_scale_init_value=1.0)))
        for p in net.parameters():
            if p.dim() > 1:
                torch.nn.init.normal_(p, std=0.1)
        opt = torch.optim.SGD(net.parameters(), lr=0.1, momentum=0.9)
        args = types.SimpleNamespace(device="cpu", fix=False, update_frequency=2, only_L=only_l,
                                     sparse_init=init, sparsity=0.4, distributed=False)
        out = {}
        loader = None
        if init == "snip":                               # one batch for SNIP(): per-pixel 8-way classification
            gl = torch.Generator().manual_seed(7)
            images = torch.randn(4, 8, 12, 12, generator=gl)
            labels = torch.randint(0, 8, (4, 12, 12), generator=gl)
            loader = [(images, labels)]
            out["snip_images"] = images.numpy().copy()
            out["snip_labels"] = labels.numpy().copy()
        T = 12
        decay = ref_sparse.CosineDecay(0.5, T)
        mask = ref_sparse.Masking(opt, train_loader=loader, prune_rate_decay=decay, prune_rate=0.5,
                                  prune_mode=prune_mode, growth_mode=growth_mode, redistribution_mode="none",
                                  args=args)
        for n, p in net.named_parameters():
            out["w_init." + n] = p.detach().numpy().copy()
        torch.manual_seed(123)                      # the stream Masking.init draws from
        mask.add_module(net)
        out["mask_names"] = np.array(sorted(mask.masks.keys()))
        for n, m in mask.masks.items():
            out["mask0." + n] = m.numpy().copy()
        for n, p in net.named_parameters():
            out["w0." + n] = p.detach().numpy().copy()
        g = torch.Generator().manual_seed(99)
        rates = []
        for step in range(1, 7):
            # deterministic pseudo-gradients, then the reference's own step()
            for p in net.parameters():
                p.grad = torch.randn(p.shape, generator=g) * 0.05
            torch.manual_seed(1000 + step)          # stream random_growth draws from
            mask.step()
            rates.append(mask.prune_rate)
            for n, m in mask.masks.items():
                out[f"mask{step}." + n] = m.numpy().copy()
            for n, p in net.named_parameters():
                out[f"w{step}." + n] = p.detach().numpy().copy()
            for n, p in net.named_parameters():
                st = opt.state[p]
                if "momentum_buffer" in st:
                    out[f"mom{step}." + n] = st["momentum_buffer"].numpy().copy()
        out["prune_rates"] = np.array(rates)
        np.savez_compressed(os.path.join(OUT, f"ref_masking_{tag}.npz"), **out)


def gen_conv_grid():
    """A slice of the reference's own test grid (test_correctness.py:16-35), torch CPU results."""
    import torch.nn.functional as F
    out = {}
    for seed in (0, 42):
        for k in (3, 7, 13, 31):
            torch.random.manual_seed(seed)
            x = torch.randn(1, 64, 16, 16)
            m = torch.nn.Conv2d(64, 64, k, groups=64, bias=False)
            y = F.conv2d(x, m.weight, padding=k // 2, groups=64)
            out[f"s{seed}_k{k}_w"] = m.weight.detach().numpy()[:4]
            out[f"s{seed}_k{k}_x"] = x.numpy()[:, :4]
            out[f"s{seed}_k{k}_y"] = y.detach().numpy()[:, :4]
    np.savez_compressed(os.path.join(OUT, "ref_conv_grid.npz"), **out)


# (N, C, H, W, R, S) of tests/test_oracle.py
HOST_CASES = [(2, 3, 9, 8, 7, 3), (1, 2, 16, 16, 13, 13), (2, 2, 14, 14, 47, 5), (1, 3, 7, 7, 5, 13), (1, 1, 1, 1, 3, 3)]


def gen_ref_host():
    """The reference's own host-side depthwise convolution (oracle/_ref/libslak_ref.so, built by oracle/Makefile from
    the reference's CUTLASS headers) on the inputs of tests/test_oracle.py and tests/test_dwconv_gpu.py."""
    sys.path.insert(0, ROOT)
    from oracle import dwconv as orc
    assert orc.ref_available(), "oracle/_ref/libslak_ref.so not built (make -C oracle)"
    out = {}
    for case in HOST_CASES:
        N, C, H, W, R, S = case
        g = torch.Generator().manual_seed(sum(case) + 1)
        x = torch.randn(N, C, H, W, generator=g).numpy()
        dy = torch.randn(N, C, H, W, generator=g).numpy()
        w = torch.randn(C, 1, R, S, generator=g).numpy()
        k = "_".join(map(str, case))
        out[k + ".fwd"] = orc.fwd_ref(x, w)
        out[k + ".bwd_data"] = orc.bwd_data_ref(dy, w)
        out[k + ".bwd_filter"] = orc.bwd_filter_ref(dy, x, w.shape)
    g = torch.Generator().manual_seed(3)                    # integer-valued fills (test_oracle.py)
    x = torch.randint(-8, 9, (3, 7, 16, 16), generator=g).float()
    w = torch.randint(-8, 9, (7, 1, 15, 5), generator=g).float()
    y = orc.fwd_ref(x.numpy(), w.numpy())
    assert np.array_equal(y, y.astype(np.int16))            # exact integer sums: stored as such
    out["int.fwd"] = y.astype(np.int16)
    g = torch.Generator().manual_seed(7)                    # the small GPU case (test_dwconv_gpu.py)
    x = torch.randn(2, 3, 12, 10, generator=g)
    torch.randn(2, 3, 12, 10, generator=g)
    w = torch.randn(3, 1, 7, 5, generator=g)
    out["small.fwd"] = orc.fwd_ref(x.numpy(), w.numpy())
    np.savez_compressed(os.path.join(OUT, "ref_host_dwconv.npz"), **out)


def gen_dropin():
    """The reference's models/SLaK.py, sparse_core.py and operator module imported with slak_b200/dropin in place of
    the CUTLASS example directory (INTEGRATION.md section 1): what they build and call, for
    tests/test_dropin_reference_cpu.py."""
    import re
    sys.path[:0] = [ROOT, os.path.join(ROOT, "slak_b200", "dropin"), REF]
    shim = types.ModuleType("timm")
    shim.__path__ = [os.path.join(HERE, "ref_shims", "timm")]
    sys.modules["timm"] = shim
    import depthwise_conv2d_implicit_gemm as op
    import models.SLaK as ref_slak
    import sparse_core as ref_sparse
    from slak_b200 import slak
    assert ref_slak.DepthWiseConv2dImplicitGEMM is op.DepthWiseConv2dImplicitGEMM
    out = {}
    ref_slak.use_sync_bn = False
    slak.use_sync_bn = False
    net = ref_slak.SLaK_tiny(kernel_size=[51, 49, 47, 13, 5], Decom=True, bn=True, width_factor=0.25)
    sd = net.state_dict()
    out["tiny.keys"] = np.array(list(sd.keys()))
    out["tiny.shapes"] = np.array([",".join(map(str, v.shape)) for v in sd.values()])
    out["tiny.dtypes"] = np.array([str(v.dtype) for v in sd.values()])
    out["tiny.dwconv_modules"] = np.array(sum(isinstance(m, op.DepthWiseConv2dImplicitGEMM) for m in net.modules()))
    torch.Tensor.cuda = lambda self, *a, **k: self
    opt = torch.optim.SGD(net.parameters(), lr=0.1, momentum=0.9)
    args = types.SimpleNamespace(device="cpu", fix=False, update_frequency=100, only_L=True, sparse_init="uniform",
                                 sparsity=0.4, distributed=False)
    mask = ref_sparse.Masking(opt, train_loader=None, prune_rate_decay=ref_sparse.CosineDecay(0.3, 100), prune_rate=0.3,
                              prune_mode="magnitude", growth_mode="random", redistribution_mode="none", args=args)
    mask.add_module(net)
    out["tiny.mask_names"] = np.array(list(mask.masks.keys()))
    # the reference's operator module: the native functions it calls and the module it builds
    ext_py = os.path.join(REF, "cutlass", "examples", "19_large_depthwise_conv2d_torch_extension",
                          "depthwise_conv2d_implicit_gemm.py")
    out["op.native_calls"] = np.array(sorted(set(re.findall(r"_extension\.(\w+)\(", open(ext_py).read()))))
    # kernel merge and BN folding (models/SLaK.py:49-58,102-122) on non-trivial statistics
    torch.manual_seed(5)
    for K, small in ((13, 5), (7, 3), (9, None)):
        kw = dict(in_channels=6, out_channels=6, kernel_size=K, stride=1, groups=6, small_kernel=small,
                  small_kernel_merged=False, Decom=False, bn=True)
        ours = slak.ReparamLargeKernelConv(**kw)
        for b in ours.branches():
            b.bn.running_mean.normal_(); b.bn.running_var.uniform_(0.5, 2.0)
            b.bn.weight.data.normal_(1, 0.2); b.bn.bias.data.normal_()
            b.conv.weight.data.normal_(0, 0.1)
        theirs = ref_slak.ReparamLargeKernelConv(**kw)
        theirs.load_state_dict(ours.state_dict())
        tag = f"merge_{K}_{small}."
        for k, v in theirs.state_dict().items():
            out[tag + "sd0." + k] = v.numpy().copy()
        k2, b2 = theirs.get_equivalent_kernel_bias()
        out[tag + "kernel"], out[tag + "bias"] = k2.detach().numpy(), b2.detach().numpy()
        theirs.merge_kernel()
        for k, v in theirs.state_dict().items():
            out[tag + "sd1." + k] = v.detach().numpy().copy()
    np.savez_compressed(os.path.join(OUT, "ref_dropin.npz"), **out)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    if len(sys.argv) > 1 and sys.argv[1] in ("host", "dropin"):   # python oracle/gen_golden.py host | dropin
        gen_ref_host() if sys.argv[1] == "host" else gen_dropin()
        sys.exit(0)
    ref_slak, ref_sparse, ref_funcs = import_reference()
    if len(sys.argv) > 1 and sys.argv[1] == "masking":      # python oracle/gen_golden.py masking [tag ...]
        gen_masking(ref_slak, ref_sparse, only=(sys.argv[2:] or None))
    else:
        gen_conv_grid()
        gen_block(ref_slak)
        gen_model(ref_slak)
        gen_masking(ref_slak, ref_sparse)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
