#!/usr/bin/env python
"""bench.py -- SLaK-T 51x51 224^2 bf16 training throughput (images/s) on N B200s, plus the
depthwise-kernel HBM roofline and the reference's CPU path timed on the same box.

  python bench.py [--gpus N --steps K --warmup W]            # this repo's CUDA path
  python bench.py --impl reference [...]                      # the reference's CPU (nn.Conv2d) path
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...   (N > 1)
  python bench.py [...] --dump-outputs DIR                    # also write what the last timed step computed

One JSON line on stdout (rank 0).  A "step" is one fwd+bwd+AdamW pass of the hot path over
one synthetic batch.  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch
import torch.nn.functional as F

NUM_CLASSES = 1000
# one metric string for BOTH arms (the driver refuses to form a ratio otherwise); `dtype` says what each arm computes in
METRIC = "SLaK-T 51x51 224x224 bf16 training images/sec"
# SURVEY.md section 8(d) "Config 1..5" (= BASELINE.json configs[0..4]); config 1 is the CPU plumbing case (tests/)
CONFIGS = {
    2: dict(model="SLaK_tiny", depths=[3, 3, 9, 3], dims=[96, 192, 384, 768], kernel_size=[51, 49, 47, 13, 5], img=224,
            batch=128, update_freq=1, sparse=False, metric=METRIC,
            what="SLaK-T 51x51 224x224 bf16 fwd+bwd+AdamW, batch 128/GPU (BASELINE.json configs[1])"),
    3: dict(model="SLaK_tiny", depths=[3, 3, 9, 3], dims=[96, 192, 384, 768], kernel_size=[51, 49, 47, 13, 5], img=224,
            batch=128, update_freq=4, sparse=False, metric="SLaK-T 51x51 224x224 bf16 DDP training images/sec (global batch 4096 at 8 GPUs)",
            what="SLaK-T 51x51 224x224 bf16 data-parallel training, 128/GPU x update_freq 4 (README.md:103-115; global "
                 "batch 4096 on 8 GPUs), one gradient all-reduce per optimizer step (BASELINE.json configs[2])"),
    4: dict(model="SLaK_base", depths=[3, 3, 27, 3], dims=[128, 256, 512, 1024], kernel_size=[51, 49, 47, 13, 5], img=384,
            batch=32, update_freq=1, sparse=False, metric="SLaK-B 51x51 384x384 bf16 training images/sec",
            what="SLaK-B 51x51 384x384 bf16 fwd+bwd+AdamW, batch 32/GPU (README.md:131; BASELINE.json configs[3])"),
    5: dict(model="SLaK_tiny", depths=[3, 3, 9, 3], dims=[96, 192, 384, 768], kernel_size=[61, 59, 57, 13, 5], img=224,
            batch=128, update_freq=1, sparse=True, metric="SLaK-T 61x61 224x224 bf16 sparse (prune-grow every 100 steps) training images/sec",
            what="SLaK-T 61x61 224x224 bf16, sparse_core.Masking(sparsity 0.4, snip init, magnitude prune, random growth, "
                 "prune_rate 0.3, update_frequency 100): mask.step() on the timed path (engine.py:79-88; BASELINE.json configs[4])"),
}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=50)
    p.add_argument("--warmup", type=int, default=20)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="SURVEY.md section 8(d) config number")
    p.add_argument("--batch", type=int, default=None, help="per-GPU batch (default: the config's)")
    p.add_argument("--width-factor", type=float, default=1.0)
    p.add_argument("--cpu-batch", type=int, default=0, help="images per CPU-arm step (0 = sized so the run takes ~2 min)")
    p.add_argument("--no-ref-ext", action="store_true", help="skip timing the reference CUTLASS ext (oracle/_ref/ext) on the GPU")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--torch-adamw", action="store_true", help="torch.optim.AdamW(fused=True) instead of slak_b200.optim.FusedAdamW")
    p.add_argument("--watchdog", type=float, default=1500.0, help="abort the process after this many seconds")
    p.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs)")
    a = p.parse_args()
    a.cfg = CONFIGS[a.config]
    if a.batch is None:
        a.batch = a.cfg["batch"]
    return a


# ---------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi fields through NVML), runs only during the timed region
# ---------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.stop_flag = [], set(), threading.Event()
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = None

    def _run(self):
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
        }
        while not self.stop_flag.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def start(self):
        if self.nv is not None:
            self.t = threading.Thread(target=self._run, daemon=True)
            self.t.start()

    def stop(self):
        self.stop_flag.set()
        if self.t is not None:
            self.t.join()
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


# ---------------------------------------------------------------------------------------
# the reference's CPU path (oracle restatement, fp32, nn.Conv2d semantics) -- checker / baseline only
# ---------------------------------------------------------------------------------------
def host_cores():
    """Threads the CPU arm may really use: the scheduler affinity, clipped by the cgroup CPU quota when the
    container has one (spinning 128 OpenMP threads on a smaller quota is what makes a CPU run crawl), or
    SLAK_CPU_THREADS when set."""
    if os.environ.get("SLAK_CPU_THREADS"):
        return max(1, int(os.environ["SLAK_CPU_THREADS"]))
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, min(n, 64))


def build_model(cfg, width_factor, drop_path_rate):
    from slak_b200 import slak
    return getattr(slak, cfg["model"])(kernel_size=cfg["kernel_size"], Decom=True, bn=True, drop_path_rate=drop_path_rate,
                                       width_factor=width_factor, num_classes=NUM_CLASSES)


def cpu_training_step_factory(cfg, width_factor, batch):
    """Returns (step_fn, cores): one fwd+bwd+AdamW step of the config's model on the host cores through the
    oracle's functional restatement of models/SLaK.py (F.conv2d depthwise, train-mode BN)."""
    from oracle import slak_model as omodel
    from slak_b200 import slak
    cores = host_cores()
    torch.set_num_threads(cores)     # explicit: torchrun exports OMP_NUM_THREADS=1 to its workers
    torch.manual_seed(0)
    slak.use_sync_bn = False
    net = build_model(cfg, width_factor, 0.0)
    sd = {}
    leaves = []
    for k, v in net.state_dict().items():
        t = v.detach().clone()
        if v.dtype.is_floating_point and "running_" not in k:
            t.requires_grad_(True)
            leaves.append(t)
        sd[k] = t
    opt = torch.optim.AdamW(leaves, lr=1e-3, weight_decay=0.05)
    x = torch.randn(batch, 3, cfg["img"], cfg["img"])
    y = torch.randint(0, NUM_CLASSES, (batch,))

    def step():
        out = omodel.forward(x, sd, cfg["depths"], training=True)
        loss = F.cross_entropy(out, y)
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
        return loss.item()

    return step, cores


def cpu_sample_batch(cfg, width_factor, total_steps, budget_s=110.0):
    """Images per CPU step such that `total_steps` steps take about `budget_s`: one probe step at batch 4 gives the
    host's images/s (the CPU arm is a BOUNDED SAMPLE of the workload, the per-step batch is reported)."""
    step, _ = cpu_training_step_factory(cfg, width_factor, 4)
    step()
    t0 = time.perf_counter()
    step()
    ips = 4.0 / (time.perf_counter() - t0)
    return max(2, min(32, int(budget_s * ips / max(total_steps, 1))))


def time_cpu(cfg, width_factor, batch, steps, warmup):
    step, cores = cpu_training_step_factory(cfg, width_factor, batch)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return batch * steps / dt, cores, dt / steps


def run_reference(args):
    """The reference's own CPU implementation of the path (nn.Conv2d semantics) on the box's host cores, through the
    oracle's restatement of models/SLaK.py (the reference's Python files cannot travel to the GPU box; the restatement
    is pinned by goldens generated from them, oracle/gen_golden.py).  Same metric / config / steps / warmup as the
    CUDA arm; every step is a bounded sample (a smaller batch) of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = args.cfg
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    batch = args.cpu_batch or cpu_sample_batch(cfg, args.width_factor, steps + warmup)
    ips, cores, sps = time_cpu(cfg, args.width_factor, batch, steps, warmup)
    sample = (f"{steps} timed + {warmup} warm-up steps x {batch} images (not {args.batch}: bounded sample) of the same "
              f"{cfg['model']} {cfg['img']}^2 fwd+bwd+AdamW step through oracle/slak_model.py (F.conv2d depthwise), fp32, {cores} threads")
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": ips, "unit": "images/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": sps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(args, args.gpus), cpu_images_per_step=batch),
        "cpu_baseline": {"value": ips, "unit": "images/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, n):
    cfg = args.cfg
    return {
        "workload": f"config {args.config}: {cfg['what']}; {cfg['model']} kernel_size={cfg['kernel_size']} Decom=True bn=True "
                    f"width_factor={args.width_factor}",
        "global_batch": args.batch * n * cfg["update_freq"], "per_gpu_batch": args.batch, "update_freq": cfg["update_freq"],
        "parallelism": f"dp{n}",
        "autocast": "bf16 (fp32 master weights, fp32 residual stream as in the reference's AMP flow)",
        "l2": "no explicit flush: one step streams >10 GB of activations, far above the 126 MB L2",
    }


# ---------------------------------------------------------------------------------------
# per-kernel roofline table from the CUDA events the fused Block records around its kernel groups
# ---------------------------------------------------------------------------------------
def roofline_table(tagged, peak_gbs, peak_tflops, replays):
    """tagged: [(tag, key, ev0, ev1)] recorded once per launch inside the step (graph: external events, re-read after
    each replay).  Returns one row per (kernel group, geometry) with the average duration, the ALGORITHMIC bytes or
    flops of the group and the fraction of the measured peak."""
    groups = {}
    for tag, key, e0, e1 in tagged:
        groups.setdefault((tag, key), []).append((e0, e1))
    rows = []
    for (tag, key), evs in groups.items():
        us = sum(a.elapsed_time(b) for a, b in evs) * 1e3 / len(evs)
        row = {"kernel": tag, "launches_per_step": len(evs), "avg_us": round(us, 2)}
        if tag.startswith("dw_"):
            N, C, H, W, KL = key
            e = N * C * H * W
            taps = C * (2 * KL * 5 + 25) * 4
            if tag == "dw_fwd":        # x read once, y1..y3 written once (bf16) + taps
                b, what = 4 * e * 2 + taps, "lk3_fwd_tc_kernel (+ statistics fold): 4 tensor passes bf16"
            elif tag == "dw_dgrad":    # dy1..dy3 bf16 in, shortcut gradient fp32 in, dx fp32 out
                b, what = e * (3 * 2 + 4 + 4) + taps, "lk_dgrad_tc_kernel x2: 3 bf16 reads + fp32 addend read + fp32 write"
            else:                      # x, dy1..dy3 bf16 in, dw out
                b, what = 4 * e * 2 + taps, "lk3_wgrad_tc_kernel (+ reduce): 4 tensor passes bf16"
            row.update(geometry=f"N{N} C{C} {H}x{W} K{KL}", bound="hbm", algorithmic_bytes=b,
                       achieved=round(b / (us * 1e-6) / 1e9, 1), unit="GB/s", frac=round(b / (us * 1e-6) / 1e9 / peak_gbs, 4),
                       what=what)
        elif tag.startswith("glue_"):  # fused elementwise / normalisation passes of the Block: HBM
            N, C, HW = key
            per = {"glue_ln_fwd": (8, "bn3_sum_ln_fwd: y1..y3 bf16 in, LayerNorm'd NHWC bf16 out"),
                   "glue_res_fwd": (12, "residual_fwd: x fp32 + h2 bf16 in, out fp32 (+ bf16 copy) out"),
                   "glue_res_bwd": (8, "residual_bwd: dout fp32 + h2 bf16 in, dh2 bf16 out"),
                   "glue_ln_bwd": (10, "bn3_sum_ln_bwd: dxn + y1..y3 bf16 in, du bf16 out"),
                   "glue_bwd_apply": (14, "bn3_bwd_apply: du + y1..y3 in, dy1..dy3 out (bf16)")}[tag]
            b = N * C * HW * per[0]
            row.update(geometry=f"N{N} C{C} HW{HW}", bound="hbm", algorithmic_bytes=b,
                       achieved=round(b / (us * 1e-6) / 1e9, 1), unit="GB/s", frac=round(b / (us * 1e-6) / 1e9 / peak_gbs, 4),
                       what=per[1])
        elif tag in ("down_ln_fwd", "down_out_fwd", "down_out_bwd", "down_ln_bwd"):   # downsampling layer, HBM passes
            N, C, HW = key
            per = {"down_ln_fwd": (6, "ln2d_patch_fwd: x fp32 in, LayerNorm'd patch rows bf16 out"),
                   "down_out_fwd": (8, "nhwc_to_nchw: GEMM output bf16 in, fp32 NCHW + bf16 copy out"),
                   "down_out_bwd": (6, "nchw_to_nhwc: dOut fp32 in, token-major bf16 out (+ bias gradient)"),
                   "down_ln_bwd": (10, "ln2d_patch_bwd: dA bf16 + x fp32 in, dx fp32 out")}[tag]
            b = N * C * HW * per[0]
            row.update(geometry=f"N{N} C{C} HW{HW}", bound="hbm", algorithmic_bytes=b,
                       achieved=round(b / (us * 1e-6) / 1e9, 1), unit="GB/s", frac=round(b / (us * 1e-6) / 1e9 / peak_gbs, 4),
                       what=per[1])
        elif tag in ("stem_patch", "stem_ln_fwd", "stem_ln_bwd"):   # stem, HBM passes
            N, C, HW = key
            if tag == "stem_patch":
                b, what = N * C * HW * 4 + N * (HW // 16) * 128, "patchify4: image fp32 in, 64-wide bf16 patch rows out"
            elif tag == "stem_ln_fwd":
                b, what = N * C * HW * 8, "ln_rows_fwd: GEMM output bf16 in, LayerNorm'd fp32 NCHW + bf16 copy out"
            else:
                b, what = N * C * HW * 8, "ln_rows_bwd: dOut fp32 + GEMM output bf16 in, dY bf16 out"
            row.update(geometry=f"N{N} C{C} HW{HW}", bound="hbm", algorithmic_bytes=b,
                       achieved=round(b / (us * 1e-6) / 1e9, 1), unit="GB/s", frac=round(b / (us * 1e-6) / 1e9 / peak_gbs, 4),
                       what=what)
        elif tag in ("stem_gemm_fwd", "stem_gemm_bwd"):             # K = 64: these are HBM passes over A and Y / dY
            M, Co, K = key
            b = M * (K + Co) * 2
            row.update(geometry=f"M{M} Co{Co} K{K}", bound="hbm", algorithmic_bytes=b,
                       achieved=round(b / (us * 1e-6) / 1e9, 1), unit="GB/s", frac=round(b / (us * 1e-6) / 1e9 / peak_gbs, 4),
                       what="stem conv as GEMM (K = 64)" if tag == "stem_gemm_fwd" else "its weight gradient (split-K over tokens)")
        elif tag in ("down_gemm_fwd", "down_gemm_bwd"):   # 2 x 2 stride-2 convolution as a GEMM over patch rows
            M, Co, K = key
            fl = (1 if tag == "down_gemm_fwd" else 2) * 2 * M * Co * K
            row.update(geometry=f"M{M} Co{Co} K{K}", bound="tensor", algorithmic_flops=fl,
                       achieved=round(fl / (us * 1e-6) / 1e12, 1), unit="TFLOP/s",
                       frac=round(fl / (us * 1e-6) / 1e12 / peak_tflops, 4),
                       what="downsampling conv as GEMM" if tag == "down_gemm_fwd" else "its data + weight gradient GEMMs")
        else:                          # pointwise MLP groups: tensor pipe
            M, Cc = key
            fl = {"mlp_fwd": 2, "mlp_bwd": 4}[tag] * 2 * M * Cc * 4 * Cc
            row.update(geometry=f"M{M} C{Cc} 4C{4 * Cc}", bound="tensor", algorithmic_flops=fl,
                       achieved=round(fl / (us * 1e-6) / 1e12, 1), unit="TFLOP/s",
                       frac=round(fl / (us * 1e-6) / 1e12 / peak_tflops, 4),
                       what="pwconv1+GELU+pwconv2 forward (2 GEMMs)" if tag == "mlp_fwd" else "their backward (4 GEMMs)")
        rows.append(row)
    rows.sort(key=lambda r: (r["kernel"], r["geometry"]))
    return rows


def ref_ext_leg(args):
    """North-star comparison target: the reference's own CUTLASS example-19 operator built for sm_100a
    (oracle/build_ref_ext.py -> oracle/_ref/ext) under stock PyTorch, timed on this GPU in a subprocess (its wrappers
    call exit() on any CUDA error).  Returns the dict tools/ref_ext_bench.py prints, or a reason string."""
    import subprocess
    so = os.path.join(ROOT, "oracle", "_ref", "ext", "_depthwise_conv2d_implicit_gemm_C.so")
    if not os.path.exists(so):
        return {"unavailable": "oracle/_ref/ext not built (python oracle/build_ref_ext.py)"}
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ref_ext_bench.py"), "--model-only",
                            "--config", str(args.config), "--batch", str(args.batch), "--steps", "3"],
                           capture_output=True, text=True, timeout=420)
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return {"unavailable": f"rc {r.returncode}: {(r.stderr or r.stdout)[-300:]}"}
    except Exception as ex:       # noqa: BLE001
        return {"unavailable": f"{type(ex).__name__}: {ex}"}


# ---------------------------------------------------------------------------------------
# outputs of the last timed step, for comparing two builds output for output
# ---------------------------------------------------------------------------------------
DUMP_SAMPLES = 4 << 20       # parameter / gradient elements kept: 2 x 16 MB of float32, whatever the model's size


def dump_outputs(path, loss, logits, params):
    """What a caller of the training step receives from its last timed step, as float32 .npy files:
    loss.npy (the loss), logits.npy (the model's output, every micro-step's batch in order), params.npy and grads.npy
    (the parameters after the optimizer update and the gradients it applied, over the concatenation of
    net.parameters() in order, at DUMP_SAMPLES positions drawn once from a fixed seed, ascending; all of them when
    the model has fewer).  The inputs and the initial weights come from fixed seeds, so two runs with the same
    arguments compute on the same data."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    sizes = [p.numel() for p in params]
    total = sum(sizes)
    if total <= DUMP_SAMPLES:
        idx = torch.arange(total)
    else:
        idx = torch.randperm(total, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLES].sort().values
    starts = torch.tensor([0] + sizes).cumsum(0)
    ps, gs = [], []
    for i, p in enumerate(params):
        lo, hi = torch.searchsorted(idx, starts[i : i + 2]).tolist()
        at = (idx[lo:hi] - starts[i]).to(p.device)
        ps.append(p.detach().flatten()[at].float())
        gs.append((p.grad.detach().flatten()[at] if p.grad is not None else torch.zeros(hi - lo, device=p.device)).float())
    arrays = {"loss": loss.detach().float().reshape(1), "logits": torch.cat([t.detach().float() for t in logits]),
              "params": torch.cat(ps), "grads": torch.cat(gs)}
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


# ---------------------------------------------------------------------------------------
# this repo's CUDA path
# ---------------------------------------------------------------------------------------
def run_ours(args):
    from slak_b200 import _lib, ddp, ops, slak
    cfg = args.cfg
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if not _lib.load().slak_device_ok():
        raise SystemExit("libslak_b200.so: no sm_100 device visible")
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    torch.backends.cudnn.benchmark = True
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True

    torch.manual_seed(0 + rank)    # main.py:232 seeds seed + rank
    slak.use_sync_bn = world > 1
    net = build_model(cfg, args.width_factor, 0.1).to(dev)
    net.train()
    params = [p for p in net.parameters()]
    UF = cfg["update_freq"]
    # data parallelism = gradient all-reduce only (main.py:374-376): flat gradient buffer, buckets all-reduced on a side
    # stream as backward produces them (slak_b200/ddp.py); identical initial weights by broadcast
    # bucket size: measured on this step (profiles/r02_bucket_sweep.txt) -- the step is bound by the SMs and HBM, and NCCL kernels
    # that overlap backward take both away from it: at N = 2 one 123 MB all-reduce after backward (16.37 ms) beats 25 MB
    # buckets overlapped with it (16.64 ms); at N = 8 the two are equal (17.18 ms).  200 MB = one bucket for SLaK-T / S.
    dp = ddp.GradientAllReducer(net, bucket_mb=float(os.environ.get("SLAK_BUCKET_MB", "200"))) if world > 1 else None
    # gradients live in one flat buffer (static addresses for the graph and for the fused optimizer's pointer tables)
    flat = dp if dp is not None else ddp.FlatGradients(net)
    if args.torch_adamw:
        opt = torch.optim.AdamW(params, lr=1e-3, weight_decay=0.05, fused=True, capturable=True)
    else:
        # this library's multi-tensor AdamW (+ mask apply when sparse): one launch, device-side step counter
        from slak_b200.optim import FusedAdamW
        decay = [p for p in params if p.dim() > 1]
        no_decay = [p for p in params if p.dim() <= 1]       # optim_factory.py:73-112: no weight decay on 1-d tensors
        opt = FusedAdamW([{"params": decay, "weight_decay": 0.05}, {"params": no_decay, "weight_decay": 0.0}], lr=1e-3)

    B = args.batch
    IMG = cfg["img"]
    x_host = torch.randn(UF * B, 3, IMG, IMG).pin_memory()
    y_host = torch.randint(0, NUM_CLASSES, (UF * B,)).pin_memory()
    x_dev = x_host.to(dev)             # static input buffers (also the CUDA-graph inputs)
    y_dev = y_host.to(dev)

    mask = None
    if cfg["sparse"]:
        import types
        from slak_b200.sparse_core import CosineDecay, Masking
        margs = types.SimpleNamespace(device=str(dev), fix=False, update_frequency=100, only_L=False, sparse_init="snip",
                                      sparsity=0.4, distributed=world > 1)
        nb = min(B, 32)
        loader = [(x_host[:nb], y_host[:nb])]      # SNIP takes one batch (sparse_core.py:11-47)
        torch.manual_seed(0)                       # same CPU RNG stream on every rank; rank 0's masks win anyway
        mask = Masking(opt, train_loader=loader, prune_rate_decay=CosineDecay(0.3, 100000), prune_rate=0.3,
                       prune_mode="magnitude", growth_mode="random", redistribution_mode="none", args=margs)
        margs.distributed = False                  # SNIP's `sampler.set_epoch` is for a real DistributedSampler
        mask.add_module(net)
        margs.distributed = world > 1
        if not args.torch_adamw:
            opt.attach_masking(mask)                   # p *= mask inside the optimizer launch

    logits = []         # the model's outputs of the latest step (in a captured graph: its static output buffers)

    def step_eager():
        # optimizer.zero_grad() as in engine.py:74-86: under graph capture the gradients live in the graph's private pool
        flat.zero_grad()
        logits.clear()
        for k in range(UF):                              # engine.py:52-80: loss /= update_freq, backward every micro-step
            with torch.autocast("cuda", dtype=torch.bfloat16):
                out = net(x_dev[k * B:(k + 1) * B])
                logits.append(out)
                loss = F.cross_entropy(out.float(), y_dev[k * B:(k + 1) * B])
                if UF > 1:
                    loss = loss / UF
            flat.arm(last_micro_step=(k == UF - 1))
            loss.backward()
        flat.finish()                                    # gradients gathered into the flat buffer (and all-reduced at N > 1)
        opt.step()
        if mask is not None and not getattr(opt, "fused_mask", False):
            mask.apply_mask()                            # Masking.step() = optimizer.step(); apply_mask(); advance()
        return loss

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (side stream, as CUDA-graph capture requires), then capture the whole step -------------
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(max(args.warmup, 3)):
            step_eager()
    torch.cuda.current_stream().wait_stream(side)
    barrier()

    graph, static_loss, static_logits, graph_note = None, None, None, "eager (no CUDA graph)"
    tagged = []
    use_graph = not args.no_graph
    launches_per_step = None
    prof_graph = None
    if use_graph:
        try:
            l_before = ops.launch_count()
            graph = torch.cuda.CUDAGraph()
            # thread_local: the NCCL watchdog thread's event queries must not invalidate this thread's capture
            with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                static_loss = step_eager()
            static_logits = list(logits)
            launches_per_step = ops.launch_count() - l_before
            # the same step once more WITH CUDA events around every kernel group: replayed only outside the timed
            # regions, for the per-kernel roofline table (the ~100 event nodes cost ~0.5 ms per replay)
            ops.profile_reset(dict(all=True, external_events=True))
            prof_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(prof_graph, capture_error_mode="thread_local"):
                step_eager()
            tagged = list(ops._prof["tagged"])
            ops.profile_reset(None)
            graph_note = "whole step (fwd+bwd+bucketed grad all-reduce+AdamW) captured in one CUDA graph and replayed"
        except Exception as ex:      # capture not possible on this software stack: fall back to eager launches
            graph, static_loss = None, None
            ops.profile_reset(None)
            torch.cuda.synchronize()
            graph_note = f"eager (CUDA graph capture failed: {type(ex).__name__})"
            print(f"[bench] rank {rank}: graph capture failed: {ex!r}", file=sys.stderr, flush=True)
        if world > 1:                # every rank must replay, or none: the captured collectives have to pair up
            ok = torch.tensor([1 if graph is not None else 0], device=dev, dtype=torch.int32)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0 and graph is not None:
                graph, static_loss = None, None
                graph_note = "eager (CUDA graph capture failed on another rank)"

    def run_step():
        if graph is not None:
            graph.replay()
            out = static_loss
            logits[:] = static_logits
        else:
            out = step_eager()
        if mask is not None:
            mask.advance()           # prune-rate schedule; every 100 steps: prune + grow (eager launches, CPU RNG)
        return out

    for _ in range(3):
        run_step()
    barrier()

    # ---- timed region 1: inputs resident in HBM ------------------------------------------
    sampler = ClockSampler(local_rank)
    launches0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    barrier()
    e0.record()
    for _ in range(args.steps):
        last_loss = run_step()
    e1.record()
    barrier()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:     # before the replays below move the weights on
        dump_outputs(args.dump_outputs, last_loss, logits, params)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)
    peak_tf = peaks.get("bf16_tflops_sustained", 1450.0)
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs / bf16_tflops_sustained)" if "hbm_gbs" in peaks else \
        "fallback 6650 GB/s, 1450 TFLOP/s (B200_PROFILING.md)"
    if graph is None:
        launches = ops.launch_count() - launches0
        ops.profile_reset(dict(all=True))
        for _ in range(2):
            step_eager()
        torch.cuda.synchronize()
        table = roofline_table(ops._prof["tagged"], peak, peak_tf, 2)
        ops.profile_reset(None)
        prof_how = "CUDA events around each kernel group in 2 eager steps right after the timed region"
    else:
        launches = launches_per_step * args.steps + (ops.launch_count() - launches0)
        # the events sit inside the captured graph: read them after the last timed replay and after 3 further replays
        acc = []
        for rep in range(5):
            prof_graph.replay()
            torch.cuda.synchronize()
            if rep:                               # the first replay warms the caches of the instrumented graph
                acc.append(roofline_table(tagged, peak, peak_tf, 1))
        table = acc[0]
        for r_i, row in enumerate(table):
            us = sum(a[r_i]["avg_us"] for a in acc) / len(acc)
            scale = row["avg_us"] / us if us > 0 else 1.0
            row["avg_us"] = round(us, 2)
            row["achieved"] = round(row["achieved"] * scale, 1)
            row["frac"] = round(row["frac"] * scale, 4)
        prof_how = ("CUDA events (external) recorded around each kernel group INSIDE a second capture of the same step "
                    "graph, replayed 4 times right after the timed region (the timed graph carries no events)")

    # ---- timed region 2: end to end through the public API with host buffers --------------
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # The way a training loop with a prefetching loader runs: batch k+1 travels pinned host -> device (staging buffer) on a
    # copy stream while step k computes, and step k's loss is read back (pinned host buffer) while step k+1 runs.  Every
    # step's inputs still cross from host memory and every step's result is read on the host inside the timed region.
    copy_stream = torch.cuda.Stream()
    x_stage, y_stage = torch.empty_like(x_dev), torch.empty_like(y_dev)
    loss_pinned = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
    ev_ready, ev_taken = torch.cuda.Event(), torch.cuda.Event()
    ev_loss = [torch.cuda.Event(), torch.cuda.Event()]
    cur = torch.cuda.current_stream()
    losses_read = 0
    f0.record()
    ev_taken.record()
    with torch.cuda.stream(copy_stream):
        copy_stream.wait_event(ev_taken)
        x_stage.copy_(x_host, non_blocking=True)     # pinned host -> device, every step
        y_stage.copy_(y_host, non_blocking=True)
        ev_ready.record()
    for k in range(args.steps):
        cur.wait_event(ev_ready)
        x_dev.copy_(x_stage, non_blocking=True)      # device -> the step's static input buffers
        y_dev.copy_(y_stage, non_blocking=True)
        ev_taken.record()
        if k + 1 < args.steps:
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ev_taken)
                x_stage.copy_(x_host, non_blocking=True)
                y_stage.copy_(y_host, non_blocking=True)
                ev_ready.record()
        loss = run_step()
        loss_pinned[k & 1].copy_(loss.detach().float(), non_blocking=True)   # device -> host read of the step's result
        ev_loss[k & 1].record()
        if k > 0:                                    # the previous step's loss, on the host, while this step runs
            ev_loss[(k - 1) & 1].synchronize()
            loss_host = float(loss_pinned[(k - 1) & 1])
            losses_read += 1
    ev_loss[(args.steps - 1) & 1].synchronize()
    loss_host = float(loss_pinned[(args.steps - 1) & 1])
    losses_read += 1
    assert losses_read == args.steps and loss_host == loss_host
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)

    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()
    total_images = UF * B * world * args.steps
    value = total_images / (ms / 1e3)
    e2e = total_images / (ms_e2e / 1e3)

    if rank == 0:
        step_ms = ms / args.steps
        for row in table:
            row["share_of_step"] = round(row["avg_us"] * 1e-3 * row["launches_per_step"] / step_ms, 4)
        head = next((r for r in table if r["kernel"] == "dw_fwd" and " 56x56 " in r["geometry"] + " "), None) or \
            next((r for r in table if r["kernel"] == "dw_fwd"), None)
        roof = {"bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": None,
                "kernel": "lk3_fwd_tc_kernel (stage-1 fused K x 5 + 5 x K + 5 x 5 depthwise forward, tcgen05) + its "
                          "statistics fold, the dominant-shape depthwise kernel of the step",
                "peak_source": peak_src, "timing": prof_how}
        if head is not None:
            roof.update(achieved=head["achieved"], frac=head["frac"], avg_us=head["avg_us"], geometry=head["geometry"],
                        algorithmic_bytes_per_launch=head["algorithmic_bytes"], launches_timed=head["launches_per_step"],
                        share_of_step=head["share_of_step"])
        try:    # DRAM bytes of one launch of this kernel from the committed `ncu --set full` capture (not measured live)
            tr = json.load(open(os.path.join(ROOT, "profiles", "headline_traffic.json")))
            if args.config == 2 and B == 128:
                roof["traffic"] = tr["dram_bytes"]
                roof["traffic_source"] = f"{tr['source']} (dram__bytes_read.sum + dram__bytes_write.sum, one launch)"
        except Exception:
            pass
        line = {
            "metric": cfg["metric"], "value": value, "unit": "images/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": dict(workload_config(args, world), launch=graph_note),
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": "images/s",
                    "h2d_bytes_per_step": x_host.numel() * 4 + y_host.numel() * 8, "d2h_bytes_per_step": 4,
                    "how": "through the model's public forward / FlatGradients / FusedAdamW API; batch k+1 is copied pinned host -> "
                           "device on a copy stream while step k computes, the loss of step k is read on the host while step k+1 runs"},
            "gpu_launches": launches,
            "roofline": roof,
            "roofline_all": table,
        }
        if mask is not None:
            line["config"]["masking"] = {"steps": mask.steps, "prune_grow_events_total": mask.steps // 100,
                                         "masked_tensors": len(mask.masks)}
        if world == 1 and not args.no_cpu_baseline:
            cb = args.cpu_batch or cpu_sample_batch(cfg, args.width_factor, 4, budget_s=20.0)
            ips, cores, _ = time_cpu(cfg, args.width_factor, cb, 3, 1)
            line["cpu_baseline"] = {
                "value": ips, "unit": "images/s", "cores": cores, "kind": "port",
                "sample": f"3 steps x {cb} images of the same {cfg['model']} {IMG}^2 fwd+bwd+AdamW step through "
                          f"oracle/slak_model.py (F.conv2d depthwise, fp32), {cores} threads"}
    if world == 1 and rank == 0 and not args.no_ref_ext:
        # free this process's GPU memory first: the reference model needs most of the card at batch 128
        del graph, static_loss, prof_graph
        opt = net = x_dev = y_dev = None
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        line["reference_cutlass_ext"] = ref_ext_leg(args)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist is not None:
        # tear down without ncclCommDestroy: with the step graph (which holds the captured all-reduces) alive the
        # communicator teardown blocks forever; the process exits right after, which frees everything
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    a = parse()
    # a run that cannot finish (a wedged collective, a dead peer rank) must not hold the GPU box forever
    _wd = threading.Timer(a.watchdog, lambda: (sys.stderr.write("[bench] watchdog: no result in time, aborting\n"), os._exit(3)))
    _wd.daemon = True
    _wd.start()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
