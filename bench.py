#!/usr/bin/env python
"""Benchmark of the hot path: med3ddram (ResNet-34) + dRAM inference on synthetic 256^3 CT volumes.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--size 256] [--impl ours|reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One step = one pass of the device-resident hot path (SURVEY §8d) over one batch of B volumes per GPU:
K8 HU window statistics -> stem (window + standardise fused into its producers) -> 37 more tcgen05 conv launches
(BN/ReLU/residual/heads fused) -> max-pool / x2 up-sampling -> dRAM (trilinear to CT size x ess mask) + lesion %.
Prints ONE JSON line (rank 0).  `value` = volumes/s with the int16 HU volumes and masks already in HBM;
`e2e` = the same through ScanRegLightningModule.predict_step with pinned HOST buffers: fp32 image + bool masks copied
host->device every step, and what the product ships copied back every step — both uint8 heat-maps of every volume
(processor.py:111-158, K f2) and the lesion percentages; `e2e_product` = the same loop fed what processor.py really
sends (int16 HU + uint8 lobe labels, 3 B/voxel; the lung / LAA-910 masks are made on the device by f1).
Multi-GPU: volumes are sharded across ranks, no data-path collective (weak scaling); time = max over ranks.

`--impl reference` times the reference's algorithm on the host cores (the oracle port of the reference's
PyTorch CPU path; /root/reference itself does not exist on the GPU box) on the same config.
`--impl cudnn` is the GPU yard-stick of SURVEY §8d: the same oracle (= the reference's ATen call sequence) on the
B200 under this image's torch/cuDNN, fp32 with TF32 convolutions (`value`) and bf16 channels_last_3d (extra field).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from argparse import Namespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ARCH = "med3ddram"
ARCH_NAMES = {"med3ddram": "med3ddram (ResNet-34)", "med3ddram18": "med3ddram18 (ResNet-18)",
              "med3ddram50": "med3ddram50 (ResNet-50 bottleneck)"}
METRIC = "CT volumes/sec med3ddram inference"


def workload_name(arch, dims, batch):
    size = f"{dims[0]}^3" if dims[0] == dims[1] == dims[2] else "x".join(str(v) for v in dims)
    return (f"{ARCH_NAMES[arch]} + dRAM inference, synthetic {size} CT volumes, batch {batch} per GPU, "
            "random-init weights (paper.ckpt is a Git-LFS pointer)")


def parse_dims(args):
    if args.dims:
        d = tuple(int(v) for v in args.dims.replace("x", ",").split(","))
        if len(d) != 3:
            raise SystemExit("--dims expects D,H,W")
        return d
    return (args.size,) * 3
FALLBACK_TFLOPS = 1590.0  # B200_PROFILING.md fallback (burst); used only when MEASURED_PEAKS.json is absent


# --------------------------------------------------------------------------------------------
# synthetic inputs (SURVEY §8d) generated on the device, and bounded random weights
# --------------------------------------------------------------------------------------------
def make_volumes(batch, dims, device, seed):
    """int16 HU [B,D,H,W], lung uint8, ess uint8: two ellipsoid lungs, emphysema-like low-HU blobs."""
    D, H, W = dims
    g = torch.Generator(device=device).manual_seed(20261018 + seed)
    z = ((torch.arange(D, device=device, dtype=torch.float32) + 0.5) / D)[:, None, None]
    y = ((torch.arange(H, device=device, dtype=torch.float32) + 0.5) / H)[None, :, None]
    x = ((torch.arange(W, device=device, dtype=torch.float32) + 0.5) / W)[None, None, :]
    lung = torch.zeros((D, H, W), dtype=torch.bool, device=device)
    for cx in (0.30, 0.70):
        lung |= ((z - 0.5) / 0.42) ** 2 + ((y - 0.5) / 0.36) ** 2 + ((x - cx) / 0.19) ** 2 <= 1.0
    hu, lungs, ess = [], [], []
    for _ in range(batch):
        ct = torch.randn((D, H, W), generator=g, device=device) * 150.0 + 20.0
        ct = torch.where(lung, torch.randn((D, H, W), generator=g, device=device) * 120.0 - 850.0, ct)
        coarse = torch.rand((1, 1, D // 8, H // 8, W // 8), generator=g, device=device)
        field = torch.nn.functional.interpolate(coarse, size=(D, H, W), mode="trilinear", align_corners=True)[0, 0]
        blob = lung & (field > 0.78)
        ct = torch.where(blob, torch.randn((D, H, W), generator=g, device=device) * 25.0 - 960.0, ct)
        ct = ct.round().clamp(-1024, 1500).to(torch.int16)
        hu.append(ct)
        lungs.append(lung.to(torch.uint8))
        ess.append(((ct < -910) & lung).to(torch.uint8))
    return torch.stack(hu), torch.stack(lungs), torch.stack(ess)


def tame_weights_(model, seed=0):
    """Random-init weights (no checkpoint can be downloaded; paper.ckpt is a Git-LFS pointer) with
    BatchNorm statistics chosen so that activations stay O(1): running_var = fan_in/fan_out of the
    preceding kaiming(fan_out) convolution, small gain on the last BN of each residual block."""
    g = torch.Generator().manual_seed(seed)
    convs = {}
    last = None
    for name, m in model.named_modules():
        if isinstance(m, torch.nn.Conv3d):
            last = m
        elif isinstance(m, torch.nn.BatchNorm3d) and last is not None:
            convs[name] = last
    with torch.no_grad():
        for name, m in model.named_modules():
            if isinstance(m, torch.nn.BatchNorm3d):
                conv = convs[name]
                k = conv.kernel_size[0] * conv.kernel_size[1] * conv.kernel_size[2]
                fan_in, fan_out = conv.in_channels * k, conv.out_channels * k
                m.running_var.fill_(max(fan_in / fan_out, 0.05))
                m.running_mean.zero_()
                m.weight.copy_(torch.rand(m.weight.shape, generator=g) * 0.5 + 0.5)
                m.bias.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
                if name.endswith("bn2") and "layer" in name:
                    m.weight.mul_(0.3)
        for fc in model.fcs:
            fc.weight.mul_(0.2)
            fc.bias.fill_(-2.0)
    return model


def build_module(device, arch=ARCH):
    import dram_b200  # noqa: F401
    from dram_b200.models import ScanRegLightningModule

    torch.manual_seed(0)
    module = ScanRegLightningModule(Namespace(model_arch=arch))
    tame_weights_(module.model)
    return module.to(device).eval()


# --------------------------------------------------------------------------------------------
# helpers
# --------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index, self.proc, self.path = gpu_index, None, None

    def start(self):
        import tempfile

        try:
            fd, self.path = tempfile.mkstemp(prefix="dram_clocks_", suffix=".csv")
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=fd, stderr=subprocess.DEVNULL)
            os.close(fd)
        except OSError:
            self.proc = None

    def mark(self):
        """Number of samples taken so far (samples before the mark belong to the warm-up)."""
        try:
            with open(self.path) as f:
                return sum(1 for _ in f)
        except (OSError, TypeError):
            return 0

    def stop(self, skip=0):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        with open(self.path) as f:
            lines = f.read().strip().splitlines()
        os.remove(self.path)
        out = "\n".join(lines[skip:] if len(lines) > skip else lines)
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        busy = [v for v in sm if v > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks(burst=False):
    """Dense 16-bit tensor peak: the sustained figure (a kernel timed inside a long step) or the burst one."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        if burst:
            return float(p.get("bf16_tflops", FALLBACK_TFLOPS)), "measured (MEASURED_PEAKS.json bf16_tflops)"
        return float(p.get("bf16_tflops_sustained", p.get("bf16_tflops"))), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    return FALLBACK_TFLOPS, "fallback (B200_PROFILING.md)"


def measured_tensor_pipe(arch, dims, batch=1):
    """Tensor-pipe utilisation per convolution family from the committed single-pass ncu capture
    (profiles/tensor_pipe.json, written by tools/summarize_tensor_pipe.py); None when no capture matches."""
    path = os.path.join(ROOT, "profiles", "tensor_pipe.json")
    if not os.path.isfile(path):
        return None
    with open(path) as f:
        t = json.load(f)
    key = f"{arch}:{'x'.join(str(v) for v in dims)}"
    return t.get(f"{key}:b{batch}", t.get(key))  # a capture at this batch size if there is one, else the batch-1 capture


def measured_traffic(arch, dims, batch):
    """DRAM bytes (read + write) of the conv launches of one step, from the committed ncu --set full capture
    (profiles/conv_traffic.json, measured per volume at batch 1); None when no capture matches the workload."""
    path = os.path.join(ROOT, "profiles", "conv_traffic.json")
    if not os.path.isfile(path):
        return None, None
    with open(path) as f:
        t = json.load(f)
    key = f"{arch}:{'x'.join(str(v) for v in dims)}"
    if key not in t:
        return None, None
    return t[key]["dram_bytes_per_volume"] * batch, t[key]["source"]


def dist_setup(n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, local, world


def barrier(world):
    if world > 1:
        import torch.distributed as dist

        dist.barrier()


def max_over_ranks(value, world, device):
    if world <= 1:
        return value
    import torch.distributed as dist

    t = torch.tensor([value], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this much in all


def dump_outputs(out_dir, arrays, seed=0):
    """Writes every tensor of `arrays` as <out_dir>/<name>.npy, float64 kept, anything else as float32, so that two
    builds can be compared output for output.  Each array gets an equal share of DUMP_BYTES; one larger than its share
    is written as a fixed sample, 1-D: its values at the flat indices
    np.unique(np.random.default_rng(seed).integers(0, numel, share // itemsize)), which depend only on numel."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 128  # less the .npy header
    for name, t in arrays.items():
        dtype = torch.float64 if t.dtype == torch.float64 else torch.float32
        itemsize = 8 if dtype == torch.float64 else 4
        t = t.detach()
        if t.numel() * itemsize > share:
            idx = np.unique(np.random.default_rng(seed).integers(0, t.numel(), share // itemsize))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.to(dtype).cpu().numpy())


# --------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference's PyTorch path on the host cores
# --------------------------------------------------------------------------------------------
def cpu_predict_seconds(sd, dims, batch=1, repeats=1, warmup=0, arch=ARCH):
    """Median seconds of one oracle predict_step (transform-equivalent standardise + network + dRAM)."""
    from oracle import pipeline_oracle as P
    from oracle import synthetic

    torch.set_num_threads(os.cpu_count() or 1)
    xs, ls, es = zip(*[synthetic.make_network_input(i, dims) for i in range(batch)])
    b = {"image": torch.stack(xs), "lung_mask": torch.stack(ls).bool(), "ess_mask": torch.stack(es).bool()}
    times = []
    with torch.no_grad():
        for i in range(warmup + repeats):
            t0 = time.perf_counter()
            P.predict_step(sd, arch, b)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    return statistics.median(times)


def cpu_state_dict(module):
    return {k: v.detach().float().cpu() if v.is_floating_point() else v.detach().cpu()
            for k, v in module.model.state_dict().items()}


def _voxels(dims):
    return dims[0] * dims[1] * dims[2]


def cpu_baseline(module, dims, arch=ARCH, budget_s=30.0):
    """Bounded sample: a sub-volume of at most 128 per axis first; the full volume only if it fits the budget."""
    sd = cpu_state_dict(module)
    small = tuple(min(v, 128) for v in dims)
    t_small = cpu_predict_seconds(sd, small, arch=arch)
    scale = _voxels(dims) / _voxels(small)
    if small == tuple(dims) or t_small * scale > budget_s:
        t = t_small * scale
        sample = (f"1 volume of {'x'.join(map(str, small))} timed ({t_small:.2f} s), scaled x{scale:.1f} by voxel "
                  f"count to {'x'.join(map(str, dims))}")
    else:
        t = cpu_predict_seconds(sd, tuple(dims), arch=arch)
        sample = f"1 full {'x'.join(map(str, dims))} volume, one pass ({t:.2f} s)"
    return {"value": 1.0 / t, "unit": "volumes/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample}


# --------------------------------------------------------------------------------------------
# GPU yard-stick: the reference's ATen call sequence (the oracle) under torch/cuDNN on the same B200
# --------------------------------------------------------------------------------------------
def cudnn_yardstick(module, dims, arch, batch, device, steps=5, warmup=2):
    """SURVEY §8d: "the unmodified reference module under torch 2.11/cuDNN on the same B200, fp32-TF32 and bf16".
    /root/reference does not exist on the GPU box, so the oracle — a functional restatement that issues the very
    ATen ops of med3d.py / models.py:430-450 — stands in for the module.  Bench-only: the product never imports it.
    Returns volumes/s for (a) fp32 tensors with TF32 convolutions (cuDNN's default since Ampere), NCDHW as the
    reference allocates them, and (b) bf16 tensors in channels_last_3d."""
    from oracle import pipeline_oracle as P
    from oracle import synthetic

    torch.backends.cudnn.benchmark = True
    sd32 = {k: v.to(device) for k, v in cpu_state_dict(module).items()}
    xs, ls, es = zip(*[synthetic.make_network_input(i, dims) for i in range(batch)])
    base = {"image": torch.stack(xs).to(device), "lung_mask": torch.stack(ls).bool().to(device),
            "ess_mask": torch.stack(es).bool().to(device)}

    def run(sd, b, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.no_grad():
            for _ in range(warmup):
                P.predict_step(sd, arch, b)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(n):
                out = P.predict_step(sd, arch, b)
            e1.record()
            torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n, out

    res = {"unit": "volumes/s", "batch": batch, "torch": torch.__version__, "cudnn": torch.backends.cudnn.version(),
           "what": "oracle.pipeline_oracle.predict_step (the reference's ATen ops: conv3d/batch_norm/relu/max_pool3d/"
                   "interpolate/cat/sigmoid) on cuda:0, cudnn.benchmark=True, inputs resident, standardised fp32 image in"}
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    ms, out32 = run(sd32, base, steps)
    res["fp32_tf32"] = {"value": batch / (ms * 1e-3), "ms_per_step": ms}
    try:
        sd16 = {k: (v.to(torch.bfloat16).contiguous(memory_format=torch.channels_last_3d) if v.dim() == 5 else
                    (v.to(torch.bfloat16) if v.is_floating_point() else v)) for k, v in sd32.items()}
        b16 = dict(base, image=base["image"].to(torch.bfloat16))
        # (the 1-channel input is channels-last by construction; every 5-D weight is, so cuDNN runs NDHWC kernels)
        ms16, out16 = run(sd16, b16, steps)
        err = (out16["cle_dense_outs"].float() - out32["cle_dense_outs"]).abs().max().item()
        res["bf16_channels_last_3d"] = {"value": batch / (ms16 * 1e-3), "ms_per_step": ms16,
                                        "dram_max_abs_vs_fp32": err}
    except Exception as exc:
        res["bf16_channels_last_3d"] = {"error": f"{type(exc).__name__}: {exc}"[:200]}
    return res


def run_cudnn_arm(args, out):
    """`--impl cudnn`: one JSON line, value = fp32/TF32 volumes/s of the yard-stick (rank 0 only)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(device)
    dims = parse_dims(args)
    module = build_module(device, args.arch)
    y = cudnn_yardstick(module, dims, args.arch, args.batch, device, steps=args.steps, warmup=max(1, args.warmup))
    line = {"impl": "cudnn", "metric": METRIC, "value": y["fp32_tf32"]["value"], "unit": "volumes/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": y["fp32_tf32"]["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (TF32 convolutions)",
            "data": "synthetic", "config": {"workload": workload_name(args.arch, dims, args.batch)}, "gpu_yardstick": y}
    out.emit(json.dumps(line))


def run_reference_arm(args, out):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import dram_b200  # noqa: F401
    from dram_b200.models import ScanRegLightningModule

    torch.manual_seed(0)
    arch, dims = args.arch, parse_dims(args)
    module = ScanRegLightningModule(Namespace(model_arch=arch))
    tame_weights_(module.model)
    sd = cpu_state_dict(module)
    # each step = one bounded sample: a full volume if (steps+warmup) of them fit ~4 minutes, else a sub-volume
    small = tuple(min(v, 128) for v in dims)
    probe = cpu_predict_seconds(sd, small, arch=arch)
    scale = _voxels(dims) / _voxels(small)
    full = probe * scale * (args.steps + args.warmup) <= 240.0
    run_dims = tuple(dims) if full else small
    vol_frac = 1.0 if full else 1.0 / scale
    t = cpu_predict_seconds(sd, run_dims, repeats=args.steps, warmup=args.warmup, arch=arch)
    value = vol_frac / t
    sample = (f"{args.steps} steps x 1 volume of {'x'.join(map(str, run_dims))}" +
              ("" if full else f" (= 1/{scale:.1f} of a full volume by voxel count)"))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "volumes/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(arch, dims, args.batch),
                   "arm": "the reference's algorithm (oracle port of its PyTorch CPU path) on the host cores, "
                          "one volume per step"},
        "cpu_baseline": {"value": value, "unit": "volumes/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "volumes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    out.emit(json.dumps(line))


# --------------------------------------------------------------------------------------------
# main arm
# --------------------------------------------------------------------------------------------
class _StdoutToStderr:
    """Everything libraries print to fd 1 while the benchmark runs (NCCL's version banner, ...) goes to
    stderr; `emit()` writes the one JSON line to the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, text):
        sys.stdout.flush()
        os.write(self.real, (text + "\n").encode())


def run_train_arm(args, out):
    """BASELINE config 5: med3ddram training, forward + loss + backward + gradient all-reduce + Adam, bf16 activations,
    one process per GPU (NCCL), per-GPU batch `--batch` (default 1 here).  Convolutions (fwd/dgrad/wgrad), train-mode
    BatchNorm(+ReLU, +residual, SyncBN exchange), max-pool, up-sampling, heads, weight re-packing, the loss with its
    gradient (K11) and Adam (K12) run on the hand-written kernels; what is left on ATen is named in `config.glue` (see
    DESIGN.md section 3, training step).  `value` = volumes/s with the batch resident in HBM, `e2e` copies the batch
    from pinned host memory every step and reads the loss back."""
    import dram_b200  # noqa: F401
    from dram_b200 import med3d, training

    rank, local, world = dist_setup(args.gpus)
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    dims = parse_dims(args)
    B = args.batch if args.batch != 4 else 1  # the inference default (4) is not a training batch: C5 is per-GPU batch 1
    torch.manual_seed(0)  # identical initial weights on every rank
    factory = {"med3ddram": med3d.resnet34segreg, "med3ddram18": med3d.resnet18segreg, "med3ddram50": med3d.resnet50segreg}
    model = factory[args.arch]().to(device).train()
    step = training.TrainStep(model, lr=1e-5, sync_bn=args.sync_bn if world > 1 else False)
    hu, lungs, ess = make_volumes(B, dims, device, seed=rank)
    v = hu.float().clamp(-1150.0, -300.0)
    v = (v + 1150.0) / 850.0
    image = (v - v.mean(dim=(1, 2, 3), keepdim=True)) / v.std(dim=(1, 2, 3), keepdim=True)
    batch = {"image": image.contiguous(), "lung_mask": lungs.bool(), "em_mask": ess.bool(),
             "cls_label": torch.full((B,), 2, device=device), "pse_label": torch.full((B,), 1, device=device)}
    bands = (torch.tensor([[0.05, 0.1]] * B, device=device), torch.tensor([[0.01, 0.05]] * B, device=device))
    w = torch.ones(B, device=device)

    def one(b):
        return step.step(b, bands[0], bands[1], w, w)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        one(batch)
    torch.cuda.synchronize()
    barrier(world)
    torch.cuda.synchronize()
    first_sample = sampler.mark() if rank == 0 else 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = one(batch)
    e1.record()
    torch.cuda.synchronize()
    barrier(world)
    ms_per_step = max_over_ranks(e0.elapsed_time(e1), world, device) / args.steps
    clocks = sampler.stop(skip=first_sample) if rank == 0 else None

    host = {k: t.cpu().pin_memory() for k, t in batch.items()}
    h2d = sum(t.numel() * t.element_size() for t in host.values())
    loss_host = torch.empty(1, dtype=torch.float32).pin_memory()
    barrier(world)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        dev_batch = {k: t.to(device, non_blocking=True) for k, t in host.items()}
        loss_host.copy_(one(dev_batch).reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()
    t1.record()
    torch.cuda.synchronize()
    barrier(world)
    e2e_ms = max_over_ranks(t0.elapsed_time(t1), world, device) / args.steps

    # one more step under the profiler (all ranks: the step holds collectives) to count this library's launches
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        one(batch)
        torch.cuda.synchronize()
    own = sum(e.count for e in prof.key_averages() if "dram::" in e.key)
    total_kernels = sum(e.count for e in prof.key_averages()
                        if e.device_type is not None and "DeviceType.CUDA" in str(e.device_type) and "Mem" not in e.key)
    if step.peer is not None:
        step.peer.check()
    ranks_identical = None
    if world > 1:  # data-parallel replicas must hold the same weights and running statistics, to the bit
        import torch.distributed as dist

        flat = torch.cat([p.detach().reshape(-1).double() for p in model.parameters()] +
                         [b.detach().reshape(-1).double() for b in model.buffers()])
        digest = torch.stack([flat.sum(), flat.abs().sum()])
        digests = [torch.zeros_like(digest) for _ in range(world)]
        dist.all_gather(digests, digest)
        ranks_identical = all(bool(torch.equal(digests[0], d)) for d in digests)
    train_flops = step.net.training_flops()  # fprop + dgrad + wgrad of every convolution; the stem has no dgrad
    peak, peak_src = measured_peaks()
    achieved = train_flops / (ms_per_step * 1e-3) / 1e12
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    line = {
        "metric": "CT volumes/sec med3ddram training (fwd+bwd+all-reduce+Adam)", "mode": "train",
        "value": world * B / (ms_per_step * 1e-3), "unit": "volumes/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16 operands / f32 accumulate, fp32 master weights and gradients", "data": "synthetic",
        "config": {"workload": f"{ARCH_NAMES[args.arch]} training step, synthetic {dims[0]}x{dims[1]}x{dims[2]} CT volumes, "
                               f"batch {B} per GPU, random-init weights",
                   "global_batch": world * B, "parallelism": f"data-parallel x{world}, bucketed NCCL gradient all-reduce"
                                                             f"{' + SyncBatchNorm (' + ('K10x peer-memory exchange' if args.sync_bn == 'peer' else 'NCCL') + ')' if world > 1 else ''}",
                   "glue": "native: conv fwd/dgrad/wgrad, BatchNorm(+ReLU,+residual), max-pool, up-sampling, heads; "
                           "weight re-packing, loss + gradient (K11), Adam (K12); ATen: shortcut-A slicing/padding, "
                           "stem weight-gradient re-layout, per-channel dtype casts",
                   "l2": "activations per step (> 10 GB) exceed the 126 MB L2; no explicit flush"},
        "clocks": clocks, "loss": float(loss), "ranks_identical": ranks_identical,
        "e2e": {"value": world * B / (e2e_ms * 1e-3), "unit": "volumes/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": e2e_ms, "api": "training.TrainStep.step(batch) with the batch copied from pinned host memory "
                                              "every step and the loss read back"},
        "gpu_launches": own * args.steps, "launches_per_step": {"dram_b200": own, "all_kernels": total_kernels},
        "roofline": {"bound": "tensor", "kernel": "whole training step (conv fprop + dgrad + wgrad FLOPs over the step time)",
                     "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": None,
                     "peak_source": peak_src, "algorithmic_flops_per_step": train_flops},
    }
    out.emit(json.dumps(line))


def training_field(device, dims, arch, steps):
    """BASELINE config 5 as an extra FIELD of the default line (N = 1 only; `--mode train` prints the full line and is
    what runs under torchrun): one training step = forward + loss + backward + Adam on the hand-written kernels, bf16
    activations, per-GPU batch 1, batch resident in HBM."""
    import dram_b200  # noqa: F401
    from dram_b200 import med3d, training

    torch.manual_seed(0)
    factory = {"med3ddram": med3d.resnet34segreg, "med3ddram18": med3d.resnet18segreg, "med3ddram50": med3d.resnet50segreg}
    model = factory[arch]().to(device).train()
    step = training.TrainStep(model, lr=1e-5, sync_bn=False)
    hu, lungs, ess = make_volumes(1, dims, device, seed=0)
    v = (hu.float().clamp(-1150.0, -300.0) + 1150.0) / 850.0
    image = (v - v.mean(dim=(1, 2, 3), keepdim=True)) / v.std(dim=(1, 2, 3), keepdim=True)
    batch = {"image": image.contiguous(), "lung_mask": lungs.bool(), "em_mask": ess.bool(),
             "cls_label": torch.full((1,), 2, device=device), "pse_label": torch.full((1,), 1, device=device)}
    bands = (torch.tensor([[0.05, 0.1]], device=device), torch.tensor([[0.01, 0.05]], device=device))
    w = torch.ones(1, device=device)
    for _ in range(3):
        step.step(batch, bands[0], bands[1], w, w)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step.step(batch, bands[0], bands[1], w, w)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    flops = step.net.training_flops()
    peak, _ = measured_peaks()
    out = {"metric": "CT volumes/sec med3ddram training (fwd+bwd+Adam), batch 1, 1 GPU", "value": 1.0 / (ms * 1e-3),
           "unit": "volumes/s", "ms_per_step": ms, "steps": steps, "dtype": "bf16 operands / f32 accumulate",
           "loss": float(loss), "roofline_frac": flops / (ms * 1e-3) / 1e12 / peak,
           "algorithmic_flops_per_step": flops, "full_line": "python bench.py --mode train (torchrun for N > 1)"}
    del step, model
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4, help="volumes per GPU per step")
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--dims", default="", help="D,H,W (overrides --size), e.g. 400,512,512")
    ap.add_argument("--arch", default=ARCH, choices=sorted(ARCH_NAMES))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "cudnn"])
    ap.add_argument("--no-train-field", dest="train_field", action="store_false",
                    help="skip the `training` field of the main line (config 5 at N=1, batch 1; ~15 s)")
    ap.add_argument("--no-yardstick", dest="yardstick", action="store_false",
                    help="skip the cuDNN yard-stick field of the main line (N=1 only; a few seconds)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sync-bn", default="peer", choices=["peer", "nccl"],
                    help="--mode train on >1 GPU: SyncBatchNorm statistics over the peer-memory kernel (K10x) or NCCL")
    ap.add_argument("--mode", default="infer", choices=["infer", "train"],
                    help="infer (default): BASELINE.json's headline metric; train: one data-parallel training step "
                         "(BASELINE config 5; additional line, not the headline)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last one returned (dRAM maps and percentages of rank "
                         "0's volumes) as DIR/<name>.npy, at most 64 MB in all: a larger map is a fixed, seeded sample "
                         "(see dump_outputs); default inference arm only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.mode != "infer"):
        ap.error("--dump-outputs applies to the default inference arm (--impl ours --mode infer)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    sink = _StdoutToStderr()
    if args.impl == "reference":
        run_reference_arm(args, sink)
        return
    if args.impl == "cudnn":
        run_cudnn_arm(args, sink)
        return
    if args.mode == "train":
        run_train_arm(args, sink)
        return

    rank, local, world = dist_setup(args.gpus)
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    from dram_b200.utils import bind_to_gpu_cpus
    cpu_binding = bind_to_gpu_cpus(local)  # before any pinned allocation: host buffers land on the GPU's NUMA node
    dims = parse_dims(args)
    B = args.batch
    module = build_module(device, args.arch)
    hu, lungs, ess = make_volumes(B, dims, device, seed=rank)
    eng = module.model.engine(B, dims, device)

    def step():
        return module.predict_step_from_hu(hu, lungs, ess)

    # ---- device-resident throughput ----------------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()  # nvidia-smi needs ~0.5 s to produce its first sample: start it before the warm-up
    for _ in range(args.warmup):
        out = step()
    torch.cuda.synchronize()
    barrier(world)
    torch.cuda.synchronize()
    first_sample = sampler.mark() if rank == 0 else 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = step()
    e1.record()
    torch.cuda.synchronize()
    barrier(world)
    ms_total = max_over_ranks(e0.elapsed_time(e1), world, device)
    clocks = sampler.stop(skip=first_sample) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)  # predict_step_from_hu allocates its outputs: `out` is the last step's
    ms_per_step = ms_total / args.steps
    value = world * B / (ms_per_step * 1e-3)
    launches_per_step = len(eng.steps) + 3 + 2  # K8 statistics + finalize + apply; the recorded steps; K7 + finalize

    # ---- end to end through the public predict_step with pinned host buffers -----------------
    from dram_b200 import ops
    from dram_b200.models import DevicePrefetcher

    win, _ = ops.window_standardize(hu, batched=True)   # the standardised fp32 volumes predict_step receives from the transforms
    host = {"image": win.cpu().pin_memory(), "lung_mask": lungs.bool().cpu().pin_memory(),
            "ess_mask": ess.bool().cpu().pin_memory()}
    del win
    h2d = sum(t.numel() * t.element_size() for t in host.values())
    D, H, W = dims
    full_box = [(0, D), (0, H), (0, W)]

    # host->device bandwidth of this box for the same buffers (explains e2e when the PCIe link is the limit)
    probe_dst = {k: torch.empty_like(v, device=device) for k, v in host.items()}
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    p0.record()
    for _ in range(3):
        for k, v in host.items():
            probe_dst[k].copy_(v, non_blocking=True)
    p1.record()
    torch.cuda.synchronize()
    h2d_gbs = 3 * h2d / (p0.elapsed_time(p1) * 1e-3) / 1e9
    del probe_dst

    e2e_diag = os.environ.get("DRAM_B200_E2E_DIAG", "")  # "" | nod2h | noh2d: A/B of the copy legs, never a bench value
    copy_streams = int(os.environ.get("DRAM_B200_COPY_STREAMS", "1"))  # DevicePrefetcher's default; > 1 = chunked over several DMA streams (A/B)

    class ResultSink:
        """The output half of the predict loop: per step the two uint8 heat-maps of every volume (f2: resample to the
        crop box, paste, window to uint8 — here the box is the whole volume) and the percentages go to pinned host
        memory on a side stream; two buffer sets, a set is reused only after its copy has finished."""

        def __init__(self):
            self.stream = torch.cuda.Stream(device=device)
            self.dev = [[torch.empty((2, B, D, H, W), dtype=torch.uint8, device=device), torch.empty((2, B), device=device)]
                        for _ in range(2)]
            self.host = [[torch.empty((2, B, D, H, W), dtype=torch.uint8).pin_memory(), torch.empty((2, B)).pin_memory()]
                         for _ in range(2)]
            self.done = [None, None]
            self.bytes_per_step = 2 * B * D * H * W + 2 * B * 4

        def push(self, i, pred):
            k = i % 2
            if self.done[k] is not None:
                self.done[k].synchronize()     # the consumer has taken step i-2's results
            maps, pct = self.dev[k]
            for m, key in enumerate(("cle_dense_outs", "pse_dense_outs")):
                for b in range(B):
                    ops.heatmap_u8(pred[key][b, 0], full_box, dims, out=maps[m, b])
            pct[0].copy_(pred["cle_precentages"])
            pct[1].copy_(pred["pse_precentages"])
            ready = torch.cuda.Event()
            ready.record()
            with torch.cuda.stream(self.stream):
                self.stream.wait_event(ready)
                if e2e_diag != "nod2h":  # diagnostic runs only (the line says so in e2e.api)
                    self.host[k][0].copy_(maps, non_blocking=True)
                    self.host[k][1].copy_(pct, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self.stream)
            self.done[k] = ev

        def finish(self):
            for ev in self.done:
                if ev is not None:
                    ev.synchronize()

    # One sink for the whole run: its pinned host buffers (2 x 134 MB) are allocated once, like a predict loop's — page-
    # locking them inside the timed region cost 7-10 % of a 20-step run at one GPU and far more with eight processes
    # pinning at once (the e2e / value ratio fell 0.95 -> 0.82 -> 0.67 at 1 / 2 / 8 GPUs with neither copy leg to blame:
    # profiles/e2e_copy_legs_r2n2c.log).
    result_sink = ResultSink()

    def e2e_pass(n_steps, batches, step_fn):
        # the user-facing predict loop: every step copies ITS host batch to the device (on the prefetcher's side
        # stream, overlapping the previous step's kernels) and every step's heat-maps + scores go back to the host
        if e2e_diag == "noh2d":  # diagnostic: the batch is staged once, no host->device copy per step
            dev_batch = {k: (v.to(device) if isinstance(v, torch.Tensor) else v) for k, v in batches.items()}
            for i in range(n_steps):
                result_sink.push(i, step_fn(dev_batch, i))
        else:
            for i, dev_batch in enumerate(DevicePrefetcher((batches for _ in range(n_steps)), device, copy_streams=copy_streams)):
                result_sink.push(i, step_fn(dev_batch, i))
        result_sink.finish()
        return result_sink.bytes_per_step

    def timed_e2e(batches, step_fn):
        e2e_pass(2, batches, step_fn)
        torch.cuda.synchronize()
        barrier(world)
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        d2h = e2e_pass(args.steps, batches, step_fn)
        t1.record()
        torch.cuda.synchronize()
        barrier(world)
        return max_over_ranks(t0.elapsed_time(t1), world, device) / args.steps, d2h

    e2e_ms, d2h = timed_e2e(host, lambda b, i: module.predict_step(b, i))
    e2e = {"value": world * B / (e2e_ms * 1e-3), "unit": "volumes/s", "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms,
           "h2d_gbs_idle_probe": h2d_gbs, "copy_streams": copy_streams,
           "api": ("" if not e2e_diag else f"DIAGNOSTIC RUN ({e2e_diag}), not an end-to-end number: ") +
                  "for batch in DevicePrefetcher(host_batches): ScanRegLightningModule.predict_step(batch) -> heatmap_u8 of "
                  "both dRAMs of every volume + percentages -> pinned host memory (fp32 image + bool masks in, "
                  "uint8 heat-maps + scores out, every step, double-buffered both ways)"}

    # the product's own wire format: int16 HU + uint8 lobe labels in (3 B/voxel); lung / ess masks made on the device
    lobes = (lungs * 3).to(torch.uint8)  # any non-zero label: dataset.py:66 only tests lobe > 0
    host_p = {"scan": hu.cpu().pin_memory(), "lobes": lobes.cpu().pin_memory()}
    h2d_p = sum(t.numel() * t.element_size() for t in host_p.values())

    crop_bufs = [(torch.empty((B, D, H, W), dtype=torch.int16, device=device),
                  torch.empty((B, D, H, W), dtype=torch.uint8, device=device),
                  torch.empty((B, D, H, W), dtype=torch.uint8, device=device)) for _ in range(2)]

    def product_step(b, i):
        im, lg, es = crop_bufs[i % 2]
        for v in range(B):  # f1 (dataset.py:66-80): blank outside the twice-dilated lung, LAA-910 mask; crop = whole volume
            ops.lung_crop(b["scan"][v], b["lobes"][v], full_box, out=(im[v], lg[v], es[v]))
        return module.predict_step_from_hu(im, lg, es)

    e2e_p_ms, d2h_p = timed_e2e(host_p, product_step)
    e2e_product = {"value": world * B / (e2e_p_ms * 1e-3), "unit": "volumes/s", "h2d_bytes_per_step": h2d_p,
                   "d2h_bytes_per_step": d2h_p, "ms_per_step": e2e_p_ms,
                   "api": "int16 HU + uint8 lobe labels from pinned host memory -> f1 lung_crop (masks on the device) -> "
                          "predict_step_from_hu -> heatmap_u8 x2 per volume -> uint8 heat-maps + percentages to the host"}
    del host, host_p, crop_bufs, result_sink

    # ---- roofline of the convolutions: per-launch CUDA events over eager launches --------------
    conv_steps = [s for s in eng.steps if s.conv_part]  # K13's gather passes count into the convolutions' time
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in conv_steps]
    conv_ms = 0.0
    reps = min(args.steps, 5)
    ops.window_standardize(hu, out=eng.image, batched=True)
    for _ in range(reps):
        ci = 0
        for s in eng.steps:
            if s.conv_part:
                evs[ci][0].record()
                s.fn()
                evs[ci][1].record()
                ci += 1
            else:
                s.fn()
        torch.cuda.synchronize()
        conv_ms += sum(a.elapsed_time(b) for a, b in evs)
    conv_ms /= reps
    conv_flops = sum(s.flops for s in conv_steps)
    exec_flops = sum(s.executed_flops for s in conv_steps)
    peak, peak_src = measured_peaks()
    burst = measured_peaks(burst=True)[0]
    achieved = conv_flops / (conv_ms * 1e-3) / 1e12
    executed = exec_flops / (conv_ms * 1e-3) / 1e12
    traffic, traffic_src = measured_traffic(args.arch, dims, B)
    roofline = {"bound": "tensor",
                "kernel": f"conv3d_stem_kernel + conv3d_slab_kernel + conv3d_stream32_kernel + conv3d_umma_kernel (+ upconv_axis_kernel of the "
                          f"commuted us1.0; {len(conv_steps)} launches/step)",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_src, "algorithmic_flops_per_step": conv_flops, "kernel_ms_per_step": conv_ms,
                "share_of_step": conv_ms / ms_per_step,
                # what the tensor pipe really executes: zero-padding taps skipped (dilated layers), border tiles and
                # the stem's K padded (343 -> 448); `achieved` above counts the reference's 2*M*N*K
                "executed_flops_per_step": exec_flops, "achieved_executed": executed, "frac_executed": executed / peak,
                "peak_burst": burst, "frac_of_burst": achieved / burst, "frac_executed_of_burst": executed / burst,
                "tensor_pipe_pct": measured_tensor_pipe(args.arch, dims, B)}

    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    line = {
        "metric": METRIC, "value": value, "unit": "volumes/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f16 operands / f32 accumulate" if eng.act_dtype == torch.float16 else "bf16 operands / f32 accumulate",
        "data": "synthetic",
        "config": {"workload": workload_name(args.arch, dims, B),
                   "global_batch": world * B, "parallelism": f"volume-sharded x{world}, no collective",
                   "l2": "inputs+activations per step (>1 GB) exceed the 126 MB L2; no explicit flush",
                   "storage_dtype": str(eng.act_dtype), "cuda_graph": ops.graphs_enabled(),
                   "cpu_binding": cpu_binding},
        "clocks": clocks, "e2e": e2e, "e2e_product": e2e_product, "gpu_launches": launches_per_step * args.steps,
        "roofline": roofline,
    }
    if not args.no_cpu_baseline and world == 1:  # reported at N=1 only
        line["cpu_baseline"] = cpu_baseline(module, dims, args.arch)
    if args.train_field and world == 1 and args.arch == ARCH:
        try:
            module.model._engines.clear()
            torch.cuda.empty_cache()
            line["training"] = training_field(device, dims, args.arch, steps=min(args.steps, 10))
        except Exception as exc:  # never at the cost of the headline line
            line["training"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    if args.yardstick and world == 1:
        try:
            line["gpu_yardstick"] = cudnn_yardstick(module, dims, args.arch, B, device, steps=min(args.steps, 5))
        except Exception as exc:  # the yard-stick must never cost the headline line
            line["gpu_yardstick"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    sink.emit(json.dumps(line))


if __name__ == "__main__":
    main()
