"""Cost of the per-lobe lesion percentages (K7l, `ops.lobe_scores`) against K7 and against a whole inference step.

    python tools/lobe_scores_bench.py [--reps 50] [--configs c3,default]

Configurations: C3 = med3ddram (ResNet-34), 256^3, batch 4; default = med3ddram, the product grid (128, 224, 288),
batch 2.  Inputs are the synthetic volumes of oracle/synthetic.py (lobe labels 1-5) and a calibrated-random checkpoint.
Kernel times are medians of CUDA-event timings of single calls, each after a 256 MB write that evicts L2 (the
labels and ess of the default grid alone would fit the 126 MB L2); step times alternate the calls with and without
labels so that both see the same machine state.  Bytes are the reduction's compulsory traffic: labels and ess once
(1 byte each per voxel) plus both fp32 maps at the ess voxels.
"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import dram_b200  # noqa: E402,F401
from dram_b200 import ops  # noqa: E402
from oracle import synthetic  # noqa: E402

CONFIGS = {"c3": ("med3ddram", (256, 256, 256), 4), "default": ("med3ddram", (128, 224, 288), 2)}


def gpu_description():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + " (power limit not readable)"


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def time_kernel(fn, reps, flush):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return median(ts)


def time_alternating(fns, reps):
    for fn in fns:
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    ts = [[] for _ in fns]
    for _ in range(reps):
        for i, fn in enumerate(fns):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts[i].append(a.elapsed_time(b))
    return [median(t) for t in ts]


def run(name, reps, flush, dev):
    from dram_b200.models import ScanRegLightningModule

    arch, dims, B = CONFIGS[name]
    module = ScanRegLightningModule(argparse.Namespace(model_arch=arch))
    module.model.load_state_dict(synthetic.make_state_dict(arch, seed=0, calib_dims=(64, 64, 64)))
    module = module.to(dev).eval()
    vols = [synthetic.make_volume(i, dims) for i in range(B)]
    hu = torch.stack([v[0] for v in vols]).to(dev)
    labels = torch.stack([v[1] for v in vols]).to(dev)
    lung = (labels > 0).to(torch.uint8)
    ess = ((hu < -910) & (lung > 0)).to(torch.uint8)
    V = dims[0] * dims[1] * dims[2]
    try:
        out = module.predict_step_from_hu(hu, lung, ess)
    except ops.ActivationOverflow:  # what processor.py does: continue with bf16 storage, and say so
        print(f"[{name}] fp16 activation overflow with this checkpoint: bf16 storage", flush=True)
        module.model.act_dtype = torch.bfloat16
        out = module.predict_step_from_hu(hu, lung, ess)
    cle, pse = out["cle_dense_outs"], out["pse_dense_outs"]
    n_ess = int(ess.sum())
    nbytes = B * V * 2 + n_ess * 8
    print(f"[{name}] {arch} {dims} batch {B}: {B * V / 1e6:.1f} M voxels, {n_ess / (B * V):.2%} in ess, "
          f"lobe voxels {int((labels > 0).sum()) / (B * V):.1%}", flush=True)
    t_lobe = time_kernel(lambda: ops.lobe_scores(cle, pse, ess, labels), reps, flush)
    print(f"[{name}] ops.lobe_scores          {t_lobe * 1e3:9.1f} us  {nbytes / 1e6:8.1f} MB  "
          f"{nbytes / t_lobe / 1e6:8.1f} GB/s  ({t_lobe * 1e3 / B:.1f} us per volume)", flush=True)
    eng = module.model.engine(B, dims, dev)
    dense = eng.run_network()
    k7_bytes = B * V * (2 + 8)  # both masks in, both maps out (the dense maps are small)
    t_k7 = time_kernel(lambda: ops.dram_upsample_mask(dense[0], dense[1], ess, lung, dims, out=(cle, pse)), reps, flush)
    print(f"[{name}] K7 dram_upsample_mask    {t_k7 * 1e3:9.1f} us  {k7_bytes / 1e6:8.1f} MB  "
          f"{k7_bytes / t_k7 / 1e6:8.1f} GB/s", flush=True)
    without, with_lab = time_alternating([lambda: module.predict_step_from_hu(hu, lung, ess),
                                          lambda: module.predict_step_from_hu(hu, lung, ess, lobe_labels=labels)], reps)
    print(f"[{name}] predict_step_from_hu     without labels {without:8.3f} ms   with labels {with_lab:8.3f} ms   "
          f"difference {(with_lab - without) / without:+.2%}; lobe_scores alone is {t_lobe / without:.2%} of the step",
          flush=True)
    module.model._engines.clear()
    del module, hu, labels, lung, ess, out, cle, pse, dense, eng
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--configs", default="c3,default")
    args = ap.parse_args()
    if args.reps < 50:
        raise SystemExit("--reps must be at least 50")
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing here is measured on the CPU")
    dev = torch.device("cuda:0")
    print(f"GPU: {gpu_description()}; torch {torch.__version__}; {args.reps} repetitions, medians", flush=True)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for name in args.configs.split(","):
        run(name, args.reps, flush, dev)


if __name__ == "__main__":
    main()
