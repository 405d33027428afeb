"""Cost of the lung and per-lobe densitometry: both device passes, the whole measurement and the pre-steps with and without it.

    python tools/densitometry_bench.py [--reps 100] [--log profiles/densitometry_bench.log]

Volumes: the synthetic CT of oracle/synthetic.py (lobe labels 1-5, ~24 % of the voxels) at 400 x 512 x 512, a
full-resolution chest scan, and at 256^3.  Kernel times are medians of CUDA-event timings of single calls, each after a
256 MB write that evicts L2 (the 105 MB of labels of the large volume would otherwise be read partly from the 126 MB L2).
Bytes are each pass's compulsory traffic: the labels once (1 byte per voxel), and for the histogram pass the HU
(2 bytes per voxel) of every 16-voxel vector that holds a lobe label.  `scan_densitometry` is the whole measurement
(counts, read-back, histograms, read-back, host arithmetic), timed on the host around a device synchronise.
`device_presteps` (host arrays in, cropped device tensors out, including the host-to-device copy of the scan and the
labels) is timed the same way, with and without densitometry, alternating the two.
"""
import argparse
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import dram_b200  # noqa: E402,F401
from dram_b200 import densitometry, ops  # noqa: E402
from dram_b200.dataset import SubtypingInference  # noqa: E402
from oracle import synthetic  # noqa: E402

SIZES = {"400x512x512": (400, 512, 512), "256^3": (256, 256, 256)}
SPACING = (1.0, 0.68, 0.68)


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


def time_host(fns, reps):
    """Host clock around each call, ending in a device synchronise; the calls alternate.  Medians in ms."""
    for fn in fns:
        fn()
    torch.cuda.synchronize()
    ts = [[] for _ in fns]
    for _ in range(reps):
        for i, fn in enumerate(fns):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts[i].append((time.perf_counter() - t0) * 1e3)
    return [median(t) for t in ts]


def run(name, reps, flush, dev, emit):
    dims = SIZES[name]
    scan, labels = synthetic.make_volume(0, dims)
    V = scan.numel()
    s, lab = scan.to(dev), labels.to(dev)
    ids = [k for k in range(1, 256) if int((labels == k).sum()) > 0]
    lung_vectors = int((labels.reshape(-1, 16) > 0).any(dim=1).sum())
    count_bytes, hist_bytes = V, V + lung_vectors * 32
    emit(f"[{name}] {V / 1e6:.1f} M voxels, lobe voxels {int((labels > 0).sum()) / V:.1%}, {len(ids)} labels, "
         f"16-voxel vectors with a lobe label {lung_vectors * 16 / V:.1%}")
    t_count = time_kernel(lambda: ops.label_counts(lab), reps, flush)
    emit(f"[{name}] ops.label_counts       {t_count * 1e3:9.1f} us  {count_bytes / 1e6:8.1f} MB  "
         f"{count_bytes / t_count / 1e6:8.1f} GB/s")
    t_hist = time_kernel(lambda: ops.hu_histograms(s, lab, ids), reps, flush)
    emit(f"[{name}] ops.hu_histograms      {t_hist * 1e3:9.1f} us  {hist_bytes / 1e6:8.1f} MB  "
         f"{hist_bytes / t_hist / 1e6:8.1f} GB/s")
    (t_all,) = time_host([lambda: densitometry.scan_densitometry(s, lab, SPACING)], reps)
    emit(f"[{name}] scan_densitometry      {t_all:9.3f} ms  (both passes, two read-backs, host arithmetic)")
    scan_np, lobe_np = scan.numpy(), labels.numpy()
    plain = SubtypingInference(".", ".", device=dev)
    dens = SubtypingInference(".", ".", device=dev, densitometry=True)
    t_plain, t_dens = time_host([lambda: plain.device_presteps(scan_np, lobe_np, SPACING, "bench"),
                                 lambda: dens.device_presteps(scan_np, lobe_np, SPACING, "bench")], max(10, reps // 5))
    emit(f"[{name}] device_presteps        without {t_plain:8.3f} ms   with densitometry {t_dens:8.3f} ms   "
         f"difference {(t_dens - t_plain) / t_plain:+.2%}")
    del s, lab
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--sizes", default=",".join(SIZES))
    ap.add_argument("--log", default=os.path.join(ROOT, "profiles", "densitometry_bench.log"))
    args = ap.parse_args()
    if args.reps < 50:
        raise SystemExit("--reps must be at least 50")
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: nothing here is measured on the CPU")
    dev = torch.device("cuda:0")
    lines = []

    def emit(line):
        print(line, flush=True)
        lines.append(line)

    emit(f"GPU: {gpu_description()}; torch {torch.__version__}; {args.reps} repetitions, medians")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for name in args.sizes.split(","):
        run(name, args.reps, flush, dev, emit)
    os.makedirs(os.path.dirname(os.path.abspath(args.log)), exist_ok=True)
    with open(args.log, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
