"""Full-resolution decoder steps dense against restricted to the dRAM's support, and the cost of the work-list builder.

    python tools/decoder_mask_bench.py [--arch med3ddram] [--batch 4] [--dims 256,256,256] [--reps 20]

Inputs: `bench.make_volumes` (the benchmark's own HU / lung / ess volumes) and `bench.build_module`'s weights.  Each
step is timed alone with CUDA events (median of `reps` single calls after warm-up); "restricted" runs the same plan with
the work list `run_network(active_ess=...)` uses.  "active" = listed work items / all work items of the step; for
us3+heads the items are (column, plane) steps.  The builder is `dram_decoder_support` on the caller's ess (eager in
front of the graph) plus one flags + compaction pass per list (inside the graph).
"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from dram_b200 import ops  # noqa: E402


def gpu_description():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "nvidia-smi: no output"
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi unavailable ({e})"


def median_ms(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return sorted(times)[len(times) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--arch", default="med3ddram")
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--dims", default="256,256,256")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    dims = tuple(int(v) for v in args.dims.split(","))
    dev = torch.device("cuda:0")
    print(f"# {torch.cuda.get_device_name(dev)} | nvidia-smi name, power.limit, clocks.max.sm: {gpu_description()}")
    print(f"# {args.arch} {dims} batch {args.batch}, bench.make_volumes(seed=0), median of {args.reps} calls")
    module = bench.build_module(dev, args.arch)
    hu, lungs, ess = bench.make_volumes(args.batch, dims, dev, seed=0)
    ess = ess.contiguous()
    module.predict_step_from_hu(hu, lungs, ess)          # builds the engine, probes, captures the graphs
    eng = module.model.engine(args.batch, dims, dev)
    ops.window_standardize(hu, out=eng.image, batched=True)
    eng.run_network()
    print(f"# ess: {ess.float().mean().item() * 100:.1f} % of voxels; decoder grid {eng.half_dims}")
    support = ops.decoder_support(ess, eng.half_dims)
    builds, rows = [], []
    for name, plan, radius, _ in eng._decoder:
        size = plan.worklist_size() if plan is not None else 0
        if size == 0:
            rows.append((name, radius, None, median_ms(eng.steps[[s.name for s in eng.steps].index(name)].fn,
                                                        args.reps), None))
            continue
        flags = torch.empty(size, dtype=torch.uint8, device=dev)
        items = torch.empty(size, dtype=torch.int32, device=dev)
        count = torch.empty(1, dtype=torch.int32, device=dev)
        build = lambda plan=plan, r=radius, f=flags, i=items, c=count: plan.build_worklist(support, r, f, i, c)  # noqa
        build()
        builds.append(build)
        frac = int(count.item()) / size
        dense = median_ms(plan.run, args.reps)
        listed = median_ms(lambda: plan.run_listed(items, count), args.reps)
        rows.append((name, radius, frac, dense, listed))
    print(f"{'step':<14}{'radius':>7}{'active':>9}{'dense ms':>10}{'restr. ms':>11}{'saved ms':>10}{'time kept':>11}")
    tot_d = tot_r = 0.0
    for name, radius, frac, dense, listed in rows:
        if frac is None:
            print(f"{name:<14}{radius:>7}{'(dense)':>9}{dense:>10.3f}")
            continue
        tot_d += dense
        tot_r += listed
        print(f"{name:<14}{radius:>7}{frac * 100:>8.1f}%{dense:>10.3f}{listed:>11.3f}{dense - listed:>10.3f}"
              f"{listed / dense * 100:>10.1f}%")
    sup = median_ms(lambda: ops.decoder_support(ess, eng.half_dims, out=support), args.reps)
    lists = median_ms(lambda: [b() for b in builds], args.reps)
    print(f"{'total':<14}{'':>7}{'':>9}{tot_d:>10.3f}{tot_r:>11.3f}{tot_d - tot_r:>10.3f}")
    print(f"builder: support {sup:.3f} ms (eager), {len(builds)} work lists {lists:.3f} ms (in the graph); "
          f"net saving {tot_d - tot_r - sup - lists:.3f} ms per step")
    step_r = median_ms(lambda: module.predict_step_from_hu(hu, lungs, ess), args.reps)
    step_d = median_ms(lambda: (ops.window_standardize(hu, out=eng.image, batched=True),
                                ops.dram_upsample_mask(*eng.run_network()[:2], ess, lungs, dims)), args.reps)
    print(f"predict_step_from_hu: restricted {step_r:.3f} ms, dense route (run_network + K7) {step_d:.3f} ms")


if __name__ == "__main__":
    main()
