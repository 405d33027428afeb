"""Per-launch CUDA-event times of one engine step's dense launches, and a before/after table of two such runs.

    python tools/conv_launch_ab.py time [arch] [D,H,W] [batch] > run.jsonl
        one JSON line per engine step: name, mean ms over `reps` dense steps, and for convolutions run by the tile
        kernels the brick (w, h, d, samples) and whether the M256 pair kernel runs it
    python tools/conv_launch_ab.py table before.jsonl[,before2.jsonl...] after.jsonl[,after2.jsonl...]
        the launches whose brick folds samples or whose kernel differs, with their times (mean over the runs given)
        and the change; the median change of the launches that run the same code in both trees is printed as the
        reference (clock and power state differ between runs at the power cap)
Dev tool: the tree it runs from decides which code is timed, so run `time` once from each tree in one session.
"""
import json
import os
import sys


def time_steps(arch, dims, batch, reps=20):
    import torch

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench

    dev = torch.device("cuda:0")
    module = bench.build_module(dev, arch)
    hu, lungs, ess = bench.make_volumes(batch, dims, dev, seed=0)
    for _ in range(2):
        module.predict_step_from_hu(hu, lungs, ess)
    eng = module.model.engine(batch, dims, dev)
    for s in eng.steps:  # warm every launch
        s.fn()
    torch.cuda.synchronize()
    tot = [0.0] * len(eng.steps)
    for _ in range(reps):
        evs = []
        for s in eng.steps:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            s.fn()
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        for i, (a, b) in enumerate(evs):
            tot[i] += a.elapsed_time(b) / reps
    for s, ms in zip(eng.steps, tot):
        plan = getattr(s.fn, "__self__", None)
        brick = getattr(plan, "brick", None)
        if brick is None and plan is not None and getattr(plan, "algo", "") == "tiles":
            brick = (0, 0, 0, 1)  # a tree before bricks could fold samples: reported as unfolded
        pair = getattr(plan, "pair", None)
        if pair is None and plan is not None:  # older tree: the M256 kernel is the 3-stage plan of a 3x3x3 filter
            pair = getattr(plan, "stages", 0) == 3 and getattr(plan, "desc", None) is not None and plan.desc.kd > 1
        print(json.dumps({"name": s.name, "ms": ms, "brick": brick, "pair": bool(pair),
                          "algo": getattr(plan, "algo", None)}))


def table(before_path, after_path):
    def load(paths):
        runs = []
        for p in paths.split(","):
            with open(p) as f:
                runs.append([json.loads(line) for line in f if line.startswith("{")])
        for r in runs[1:]:
            assert [x["name"] for x in r] == [x["name"] for x in runs[0]], "the runs time different step lists"
        for i, x in enumerate(runs[0]):
            x["ms"] = sum(r[i]["ms"] for r in runs) / len(runs)
        return runs[0]

    before, after = load(before_path), load(after_path)
    assert [r["name"] for r in before] == [r["name"] for r in after], "the runs time different step lists"
    same = sorted(a["ms"] / b["ms"] for b, a in zip(before, after)
                  if not (a["brick"] and a["brick"][3] > 1) and a["pair"] == b["pair"])
    print(f"{'launch':22s} {'brick after':18s} {'pair':>5s} {'before ms':>10s} {'after ms':>9s} {'change':>8s}")
    tb = ta = 0.0
    for b, a in zip(before, after):
        if not (a["brick"] and a["brick"][3] > 1) and a["pair"] == b["pair"]:
            continue  # same code in both trees: not a tile-kernel launch, or its brick did not fold
        tb += b["ms"]
        ta += a["ms"]
        print(f"{a['name']:22s} {str(tuple(a['brick'])):18s} {str(a['pair']):>5s} {b['ms']:10.3f} {a['ms']:9.3f} "
              f"{100.0 * (a['ms'] / b['ms'] - 1.0):+7.1f}%")
    print(f"{'changed launches':22s} {'':18s} {'':>5s} {tb:10.3f} {ta:9.3f} {100.0 * (ta / tb - 1.0):+7.1f}%")
    print(f"{'unchanged launches':22s} {'':18s} {'':>5s} {'':>10s} {'':>9s} {100.0 * (same[len(same) // 2] - 1.0):+7.1f}%"
          f"  (median of {len(same)})")
    print(f"{'whole dense step':22s} {'':18s} {'':>5s} {sum(r['ms'] for r in before):10.3f} "
          f"{sum(r['ms'] for r in after):9.3f}")


if __name__ == "__main__":
    if sys.argv[1] == "time":
        arch = sys.argv[2] if len(sys.argv) > 2 else "med3ddram"
        dims = tuple(int(v) for v in sys.argv[3].split(",")) if len(sys.argv) > 3 else (256, 256, 256)
        batch = int(sys.argv[4]) if len(sys.argv) > 4 else 4
        time_steps(arch, dims, batch)
    else:
        table(sys.argv[2], sys.argv[3])
