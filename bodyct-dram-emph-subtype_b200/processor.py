"""Inference CLI with the reference's surface (processor.py:55-177 / run.sh):

    python processor.py --scan_path DIR --lobe_path DIR --output_path DIR [--ngpus N]
                        [--model_arch med3ddram] [--batch_size 2] [--target_size 128,224,288] [--workers 0]
                        [--lobe_scores] [--densitometry]

Outputs (same names, including the reference's `araseptal-` typo, processor.py:77):
    <out>/images/centrilobular-emphysema-heatmap/<uid>.mha   uint8
    <out>/images/paraseptal-emphysema-heatmap/<uid>.mha      uint8
    <out>/centrilobular-emphysema-score.json, <out>/araseptal-emphysema-score.json, <out>/results.json

Differences, all deliberate (SURVEY §8a quirks): no Lightning Trainer — one process per GPU is spawned
here for --ngpus > 1, each takes the DistributedSampler(shuffle=False) shard of the sorted scan list, and
rank 0 merges the per-rank records (the reference lets every rank overwrite results.json, Q8);
classification architectures (med3d*) are routed to ScanCLSLightningModule and emit argmax classes
(the reference crashes on them, Q4); --target_size is parseable (Q7); unknown Trainer flags are ignored.

`--lobe_scores` (not in the reference; *dram architectures only) adds to every results.json record
    "lobe_metrics": {"<label>": {"cle_lesion_percentage": "x.xxx", "pse_lesion_percentage": "y.yyy"}, ...}
for each label >= 1 of the lobe segmentation that has voxels in the network's grid: the lesion fraction of that
lobe, in the unit of `*_lesion_percentage_per_lung`.

`--densitometry` (not in the reference; every architecture) adds to every results.json record
    "densitometry": {"lung": {...}, "lobes": {"<label>": {...}, ...}}
with "volume_ml", "laa950_percentage", "laa910_percentage", "perc15_hu" and "mean_hu" of the lung (all labels >= 1)
and of each label >= 1 that has voxels, measured on the full-resolution scan (definitions in densitometry.py).
"""
import json
import logging
import os
import subprocess
import sys
import warnings
from argparse import ArgumentParser
from pathlib import Path

if __package__ in (None, ""):  # executed as a script: import the package under its shim name
    _here = os.path.dirname(os.path.abspath(__file__))
    sys.path.insert(0, os.path.dirname(_here))
    import importlib

    importlib.import_module("dram_b200")
    __package__ = "dram_b200"

import numpy as np  # noqa: E402
import torch  # noqa: E402

from . import mha_io, ops  # noqa: E402
from .densitometry import format_densitometry  # noqa: E402
from .models import (CLE_RATIO_MAP, PSE_RATIO_MAP, RunningStage, ScanCLSLightningModule,  # noqa: E402
                     ScanRegLightningModule, SubtypeDataModule, ratio_to_label)
from .utils import load_state_dict_greedy, windowing, write_array_to_mha_itk  # noqa: E402

warnings.filterwarnings("ignore")
logging.basicConfig(level=logging.ERROR, format="%(asctime)s [%(levelname)s] %(message)s",
                    handlers=[logging.StreamHandler()])


def _size(text):
    if isinstance(text, (tuple, list)):
        return tuple(int(v) for v in text)
    return tuple(int(v) for v in str(text).replace("x", ",").strip("()[] ").split(","))


def build_parser():
    p = ArgumentParser()
    p.add_argument("--ngpus", default=1, type=int)
    p.add_argument("--model_arch", default="med3ddram", type=str)
    p.add_argument("--workers", default=0, type=int)
    p.add_argument("--batch_size", default=2, type=int)
    p.add_argument("--target_size", default=(128, 224, 288), type=_size)
    p.add_argument("--scan_path", default="/input/images/ct/", type=str)
    p.add_argument("--lobe_path", default="/input/images/pulmonary-lobes/", type=str)
    p.add_argument("--output_path", default="/output", type=str)
    p.add_argument("--local_rank", default=0, type=int, help="not used; kept for compatibility")
    p.add_argument("--ckpt_path", default="best.ckpt", type=str, help="Lightning checkpoint (state_dict under 'state_dict')")
    p.add_argument("--allow_random_init", action="store_true",
                   help="tests/benchmarks only: run with random-init weights when the checkpoint is missing or a Git-LFS "
                        "pointer (recorded in every result's error_messages); without it that is a fatal error")
    p.add_argument("--lobe_scores", action="store_true",
                   help="also report CLE and PSE lesion percentages per lobe label (lobe_metrics in results.json); "
                        "*dram architectures only")
    p.add_argument("--densitometry", action="store_true",
                   help="also report lung and per-lobe volume, %%LAA-950, %%LAA-910, Perc15 and mean HU of the "
                        "full-resolution scan (densitometry in results.json); every architecture")
    return p


def check_args(args):
    """Refuses option combinations that cannot run, before any GPU work."""
    if args.lobe_scores and "dram" not in args.model_arch:
        raise ValueError(f"--lobe_scores needs a *dram (regression) architecture; {args.model_arch} is a "
                         "classification architecture without dRAM maps")


class CheckpointError(RuntimeError):
    """The checkpoint the predictions depend on could not be loaded."""


RANDOM_INIT_NOTE = "checkpoint missing: predictions come from RANDOM-INIT weights (--allow_random_init)"


def _read_checkpoint(path):
    """A reference checkpoint is what Lightning's ModelCheckpoint wrote under torch 1.12: besides `state_dict` it holds
    `hyper_parameters = {'args': argparse.Namespace(...)}` (models.py:166 `save_hyperparameters()`), callback and
    optimiser states.  torch >= 2.6 defaults to `weights_only=True`, which rejects the Namespace: allow-list it, and fall
    back to the full unpickler (what processor.py:85 of the reference does) for anything else in this trusted file."""
    import argparse
    import pickle

    try:
        with torch.serialization.safe_globals([argparse.Namespace]):
            return torch.load(path, map_location="cpu", weights_only=True)
    except pickle.UnpicklingError as exc:
        logging.warning(f"checkpoint '{path}' needs the full unpickler ({str(exc).splitlines()[0]}); it ships with the "
                        "model and is trusted")
        return torch.load(path, map_location="cpu", weights_only=False)


def load_checkpoint(module, path, allow_random_init=False):
    """processor.py:85-87.  The reference checkout ships Git-LFS pointers; a pointer or a missing file is a fatal
    `CheckpointError` (the reference's torch.load fails there too) unless `allow_random_init` — then the random
    initialisation stays, False is returned and the caller records it in every result."""
    if not os.path.isfile(path) or os.path.getsize(path) < 4096:
        msg = (f"checkpoint '{os.path.abspath(path)}' is missing or a Git-LFS pointer (the default 'best.ckpt' is relative "
               "to the working directory)")
        if not allow_random_init:
            raise CheckpointError(msg + "; refusing to write scores from random-init weights "
                                        "(--allow_random_init overrides, for tests and benchmarks)")
        logging.error(msg + ": running with random-init weights")
        return False
    ckpt = _read_checkpoint(path)
    load_state_dict_greedy(module, ckpt["state_dict"] if "state_dict" in ckpt else ckpt)
    return True


def lobe_metrics(voxels, cle_pct, pse_pct):
    """The `lobe_metrics` field of one record from predict_step's per-label outputs of one sample (voxels [256],
    percentages [256]): labels >= 1 that have voxels, percentages formatted like the whole-lung ones."""
    voxels, cle_pct, pse_pct = (torch.as_tensor(v).cpu().tolist() for v in (voxels, cle_pct, pse_pct))
    return {str(k): {"cle_lesion_percentage": "{:.3f}".format(cle_pct[k]),
                     "pse_lesion_percentage": "{:.3f}".format(pse_pct[k])}
            for k in range(1, len(voxels)) if voxels[k] > 0}


def postprocess_reg(pred, data_module, out_cle, out_pse, writer=None):
    """processor.py:111-158 for one batch of predictions; returns the result records.  `writer`: a
    `mha_io.BackgroundWriter` that takes the file writes off this thread (`--workers N`)."""
    records = []
    meta_cache = data_module.datasets[RunningStage.PREDICTING].scan_meta_cache
    B = pred["cle_dense_outs"].shape[0]
    lobes = None
    if "lobe_voxels" in pred:
        lobes = [pred[k].cpu() for k in ("lobe_voxels", "cle_lobe_percentages", "pse_lobe_percentages")]
    for b in range(B):
        crop = pred["crop_slices"][b]
        orig = tuple(int(v) for v in pred["original_size"][b])
        uid = pred["uids"][b]
        # f2: resample to the crop, paste into the full volume and window to uint8 in one kernel per map;
        # only uint8 leaves the GPU (processor.py:115-122, 143, 152 of the reference do this in numpy/float64)
        heat = [ops.heatmap_u8(pred[k][b, 0].contiguous(), crop.tolist(), orig).cpu().numpy()
                for k in ("cle_dense_outs", "pse_dense_outs")]
        cle_pct, pse_pct = pred["cle_precentages"][b].item(), pred["pse_precentages"][b].item()
        metrics = {
            "cle_severity_score": "{:d}".format(ratio_to_label(cle_pct, CLE_RATIO_MAP)),
            "cle_lesion_percentage_per_lung": "{:.3f}".format(cle_pct),
            "pse_severity_score": "{:d}".format(ratio_to_label(pse_pct, PSE_RATIO_MAP)),
            "pse_lesion_percentage_per_lung": "{:.3f}".format(pse_pct),
        }
        record = {"entity": uid, "metrics": metrics, "error_messages": []}
        if lobes is not None:
            record["lobe_metrics"] = lobe_metrics(lobes[0][b], lobes[1][b], lobes[2][b])
        add_densitometry(record, data_module)
        records.append(record)
        meta = meta_cache[uid]
        kw = dict(type=np.uint8, origin=meta["origin"][::-1], spacing=meta["spacing"][::-1],
                  direction=np.asarray(meta["direction"]).reshape(3, 3)[::-1].flatten().tolist())
        for full, folder in zip(heat, (out_cle, out_pse)):
            if writer is None:
                write_array_to_mha_itk(folder, [full], [uid], **kw)
            else:
                writer.submit(write_array_to_mha_itk, folder, [full], [uid], **kw)
    return records


def postprocess_cls(pred, data_module=None):
    records = []
    for b, uid in enumerate(pred["uids"]):
        metrics = {"cle_severity_score": "{:d}".format(int(pred["cle_labels"][b])),
                   "pse_severity_score": "{:d}".format(int(pred["pse_labels"][b]))}
        record = {"entity": uid, "metrics": metrics, "error_messages": []}
        if data_module is not None:
            add_densitometry(record, data_module)
        records.append(record)
    return records


def add_densitometry(record, data_module):
    """Adds the `densitometry` field to a record when the dataset measured its scan (`--densitometry`)."""
    ds = data_module.datasets[RunningStage.PREDICTING]
    if getattr(ds, "densitometry", False):
        record["densitometry"] = format_densitometry(ds.densitometry_cache[record["entity"]])


def run_rank(args, rank, world_size):
    device = torch.device("cuda", rank % max(1, torch.cuda.device_count()))
    torch.cuda.set_device(device)
    if world_size > 1:  # one process per GPU: keep its host buffers and reader / writer threads on the GPU's NUMA node
        from .utils import bind_to_gpu_cpus
        bind_to_gpu_cpus(device.index)
    args.device = device
    is_reg = "dram" in args.model_arch  # the split train.py:72 / test.py:62 make
    module = (ScanRegLightningModule if is_reg else ScanCLSLightningModule)(args)
    loaded = load_checkpoint(module, args.ckpt_path, allow_random_init=bool(getattr(args, "allow_random_init", False)))
    module = module.to(device).eval()
    data_module = SubtypeDataModule(args)
    out_cle = f"{args.output_path}/images/centrilobular-emphysema-heatmap/"
    out_pse = f"{args.output_path}/images/paraseptal-emphysema-heatmap/"
    Path(out_cle).mkdir(parents=True, exist_ok=True)
    Path(out_pse).mkdir(parents=True, exist_ok=True)
    records, notes = [], []
    workers = int(getattr(args, "workers", 0) or 0)
    with mha_io.BackgroundWriter(workers) as writer:  # workers == 0: writes happen in place, as before
        for i, batch in enumerate(data_module.predict_dataloader(rank, world_size)):
            try:
                pred = module.predict_step(batch, i)
            except ops.ActivationOverflow as exc:
                # fp16 storage (more mantissa, DESIGN.md section 2) cannot hold this checkpoint's activations:
                # continue in bf16 (fp32's exponent range) and say so in every record
                logging.error(f"{exc}; switching this run to bf16 storage")
                module.model.act_dtype = torch.bfloat16
                notes.append("fp16 activation overflow detected: run continued with bf16 storage (coarser dRAM values)")
                pred = module.predict_step(batch, i)
            if is_reg:
                records += postprocess_reg(pred, data_module, out_cle, out_pse, writer if workers > 0 else None)
            else:
                records += postprocess_cls(pred, data_module)
    if not loaded:
        notes.append(RANDOM_INIT_NOTE)
    for r in records:
        r["error_messages"] += notes
    return records


def write_results(args, records):
    """processor.py:160-177 (first record feeds the two per-algorithm score files)."""
    seen, merged = set(), []
    for r in records:  # drop the wrap-around duplicates DistributedSampler padding produces
        if r["entity"] not in seen:
            seen.add(r["entity"])
            merged.append(r)
    merged.sort(key=lambda r: r["entity"])
    if merged:
        m = merged[0]["metrics"]
        with open(f"{args.output_path}/centrilobular-emphysema-score.json", "w") as f:
            f.write(json.dumps({"score": int(float(m["cle_severity_score"])),
                                "percentage": float(m.get("cle_lesion_percentage_per_lung", "nan"))}))
        with open(f"{args.output_path}/araseptal-emphysema-score.json", "w") as f:
            f.write(json.dumps({"score": int(float(m["pse_severity_score"])),
                                "percentage": float(m.get("pse_lesion_percentage_per_lung", "nan"))}))
    with open(f"{args.output_path}/results.json", "w") as f:
        f.write(json.dumps(merged))
    return merged


def run_testing_job(argv=None):
    args, _ignored_trainer_flags = build_parser().parse_known_args(argv)
    check_args(args)
    Path(args.output_path).mkdir(parents=True, exist_ok=True)
    rank = int(os.environ.get("DRAM_B200_RANK", "-1"))
    if rank >= 0:  # worker of a multi-GPU job
        records = run_rank(args, rank, int(os.environ["DRAM_B200_WORLD"]))
        with open(f"{args.output_path}/results.rank{rank}.json", "w") as f:
            json.dump(records, f)
        return records
    if args.ngpus <= 1:
        return write_results(args, run_rank(args, 0, 1))
    procs = []
    for r in range(args.ngpus):  # one process per GPU; no collective: volumes are independent
        env = dict(os.environ, DRAM_B200_RANK=str(r), DRAM_B200_WORLD=str(args.ngpus))
        procs.append(subprocess.Popen([sys.executable, os.path.abspath(__file__)] + (argv or sys.argv[1:]), env=env))
    failed = [r for r, p in enumerate(procs) if p.wait() != 0]
    if failed:
        raise RuntimeError(f"inference workers {failed} failed")
    records = []
    for r in range(args.ngpus):
        part = f"{args.output_path}/results.rank{r}.json"
        with open(part) as f:
            records += json.load(f)
        os.remove(part)
    return write_results(args, records)


if __name__ == "__main__":
    print("Docker start running testing job.")
    print("results:", run_testing_job())
