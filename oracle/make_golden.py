"""Generates tests/golden/* by running the UNMODIFIED reference on CPU.  TEST INFRASTRUCTURE.

    DRAM_REFERENCE_DIR=<upstream checkout> python -m oracle.make_golden      (from the repo root)

Every fixture records the seeds/dims that regenerate its inputs with oracle/synthetic.py, a
fingerprint of the weights, and the reference's outputs.  Nothing here is imported by product code;
the fixtures travel to the GPU box, the reference does not.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import pipeline_oracle as P  # noqa: E402
from oracle import ref_shim, synthetic  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")

# (arch, batch, dims, with_lungs)
FORWARD_CASES = [
    ("med3ddram18", 2, (32, 32, 32), True),
    ("med3ddram18", 1, (32, 32, 32), False),
    ("med3d18", 1, (32, 32, 32), False),
    ("med3ddram", 1, (32, 40, 48), True),
    ("med3d", 1, (32, 32, 32), False),
    ("med3ddram50", 1, (32, 32, 32), True),
    ("med3d50", 1, (24, 32, 32), False),
]


def case_name(arch, batch, dims, with_lungs):
    return f"forward_{arch}_b{batch}_{dims[0]}x{dims[1]}x{dims[2]}_{'lungs' if with_lungs else 'nolungs'}"


def batch_inputs(batch, dims):
    xs, ls, es = zip(*[synthetic.make_network_input(i, dims) for i in range(batch)])
    return torch.stack(xs), torch.stack(ls), torch.stack(es)


def gen_layouts(ref):
    out = {}
    for arch in ["med3d", "med3d18", "med3d50", "med3ddram", "med3ddram18", "med3ddram50"]:
        m = ref_shim.model(arch)
        sd = m.state_dict()
        out[arch] = {
            "keys": [[k, list(v.shape), str(v.dtype)] for k, v in sd.items()],
            "params": sum(p.numel() for p in m.parameters()),
            "class": type(m).__name__,
        }
    with open(os.path.join(GOLDEN, "state_layouts.json"), "w") as f:
        json.dump(out, f)
    print("state_layouts.json", {k: (len(v["keys"]), v["params"]) for k, v in out.items()})


def gen_forward(ref):
    for arch, batch, dims, with_lungs in FORWARD_CASES:
        sd = synthetic.make_state_dict(arch, seed=0, calib_dims=dims)
        model = ref_shim.model(arch)
        ref.utils.load_state_dict_greedy(model, sd)
        model.eval()
        x, lung, _ = batch_inputs(batch, dims)
        with torch.no_grad():
            dense, scores = model(x.unsqueeze(1).clone(), lung.unsqueeze(1).float() if with_lungs else None)
        fix = {
            "arch": arch, "batch": batch, "dims": dims, "with_lungs": with_lungs, "weight_seed": 0,
            "weight_checksum": synthetic.state_dict_checksum(sd),
            "dense_outs": [d.clone() for d in dense],
            "scores": [s.clone() for s in scores],
        }
        name = case_name(arch, batch, dims, with_lungs)
        torch.save(fix, os.path.join(GOLDEN, name + ".pt"))
        print(name, [tuple(d.shape) for d in dense], [s.flatten().tolist()[:3] for s in scores])


# (arch, dims): the reference's OWN initialisation (med3d.py:334-339: kaiming-normal fan_out convolutions, BatchNorm
# weight 1 / bias 0 and default running statistics, PyTorch-default conv biases) under torch.manual_seed(REF_INIT_SEED).
# dram_b200.med3d draws the same random stream (module construction order and init calls are the same), so the GPU
# test rebuilds these weights from the seed alone; `weight_checksum` guards that.
REF_INIT_SEED = 20261018
REF_INIT_CASES = [("med3d", (32, 32, 32)), ("med3d18", (32, 32, 32)), ("med3d50", (24, 32, 32)),
                  ("med3ddram", (32, 32, 32)), ("med3ddram18", (32, 40, 48)), ("med3ddram50", (32, 32, 32))]


def gen_reference_init(ref):
    for arch, dims in REF_INIT_CASES:
        torch.manual_seed(REF_INIT_SEED)
        model = ref_shim.model(arch)
        sd = model.state_dict()
        x, lung, _ = batch_inputs(1, dims)
        logits, acts = [], {}
        hooks = [fc.register_forward_hook(lambda mod, i, o: logits.append(o.detach().clone())) for fc in model.fcs]
        for n, mod in model.named_modules():
            if isinstance(mod, torch.nn.Conv3d):
                hooks.append(mod.register_forward_hook(lambda mod, i, o, n=n: acts.__setitem__(n, float(o.abs().max()))))
        with torch.no_grad():
            dense, scores = model(x.unsqueeze(1).clone(), lung.unsqueeze(1).float())
        for h in hooks:
            h.remove()
        fix = {"arch": arch, "dims": dims, "batch": 1, "with_lungs": True, "init_seed": REF_INIT_SEED,
               "weight_checksum": synthetic.state_dict_checksum(sd),
               "dense_outs": [d.clone() for d in dense], "scores": [s.clone() for s in scores],
               "logits": logits, "max_conv_output": max(acts.values())}
        torch.save(fix, os.path.join(GOLDEN, f"refinit_{arch}.pt"))
        print("refinit", arch, dims, "max |conv out|", fix["max_conv_output"], "logit absmax",
              [float(l.abs().max()) for l in logits], "scores", [sc.flatten().tolist()[:3] for sc in scores])


def gen_predict_step(ref):
    from argparse import Namespace

    arch, dims, batch = "med3ddram18", (16, 32, 48), 2
    sd = synthetic.make_state_dict(arch, seed=1, calib_dims=dims, prefix="model.")
    with ref_shim.reference_cwd():
        module = ref.models.ScanRegLightningModule(Namespace(model_arch=arch))
    ref.utils.load_state_dict_greedy(module, sd)  # the processor.py:85-87 path, `model.` prefixed keys
    module.eval()
    x, lung, ess = batch_inputs(batch, dims)
    b = {
        "image": x, "lung_mask": lung.bool(), "ess_mask": ess.bool(),
        "crop_slice": torch.tensor([[[0, d] for d in dims]] * batch), "original_size": torch.tensor([dims] * batch),
        "uid": [f"v{i}" for i in range(batch)],
    }
    out = module.predict_step(b, 0)
    fix = {
        "arch": arch, "dims": dims, "batch": batch, "weight_seed": 1,
        "weight_checksum": synthetic.state_dict_checksum(sd),
        "cle_dense_outs": out["cle_dense_outs"], "pse_dense_outs": out["pse_dense_outs"],
        "cle_precentages": out["cle_precentages"], "pse_precentages": out["pse_precentages"],
        "keys": list(out.keys()),
        "cle_labels": module._ratio_to_label(out["cle_precentages"], ref.dataset.COPDGeneSubtyping.cle_ratio_map),
        "pse_labels": module._ratio_to_label(out["pse_precentages"], ref.dataset.COPDGeneSubtyping.pse_ratio_map),
    }
    torch.save(fix, os.path.join(GOLDEN, "predict_step_med3ddram18.pt"))
    print("predict_step", fix["cle_precentages"].tolist(), fix["pse_precentages"].tolist(), fix["cle_labels"].tolist())


def reference_train_step(ref, case):
    """One training step of the UNMODIFIED reference network (train mode) with the reference's own loss code
    (models.py:477-518, 547-565; metrics.py) on CPU -> (loss, [four terms], bands, dense, regs, {name: gradient})."""
    from types import SimpleNamespace

    arch, B = case["arch"], case["batch"]
    model = ref_shim.model(arch)
    ref.utils.load_state_dict_greedy(model, case["sd"])
    model.train()
    lm = ref.models.ScanRegLightningModule
    me = SimpleNamespace(beta=0.7338, gamma=0.2578, dice_score=ref.models.BinaryDice(1e-7), bce=ref.models.BinaryCrossEntropy())
    ds = ref.dataset.COPDGeneSubtyping

    def bands(labels, mapping):  # models.py:477-493 without the .cuda()
        out = []
        for c in labels:
            lo, hi = mapping[int(c)]
            if lo < 1e-7:
                out.append((0.0, 0.0))
            else:
                m, span = (lo + hi) / 2.0, (hi - lo) * 1.0 / 2.0
                out.append((m - span, m + span))
        return torch.FloatTensor(out)

    scans = case["image"].unsqueeze(1)
    lungs = case["lung_mask"].unsqueeze(1).float()
    ems = case["em_mask"].unsqueeze(1).float()
    cle, pse = case["cls_label"], case["pse_label"]
    cle_b, pse_b = bands(cle, ds.cle_ratio_map), bands(pse, ds.pse_ratio_map)
    dense, regs = model(scans, lungs)
    loss_cle = lm._interval_regression_loss(me, regs[0], cle_b, case["cle_weights"])
    loss_pse = lm._interval_regression_loss(me, regs[1], pse_b, case["pse_weights"])
    binary = torch.logical_or(cle > 0, pse > 0).long()
    seg_labels = torch.nn.functional.interpolate(ems * binary.float().view(B, 1, 1, 1, 1), dense[0].shape[-3:],
                                                 mode="nearest").detach()
    lung_labels = torch.nn.functional.interpolate(lungs, size=dense[0].shape[-3:], mode="nearest")
    mul_loss, seg_loss = lm._segmentation_loss(me, dense[0], dense[1], seg_labels, lung_labels)
    loss = loss_cle + loss_pse + 2.0 * mul_loss + seg_loss
    loss.backward()
    grads = {n: p.grad for n, p in model.named_parameters()}
    parts = [float(v.detach()) for v in (loss_cle, loss_pse, mul_loss, seg_loss)]
    return loss.detach(), parts, (cle_b, pse_b), [d.detach() for d in dense], [r.detach() for r in regs], grads


def gen_train_step(ref):
    from oracle import training_oracle as T

    case = T.train_case()
    arch, B = case["arch"], case["batch"]
    loss, parts, (cle_b, pse_b), dense, regs, grads = reference_train_step(ref, case)
    small = {n: g.clone() for n, g in grads.items() if g.numel() <= 4096}
    fix = {
        "arch": arch, "dims": case["dims"], "batch": B, "weight_seed": case["weight_seed"],
        "weight_checksum": synthetic.state_dict_checksum(case["sd"]),
        "loss": float(loss), "parts": parts,
        "cle_bands": cle_b, "pse_bands": pse_b,
        "dense_outs": [d.clone() for d in dense], "reg_outs": [r.clone() for r in regs],
        "grad_summary": T.grad_summary(grads), "small_grads": small,
    }
    torch.save(fix, os.path.join(GOLDEN, "train_step_med3ddram18.pt"))
    print("train_step loss", fix["loss"], fix["parts"], "params", len(grads))


def gen_transforms(ref):
    from argparse import Namespace

    scan_dims, target = (44, 52, 60), (32, 40, 48)
    ct, lobes = synthetic.make_volume(3, scan_dims)
    sample = P.lung_crop_sample(ct.numpy(), lobes.numpy(), spacing=(1.0, 1.0, 1.0), crop_border=5, uid="s3")
    # utils.find_crops itself cannot run here: scipy 1.18's find_objects rejects the bool array that
    # `mask > 0` (utils.py:54) produces, so the crop arithmetic is pinned through scipy directly.
    from scipy import ndimage
    obj = ndimage.find_objects((lobes.numpy() > 0).astype(np.int32))[0]
    ref_crop = tuple(slice(max(0, o.start - 5), min(n, o.stop + 5)) for o, n in zip(obj, scan_dims))
    dm = ref.models.SubtypeDataModule(Namespace(target_size=target))
    tf = dm._make_transforms(ref.models.TEST_PHASE)
    out = tf({k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in sample.items()})
    fix = {
        "scan_index": 3, "scan_dims": scan_dims, "target_size": target,
        "ref_crop": [[s.start, s.stop] for s in ref_crop],
        "image": out["image"], "original_image": out["original_image"],
        "lung_mask": out["lung_mask"], "ess_mask": out["ess_mask"],
        "crop_slice": out["crop_slice"], "original_size": out["original_size"],
    }
    torch.save(fix, os.path.join(GOLDEN, "transforms.pt"))
    print("transforms", tuple(out["image"].shape), out["image"].dtype, out["lung_mask"].dtype,
          float(out["image"].mean()), int(out["ess_mask"].sum()))


def gen_index_luts():
    """ATen's index rules the kernels must reproduce bit-exactly (SURVEY H7)."""
    import torch.nn.functional as F

    cases = {"nearest": {}, "slice": {}, "linear_ac": {}}
    for n_in, n_out in [(40, 32), (32, 40), (128, 64), (100, 37), (37, 100), (288, 144), (57, 224), (224, 57), (7, 3)]:
        src = torch.arange(n_in, dtype=torch.float32).view(1, 1, n_in)
        cases["nearest"][f"{n_in}->{n_out}"] = F.interpolate(src, size=n_out, mode="nearest").long().flatten().tolist()
        cases["slice"][f"{n_in}->{n_out}"] = torch.linspace(0, n_in - 1, n_out).long().tolist()
    with open(os.path.join(GOLDEN, "index_luts.json"), "w") as f:
        json.dump(cases, f)
    print("index_luts.json")


def gen_labels(ref):
    ratios = [0.0, 0.0099, 0.01, 0.0100001, 0.03, 0.049999, 0.05, 0.0999, 0.1, 0.15, 0.2, 0.25, 0.2999, 0.3, 0.7, 1.0]
    from argparse import Namespace

    with ref_shim.reference_cwd():
        module = ref.models.ScanRegLightningModule(Namespace(model_arch="med3ddram18"))
    cm, pm = ref.dataset.COPDGeneSubtyping.cle_ratio_map, ref.dataset.COPDGeneSubtyping.pse_ratio_map
    t = torch.tensor(ratios, dtype=torch.float32)
    out = {"ratios": ratios, "cle": module._ratio_to_label(t, cm).tolist(), "pse": module._ratio_to_label(t, pm).tolist(),
           "cle_map": {str(k): list(v) for k, v in cm.items()}, "pse_map": {str(k): list(v) for k, v in pm.items()}}
    with open(os.path.join(GOLDEN, "labels.json"), "w") as f:
        json.dump(out, f)
    print("labels.json", out["cle"], out["pse"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="")
    args = ap.parse_args()
    os.makedirs(GOLDEN, exist_ok=True)
    torch.manual_seed(0)
    ref = ref_shim.load()
    steps = {"layouts": gen_layouts, "forward": gen_forward, "predict": gen_predict_step,
             "transforms": gen_transforms, "labels": gen_labels, "train": gen_train_step, "refinit": gen_reference_init}
    for name, fn in steps.items():
        if not args.only or name in args.only.split(","):
            fn(ref)
    if not args.only or "luts" in args.only:
        gen_index_luts()


if __name__ == "__main__":
    main()
