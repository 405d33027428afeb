"""Per-lobe lesion percentages on the GPU: the K7l reduction and the label resize against the fp64 oracle, the
invariants against K7, reproducibility, guard bands, the custom op, predict_step / predict_step_from_hu with labels,
the processor CLI with --lobe_scores, and C3 at full size."""
import json
import os
from argparse import Namespace

import numpy as np
import pytest
import torch

from oracle import lobe_oracle as L
from oracle import pipeline_oracle as P
from oracle import synthetic

pytestmark = pytest.mark.gpu

SHAPES = [(1, 64, 64, 64), (2, 63, 67, 250), (3, 16, 16, 17), (1, 128, 224, 288)]
CASES = ["lobes", "random", "one_sample", "zero_sample"]


def _inputs(shape, case, seed=0):
    """(cle, pse fp32 [B,1,D,H,W], ess uint8, labels uint8 [B,D,H,W]) on the CPU.  The maps are NOT zero outside ess:
    the reduction must read them only where ess is set."""
    B, D, H, W = shape
    g = torch.Generator().manual_seed(seed)
    if case == "random":
        palette = torch.tensor([0, 1, 2, 7, 200, 255], dtype=torch.uint8)
        labels = palette[torch.randint(0, len(palette), (B, D, H, W), generator=g)]
    else:
        labels = torch.stack([synthetic.make_volume(50 + b, (D, H, W))[1] for b in range(B)])
    if case == "one_sample":
        labels[0, : D // 2, : H // 3] = 9            # label 9 exists in sample 0 only
    if case == "zero_sample":
        labels[-1] = 0
    ess = (torch.rand((B, D, H, W), generator=g) < 0.05).to(torch.uint8)
    cle = torch.rand((B, 1, D, H, W), generator=g)
    pse = torch.rand((B, 1, D, H, W), generator=g) * 0.1
    return cle, pse, ess, labels


def _check_against_oracle(pct, voxels, cle, pse, ess, labels, rel=1e-6):
    ref_pct, ref_vox, _ = L.lobe_scores(cle, pse, ess, labels)
    assert voxels.dtype == torch.int64 and pct.dtype == torch.float32
    assert torch.equal(voxels.cpu(), ref_vox), "voxel counts differ"
    got = pct.cpu().double()
    assert torch.equal(torch.isnan(got), torch.isnan(ref_pct)), "NaN pattern differs"
    fin = ~torch.isnan(ref_pct)
    err = ((got[fin] - ref_pct[fin]).abs() / ref_pct[fin].abs().clamp_min(1e-30)).max().item()
    assert err <= rel, err
    return ref_pct, ref_vox


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("shape", SHAPES)
def test_lobe_scores_match_oracle_and_repeat_bit_for_bit(cuda, lib, shape, case):
    from dram_b200 import ops

    cle, pse, ess, labels = _inputs(shape, case)
    dev = [t.to(cuda) for t in (cle, pse, ess, labels)]
    pct, voxels = ops.lobe_scores(*dev)
    _, ref_vox = _check_against_oracle(pct, voxels, cle, pse, ess, labels)
    if case == "zero_sample":
        assert ref_vox[-1, 0] == ref_vox[-1].sum() and torch.isnan(pct[:, -1, 1:].cpu()).all()
    if case == "one_sample" and shape[0] > 1:
        assert voxels[0, 9].item() > 0 and (voxels[1:, 9] == 0).all()
    pct2, voxels2 = ops.lobe_scores(*dev)
    assert torch.equal(pct.view(torch.int32), pct2.view(torch.int32)) and torch.equal(voxels, voxels2)
    # bool ess takes the same path
    pct3, _ = ops.lobe_scores(dev[0], dev[1], dev[2].bool(), dev[3])
    assert torch.equal(pct.view(torch.int32), pct3.view(torch.int32))


@pytest.mark.parametrize("shape", [(2, 40, 48, 56), (3, 16, 16, 17), (1, 128, 224, 288)])
def test_lobe_scores_invariants_against_k7(cuda, lib, shape):
    """With lung == (labels > 0): the label counts >= 1 add up to K7's lung count, and the count-weighted per-label
    percentages add up to K7's per-sample percentage (ess lies inside the lung)."""
    from dram_b200 import ops

    B, D, H, W = shape
    labels = torch.stack([synthetic.make_volume(60 + b, (D, H, W))[1] for b in range(B)])
    g = torch.Generator().manual_seed(5)
    lung = (labels > 0).to(torch.uint8)
    ess = ((torch.rand((B, D, H, W), generator=g) < 0.1) & (lung > 0)).to(torch.uint8)
    dense = [torch.rand((B, 1, D // 2, H // 2, W // 2), generator=g).to(cuda) for _ in range(2)]
    cle, pse, k7 = ops.dram_upsample_mask(dense[0], dense[1], ess.to(cuda), lung.to(cuda), (D, H, W),
                                          per_sample_denominator=True)
    pct, voxels = ops.lobe_scores(cle, pse, ess.to(cuda), labels.to(cuda))
    lung_count = lung.reshape(B, -1).sum(-1)
    assert torch.equal(voxels[:, 1:].sum(-1).cpu(), lung_count)
    vox = voxels.cpu().double()
    for m in range(2):
        num = torch.nan_to_num(pct[m].cpu().double()) * vox
        recon = num.sum(-1) / vox[:, 1:].sum(-1)
        rel = ((recon - k7[m].cpu().double()).abs() / k7[m].cpu().double()).max().item()
        assert rel <= 1e-6, (m, rel)


@pytest.mark.parametrize("src,size", [((40, 60, 70), (32, 48, 56)), ((20, 30, 40), (31, 63, 127)),
                                      ((64, 64, 64), (63, 63, 63)), ((17, 33, 9), (15, 16, 23))])
def test_resize_labels_bit_exact(cuda, lib, src, size):
    from dram_b200 import ops

    g = torch.Generator().manual_seed(7)
    palette = torch.tensor([0, 1, 3, 5, 200, 255], dtype=torch.uint8)
    lab = palette[torch.randint(0, len(palette), src, generator=g)]
    got = ops.resize_labels(lab.to(cuda), size)
    assert torch.equal(got.cpu(), L.interpolate_labels(lab, size))
    assert torch.equal(got > 0, ops.resize_mask((lab > 0).to(torch.uint8).to(cuda), size) > 0)


def _module(arch, sd, cuda):
    from dram_b200.models import ScanRegLightningModule

    module = ScanRegLightningModule(Namespace(model_arch=arch))
    module.model.load_state_dict(sd)
    return module.to(cuda).eval()


def test_predict_step_with_lobe_labels(cuda, lib):
    from dram_b200 import ops

    arch, dims = "med3ddram18", (32, 48, 40)
    sd = synthetic.make_state_dict(arch, seed=6, calib_dims=dims)
    module = _module(arch, sd, cuda)
    vols = [synthetic.make_volume(20 + i, dims) for i in range(2)]
    hu = torch.stack([v[0] for v in vols]).to(cuda)
    labels = torch.stack([v[1] for v in vols]).to(cuda)
    lung = labels > 0
    ess = (hu < -910) & lung
    image = torch.stack([P.standardize(P.intensity_window(h)) for h in hu.cpu()]).to(cuda)
    batch = {"image": image, "lung_mask": lung, "ess_mask": ess, "crop_slice": torch.zeros(2, 3, 2), "uid": ["a", "b"],
             "original_size": torch.tensor([dims] * 2)}
    plain = module.predict_step(batch, 0)
    with_lab = module.predict_step(dict(batch, lobe_labels=labels), 0)
    plain_hu = module.predict_step_from_hu(hu, lung, ess)
    with_hu = module.predict_step_from_hu(hu, lung, ess, lobe_labels=labels)
    new = ["lobe_voxels", "cle_lobe_percentages", "pse_lobe_percentages"]
    for a, b in ((plain, with_lab), (plain_hu, with_hu)):
        assert list(b.keys()) == list(a.keys()) + new
        for k, v in a.items():
            if isinstance(v, torch.Tensor):
                assert torch.equal(v, b[k]), k
            else:
                assert v == b[k], k
        pct, vox = ops.lobe_scores(b["cle_dense_outs"], b["pse_dense_outs"], ess.to(torch.uint8), labels)
        assert torch.equal(b["lobe_voxels"], vox) and b["lobe_voxels"].shape == (2, 256)
        assert torch.equal(b["cle_lobe_percentages"].view(torch.int32), pct[0].view(torch.int32))
        assert torch.equal(b["pse_lobe_percentages"].view(torch.int32), pct[1].view(torch.int32))


def test_new_kernels_stay_inside_their_output(cuda, lib):
    """Guard bands around the outputs, inputs that start one byte off a 16-byte boundary (the byte path), ragged W."""
    from dram_b200 import ops

    PAD = 4096
    B, D, H, W = 2, 9, 13, 31
    cle, pse, ess, labels = _inputs((B, D, H, W), "random", seed=3)

    def guarded(numel, dtype):
        item = torch.empty((), dtype=dtype).element_size()
        raw = torch.full((2 * PAD + numel * item,), 0xA5, dtype=torch.uint8, device=cuda)
        return raw, raw[PAD:PAD + numel * item].view(dtype)

    def intact(raw, numel_bytes, what):
        torch.cuda.synchronize()
        assert bool((raw[:PAD] == 0xA5).all()) and bool((raw[PAD + numel_bytes:] == 0xA5).all()), what

    def offset_copy(t):  # contiguous view starting one byte after an aligned address
        raw = torch.zeros(t.numel() + 1, dtype=torch.uint8, device=cuda)
        v = raw[1:].view(t.shape)
        v.copy_(t)
        return v

    ess_u, lab_u = offset_copy(ess.to(cuda)), offset_copy(labels.to(cuda))
    assert ess_u.data_ptr() % 16 == 1
    raw_p, pct = guarded(2 * B * 256, torch.float32)
    raw_v, vox = guarded(B * 256, torch.int64)
    ops.lobe_scores(cle.to(cuda), pse.to(cuda), ess_u, lab_u, out=(pct.view(2, B, 256), vox.view(B, 256)))
    intact(raw_p, 2 * B * 256 * 4, "lobe_scores pct")
    intact(raw_v, B * 256 * 8, "lobe_scores voxels")
    _check_against_oracle(pct.view(2, B, 256), vox.view(B, 256), cle, pse, ess, labels)
    size = (7, 17, 29)
    raw_r, out = guarded(7 * 17 * 29, torch.uint8)
    ops.resize_labels(lab_u[0], size, out=out.view(size))
    intact(raw_r, 7 * 17 * 29, "resize_labels")
    assert torch.equal(out.view(size).cpu(), L.interpolate_labels(labels[0], size))


def test_lobe_scores_op_opcheck_and_graph_capture(cuda, lib):
    from dram_b200 import ops

    cle, pse, ess, labels = [t.to(cuda) for t in _inputs((2, 16, 24, 32), "lobes", seed=4)]
    pct, vox = torch.ops.dram_b200.lobe_scores(cle, pse, ess, labels)
    ref = ops.lobe_scores(cle, pse, ess, labels)
    assert torch.equal(pct.view(torch.int32), ref[0].view(torch.int32)) and torch.equal(vox, ref[1])
    # opcheck compares outputs with NaN != NaN: give every one of the 256 labels voxels in every sample
    every = (torch.arange(labels.numel(), device=cuda) % 256).to(torch.uint8).view(labels.shape)
    torch.library.opcheck(torch.ops.dram_b200.lobe_scores.default, (cle, pse, ess, every))
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gp, gv = torch.ops.dram_b200.lobe_scores(cle, pse, ess, labels)
    new = _inputs((2, 16, 24, 32), "random", seed=8)
    for dst, src in zip((cle, pse, ess, labels), new):
        dst.copy_(src.to(cuda))
    graph.replay()
    torch.cuda.synchronize()
    eager = ops.lobe_scores(cle, pse, ess, labels)
    assert torch.equal(gp.view(torch.int32), eager[0].view(torch.int32)) and torch.equal(gv, eager[1])


def _write_scans(tmp_path, scan_dims, label_dtype):
    from dram_b200 import mha_io

    scan_dir, lobe_dir = tmp_path / "ct", tmp_path / "lobes"
    scan_dir.mkdir(exist_ok=True)
    lobe_dir.mkdir(exist_ok=True)
    vols = {}
    for i in range(3):
        ct, lobes = synthetic.make_volume(40 + i, scan_dims)
        mha_io.write_mha(str(scan_dir / f"scan{i}.mha"), ct.numpy(), spacing=(1.0, 1.0, 1.0), origin=(1.0, 2.0, 3.0))
        mha_io.write_mha(str(lobe_dir / f"scan{i}.mha"), lobes.numpy().astype(label_dtype), spacing=(1.0, 1.0, 1.0),
                         origin=(1.0, 2.0, 3.0))
        vols[f"scan{i}"] = (ct, lobes)
    return scan_dir, lobe_dir, vols


def _run(argv_base, out_dir, extra=()):
    from dram_b200 import processor

    records = processor.run_testing_job(argv_base + ["--output_path", str(out_dir)] + list(extra))
    heat = {}
    for folder in ("centrilobular-emphysema-heatmap", "paraseptal-emphysema-heatmap"):
        for f in sorted(os.listdir(out_dir / "images" / folder)):
            heat[(folder, f)] = open(out_dir / "images" / folder / f, "rb").read()
    return records, heat


@pytest.mark.parametrize("workers,label_dtype", [(0, np.uint8), (2, np.uint8), (0, np.int16)])
def test_processor_lobe_scores_end_to_end(cuda, lib, tmp_path, workers, label_dtype):
    arch, scan_dims, target = "med3ddram18", (40, 48, 56), (32, 40, 48)
    scan_dir, lobe_dir, vols = _write_scans(tmp_path, scan_dims, label_dtype)
    sd = synthetic.make_state_dict(arch, seed=7, calib_dims=target, prefix="model.")
    ckpt = tmp_path / "best.ckpt"
    torch.save({"state_dict": sd}, ckpt)
    argv = ["--scan_path", str(scan_dir), "--lobe_path", str(lobe_dir), "--model_arch", arch, "--target_size",
            "32,40,48", "--batch_size", "2", "--ckpt_path", str(ckpt), "--workers", str(workers)]
    plain, heat_plain = _run(argv, tmp_path / "plain")
    got, heat_got = _run(argv, tmp_path / "lobes", ["--lobe_scores"])
    assert heat_got == heat_plain, "heat-maps changed with --lobe_scores"
    assert [{k: v for k, v in r.items() if k != "lobe_metrics"} for r in got] == plain
    on_disk = json.load(open(tmp_path / "lobes" / "results.json"))
    assert on_disk == got
    plain_sd = {k[len("model."):]: v for k, v in sd.items()}
    worst = 0.0
    for rec in got:
        ct, lobes = vols[rec["entity"]]
        cropped = P.lung_crop_sample(ct.numpy(), lobes.numpy(), crop_border=5, uid=rec["entity"])
        sample = P.inference_transform(cropped, target)
        lab = L.interpolate_labels(L.crop_labels(lobes.numpy(), cropped["crop_slice"]), target)
        ref = P.predict_step(plain_sd, arch, {k: sample[k][None] for k in ("image", "lung_mask", "ess_mask")})
        ref_pct, ref_vox, _ = L.lobe_scores(ref["cle_dense_outs"], ref["pse_dense_outs"], sample["ess_mask"][None],
                                            lab[None])
        assert torch.equal(lab > 0, sample["lung_mask"])
        want = {str(k) for k in range(1, 256) if ref_vox[0, k] > 0}
        assert set(rec["lobe_metrics"]) == want == {"1", "2", "3", "4", "5"}
        for k, m in rec["lobe_metrics"].items():
            for j, name in enumerate(("cle_lesion_percentage", "pse_lesion_percentage")):
                r = ref_pct[j, 0, int(k)].item()
                # the 1e-2 relative bar of the scores, plus the half unit of the 3-decimal formatting
                err = abs(float(m[name]) - r)
                assert err <= 1e-2 * abs(r) + 5e-4 + 1e-9, (rec["entity"], k, name, m[name], r)
                worst = max(worst, err)
    print(f"lobe_metrics vs oracle: worst abs difference {worst:.3g}")


def test_processor_lobe_scores_two_gpus_equal_one(cuda, lib, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    arch = "med3ddram18"
    scan_dir, lobe_dir, _ = _write_scans(tmp_path, (40, 48, 56), np.uint8)
    sd = synthetic.make_state_dict(arch, seed=7, calib_dims=(32, 40, 48), prefix="model.")
    torch.save({"state_dict": sd}, tmp_path / "best.ckpt")
    argv = ["--scan_path", str(scan_dir), "--lobe_path", str(lobe_dir), "--model_arch", arch, "--target_size",
            "32,40,48", "--batch_size", "1", "--ckpt_path", str(tmp_path / "best.ckpt"), "--lobe_scores"]
    one, _ = _run(argv, tmp_path / "one")
    two, _ = _run(argv, tmp_path / "two", ["--ngpus", "2"])
    assert two == one and all("lobe_metrics" in r for r in two)


def test_c3_256cube_lobe_scores_match_oracle(cuda, lib):
    """C3 (med3ddram, ResNet-34) on one 256^3 volume with the synthetic lobes 1-5: the per-lobe percentages of the
    module against the oracle's dRAM maps reduced with the oracle's lobe_scores."""
    arch, dims = "med3ddram", (256, 256, 256)
    sd = synthetic.make_state_dict(arch, seed=0, calib_dims=(64, 64, 64))
    module = _module(arch, sd, cuda)
    x, lung, ess = synthetic.make_network_input(3, dims)
    labels = synthetic.make_volume(3, dims)[1]
    batch = {"image": x[None], "lung_mask": lung[None].bool(), "ess_mask": ess[None].bool()}
    torch.set_num_threads(os.cpu_count() or 1)
    ref = P.predict_step(sd, arch, batch)
    ref_pct, ref_vox, _ = L.lobe_scores(ref["cle_dense_outs"], ref["pse_dense_outs"], ess[None], labels[None])
    got = module.predict_step(dict({k: v.to(cuda) for k, v in batch.items()}, lobe_labels=labels[None].to(cuda)), 0)
    assert torch.equal(got["lobe_voxels"].cpu(), ref_vox)
    worst = 0.0
    for j, key in enumerate(("cle_lobe_percentages", "pse_lobe_percentages")):
        g, r = got[key][0, 1:6].cpu().double(), ref_pct[j, 0, 1:6]
        rel = ((g - r).abs() / r.abs().clamp_min(1e-6)).max().item()
        print(f"C3 {key} lobes 1-5: got {g.tolist()} ref {r.tolist()} rel {rel:.3g} (bar 1e-2: headroom "
              f"{1e-2 / max(rel, 1e-12):.1f}x)")
        worst = max(worst, rel)
    assert worst <= 1e-2, worst
    module.model._engines.clear()
    torch.cuda.empty_cache()
