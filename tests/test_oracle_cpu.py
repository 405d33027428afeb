"""Pins the CPU oracle (oracle/*.py) against golden vectors produced by the unmodified reference
(oracle/make_golden.py) and — where DRAM_REFERENCE_DIR names an upstream checkout — against the live reference.
No GPU needed."""
import glob
import json
import os

import numpy as np
import pytest
import torch

from oracle import med3d_oracle as M
from oracle import pipeline_oracle as P
from oracle import ref_shim, synthetic

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FORWARD_FIXTURES = sorted(glob.glob(os.path.join(GOLDEN, "forward_*.pt")))
REF_SKIP = "needs DRAM_REFERENCE_DIR: a checkout of the upstream project"


@pytest.fixture(autouse=True)
def _eight_cpu_threads():
    """The goldens were computed multi-threaded.  With 4 threads or fewer ATen's CPU kernels sum in another order, and
    that moves the saturating reference-init maps and the gradient of a bias that feeds train-mode BatchNorm (zero up
    to rounding) past the tolerances.  So the thread count is fixed here, not left to the host or an earlier test."""
    before = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(before)


def test_state_layout_matches_reference_modules():
    with open(os.path.join(GOLDEN, "state_layouts.json")) as f:
        layouts = json.load(f)
    assert set(layouts) == set(M.ARCHS)
    for arch, info in layouts.items():
        mine = M.state_layout(arch)
        assert [k for k, _, _ in mine] == [k for k, _, _ in info["keys"]], arch
        assert [list(s) for _, s, _ in mine] == [s for _, s, _ in info["keys"]], arch
        n_params = sum(int(np.prod(s)) for k, s, kind in mine if kind in ("conv_w", "conv_b", "bn_w", "bn_b"))
        assert n_params == info["params"], arch
    assert len(layouts["med3ddram18"]["keys"]) == 141 and len(layouts["med3ddram"]["keys"]) == 237
    assert len(layouts["med3ddram50"]["keys"]) == 333


@pytest.mark.parametrize("path", FORWARD_FIXTURES, ids=[os.path.basename(p)[:-3] for p in FORWARD_FIXTURES])
def test_forward_oracle_matches_reference_golden(path):
    fix = torch.load(path)
    arch, dims, batch = fix["arch"], tuple(fix["dims"]), fix["batch"]
    sd = synthetic.make_state_dict(arch, seed=fix["weight_seed"], calib_dims=dims)
    assert abs(synthetic.state_dict_checksum(sd) - fix["weight_checksum"]) <= 1e-6 * abs(fix["weight_checksum"]), \
        "synthetic weights drifted from the ones the golden vectors were made with"
    xs, ls, _ = zip(*[synthetic.make_network_input(i, dims) for i in range(batch)])
    x = torch.stack(xs).unsqueeze(1)
    lungs = torch.stack(ls).unsqueeze(1).float() if fix["with_lungs"] else None
    dense, scores = M.forward(sd, arch, x, lungs)
    for got, ref in zip(dense, fix["dense_outs"]):
        assert got.shape == ref.shape
        assert (got - ref).abs().max().item() <= 2e-5 * max(1.0, ref.abs().max().item())
    for got, ref in zip(scores, fix["scores"]):
        assert torch.allclose(got, ref, rtol=1e-4, atol=1e-5)
    if M.ARCHS[arch][2] == "cls":
        for got, ref in zip(scores, fix["scores"]):
            assert torch.equal(got.argmax(-1), ref.argmax(-1))


REFINIT_FIXTURES = sorted(glob.glob(os.path.join(GOLDEN, "refinit_*.pt")))


@pytest.mark.parametrize("path", REFINIT_FIXTURES, ids=[os.path.basename(p)[:-3] for p in REFINIT_FIXTURES])
def test_reference_init_fixture_is_reproducible_and_oracle_matches(path):
    """The reference's OWN initialisation (med3d.py:334-339) under a fixed seed: the drop-in module draws the very
    same weights (so the GPU test needs only the seed), and the oracle reproduces the reference's outputs on them —
    including the large, saturating logits this initialisation produces."""
    import dram_b200  # noqa: F401
    from dram_b200.utils import get_model_by_name

    fix = torch.load(path)
    arch, dims = fix["arch"], tuple(fix["dims"])
    torch.manual_seed(fix["init_seed"])
    sd = get_model_by_name(arch).state_dict()
    assert abs(synthetic.state_dict_checksum(sd) - fix["weight_checksum"]) <= 1e-9 * abs(fix["weight_checksum"]), \
        "dram_b200.med3d no longer draws the reference's random-init weights from the same seed"
    x, lung, _ = synthetic.make_network_input(0, dims)
    dense, scores = M.forward(sd, arch, x[None, None], lung[None, None].float())
    for got, ref in zip(dense, fix["dense_outs"]):
        assert (got - ref).abs().max().item() <= 2e-5 * max(1.0, ref.abs().max().item())
    for got, ref in zip(scores, fix["scores"]):
        assert torch.allclose(got, ref, rtol=1e-4, atol=1e-5)
    assert fix["max_conv_output"] < 65504.0  # this initialisation stays inside the fp16 range (by a factor > 100)


def test_predict_step_oracle_matches_reference_golden():
    fix = torch.load(os.path.join(GOLDEN, "predict_step_med3ddram18.pt"))
    dims, batch = tuple(fix["dims"]), fix["batch"]
    sd = synthetic.make_state_dict(fix["arch"], seed=fix["weight_seed"], calib_dims=dims)
    xs, ls, es = zip(*[synthetic.make_network_input(i, dims) for i in range(batch)])
    out = P.predict_step(sd, fix["arch"], {"image": torch.stack(xs), "lung_mask": torch.stack(ls).bool(),
                                           "ess_mask": torch.stack(es).bool()})
    assert list(out.keys()) == fix["keys"]  # 7 keys, reference spelling (`precentages`)
    for k in ("cle_dense_outs", "pse_dense_outs"):
        assert (out[k] - fix[k]).abs().max().item() < 2e-5
        assert torch.equal(out[k] == 0, fix[k] == 0)
    for k in ("cle_precentages", "pse_precentages"):
        assert torch.allclose(out[k], fix[k], rtol=1e-4)
    cle = [P.ratio_to_label(r.item(), P.CLE_RATIO_MAP) for r in out["cle_precentages"]]
    pse = [P.ratio_to_label(r.item(), P.PSE_RATIO_MAP) for r in out["pse_precentages"]]
    assert cle == fix["cle_labels"].tolist() and pse == fix["pse_labels"].tolist()


def test_transforms_oracle_matches_reference_golden():
    fix = torch.load(os.path.join(GOLDEN, "transforms.pt"))
    ct, lobes = synthetic.make_volume(fix["scan_index"], tuple(fix["scan_dims"]))
    sample = P.lung_crop_sample(ct.numpy(), lobes.numpy(), crop_border=5, uid="s3")
    assert sample["crop_slice"].tolist() == fix["ref_crop"]
    out = P.inference_transform(sample, tuple(fix["target_size"]))
    assert torch.equal(out["lung_mask"], fix["lung_mask"]) and out["lung_mask"].dtype == torch.bool
    assert torch.equal(out["ess_mask"], fix["ess_mask"])
    assert (out["image"] - fix["image"]).abs().max().item() < 1e-6
    assert (out["original_image"] - fix["original_image"]).abs().max().item() < 1e-6
    assert out["image"].dtype == torch.float32
    assert torch.equal(torch.as_tensor(out["crop_slice"]), torch.as_tensor(fix["crop_slice"]))


def test_labels_match_reference_golden():
    with open(os.path.join(GOLDEN, "labels.json")) as f:
        fix = json.load(f)
    ratios = torch.tensor(fix["ratios"], dtype=torch.float32)
    assert [P.ratio_to_label(r.item(), P.CLE_RATIO_MAP) for r in ratios] == fix["cle"]
    assert [P.ratio_to_label(r.item(), P.PSE_RATIO_MAP) for r in ratios] == fix["pse"]
    assert {str(k): list(v) for k, v in P.CLE_RATIO_MAP.items()} == fix["cle_map"]
    assert {str(k): list(v) for k, v in P.PSE_RATIO_MAP.items()} == fix["pse_map"]
    with pytest.raises(IndexError):
        P.ratio_to_label(1.5, P.CLE_RATIO_MAP)


def test_slice_pick_matches_golden():
    with open(os.path.join(GOLDEN, "index_luts.json")) as f:
        fix = json.load(f)
    for key, ref in fix["slice"].items():
        a, b = (int(v) for v in key.split("->"))
        assert P.slice_indices(a, b).tolist() == ref


def test_conv_flops_match_survey():
    # SURVEY.md §8d / Appendix A: algorithmic conv FLOPs per volume
    assert abs(M.conv_flops("med3ddram", (256, 256, 256)) / 1e12 - 6.746) < 2e-3
    assert abs(M.conv_flops("med3ddram18", (256, 256, 256)) / 1e12 - 4.658) < 2e-3
    assert abs(M.conv_flops("med3d18", (128, 128, 128)) / 1e12 - 0.582) < 1e-3
    assert abs(M.conv_flops("med3ddram50", (400, 512, 512)) / 1e12 - 43.164) < 2e-2


def test_synthetic_volume_statistics():
    ct, lobes = synthetic.make_volume(0, (48, 48, 48))
    assert ct.dtype == torch.int16 and lobes.dtype == torch.uint8
    assert set(lobes.unique().tolist()) == {0, 1, 2, 3, 4, 5}
    lung = lobes > 0
    assert 0.18 < lung.float().mean().item() < 0.30
    ess = (ct < -910) & lung
    assert 0.15 < ess.sum().item() / lung.sum().item() < 0.6
    ct2, _ = synthetic.make_volume(0, (48, 48, 48))
    assert torch.equal(ct, ct2)


LIVE_CASES = [
    # arch, (D, H, W), batch, with lobe mask
    ("med3ddram18", (16, 24, 32), 1, True),
    ("med3ddram", (24, 16, 40), 2, True),      # ResNet-34, batch 2
    ("med3ddram50", (16, 16, 24), 1, True),    # bottleneck blocks, shortcut A on four stages
    ("med3ddram18", (16, 16, 16), 2, False),   # lungs=None: the plain mean (med3d.py:383-384, quirk Q3)
    ("med3d18", (16, 24, 16), 1, False),       # classification heads, global average pool
    ("med3d", (16, 16, 24), 2, False),
    ("med3d50", (16, 16, 16), 1, False),
]


@pytest.mark.skipif(not ref_shim.available(), reason=REF_SKIP)
@pytest.mark.parametrize("arch,dims,batch,with_mask", LIVE_CASES)
def test_oracle_against_live_reference(arch, dims, batch, with_mask):
    """The oracle's forward against the unmodified reference module executed here (through oracle/ref_shim.py) on the
    same seeded weights and inputs: bit-identical dense maps and scores for all six architectures, ragged sizes,
    batches of two and the lungs=None path.  (Only runs with DRAM_REFERENCE_DIR set; these cases have no golden
    vectors, the forward goldens above cover other shapes to 2e-5.)"""
    sd = synthetic.make_state_dict(arch, seed=3, calib_dims=dims)
    ref = ref_shim.model(arch)
    ref.load_state_dict(sd)
    ref.eval()
    xs, lungs = zip(*[synthetic.make_network_input(5 + i, dims)[:2] for i in range(batch)])
    x = torch.stack(xs)[:, None]
    lung = torch.stack(lungs)[:, None].float() if with_mask else None
    with torch.no_grad():
        d_ref, r_ref = ref(x.clone(), None if lung is None else lung.clone())
    d_or, r_or = M.forward(sd, arch, x, lung)
    assert len(d_ref) == len(d_or) == 2 and len(r_ref) == len(r_or) == 2
    for a, b in zip(d_ref, d_or):
        assert torch.equal(a, b)
    for a, b in zip(r_ref, r_or):
        assert torch.equal(a, b)


@pytest.mark.skipif(not ref_shim.available(), reason=REF_SKIP)
@pytest.mark.parametrize("arch,dims,batch", [("med3ddram", (16, 24, 32), 3), ("med3ddram50", (16, 16, 24), 1),
                                              ("med3ddram18", (24, 16, 16), 2)])
def test_predict_step_oracle_against_live_reference(arch, dims, batch):
    """`ScanRegLightningModule.predict_step` of the unmodified reference (models.py:430-450, weights loaded the
    processor.py:85-87 way) against the oracle: dRAM maps, percentages with the batch-wide denominator (quirk Q1),
    key order and spelling, labels."""
    from argparse import Namespace

    ref = ref_shim.load()
    sd = synthetic.make_state_dict(arch, seed=4, calib_dims=dims)
    with ref_shim.reference_cwd():
        module = ref.models.ScanRegLightningModule(Namespace(model_arch=arch))
    ref.utils.load_state_dict_greedy(module, {"model." + k: v for k, v in sd.items()})
    module.eval()
    xs, ls, es = zip(*[synthetic.make_network_input(20 + i, dims) for i in range(batch)])
    b = {"image": torch.stack(xs), "lung_mask": torch.stack(ls).bool(), "ess_mask": torch.stack(es).bool(),
         "crop_slice": torch.tensor([[[0, d] for d in dims]] * batch), "original_size": torch.tensor([dims] * batch),
         "uid": [f"v{i}" for i in range(batch)]}
    with torch.no_grad():
        want = module.predict_step({k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in b.items()}, 0)
    got = P.predict_step(sd, arch, {k: b[k] for k in ("image", "lung_mask", "ess_mask")})
    assert list(got.keys()) == list(want.keys())
    for k in ("cle_dense_outs", "pse_dense_outs"):
        assert (got[k] - want[k]).abs().max().item() < 2e-5 and torch.equal(got[k] == 0, want[k] == 0)
    for k in ("cle_precentages", "pse_precentages"):
        assert torch.allclose(got[k], want[k], rtol=1e-4)
    cle_map, pse_map = ref.dataset.COPDGeneSubtyping.cle_ratio_map, ref.dataset.COPDGeneSubtyping.pse_ratio_map
    assert [P.ratio_to_label(r.item(), P.CLE_RATIO_MAP) for r in got["cle_precentages"]] == \
        module._ratio_to_label(want["cle_precentages"], cle_map).tolist()
    assert [P.ratio_to_label(r.item(), P.PSE_RATIO_MAP) for r in got["pse_precentages"]] == \
        module._ratio_to_label(want["pse_precentages"], pse_map).tolist()


@pytest.mark.skipif(not ref_shim.available(), reason=REF_SKIP)
@pytest.mark.parametrize("scan_dims,target", [((40, 48, 56), (24, 32, 40)), ((30, 36, 44), (32, 48, 40)),
                                               ((33, 47, 51), (16, 47, 64))])
def test_transforms_oracle_against_live_reference(scan_dims, target):
    """The reference's own transform chain (`SubtypeDataModule._make_transforms(TEST)`, models.py:55-63: window,
    standardise, in-plane resize + slice pick; down- and up-sampling targets, odd sizes) against the oracle: masks
    bit-exact, images to 1e-6."""
    from argparse import Namespace

    ref = ref_shim.load()
    ct, lobes = synthetic.make_volume(7, scan_dims)
    sample = P.lung_crop_sample(ct.numpy(), lobes.numpy(), spacing=(1.0, 1.0, 1.0), crop_border=5, uid="s7")
    tf = ref.models.SubtypeDataModule(Namespace(target_size=target))._make_transforms(ref.models.TEST_PHASE)
    want = tf({k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in sample.items()})
    got = P.inference_transform(sample, target)
    assert tuple(got["image"].shape) == tuple(want["image"].shape) == tuple(target)
    assert torch.equal(got["lung_mask"], want["lung_mask"]) and torch.equal(got["ess_mask"], want["ess_mask"])
    assert (got["image"] - want["image"]).abs().max().item() < 1e-6
    assert (got["original_image"] - want["original_image"]).abs().max().item() < 1e-6


# ------------------------------------------------------------------------------------------
# training step (SURVEY §8f f4): the oracle against the unmodified reference's loss and gradients
# ------------------------------------------------------------------------------------------
def test_training_oracle_matches_reference_golden():
    from oracle import training_oracle as T

    fix = torch.load(os.path.join(GOLDEN, "train_step_med3ddram18.pt"), weights_only=False)
    case = T.train_case()
    assert (case["arch"], tuple(case["dims"]), case["batch"]) == (fix["arch"], tuple(fix["dims"]), fix["batch"])
    assert abs(synthetic.state_dict_checksum(case["sd"]) - fix["weight_checksum"]) <= 1e-6 * abs(fix["weight_checksum"])
    loss, grads, dense, regs = T.train_step_grads(
        case["sd"], case["arch"], case["image"], case["lung_mask"], case["em_mask"], case["cls_label"],
        case["pse_label"], fix["cle_bands"], fix["pse_bands"], case["cle_weights"], case["pse_weights"])
    assert abs(float(loss) - fix["loss"]) <= 1e-5 * abs(fix["loss"])
    for a, b in zip(dense + regs, fix["dense_outs"] + fix["reg_outs"]):
        assert torch.allclose(a, b, rtol=1e-4, atol=1e-6)
    assert set(grads) == set(fix["grad_summary"])
    summ = T.grad_summary(grads)
    scale = max(v[0] for v in fix["grad_summary"].values())
    for name, (norm, proj) in fix["grad_summary"].items():
        assert abs(summ[name][0] - norm) <= 2e-3 * norm + 1e-6 * scale, (name, summ[name], norm)
        assert abs(summ[name][1] - proj) <= 2e-3 * norm + 1e-6 * scale, (name, summ[name], proj)
    for name, g in fix["small_grads"].items():
        assert torch.allclose(grads[name], g, rtol=2e-3, atol=2e-3 * float(g.abs().max()) + 1e-9), name


def test_label_bands_follow_the_ratio_maps():
    from oracle import training_oracle as T

    fix = torch.load(os.path.join(GOLDEN, "train_step_med3ddram18.pt"), weights_only=False)
    labels = json.load(open(os.path.join(GOLDEN, "labels.json")))
    case = T.train_case()
    for key, lab, want in (("cle_map", case["cls_label"], fix["cle_bands"]), ("pse_map", case["pse_label"], fix["pse_bands"])):
        mapping = {int(k): tuple(v) for k, v in labels[key].items()}
        assert torch.equal(T.label_bands(lab, mapping), want)


@pytest.mark.skipif(not ref_shim.available(), reason=REF_SKIP)
@pytest.mark.parametrize("arch,dims,batch", [("med3ddram50", (16, 16, 16), 2), ("med3ddram", (16, 16, 24), 1)])
def test_training_oracle_against_live_reference(arch, dims, batch):
    """The training oracle (train-mode BatchNorm, detached shortcut A, the reference's loss) against one training step
    of the unmodified reference network with the reference's own loss code, executed here: loss to 1e-5, every
    parameter gradient to 2e-3 of the largest gradient — on the bottleneck network (shortcut A on four stages) and on
    ResNet-34, beyond the committed med3ddram18 golden step."""
    from oracle import make_golden
    from oracle import training_oracle as T

    case = T.train_case(batch=batch, dims=dims, arch=arch, seed=6)
    loss_ref, parts, (cle_b, pse_b), dense_ref, regs_ref, grads_ref = make_golden.reference_train_step(ref_shim.load(), case)
    loss, grads, dense, regs = T.train_step_grads(case["sd"], arch, case["image"], case["lung_mask"], case["em_mask"],
                                                  case["cls_label"], case["pse_label"], cle_b, pse_b,
                                                  case["cle_weights"], case["pse_weights"])
    assert abs(float(loss) - float(loss_ref)) <= 1e-5 * abs(float(loss_ref)), (float(loss), float(loss_ref), parts)
    for a, b in zip(dense, dense_ref):
        assert (a - b).abs().max().item() < 2e-5
    for a, b in zip(regs, regs_ref):
        assert torch.allclose(a, b, rtol=1e-5)
    top = max(float(g.abs().max()) for g in grads_ref.values() if g is not None)
    assert set(grads) == {n for n, g in grads_ref.items() if g is not None}
    for name, g in grads.items():
        err = float((g - grads_ref[name]).abs().max())
        assert err <= 2e-3 * top, (name, err, top)


@pytest.mark.parametrize("dims,mdims", [((8, 6, 10), (16, 12, 20)), ((5, 7, 9), (13, 14, 30))])
def test_closed_form_loss_gradient_equals_autograd(dims, mdims):
    """K11's derivation (training_oracle.loss_closed_form: seven sums per scan, scalar step, closed-form gradient) against
    autograd of the restated reference loss `total_loss` (models.py:547-565), including map sums above 1 and values at
    the 1e-6 clamp of the cross entropy where ATen's clamp stops the gradient."""
    import torch.nn.functional as F

    from oracle import training_oracle as T

    B = 2
    g = torch.Generator().manual_seed(dims[0])
    d0, d1 = torch.rand((B, 1) + dims, generator=g) * 0.8, torch.rand((B, 1) + dims, generator=g) * 0.8
    d0.view(-1)[:5], d1.view(-1)[:5] = 3e-7, 2e-7
    lungs = (torch.rand((B, 1) + mdims, generator=g) > 0.5).float()
    ems = (torch.rand((B, 1) + mdims, generator=g) > 0.7).float()
    cl, pl = torch.tensor([3, 0]), torch.tensor([1, 0])
    cb, pb = torch.tensor([[0.1, 0.2], [0.0, 0.0]]), torch.tensor([[0.01, 0.05], [0.0, 0.0]])
    cw, pw = torch.tensor([1.0, 2.0]), torch.tensor([1.5, 0.5])
    a, b = d0.clone().requires_grad_(True), d1.clone().requires_grad_(True)
    lm = F.interpolate(lungs, dims, mode="nearest")
    regs = [(x * lm).view(B, -1).sum(-1) / lm.view(B, -1).sum(-1) for x in (a, b)]
    loss = T.total_loss([a, b], regs, lungs, ems, cl, pl, cb, pb, cw, pw)
    loss.backward()
    got, grads, got_regs = T.loss_closed_form([d0, d1], lungs, ems, cl, pl, cb, pb, cw, pw)
    assert abs(float(got) - float(loss.detach())) <= 1e-5 * abs(float(loss.detach()))
    for k, ref in enumerate((a.grad, b.grad)):
        assert float((grads[k] - ref).abs().max()) <= 1e-5 * float(ref.abs().max()), k
        assert torch.allclose(got_regs[k], regs[k].detach(), rtol=1e-6)
