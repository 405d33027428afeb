"""Per-lobe lesion percentages, host side: CLI flag, record formatting and merging, the label dtype rule and the
custom op's fake kernel.  No GPU needed."""
import json
from argparse import Namespace

import numpy as np
import pytest
import torch


def test_parser_has_lobe_scores_off_by_default():
    from dram_b200 import processor

    assert processor.build_parser().parse_args([]).lobe_scores is False
    assert processor.build_parser().parse_args(["--lobe_scores"]).lobe_scores is True


def _pred_lobes():
    voxels = torch.zeros(256, dtype=torch.int64)
    cle = torch.full((256,), float("nan"))
    pse = torch.full((256,), float("nan"))
    voxels[0], cle[0], pse[0] = 1000, 0.5, 0.5       # background: never reported
    voxels[1], cle[1], pse[1] = 40, 0.12345, 0.0004
    voxels[5], cle[5], pse[5] = 7, 0.3, 0.02
    voxels[200], cle[200], pse[200] = 3, 0.0, 0.9996
    return voxels, cle, pse


def test_lobe_metrics_formatting():
    from dram_b200 import processor

    got = processor.lobe_metrics(*_pred_lobes())
    assert got == {"1": {"cle_lesion_percentage": "0.123", "pse_lesion_percentage": "0.000"},
                   "5": {"cle_lesion_percentage": "0.300", "pse_lesion_percentage": "0.020"},
                   "200": {"cle_lesion_percentage": "0.000", "pse_lesion_percentage": "1.000"}}
    assert processor.lobe_metrics(torch.zeros(256, dtype=torch.int64), torch.zeros(256), torch.zeros(256)) == {}


def test_lobe_metrics_survive_the_multi_rank_merge(tmp_path):
    from dram_b200 import processor

    lobes = processor.lobe_metrics(*_pred_lobes())
    rec = lambda uid: {"entity": uid, "error_messages": [], "lobe_metrics": lobes, "metrics": {  # noqa: E731
        "cle_severity_score": "2", "cle_lesion_percentage_per_lung": "0.070",
        "pse_severity_score": "1", "pse_lesion_percentage_per_lung": "0.020"}}
    # what the ranks of --ngpus 2 leave behind, read back the way the merge reads them
    parts = [json.loads(json.dumps([rec("b"), rec("a")])), json.loads(json.dumps([rec("c"), rec("b")]))]
    merged = processor.write_results(Namespace(output_path=str(tmp_path)), parts[0] + parts[1])
    assert [r["entity"] for r in merged] == ["a", "b", "c"]
    on_disk = json.load(open(tmp_path / "results.json"))
    assert [r["lobe_metrics"] for r in on_disk] == [lobes] * 3


def test_classification_architecture_with_lobe_scores_is_refused(tmp_path):
    from dram_b200 import processor

    argv = ["--model_arch", "med3d18", "--lobe_scores", "--scan_path", str(tmp_path), "--lobe_path", str(tmp_path),
            "--output_path", str(tmp_path / "out")]
    with pytest.raises(ValueError, match="--lobe_scores"):
        processor.run_testing_job(argv)
    assert not (tmp_path / "out").exists()
    processor.check_args(processor.build_parser().parse_args(["--model_arch", "med3d18"]))   # the flag off: fine
    processor.check_args(processor.build_parser().parse_args(["--lobe_scores"]))            # med3ddram: fine


def test_label_dtype_rule():
    from dram_b200.dataset import labels_as_u8

    u8 = np.arange(6, dtype=np.uint8).reshape(1, 2, 3)
    assert labels_as_u8(u8, "s") is u8
    i16 = np.array([[[0, 1, 5], [200, 255, 3]]], dtype=np.int16)
    got = labels_as_u8(i16, "s")
    assert got.dtype == np.uint8 and np.array_equal(got, i16.astype(np.uint8))
    assert labels_as_u8(np.array([0, 7], dtype=np.int64), "s").tolist() == [0, 7]
    for bad in (300, -1):
        arr = i16.copy()
        arr[0, 0, 0] = bad
        with pytest.raises(ValueError, match="scan_17"):
            labels_as_u8(arr, "scan_17")
    with pytest.raises(ValueError, match="scan_18"):
        labels_as_u8(np.zeros((2, 2, 2), dtype=np.float32), "scan_18")


def test_lobe_scores_fake_kernel_shapes():
    from torch._subclasses.fake_tensor import FakeTensorMode

    from dram_b200 import custom_ops  # noqa: F401

    assert "lobe_scores" in custom_ops.REGISTERED and hasattr(torch.ops.dram_b200, "lobe_scores")
    with FakeTensorMode():
        m = torch.empty((3, 1, 16, 16, 17), device="cuda")
        u8 = torch.empty((3, 16, 16, 17), dtype=torch.uint8, device="cuda")
        pct, voxels = torch.ops.dram_b200.lobe_scores(m, m, u8, u8)
        assert pct.shape == (2, 3, 256) and pct.dtype == torch.float32
        assert voxels.shape == (3, 256) and voxels.dtype == torch.int64


def test_oracle_lobe_scores_definitions():
    """The fp64 restatement the GPU tests compare against: counts, NaN for absent labels, and the invariants."""
    from oracle import lobe_oracle as L
    from oracle import pipeline_oracle as P

    g = torch.Generator().manual_seed(3)
    labels = torch.randint(0, 6, (2, 5, 6, 7), generator=g, dtype=torch.uint8)
    labels[1] = 0
    ess = (torch.rand((2, 5, 6, 7), generator=g) < 0.3) & (labels > 0)
    cle, pse = torch.rand((2, 1, 5, 6, 7), generator=g) * ess[:, None], torch.rand((2, 1, 5, 6, 7), generator=g) * ess[:, None]
    pct, voxels, sums = L.lobe_scores(cle, pse, ess, labels)
    assert voxels.dtype == torch.int64 and voxels[0, :6].sum() == 210 and voxels[1, 0] == 210
    assert torch.isnan(pct[:, 0, 6:]).all() and torch.isnan(pct[:, 1, 1:]).all()
    assert torch.allclose(sums[0].sum(-1), cle.double().reshape(2, -1).sum(-1))
    assert torch.allclose(pct[1, 0, 3], pse[0, 0][labels[0] == 3].double().sum() / (labels[0] == 3).sum())
    m = torch.arange(24, dtype=torch.uint8).reshape(2, 3, 4)
    assert torch.equal(L.interpolate_labels(m, (2, 6, 8)) > 0, P.interpolate_mask(m > 0, (2, 6, 8)))
    from oracle import synthetic

    ct, lobes = synthetic.make_volume(41, (20, 24, 28))
    sample = P.lung_crop_sample(ct.numpy(), lobes.numpy(), crop_border=2)
    cropped = L.crop_labels(lobes.numpy(), sample["crop_slice"])
    assert torch.equal(cropped > 0, torch.as_tensor(sample["lung_mask"]))
    assert set(torch.unique(cropped).tolist()) == {0, 1, 2, 3, 4, 5}
