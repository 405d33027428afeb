"""Lung and per-lobe densitometry, host side: the histogram -> measures arithmetic against the numpy oracle, the record
formatting, the CLI flag for regression and classification architectures, the multi-rank merge, the custom ops' fake
kernels and the C-ABI argument checks.  No GPU needed."""
import json
from argparse import Namespace

import numpy as np
import pytest
import torch

from oracle import densitometry_oracle as O


def _measures_via_histogram(v, spacing):
    from dram_b200 import densitometry

    labels = np.ones(v.shape, dtype=np.uint8)
    hist, sums = O.hu_histograms(v, labels, [1])
    return densitometry.metrics_from_histogram(hist[0], int(sums[0]), v.size, spacing)


@pytest.mark.parametrize("n", list(range(1, 61)) + [101, 1000, 4097])
def test_histogram_measures_equal_the_oracle_bit_for_bit(n):
    """Every n from 1 to 60 walks the virtual index (n - 1) * 0.15 over exact order statistics, fractions below and
    above one half, and ties; the values reach past both clamp bounds."""
    g = np.random.default_rng(n)
    v = g.integers(-1300, 1300, size=n).astype(np.int16)
    if n % 3 == 0:
        v = g.choice(np.array([-3024, -1024, -1000, -951, -950, -911, -910, -850, 1023, 3071], dtype=np.int16), size=n)
    spacing = (1.25, 0.7, 0.7)
    assert _measures_via_histogram(v, spacing) == O.measures(v, spacing)


def test_perc15_at_order_statistic_boundaries_and_clamps():
    from dram_b200 import densitometry

    spacing = (1.0, 1.0, 1.0)
    for n in (21, 41, 61, 81):                      # (n - 1) * 0.15 lands on (or next to) an integer
        v = np.arange(n, dtype=np.int16) * 7 - 900
        assert _measures_via_histogram(v, spacing)["perc15_hu"] == float(np.percentile(v, 15))
    one = np.array([-777], dtype=np.int16)
    m = _measures_via_histogram(one, spacing)
    assert m == O.measures(one, spacing)
    assert m["perc15_hu"] == -777.0 and m["mean_hu"] == -777.0 and m["volume_ml"] == 0.001
    low = np.array([-3024] * 30 + [-500] * 3, dtype=np.int16)
    m = _measures_via_histogram(low, spacing)
    assert m["perc15_hu"] == -1024.0, "a Perc15 below the clamp is reported as the bound"
    assert m["mean_hu"] == (30 * -3024 + 3 * -500) / 33, "the mean uses the unclamped HU"
    assert m["laa950_percentage"] == m["laa910_percentage"] == 100 * 30 / 33
    high = np.array([3071] * 9, dtype=np.int16)
    m = _measures_via_histogram(high, spacing)
    assert m["perc15_hu"] == 1023.0 and m["mean_hu"] == 3071.0 and m["laa950_percentage"] == 0.0
    # strict <: -950 is not below -950, -951 is
    edge = np.array([-950, -951, -910, -911], dtype=np.int16)
    m = _measures_via_histogram(edge, spacing)
    assert m["laa950_percentage"] == 25.0 and m["laa910_percentage"] == 75.0
    assert densitometry.metrics_from_histogram(np.zeros(2048, dtype=np.int64), 0, 0, spacing) is None
    with pytest.raises(ValueError):
        densitometry.percentile15(np.zeros(2048, dtype=np.int64))


def test_lung_is_the_union_of_the_labels():
    """scan_densitometry adds the label histograms into the lung's; the same on the voxels is the oracle's lung."""
    from dram_b200 import densitometry

    g = np.random.default_rng(5)
    labels = g.choice(np.array([0, 1, 2, 7, 255], dtype=np.uint8), size=(6, 7, 9))
    scan = g.integers(-1200, 200, size=labels.shape).astype(np.int16)
    spacing = (1.25, 0.7, 0.7)
    counts = O.label_counts(labels)
    ids = [k for k in range(1, 256) if counts[k]]
    hist, sums = O.hu_histograms(scan, labels, ids)
    lung = densitometry.metrics_from_histogram(hist.sum(0), int(sums.sum()), int(counts[1:].sum()), spacing)
    ref = O.densitometry(scan, labels, spacing)
    assert lung == ref["lung"] and sorted(ref["lobes"]) == ids == [1, 2, 7, 255]


def _result():
    lung = {"volume_ml": 5123.456, "laa950_percentage": 12.34567, "laa910_percentage": 40.0, "perc15_hu": -953.85,
            "mean_hu": -851.04999}
    lobe = {"volume_ml": 0.001, "laa950_percentage": 0.0, "laa910_percentage": 100.0, "perc15_hu": -1024.0,
            "mean_hu": -3024.0}
    return {"lung": lung, "lobes": {5: lobe, 1: lung}}


def test_format_densitometry():
    from dram_b200 import densitometry

    want_lung = {"volume_ml": "5123.5", "laa950_percentage": "12.346", "laa910_percentage": "40.000",
                 "perc15_hu": "-953.9", "mean_hu": "-851.0"}
    got = densitometry.format_densitometry(_result())
    assert got == {"lung": want_lung, "lobes": {"1": want_lung, "5": {
        "volume_ml": "0.0", "laa950_percentage": "0.000", "laa910_percentage": "100.000", "perc15_hu": "-1024.0",
        "mean_hu": "-3024.0"}}}
    assert list(got["lobes"]) == ["1", "5"] and list(got["lung"]) == list(densitometry.METRICS)
    assert densitometry.format_densitometry({"lung": None, "lobes": {}}) == {"lung": {}, "lobes": {}}


def test_parser_flag_off_by_default_and_allowed_for_every_architecture():
    from dram_b200 import processor
    from dram_b200.models import SubtypeDataModule

    assert processor.build_parser().parse_args([]).densitometry is False
    for arch in ("med3ddram", "med3ddram18", "med3d18", "med3d50"):
        args = processor.build_parser().parse_args(["--densitometry", "--model_arch", arch])
        processor.check_args(args)
        ds = SubtypeDataModule(args).predict_dataset()
        assert ds.densitometry is True and ds.lobe_labels is False and ds.densitometry_cache == {}
    ds = SubtypeDataModule(processor.build_parser().parse_args([])).predict_dataset()
    assert ds.densitometry is False


class _DataModule:
    def __init__(self, densitometry, cache):
        from dram_b200.models import RunningStage

        ds = Namespace(densitometry=densitometry, densitometry_cache=cache)
        self.datasets = {RunningStage.PREDICTING: ds}


def test_classification_records_carry_the_field_only_with_the_flag():
    from dram_b200 import densitometry, processor

    pred = {"uids": ["a", "b"], "cle_labels": torch.tensor([3, 0]), "pse_labels": torch.tensor([1, 2])}
    plain = processor.postprocess_cls(pred)
    assert processor.postprocess_cls(pred, _DataModule(False, {})) == plain
    cache = {"a": _result(), "b": {"lung": _result()["lung"], "lobes": {}}}
    got = processor.postprocess_cls(pred, _DataModule(True, cache))
    assert [{k: v for k, v in r.items() if k != "densitometry"} for r in got] == plain
    assert [list(r) for r in got] == [["entity", "metrics", "error_messages", "densitometry"]] * 2
    assert got[0]["densitometry"] == densitometry.format_densitometry(cache["a"])
    assert got[1]["densitometry"]["lobes"] == {}


def test_densitometry_survives_the_multi_rank_merge(tmp_path):
    from dram_b200 import densitometry, processor

    field = densitometry.format_densitometry(_result())
    rec = lambda uid: {"entity": uid, "error_messages": [], "densitometry": field, "metrics": {  # noqa: E731
        "cle_severity_score": "2", "cle_lesion_percentage_per_lung": "0.070",
        "pse_severity_score": "1", "pse_lesion_percentage_per_lung": "0.020"}}
    parts = [json.loads(json.dumps([rec("b"), rec("a")])), json.loads(json.dumps([rec("c"), rec("b")]))]
    merged = processor.write_results(Namespace(output_path=str(tmp_path)), parts[0] + parts[1])
    assert [r["entity"] for r in merged] == ["a", "b", "c"]
    on_disk = json.load(open(tmp_path / "results.json"))
    assert [r["densitometry"] for r in on_disk] == [field] * 3


def test_densitometry_fake_kernel_shapes():
    from torch._subclasses.fake_tensor import FakeTensorMode

    from dram_b200 import custom_ops  # noqa: F401

    assert {"label_counts", "hu_histograms"} <= set(custom_ops.REGISTERED)
    with FakeTensorMode():
        lab = torch.empty((7, 9, 11), dtype=torch.uint8, device="cuda")
        scan = torch.empty((7, 9, 11), dtype=torch.int16, device="cuda")
        counts = torch.ops.dram_b200.label_counts(lab)
        assert counts.shape == (256,) and counts.dtype == torch.int64
        hist, sums = torch.ops.dram_b200.hu_histograms(scan, lab, [1, 2, 3, 200, 255])
        assert hist.shape == (5, 2048) and hist.dtype == torch.int64
        assert sums.shape == (5,) and sums.dtype == torch.int64


def test_densitometry_argument_validation_without_gpu(lib):
    from dram_b200 import _capi

    table = bytes([0, 1] + [0xFF] * 254)
    assert lib.dram_label_counts(None, 16, 16, None) == -1 and "null pointer" in _capi.last_error()
    assert lib.dram_label_counts(16, 16, None, None) == -1 and "null pointer" in _capi.last_error()
    assert lib.dram_label_counts(16, -1, 16, None) == -1 and "count -1" in _capi.last_error()
    assert lib.dram_label_hu_hist(None, 16, 16, table, 2, 16, 16, None) == -1 and "null pointer" in _capi.last_error()
    assert lib.dram_label_hu_hist(16, 16, 16, None, 2, 16, 16, None) == -1 and "null pointer" in _capi.last_error()
    assert lib.dram_label_hu_hist(16, 16, 16, table, 2, 16, None, None) == -1 and "null pointer" in _capi.last_error()
    for nslots in (0, -1, 17):
        assert lib.dram_label_hu_hist(16, 16, 16, table, nslots, 16, 16, None) == -1
        assert f"nslots {nslots}" in _capi.last_error()
    assert lib.dram_label_hu_hist(16, 16, -5, table, 2, 16, 16, None) == -1 and "count -5" in _capi.last_error()
    bad = bytes([0, 1, 2] + [0xFF] * 253)                    # slot 2 of 2
    assert lib.dram_label_hu_hist(16, 16, 16, bad, 2, 16, 16, None) == -1 and "label 2" in _capi.last_error()


def test_ops_need_cuda_tensors():
    from dram_b200 import ops

    with pytest.raises(RuntimeError, match="CUDA tensor"):
        ops.label_counts(torch.zeros(4, dtype=torch.uint8))
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        ops.hu_histograms(torch.zeros(4, dtype=torch.int16), torch.zeros(4, dtype=torch.uint8), [1])
