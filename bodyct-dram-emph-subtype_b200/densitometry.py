"""Quantitative-CT densitometry of the lung and of each lobe label, on the full-resolution scan (not in the reference).

For every label k >= 1 that has voxels in the lobe segmentation, and for "lung" (the union of all labels >= 1):
    N                   #{label == k}, exact
    volume_ml           N * s_z * s_y * s_x / 1000, s = the scan's spacing in mm
    laa950_percentage   100 * #{HU < -950} / N     (the usual emphysema index)
    laa910_percentage   100 * #{HU < -910} / N     (the threshold of the pipeline's `ess` mask)
    perc15_hu           numpy.percentile(v, 15) with the default linear method, v = the label's HU clamped to
                        [-1024, 1023]; a Perc15 on a clamp bound is reported as that bound
    mean_hu             the exact integer sum of the label's unclamped HU / N
The device makes two memory-bound passes over the scan it already holds for the pre-steps (`ops.label_counts`,
`ops.hu_histograms`); the histograms hold every number above exactly, and this module does the arithmetic on the host.
The full-resolution grid is the one on which voxel counts times spacing are physical volumes and HU values are not
resampled.
"""
import math

import numpy as np

from . import ops

HU_LO = -1024                       # the value of histogram bin 0; bin b holds HU b - 1024
METRICS = ("volume_ml", "laa950_percentage", "laa910_percentage", "perc15_hu", "mean_hu")
FORMATS = {"volume_ml": "{:.1f}", "laa950_percentage": "{:.3f}", "laa910_percentage": "{:.3f}", "perc15_hu": "{:.1f}",
           "mean_hu": "{:.1f}"}


def percentile15(hist):
    """numpy.percentile(v, 15) (linear method) of the values a 2048-bin histogram holds, with numpy's arithmetic:
    virtual index (n - 1) * 0.15 between the order statistics a = v[lo] and b = v[lo + 1], a + (b - a) * g below
    g = 0.5 and b - (b - a) * (1 - g) from there on."""
    cum = np.cumsum(np.asarray(hist, dtype=np.int64))
    n = int(cum[-1])
    if n <= 0:
        raise ValueError("percentile15 of an empty histogram")

    def value_of_rank(r):
        return int(np.searchsorted(cum, r, side="right")) + HU_LO

    virtual = (n - 1) * 0.15
    if virtual >= n - 1:
        return float(value_of_rank(n - 1))
    lo = math.floor(virtual)
    gamma = virtual - lo
    a, b = value_of_rank(lo), value_of_rank(lo + 1)
    diff = b - a
    return float(b - diff * (1 - gamma)) if gamma >= 0.5 else float(a + diff * gamma)


def metrics_from_histogram(hist, hu_sum, voxels, spacing):
    """The five measures of one label from its HU histogram (2048 bins), exact HU sum and voxel count; None without
    voxels.  `spacing`: (s_z, s_y, s_x) in mm."""
    voxels = int(voxels)
    if voxels <= 0:
        return None
    hist = np.asarray(hist, dtype=np.int64)
    sz, sy, sx = (float(s) for s in spacing)
    return {
        "volume_ml": voxels * sz * sy * sx / 1000,
        "laa950_percentage": 100 * int(hist[:-950 - HU_LO].sum()) / voxels,
        "laa910_percentage": 100 * int(hist[:-910 - HU_LO].sum()) / voxels,
        "perc15_hu": percentile15(hist),
        "mean_hu": int(hu_sum) / voxels,
    }


def scan_densitometry(scan_d, labels_d, spacing):
    """Densitometry of one scan: int16 HU and uint8 lobe labels of the full-resolution grid on the device, spacing
    (z, y, x) in mm.  One counting pass, one read-back of the 256 counts, one histogram pass per 16 labels present, then
    the arithmetic on the host.  Returns {"lung": measures or None, "lobes": {label: measures}}."""
    counts = ops.label_counts(labels_d).cpu().tolist()
    ids = [k for k in range(1, len(counts)) if counts[k] > 0]
    hist, hu_sum = ops.hu_histograms(scan_d, labels_d, ids)
    hist, hu_sum = hist.cpu().numpy(), hu_sum.cpu().tolist()
    lobes = {k: metrics_from_histogram(hist[i], hu_sum[i], counts[k], spacing) for i, k in enumerate(ids)}
    lung = metrics_from_histogram(hist.sum(axis=0), sum(hu_sum), sum(counts[k] for k in ids), spacing)
    return {"lung": lung, "lobes": lobes}


def _format(measures):
    return {name: FORMATS[name].format(measures[name]) for name in METRICS}


def format_densitometry(result):
    """The `densitometry` field of a results.json record from `scan_densitometry`'s result: strings formatted like
    the other metrics ({:.1f} for mL and HU, {:.3f} for percentages on the 0-100 scale); lobes keyed by str(label)."""
    lung = result["lung"]
    return {"lung": _format(lung) if lung is not None else {},
            "lobes": {str(k): _format(m) for k, m in sorted(result["lobes"].items())}}
