"""CPU oracle of the lung and per-lobe densitometry (not in the reference, which reports no densitometry).
TEST INFRASTRUCTURE (see oracle/__init__.py).  A restatement of the definitions on the voxel arrays themselves:
  label_counts      np.bincount of the labels (int64 [256])
  hu_histograms     per label: np.bincount of the HU clamped to [-1024, 1023] (2048 bins) and the exact int64 HU sum
  measures          volume_ml, laa950/laa910 percentages (strict <), np.percentile(clamped, 15), exact mean HU
  densitometry      {"lung": measures of labels >= 1, "lobes": {label: measures}} of one scan
"""
import numpy as np

HU_LO, HU_HI = -1024, 1023


def label_counts(labels):
    return np.bincount(np.asarray(labels, dtype=np.uint8).ravel(), minlength=256).astype(np.int64)


def hu_histograms(scan, labels, label_ids):
    scan = np.asarray(scan).ravel().astype(np.int64)
    labels = np.asarray(labels).ravel()
    hist = np.zeros((len(label_ids), HU_HI - HU_LO + 1), dtype=np.int64)
    sums = np.zeros(len(label_ids), dtype=np.int64)
    for i, k in enumerate(label_ids):
        v = scan[labels == k]
        hist[i] = np.bincount(np.clip(v, HU_LO, HU_HI) - HU_LO, minlength=HU_HI - HU_LO + 1)
        sums[i] = v.sum(dtype=np.int64)
    return hist, sums


def measures(v, spacing):
    """The five measures of the HU values `v` (any integer dtype) of one label; None when it is empty."""
    v = np.asarray(v)
    n = v.size
    if n == 0:
        return None
    sz, sy, sx = (float(s) for s in spacing)
    return {
        "volume_ml": n * sz * sy * sx / 1000,
        "laa950_percentage": 100 * int(np.count_nonzero(v < -950)) / n,
        "laa910_percentage": 100 * int(np.count_nonzero(v < -910)) / n,
        "perc15_hu": float(np.percentile(np.clip(v, HU_LO, HU_HI), 15)),
        "mean_hu": float(np.sum(v, dtype=np.int64) / n),
    }


def densitometry(scan, labels, spacing):
    """Densitometry of one scan (HU and lobe labels of one shape, spacing (z, y, x) in mm)."""
    scan, labels = np.asarray(scan), np.asarray(labels)
    ids = [int(k) for k in np.unique(labels) if k > 0]
    return {"lung": measures(scan[labels > 0], spacing),
            "lobes": {k: measures(scan[labels == k], spacing) for k in ids}}
