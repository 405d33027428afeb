"""`SubtypingInference`: the reference's inference dataset (dataset.py:14-92) on the native .mha reader.

Per scan: read CT + lobe segmentation, lung = lobe > 0, blank everything outside the lung dilated by
two 3x3x3 steps (== one 5x5x5 box) to -2048, crop to the lung bounding box + 5 mm, derive the LAA-910
`ess` mask, and hand the dict to the transform.  With a CUDA `device` these pre-steps run on the GPU
(`ops.mask_bbox` + `ops.lung_crop`, SURVEY §8f row f1): the scan and the lobe labels are copied to the device
once (3 bytes per voxel), only the 6 bounding-box integers come back, and the cropped tensors go straight
into the GPU transform.  There is no CPU path (the CPU restatement of these steps is oracle/pipeline_oracle.py,
test infrastructure).
"""
import glob
import math
import os
from pathlib import Path

import numpy as np
import torch

from . import mha_io


def grow_bbox(bbox, shape, spacing, border):
    """utils.py:55-60: pad the find_objects box by ceil(border/spacing) voxels per axis, clipped to the volume."""
    out = []
    for ax in range(3):
        lo, hi = int(bbox[2 * ax]), int(bbox[2 * ax + 1])
        pad = int(math.ceil(border / spacing[ax])) if border > 0 else 0
        out.append((max(0, lo - pad), min(int(shape[ax]), hi + pad)))
    return out


def labels_as_u8(lobe, uid):
    """The lobe segmentation as a uint8 label volume: uint8 as it is; another integer (or bool) type when every value
    lies in 0..255; anything else raises ValueError naming the scan."""
    lobe = np.asarray(lobe)
    if lobe.dtype == np.uint8:
        return lobe
    if lobe.dtype.kind not in "iub":
        raise ValueError(f"{uid}: lobe labels of type {lobe.dtype} are not integers")
    if lobe.size and (int(lobe.min()) < 0 or int(lobe.max()) > 255):
        raise ValueError(f"{uid}: lobe labels span {int(lobe.min())}..{int(lobe.max())}, outside 0..255")
    return lobe.astype(np.uint8)


class SubtypingInference(torch.utils.data.Dataset):
    label_to_cle = {0: "absent", 1: "trace", 2: "mild", 3: "moderate", 4: "confluence", 5: "destructive"}
    label_to_pse = {0: "absent", 1: "mild", 2: "substantial"}

    def __init__(self, scan_path, lobe_path, transforms=None, keep_sorted=True, crop_border=5, device=None,
                 lobe_labels=False, densitometry=False):
        """`lobe_labels=True`: every sample also carries `lobe_labels`, the uint8 label volume cropped like the masks
        (for the per-lobe percentages).  `densitometry=True`: the pre-steps also measure the lung and every lobe label
        on the full-resolution scan (`densitometry.scan_densitometry`) into `densitometry_cache[uid]`."""
        super().__init__()
        self.device = torch.device(device) if device is not None else getattr(transforms, "device", None)
        self.scan_path, self.lobe_path = scan_path, lobe_path
        self.keep_sorted, self.transforms, self.crop_border = keep_sorted, transforms, crop_border
        self.lobe_labels, self.densitometry = lobe_labels, densitometry
        self.scan_files = sorted(glob.glob(os.path.join(scan_path, "*.mha")))
        self.lobe_files = sorted(glob.glob(os.path.join(lobe_path, "*.mha")))
        self.scan_meta_cache = {}
        self.densitometry_cache = {}

    def __len__(self):
        return len(self.scan_files)

    def __getitem__(self, index):
        return self.get_data(index)

    def read_image(self, path):
        """(array [z,y,x], origin, spacing, direction) with the metadata reversed to z-y-x like dataset.py:49-55."""
        arr, meta = mha_io.read_mha(path)
        direction = np.asarray(meta["direction"]).reshape(3, 3)[::-1].flatten().tolist()
        return arr, meta["origin"][::-1], meta["spacing"][::-1], direction

    def device_presteps(self, scan, lobe, spacing, uid):
        """dataset.py:66-83 on the GPU; returns the same dict with device tensors (masks as bool)."""
        from . import ops

        dev = self.device
        scan_d = torch.as_tensor(np.ascontiguousarray(scan)).to(torch.int16).to(dev, non_blocking=True)
        if self.lobe_labels or self.densitometry:  # values kept: lung_crop takes labels > 0 itself
            lobe_d = torch.as_tensor(np.ascontiguousarray(labels_as_u8(lobe, uid))).to(dev, non_blocking=True)
        else:
            lobe_d = torch.as_tensor(np.ascontiguousarray(lobe))
            lobe_d = (lobe_d.to(torch.uint8) if lobe_d.dtype in (torch.uint8, torch.int8, torch.bool)
                      else (lobe_d > 0).to(torch.uint8)).to(dev, non_blocking=True)
        bbox = ops.mask_bbox(lobe_d).cpu().tolist()
        if bbox[1] <= bbox[0]:
            raise IndexError(f"{uid}: empty lobe segmentation (the reference fails in find_objects here)")
        crop = grow_bbox(bbox, scan.shape, spacing, self.crop_border)
        image, lung, ess = ops.lung_crop(scan_d, lobe_d, crop)
        if self.densitometry:
            from .densitometry import scan_densitometry

            self.densitometry_cache[uid] = scan_densitometry(scan_d, lobe_d, spacing)
        sample = {
            "image": image,
            "lung_mask": lung.view(torch.bool),
            "ess_mask": ess.view(torch.bool),
            "crop_slice": np.asarray(crop),
            "original_size": np.asarray(scan.shape),
            "uid": uid,
        }
        if self.lobe_labels:
            (z0, z1), (y0, y1), (x0, x1) = crop
            sample["lobe_labels"] = lobe_d[z0:z1, y0:y1, x0:x1].contiguous()
        return sample

    def load_raw(self, index):
        """The file half of `get_data` (dataset.py:57-65): read CT + lobes.  Host only and thread-safe, so the
        processor's `--workers N` can read ahead on N threads (zlib releases the GIL)."""
        scan_file, lobe_file = self.scan_files[index], self.lobe_files[index]
        uid = Path(scan_file).stem
        scan, origin, spacing, direction = self.read_image(scan_file)
        lobe, _, _, _ = self.read_image(lobe_file)
        assert lobe.shape == scan.shape, "scan and lobe segmentation have different shapes."
        return {"uid": uid, "scan": scan, "lobe": lobe, "origin": origin, "spacing": spacing, "direction": direction}

    def get_data(self, index, raw=None):
        raw = self.load_raw(index) if raw is None else raw
        uid, scan, lobe, spacing = raw["uid"], raw["scan"], raw["lobe"], raw["spacing"]
        self.scan_meta_cache[uid] = {"spacing": spacing, "origin": raw["origin"], "direction": raw["direction"]}
        if self.device is None and torch.cuda.is_available():
            # the GPU transform follows: the pre-steps run on the same device
            self.device = self.transforms._dev() if hasattr(self.transforms, "_dev") else \
                torch.device("cuda", torch.cuda.current_device())
        if self.device is None or self.device.type != "cuda":
            raise RuntimeError("SubtypingInference needs a CUDA device: the pre-steps of dataset.py:66-83 run on the GPU "
                               "(ops.mask_bbox / ops.lung_crop); there is no CPU path")
        sample = self.device_presteps(scan, lobe, spacing, uid)
        return self.transforms(sample) if self.transforms else sample
