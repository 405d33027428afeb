"""CPU oracle of the per-lobe lesion percentages (not in the reference, which reports whole-lung numbers only).
TEST INFRASTRUCTURE (see oracle/__init__.py).  Builds on pipeline_oracle:
  crop_labels           the lobe labels cut with the crop window of pipeline_oracle.lung_crop_sample
  interpolate_labels    pipeline_oracle.interpolate_mask without the bool cast (label values kept)
  lobe_scores           fp64 bincount restatement of the per-label voxel counts and lesion percentages
"""
import numpy as np
import torch
import torch.nn.functional as F

from .pipeline_oracle import slice_indices


def crop_labels(lobe, crop_slice):
    """uint8 labels of the crop window ((z0, z1), (y0, y1), (x0, x1)), e.g. a dataset dict's `crop_slice`."""
    sl = tuple(slice(int(a), int(b)) for a, b in np.asarray(crop_slice))
    return torch.as_tensor(np.asarray(lobe)[sl].astype(np.uint8))


def interpolate_labels(m, target_size):
    """[D,H,W] uint8 labels -> target: the voxel `interpolate_mask` picks, its value kept (no bool cast)."""
    y = F.interpolate(m[None].float(), size=tuple(target_size[1:]), mode="nearest")
    return y[:, slice_indices(m.shape[0], target_size[0])][0].to(torch.uint8)


def lobe_scores(cle, pse, ess, labels, nlabels=256):
    """voxels[b, k] = #{labels == k} (int64); sums[m, b, k] = sum of map m over {labels == k and ess} in fp64;
    pct = sums / voxels (NaN without voxels).  Maps [B,1,D,H,W] or [B,D,H,W].  Returns (pct, voxels, sums)."""
    B = labels.shape[0]
    lab = labels.reshape(B, -1).long().cpu()
    e = ess.reshape(B, -1).bool().cpu()
    voxels = torch.stack([torch.bincount(lab[b], minlength=nlabels) for b in range(B)])
    sums = torch.stack([torch.stack([torch.bincount(lab[b][e[b]], weights=m.reshape(B, -1)[b].cpu().double()[e[b]],
                                                    minlength=nlabels) for b in range(B)]) for m in (cle, pse)])
    return sums / voxels.double(), voxels, sums
