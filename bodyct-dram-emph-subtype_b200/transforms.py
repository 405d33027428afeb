"""The inference transform of the reference (models.py:55-63: NumpyToTensor -> IntensityWindow(-1150,-300
-> 0,1) -> Standardize -> Interpolate(target_size, align_corners=True, only_in_plane=True)) as two GPU
kernels per image (K8 window+standardise, K8b in-plane bilinear + slice pick) and one per mask (K8b
legacy-nearest + slice pick).  Dispatch is by key substring exactly like base.py:119-133: keys containing
"image" take the image path, keys containing "mask" the mask path, everything else passes through.  One key is
matched exactly before that: `lobe_labels` (not in the reference) takes the mask path with the label values kept.
"""
import numpy as np
import torch

from . import ops

WINDOW = (-1150.0, -300.0)  # models.py:60


class InferenceTransform:
    def __init__(self, target_size=(128, 224, 288), device=None, keep_original_image=False):
        self.target_size = tuple(int(v) for v in target_size)
        self.device = torch.device(device) if device is not None else None
        self.keep_original_image = keep_original_image

    def _dev(self):
        if self.device is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        return self.device

    def apply_to_image(self, data):
        """int16 HU [D,H,W] (numpy or tensor) -> fp32 standardised window at target size, on the GPU."""
        t = torch.as_tensor(data)
        if t.dtype != torch.int16:
            t = t.to(torch.int16)
        t = t.to(self._dev(), non_blocking=True).contiguous()
        win, _ = ops.window_standardize(t, WINDOW[0], WINDOW[1])
        return ops.resize_image(win, self.target_size)

    def apply_to_mask(self, data):
        t = torch.as_tensor(data)
        t = (t != 0).to(torch.uint8) if t.dtype != torch.bool else t.view(torch.uint8)
        t = t.to(self._dev(), non_blocking=True).contiguous()
        return ops.resize_mask(t, self.target_size).view(torch.bool)

    def apply_to_labels(self, data):
        """uint8 lobe labels: the mask path with the label values kept."""
        t = torch.as_tensor(data).to(self._dev(), non_blocking=True).contiguous()
        return ops.resize_labels(t, self.target_size)

    def __call__(self, sample):
        out = {}
        for key, val in sample.items():
            is_array = isinstance(val, (np.ndarray, torch.Tensor))
            if is_array and key == "lobe_labels":
                out[key] = self.apply_to_labels(val)
            elif is_array and "image" in key:
                if key == "original_image" and not self.keep_original_image:
                    continue  # never read by predict_step / the processor; skipped unless asked for
                out[key] = self.apply_to_image(val)
            elif is_array and "mask" in key:
                out[key] = self.apply_to_mask(val)
            elif isinstance(val, np.ndarray):
                out[key] = torch.as_tensor(val)
            else:
                out[key] = val
        return out
