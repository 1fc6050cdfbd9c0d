"""Device-resident version of the numeric path of the reference's single-image inference (infer.py:16-28,72-103; SURVEY.md
section 8 row f2): image + amodal mask -> observation depth (un-guided model) -> amodal depth (guided model) -> blended
depth with a smoothed seam. In the reference every step between the two networks goes through the host
(`.detach().cpu()` at infer.py:19,94, numpy blend + cv2.blur at :30-44); here the image and the mask are uploaded once
and everything else runs as kernels on the current stream. Colour maps / PNG writing (infer.py:24-27,105-121) stay with
the caller: they are presentation, not part of the depth result.

`batch` runs the same path over lists of images of any size: one upload of the packed images and masks, then the
resize of infer.py:17 (cv2's bilinear, bit-exact) and every other step as kernels over the batch, with both networks at
batch B. The models are batch-invariant, so each image's result is bit-equal to a single-image call on it.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops


class AmodalInference:
    def __init__(self, model_raw, depth_amodal_model, size: int = 518, cuda_graph: bool = True):
        self.model_raw = model_raw.set_graph(cuda_graph)      # one image per call is launch bound: replay as CUDA graphs
        self.model = depth_amodal_model.set_graph(cuda_graph)
        self.size = size
        self.device = next(depth_amodal_model.parameters()).device
        self._staging = ops.Staging(self.device)   # reused host staging of batch(): packed images + masks, descriptors

    def _upload_u8(self, a: np.ndarray) -> torch.Tensor:
        t = torch.from_numpy(np.ascontiguousarray(a))
        return t.to(self.device, non_blocking=True)

    @torch.no_grad()
    def predict_base_depth(self, image_u8_hwc: np.ndarray):
        """infer.py:16-23 -> (base01 [S,S], observation = base01*2-1 [1,1,S,S]) on the device."""
        S = self.size
        img = image_u8_hwc
        if img.shape[:2] != (S, S):  # infer.py:17 resizes the uint8 image on the host with cv2 (bilinear, fixed point)
            import cv2
            img = cv2.resize(img, (S, S))
        x = ops.image_nearest(self._upload_u8(img), S, S, normalize=True)       # infer.py:18 (identity sampling)
        depth_raw = self.model_raw(x)                                            # [1,S,S], infer.py:19
        base, obs = ops.minmax_normalize(depth_raw)                              # infer.py:20-22
        return base[0], obs.unsqueeze(1)

    @torch.no_grad()
    def __call__(self, image_u8_hwc: np.ndarray, amodal_mask: np.ndarray):
        """infer.py:72-103. image: uint8 [H0,W0,3] as cv2.imread returns it; amodal_mask: [H0,W0], non-zero = object.
        Returns device tensors: base_depth [S,S] in [0,1], pred [1,1,S,S], depth_agg [S,S]."""
        S = self.size
        base, obs = self.predict_base_depth(image_u8_hwc)
        rgb = ops.image_nearest(self._upload_u8(image_u8_hwc), S, S)                                # infer.py:84-86
        m01, guide = ops.mask_nearest(self._upload_u8((np.asarray(amodal_mask) > 0).astype(np.uint8)), S, S)   # :80-87
        pred = self.model(rgb, guide_rgb=None, guide_mask=guide, observation=obs)                   # infer.py:88-93
        agg = ops.blend_seam(base, pred[0, 0], m01[0, 0])                                           # infer.py:97-103
        return dict(base_depth=base, pred=pred, depth_agg=agg)

    @torch.no_grad()
    def batch(self, images, masks, max_batch: int = 32):
        """__call__ over lists: images[i] uint8 [H0,W0,3] (cv2 order) with masks[i] [h0,w0] (any dtype, non-zero = object;
        sizes may differ between images and from the image). Returns device tensors base_depth [B,S,S], pred [B,1,S,S],
        depth_agg [B,S,S]; image i is bit-equal to self(images[i], masks[i]). Lists longer than max_batch run in chunks of
        max_batch images. After the upload nothing synchronises with the host."""
        assert len(images) == len(masks) and len(images) > 0 and max_batch > 0
        outs = [self._batch(images[i:i + max_batch], masks[i:i + max_batch]) for i in range(0, len(images), max_batch)]
        if len(outs) == 1:
            return outs[0]
        return {k: torch.cat([o[k] for o in outs]) for k in outs[0]}

    def _stage(self, images, masks):
        """Packs the images and the thresholded masks into the pinned staging buffer and uploads it and the descriptor
        table (ada_img_desc rows: images, masks, then the [B,S,S,3] resized batch), one copy each."""
        S, B = self.size, len(images)
        imgs = [np.asarray(a) for a in images]
        ms = [np.asarray(m) for m in masks]
        for a, m in zip(imgs, ms):
            assert a.dtype == np.uint8 and a.ndim == 3 and a.shape[2] == 3, "images must be uint8 [H0,W0,3]"
            assert m.ndim == 2, "masks must be [h0,w0]"
        rows_img, end = ops.pack_layout([a.shape for a in imgs])
        rows_mask, end = ops.pack_layout([m.shape for m in ms], end)
        rows = rows_img + rows_mask + [(b * S * S * 3, S, S) for b in range(B)]

        def fill(host):
            for (o, _, _), a in zip(rows_img, imgs):
                np.copyto(host[o:o + a.size].reshape(a.shape), a)
            for (o, _, _), m in zip(rows_mask, ms):
                np.greater(m, 0, out=host[o:o + m.size].reshape(m.shape).view(np.bool_))   # as __call__ thresholds
        data, desc = self._staging.upload(end, rows, fill)
        return data, desc[:B], desc[B:2 * B], desc[2 * B:]

    def _batch(self, images, masks):
        S = self.size
        with torch.cuda.device(self.device):
            data, d_img, d_mask, d_resized = self._stage(images, masks)
            resized = ops.resize_linear_batch(data, d_img, S, S)                                     # infer.py:17
            x = ops.image_nearest_batch(resized.view(-1), d_resized, S, S, normalize=True)            # infer.py:18
            rgb = ops.image_nearest_batch(data, d_img, S, S)                                         # infer.py:84-86
            m01, guide = ops.mask_nearest_batch(data, d_mask, S, S)                                  # infer.py:80-87
            depth_raw = self.model_raw(x)                                                            # [B,S,S], infer.py:19
            base, obs = ops.minmax_normalize_batch(depth_raw)                                        # infer.py:20-22
            pred = self.model(rgb, guide_rgb=None, guide_mask=guide, observation=obs.unsqueeze(1))   # infer.py:88-93
            agg = ops.blend_seam_batch(base, pred[:, 0], m01[:, 0])                                  # infer.py:97-103
        return dict(base_depth=base, pred=pred, depth_agg=agg)
