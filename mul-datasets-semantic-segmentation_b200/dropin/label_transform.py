"""Host side of the GPU data pipeline (SURVEY.md §8 f3): the random draws of the reference's training transforms,
turned into the integers and tables ``ops.label_pipeline`` and ``ops.image_pipeline`` consume.

The reference transforms one (image, label) pair at a time on a DataLoader worker (lib/transform_cv2.py): the label
goes through ``lb_map`` (lib/base_dataset.py:81-82), ``RandomResizedCrop`` (nearest resize, 255-padding, crop,
:14-62) and ``RandomHorizontalFlip`` (:66-77).  Only the *numbers* are decided on the host here — with the same
``np.random`` calls in the same order, so a seeded run crops exactly where the reference would — and the pixels are
produced by one kernel for the whole batch, uint8 in HBM end to end.  ``TrainPipeline`` does the same for both
branches, images included: a DataLoader worker then only decodes.
"""
import math

import numpy as np
import torch

from .. import ops


class RandomResizedCropPlan:
    """``RandomResizedCrop(scales, size)`` of lib/transform_cv2.py:14-62, label branch: ``plan(shape)`` draws
    ``np.random.uniform`` (scale) and ``np.random.random(2)`` (crop origin) like ``__call__`` does."""

    def __init__(self, scales=(0.5, 1.), size=(384, 384)):
        self.scales, self.size = scales, size

    def plan(self, shape, rng=np.random):
        H, W = shape
        crop_h, crop_w = self.size
        scale = rng.uniform(min(self.scales), max(self.scales))
        if np.min([H, W]) < 1080:  # :36-37
            scale = scale * (1080 / np.min([H, W]))
        im_h, im_w = [math.ceil(el * scale) for el in (H, W)]
        if (im_h, im_w) == (crop_h, crop_w):  # :45, no crop-origin draw in this case
            return dict(im_h=im_h, im_w=im_w, pad_top=0, pad_left=0, crop_y=0, crop_x=0)
        pad_h = (crop_h - im_h) // 2 + 1 if im_h < crop_h else 0
        pad_w = (crop_w - im_w) // 2 + 1 if im_w < crop_w else 0
        sh, sw = rng.random(2)
        sh, sw = int(sh * (im_h + 2 * pad_h - crop_h)), int(sw * (im_w + 2 * pad_w - crop_w))
        return dict(im_h=im_h, im_w=im_w, pad_top=pad_h, pad_left=pad_w, crop_y=sh, crop_x=sw)


class RandomHorizontalFlipPlan:
    """``RandomHorizontalFlip(p)`` of lib/transform_cv2.py:66-77: one ``np.random.random()`` draw; the pair is
    flipped when the draw is NOT below p (the reference returns the input unchanged when it is)."""

    def __init__(self, p=0.5):
        self.p = p

    def plan(self, rng=np.random):
        return not (rng.random() < self.p)


class LabelPipeline:
    """Batch-level label branch: ``LabelPipeline(scales, size, p)(raw_labels, lut_ids)`` -> ``[B, crop_h, crop_w]``.

    raw_labels: list of uint8 CUDA tensors as decoded from disk (``cv2.imread(lbpth, 0)``); luts: uint8
    ``[n_datasets, 256]`` holding every dataset's ``lb_map``; lut_ids[b] = dataset of image b.  The per-image order
    of random draws is the reference's per-sample order: crop draws, then the flip draw (``TransformationTrain``,
    lib/transform_cv2.py:257-270, skipping ColorJitter which only draws for the image)."""

    def __init__(self, scales, size, p=0.5, luts=None, out_dtype=None, image_draws=3):
        import torch
        self.crop, self.flip, self.size = RandomResizedCropPlan(scales, size), RandomHorizontalFlipPlan(p), size
        self.luts, self.out_dtype = luts, out_dtype or torch.int64
        # ColorJitter(brightness, contrast, saturation) draws one np.random.uniform per enabled term after the flip
        # (lib/transform_cv2.py:94-103); they are drawn and dropped here so that the stream stays aligned with a
        # reference worker that also transforms the image
        self.image_draws = image_draws

    def plans(self, shapes, rng=np.random):
        out = []
        for shape in shapes:
            pl = self.crop.plan(shape, rng)
            pl["flip"] = self.flip.plan(rng)
            for _ in range(self.image_draws):
                rng.uniform(0.0, 1.0)
            out.append(pl)
        return out

    def __call__(self, raw_labels, lut_ids=None, rng=np.random, plans=None):
        plans = plans or self.plans([tuple(t.shape) for t in raw_labels], rng)
        return ops.label_pipeline(raw_labels, plans, self.size, luts=self.luts, lut_ids=lut_ids,
                                  out_dtype=self.out_dtype)


class ColorJitterPlan:
    """``ColorJitter(brightness, contrast, saturation)`` of lib/transform_cv2.py: ``plan(rng)`` draws one
    ``np.random.uniform(max(1 - f, 0), 1 + f)`` per enabled term, in the order brightness, contrast, saturation — the
    same stream consumption as ``LabelPipeline``'s dropped draws — and turns the rates into what
    ``ops.image_pipeline`` consumes, each with the reference's own expression:
    ``lut`` = contrast_table[brightness_table] (uint8[256]) and ``sat`` = float32 (1 + 2r, 1 - r), the two distinct
    entries of adj_saturation's matrix (None when saturation is off)."""

    def __init__(self, brightness=None, contrast=None, saturation=None):
        def rng_of(f):
            return [max(1 - f, 0), 1 + f] if f is not None and f > 0 else None
        self.ranges = [rng_of(brightness), rng_of(contrast), rng_of(saturation)]

    def plan(self, rng=np.random):
        rb, rc, rs = [rng.uniform(*r) if r is not None else None for r in self.ranges]
        lut = np.arange(256).astype(np.uint8)
        if rb is not None:
            lut = np.array([i * rb for i in range(256)]).clip(0, 255).astype(np.uint8)[lut]
        if rc is not None:
            lut = np.array([74 + (i - 74) * rc for i in range(256)]).clip(0, 255).astype(np.uint8)[lut]
        sat = None
        if rs is not None:
            m = np.float32([[1 + 2 * rs, 1 - rs, 1 - rs]])
            sat = (m[0, 0], m[0, 1])
        return dict(brightness=rb, contrast=rc, saturation=rs, lut=lut, sat=sat)


class TrainPipeline:
    """Both branches of the reference's training transforms (``TransformationTrain``: RandomResizedCrop,
    RandomHorizontalFlip, ColorJitter, then ToTensor; lib/get_dataloader.py, lib/transform_cv2.py) for a batch:
    ``TrainPipeline(scales, size)(raw_images, raw_labels, dataset_ids, rng)`` -> ``(im, lb)``, what
    ``to_tensor(trans(...))`` gives per sample, stacked.

    raw_images: uint8 CUDA tensors [H, W, 3] as cv2.imread decodes them (BGR); raw_labels: uint8 CUDA tensors
    [H, W]; dataset_ids[b] selects the row of `luts` (each dataset's ``lb_map``, uint8 [n_datasets, 256]) and of
    `norms` (one ``(mean, std)`` per dataset, the reader's ToTensor arguments; None: mean 0, std 1).  Per sample the
    random draws come in the reference's order — crop, flip, jitter — from `rng`, and ONE list of plans drives
    ``ops.image_pipeline`` and ``ops.label_pipeline``.  Returns fp32 [B, 3, crop_h, crop_w] in `memory_format` and
    `label_dtype` [B, crop_h, crop_w]."""

    def __init__(self, scales, size, p=0.5, jitter=(0.4, 0.4, 0.4), luts=None, norms=None, label_dtype=torch.int64,
                 memory_format=torch.contiguous_format):
        self.crop, self.flip, self.size = RandomResizedCropPlan(scales, size), RandomHorizontalFlipPlan(p), size
        self.jitter = ColorJitterPlan(*jitter) if jitter is not None else None
        self.luts, self.norms = luts, norms
        self.label_dtype, self.memory_format = label_dtype, memory_format
        self._tables = {}

    def plans(self, shapes, rng=np.random):
        out = []
        for shape in shapes:
            pl = self.crop.plan(shape, rng)
            pl["flip"] = self.flip.plan(rng)
            pl["jitter"] = self.jitter.plan(rng) if self.jitter is not None else None
            out.append(pl)
        return out

    def __call__(self, raw_images, raw_labels, dataset_ids=None, rng=np.random, plans=None):
        if len(raw_images) != len(raw_labels):
            raise ValueError("TrainPipeline: one label per image")
        for im, lb in zip(raw_images, raw_labels):
            if tuple(im.shape[:2]) != tuple(lb.shape[:2]):  # the reference asserts this in RandomResizedCrop
                raise ValueError("TrainPipeline: image and label sizes differ")
        plans = plans or self.plans([tuple(t.shape[:2]) for t in raw_images], rng)
        dev = raw_images[0].device
        norms, norm_ids = None, None
        if self.norms is not None:
            if dev not in self._tables:
                self._tables[dev] = ops.to_tensor_tables(self.norms, dev)
            norms, norm_ids = self._tables[dev], dataset_ids
        im = ops.image_pipeline(raw_images, plans, self.size, jitter=[pl["jitter"] for pl in plans], norms=norms,
                                norm_ids=norm_ids, bgr=True, memory_format=self.memory_format)
        lb = ops.label_pipeline(raw_labels, plans, self.size, luts=self.luts,
                                lut_ids=dataset_ids if self.luts is not None else None, out_dtype=self.label_dtype)
        return im, lb
