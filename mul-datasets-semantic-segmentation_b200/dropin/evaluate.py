"""Drop-in for the evaluator tail of evaluate.py (``MscEvalV0`` :45-98 and its multi-scale siblings :100-192).

``MscEvalV0(scales, flip, ignore_label)(net, dl, n_classes, dataset_id) -> float`` keeps the reference
signature.  Per image the reference up-samples every (scale, flip) pass to label size, soft-maxes, sums,
arg-maxes, copies label and prediction to the host and calls ``np.bincount``; here all passes of an image go
through two kernels that keep the probability accumulators in registers, take the arg-max and update an
exact int64 confusion matrix on the device (``ops.eval_fused``; more than 16 passes or mixed dtypes fall
back to one upsample+softmax+accumulate kernel per pass), and the only collective is one all-reduce of that matrix.
"""
import math

import numpy as np
import torch
import torch.distributed as dist
import torch.nn.functional as F

from .. import ops


def get_round_size(size, divisor=32):
    return [math.ceil(el / divisor) * divisor for el in size]


class SegHist:
    """Device-side confusion matrix of one dataset: update(label, logits passes) / all_reduce / miou."""

    def __init__(self, n_classes, device, ignore_label=255, lb_map=None):
        self.n_classes, self.ignore_label, self.lb_map = n_classes, ignore_label, lb_map
        self.hist = torch.zeros(n_classes, n_classes, dtype=torch.int64, device=device)

    @torch.no_grad()
    def update_from_passes(self, label, passes):
        """label [H, W]; passes: iterable of (logits [C, h, w], flip) — evaluate.py:64-93 for one image."""
        H, W = label.shape[-2:]
        passes = list(passes)
        if ops.eval_fused_fits(self.n_classes, len(passes)) and len({p[0].dtype for p in passes}) == 1:
            # every pass of the image at once, no [C, H, W] probability tensor
            return ops.eval_fused(passes, (H, W), label=label.reshape(H, W), hist=self.hist, lut=self.lb_map,
                                  ignore=self.ignore_label)[0]
        probs = torch.empty(self.n_classes, H, W, dtype=torch.float32, device=label.device)
        first = True
        for logits, flip in passes:
            ops.eval_accum(logits, probs, flip=flip, first=first)
            first = False
        return ops.argmax_hist(probs, label=label.reshape(H, W), hist=self.hist, lut=self.lb_map,
                               ignore=self.ignore_label)

    @torch.no_grad()
    def update(self, label, pred):
        """hist += bincount(label[keep] * C + pred[keep]) (evaluate.py:89-93)."""
        ops.confusion(label, pred, self.n_classes, lut=self.lb_map, ignore=self.ignore_label, hist=self.hist)

    def all_reduce(self):
        if dist.is_available() and dist.is_initialized():
            dist.all_reduce(self.hist, dist.ReduceOp.SUM)  # evaluate.py:94-95, exact in int64

    def ious(self):
        return ops.miou(self.hist)

    def miou(self):
        ops.check_errors(self.hist.device)
        return float(self.ious()[1])


class MscEvalV0:
    def __init__(self, scales=(0.5,), flip=False, ignore_label=255):
        self.scales, self.flip, self.ignore_label = scales, flip, ignore_label

    @torch.no_grad()
    def __call__(self, net, dl, n_classes, dataset_id):
        dev = torch.device("cuda", torch.cuda.current_device())
        acc = SegHist(n_classes, dev, self.ignore_label)
        for imgs, label in dl:
            N_, _, H, W = label.shape
            label = label.squeeze(1).to(dev, non_blocking=True)
            per_image = [[] for _ in range(N_)]
            for scale in self.scales:
                sH, sW = get_round_size((int(scale * H), int(scale * W)))
                im_sc = F.interpolate(imgs, size=(sH, sW), mode='bilinear', align_corners=True).to(dev)
                logits = net(im_sc, dataset=dataset_id)[0]
                for b in range(N_):
                    per_image[b].append((logits[b], False))
                if self.flip:
                    logits = net(torch.flip(im_sc, dims=(3,)), dataset=dataset_id)[0]
                    for b in range(N_):
                        per_image[b].append((logits[b], True))  # un-flipped inside the kernel
            for b in range(N_):
                acc.update_from_passes(label[b], per_image[b])
        acc.all_reduce()
        return acc.miou()


class MscEvalCrop:
    """evaluate.py:650-753 — sliding-window multi-scale evaluator (upstream BiSeNet's cropped evaluation):
    ``MscEvalCrop(cropsize, cropstride, flip, scales, lb_ignore)(net, dl, n_classes) -> float``.  The net returns
    full-resolution logits (``net(crop)[0]``).  Per chip the soft-max(es), the reference's ``exp`` of the flipped sum
    (:689, kept) and the add into the scale-level map are one kernel; per scale the bilinear resize of that map to
    the label size and the add into the image-level map another; arg-max + int64 confusion matrix + one all-reduce
    as in the other evaluators."""

    def __init__(self, cropsize=1024, cropstride=2. / 3, flip=True, scales=(0.5, 0.75, 1, 1.25, 1.5, 1.75), lb_ignore=255):
        self.scales, self.ignore_label, self.flip = scales, lb_ignore, flip
        self.distributed = dist.is_available() and dist.is_initialized()
        self.cropsize = tuple(cropsize) if isinstance(cropsize, (list, tuple)) else (cropsize, cropsize)
        self.cropstride = cropstride

    def pad_tensor(self, inten):
        """:667-679 — centre the image in a zero canvas at least as large as the crop."""
        N_, C_, H, W = inten.shape
        cropH, cropW = self.cropsize
        if cropH < H and cropW < W:
            return inten, [0, H, 0, W]
        padH, padW = max(cropH, H), max(cropW, W)
        out = torch.zeros(N_, C_, padH, padW, device=inten.device, dtype=inten.dtype)
        hst, wst = (padH - H) // 2, (padW - W) // 2
        out[:, :, hst:hst + H, wst:wst + W] = inten
        return out, [hst, hst + H, wst, wst + W]

    def chips(self, H, W):
        """:697-709 — chip origins of the padded scale-level image."""
        cropH, cropW = self.cropsize
        strdH, strdW = math.ceil(cropH * self.cropstride), math.ceil(cropW * self.cropstride)
        n_h, n_w = math.ceil((H - cropH) / strdH) + 1, math.ceil((W - cropW) / strdW) + 1
        for i in range(n_h):
            for j in range(n_w):
                endH, endW = min(H, strdH * i + cropH), min(W, strdW * j + cropW)
                yield endH - cropH, endH, endW - cropW, endW

    @torch.no_grad()
    def __call__(self, net, dl, n_classes):
        dev = torch.device("cuda", torch.cuda.current_device())
        acc = SegHist(n_classes, dev, self.ignore_label)
        for imgs, label in dl:
            imgs = imgs.to(dev)
            label = label.squeeze(1).to(dev, non_blocking=True)
            N_, H, W = label.shape
            probs = torch.empty(N_, n_classes, H, W, dtype=torch.float32, device=dev)
            for si, sc in enumerate(self.scales):
                im = F.interpolate(imgs, [int(H * sc), int(W * sc)], mode='bilinear', align_corners=True)
                im, window = self.pad_tensor(im)
                PH, PW = im.shape[-2:]
                pmap = torch.zeros(N_, n_classes, PH, PW, dtype=torch.float32, device=dev)
                for y0, y1, x0, x1 in self.chips(PH, PW):
                    chip = im[:, :, y0:y1, x0:x1]
                    lg = net(chip)[0]
                    lgf = net(torch.flip(chip, dims=(3,)))[0] if self.flip else None
                    for b in range(N_):
                        ops.eval_chip_accum(lg[b], pmap[b], y0, x0, None if lgf is None else lgf[b], exp_after=self.flip)
                for b in range(N_):
                    ops.prob_resize_accum(pmap[b], window, probs[b], first=(si == 0))
            for b in range(N_):
                ops.argmax_hist(probs[b], label=label[b], hist=acc.hist, ignore=self.ignore_label, want_pred=False)
        acc.all_reduce()
        return acc.miou()


class MscEvalV0_Contrast:
    """evaluate.py:101-192 — the evaluator ``eval_model_contrast`` (:1127) and tools/eval_snp.py build as
    ``MscEvalV0_Contrast(configer, (0.5,), False)``.  The net returns the logits tensor itself.  With
    ``ori_scales=False`` (the default) the probabilities stay at the resolution of the logits and the *label* is
    resized to it with torch's legacy 'nearest' rule, once per scale and cumulatively (:156-157); with
    ``ori_scales=True`` the logits are up-sampled to the label as in ``MscEvalV0``."""

    def __init__(self, configer, scales=(0.5,), flip=False, ignore_label=255, ori_scales=False):
        self.configer, self.scales, self.flip = configer, scales, flip
        self.ignore_label, self.ori_scales = ignore_label, ori_scales

    @torch.no_grad()
    def __call__(self, net, dl, n_classes, dataset_id):
        dev = torch.device("cuda", torch.cuda.current_device())
        acc = SegHist(n_classes, dev, self.ignore_label)
        for imgs, label in dl:
            N_, _, H, W = label.shape
            label = label.squeeze(1).to(dev, non_blocking=True)
            per_image = [[] for _ in range(N_)]
            psize = (H, W)
            for scale in self.scales:
                sH, sW = get_round_size((int(scale * H), int(scale * W)))
                im_sc = F.interpolate(imgs, size=(sH, sW), mode='bilinear', align_corners=True).to(dev)
                logits = net(im_sc, dataset=dataset_id)
                lH, lW = logits.shape[-2:]
                if not self.ori_scales:
                    if per_image[0] and psize != (lH, lW):
                        # the reference's `probs += softmax(logits)` fails on the shape mismatch here (:163)
                        raise RuntimeError(f"ori_scales=False: logits of size {(lH, lW)} after probabilities of size {psize}")
                    label = ops.label_nearest(label, (lH, lW))
                    psize = (lH, lW)
                for b in range(N_):
                    per_image[b].append((logits[b], False))
                if self.flip:
                    if psize != (H, W):
                        raise RuntimeError("ori_scales=False with flip: the reference up-samples the flipped pass to the "
                                           "label size (:169) and fails on the shape mismatch")
                    logits = net(torch.flip(im_sc, dims=(3,)), dataset=dataset_id)
                    for b in range(N_):
                        per_image[b].append((logits[b], True))
            for b in range(N_):
                acc.update_from_passes(label[b], per_image[b])
        acc.all_reduce()
        return acc.miou()


class MscEvalV0_AutoLink:
    """evaluate.py:582-640 — rectangular ``[n_classes, n_cats_k]`` confusion matrices of this dataset's labels
    against the arg-max of every *other* dataset's head (first scale only, no flip); returns, per dataset, the
    row arg-max (identity rows for the dataset itself)."""

    def __init__(self, configer, scales=(0.5,), flip=False, ignore_label=255):
        self.configer, self.n_datasets = configer, configer.get('n_datasets')
        self.scales, self.flip, self.ignore_label = scales, flip, ignore_label

    @torch.no_grad()
    def __call__(self, net, dl, n_classes, dataset_id):
        dev = torch.device("cuda", torch.cuda.current_device())
        n_cats = [self.configer.get('dataset' + str(k + 1), 'n_cats') for k in range(self.n_datasets)]
        hists = [None if k == dataset_id else torch.zeros(n_classes, n_cats[k], dtype=torch.int64, device=dev)
                 for k in range(self.n_datasets)]
        scale = self.scales[0]
        for imgs, label in dl:
            N_, _, H, W = label.shape
            label = label.squeeze(1).to(dev, non_blocking=True)
            sH, sW = get_round_size((int(scale * H), int(scale * W)))
            im_sc = F.interpolate(imgs, size=(sH, sW), mode='bilinear', align_corners=True).to(dev)
            all_logits = net(im_sc)
            for k in range(self.n_datasets):
                if k == dataset_id:
                    continue
                for b in range(N_):
                    # softmax is monotone: arg-max of the up-sampled logits through the one-pass fused kernel
                    pred = ops.eval_fused([(all_logits[k][b], False)], (H, W))[0]
                    ops.confusion(label[b], pred, n_classes, n_cats[k], ignore=self.ignore_label, hist=hists[k])
        ops.check_errors(dev)
        eye = torch.eye(n_classes, device=dev)
        return [torch.argmax(eye if h is None else h, dim=1) for h in hists]


def target_bipart_from_hist(hist, bipart_graph, ignore_index=255):
    """The bucket rules of evaluate.py:1886-1925, vectorised on the device.  Every unified class (column) belongs to
    the dataset class with the largest graph weight (columns whose weights are all zero are skipped); within the
    bucket of class k a column u becomes 0 when it holds < 10 % of the bucket's pixels or class k is < 10 % of the
    pixels predicted as u, 1 when it holds > 50 % of the bucket, and stays `ignore_index` otherwise (also when the
    bucket saw no pixel).  `hist` is the [n_cats, C_uni] label x unified-prediction histogram."""
    h = hist.to(torch.float32)  # the reference accumulates in a float32 tensor (:1815)
    max_value, max_index = torch.max(bipart_graph, dim=0)
    cols = torch.arange(h.shape[1], device=h.device)
    valid = max_value != 0
    own = h[max_index, cols]
    total = torch.zeros(h.shape[0], dtype=torch.float32, device=h.device).index_add_(0, max_index[valid], own[valid])
    tot = total[max_index]
    rate, share = own / tot, own / h.sum(dim=0)
    zero = (rate < 0.1) | (share < 0.1)
    one = ~zero & (rate > 0.5)
    live = valid & (tot != 0)
    out = ignore_index * torch.ones_like(bipart_graph)
    val = torch.where(zero, torch.zeros_like(own), torch.where(one, torch.ones_like(own), ignore_index * torch.ones_like(own)))
    out[max_index[live], cols[live]] = val[live].to(out.dtype)
    return out


@torch.no_grad()
def eval_find_use_and_unuse_label(configer, net, dls=None):
    """evaluate.py:1788-1930 — per dataset the rectangular ``[n_cats, C_uni]`` histogram of the labels against the
    arg-max of the UNIFIED logits (prototype einsum -> bilinear up-sampling -> soft-max -> arg-max), then the
    bucket rules that produce ``target_bi_graph`` for the GNN stage.  The prototype einsum runs on tcgen05 (ops.prototype_head;
    a channels_last bf16 / fp16 embedding is read as it is, without a layout copy);
    up-sampling + arg-max (soft-max is monotone, no [C_uni, H, W] tensor) and the histogram run in libmdseg_b200.so.
    `dls` defaults to the reference's ``get_data_loader(configer, aux_mode='train', distributed=..., stage=2)``."""
    org_aux = net.aux_mode
    n_datasets = configer.get("n_datasets")
    ignore_index = configer.get('loss', 'ignore_index')
    net.aux_mode = 'train'
    net.eval()
    unify_prototype, bipart_graph = net.unify_prototype, net.bipartite_graphs
    if dls is None:
        from lib.get_dataloader import get_data_loader  # the reference's loaders
        dls = get_data_loader(configer, aux_mode='train', distributed=dist.is_initialized(), stage=2)
    total_cats = int(sum(configer.get("dataset" + str(i + 1), "n_cats") for i in range(n_datasets))
                     * configer.get('GNN', 'unify_ratio'))
    dev = torch.device("cuda", torch.cuda.current_device())
    target_bipart = []
    for i in range(n_datasets):
        n_classes = configer.get(f'dataset{i + 1}', 'n_cats')
        hist = torch.zeros(n_classes, total_cats, dtype=torch.int64, device=dev)
        for imgs, label in dls[i]:
            label = label.squeeze(1).to(dev, non_blocking=True)
            H, W = label.shape[-2:]
            emb = net(imgs.to(dev), dataset=i)
            logits = ops.prototype_head(emb['seg'], unify_prototype.to(dev))  # semseg.py:342-343 on tcgen05
            for b in range(label.shape[0]):
                pred = ops.eval_fused([(logits[b], False)], (H, W))[0]
                ops.confusion(label[b], pred, n_classes, total_cats, ignore=255, hist=hist)
        ops.check_errors(dev)
        target_bipart.append(target_bipart_from_hist(hist, bipart_graph[i].to(dev), ignore_index))
    net.aux_mode = org_aux
    return ['single_scale'], [], target_bipart
