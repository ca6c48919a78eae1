"""Torch-facing operators over the C ABI (``native.py``).

PyTorch is plumbing here: it owns device memory, streams and autograd
bookkeeping; every computation on the path is a hand-written sm_100a kernel in
libmdseg_b200.so.  Nothing in this module synchronises the host except
``check_errors`` (explicit) and the graph cache (only when a bipartite graph
tensor changed).
"""
import ctypes as C
import math

import numpy as np
import torch

from . import native as N

_DT = {
    torch.float32: N.F32, torch.bfloat16: N.BF16, torch.float16: N.F16,
    torch.uint8: N.U8, torch.int32: N.I32, torch.int64: N.I64,
}
STATE_BYTES = C.sizeof(N.OhemState)
assert STATE_BYTES == 128 == N.lib.mdseg_ohem_state_bytes()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return None if t is None else t.data_ptr()


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("mdseg_b200 ops run on CUDA tensors only (no CPU fallback)")


def _labels(lb):
    """Labels as a contiguous u8 / i32 / i64 tensor (reference labels are int64, transform_cv2.py:300)."""
    if lb.dtype not in (torch.uint8, torch.int32, torch.int64):
        lb = lb.long()
    return lb.contiguous()


_IDENTITY_LUT = {}


def _compact_labels(labels, c_max, ignore):
    """int labels -> uint8 once (the kernels stage label rows as bytes; 8x less label traffic in every later
    pass).  Values outside [0, 255] become a byte that is >= c_max and != ignore, so they are still flagged."""
    if labels.dtype == torch.uint8:
        return labels
    oob = 254 if ignore != 254 else 253
    if c_max > oob or not 0 <= ignore <= 255:
        return labels
    key = labels.device
    if key not in _IDENTITY_LUT:
        _IDENTITY_LUT[key] = torch.arange(256, dtype=torch.uint8, device=labels.device)
    return lut_remap(labels, _IDENTITY_LUT[key], out_dtype=torch.uint8, oob=oob)


# ---- lazily checked device-side data errors -----------------------------------
_err_flags = {}


def err_flag(device):
    key = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
    if key not in _err_flags:
        _err_flags[key] = torch.zeros(1, dtype=torch.int32, device=f"cuda:{key}")
    return _err_flags[key]


def check_errors(device=None):
    """Host sync.  Raises if any kernel since the last check saw a bad label / prediction / dataset id
    (the reference would have hit a device assert in nll_loss or a reshape error after np.bincount)."""
    flag = err_flag(device if device is not None else torch.cuda.current_device())
    v = int(flag.item())
    if v:
        flag.zero_()
        names = [n for n, bit in (("label out of range", 1), ("prediction out of range", 2),
                                  ("top-k larger than the loss vector", 4), ("dataset id out of range", 8),
                                  ("a graph declared column-one-hot 0/1 is not", 16)) if v & bit]
        raise RuntimeError("mdseg_b200 device-side data error: " + ", ".join(names))


def read_states(states):
    """Copy OHEM state(s) to the host (sync) as a list of native.OhemState — for tests / logging."""
    raw = states.detach().cpu().numpy().tobytes()
    n = len(raw) // STATE_BYTES
    return [N.OhemState.from_buffer_copy(raw[i * STATE_BYTES:(i + 1) * STATE_BYTES]) for i in range(n)]


# ---- a1 / a2: LUT remap ----------------------------------------------------------
def lut_remap(x, lut, out_dtype=None, oob=255):
    """out = lut[x] with a uint8[256] table (lib/base_dataset.py:81-82, lib/class_remap.py:34-66)."""
    _require_cuda(x)
    x = x.contiguous()
    if x.dtype not in (torch.uint8, torch.int32, torch.int64):
        raise TypeError(f"lut_remap: unsupported input dtype {x.dtype}")
    out_dtype = out_dtype or x.dtype
    lut = torch.as_tensor(lut).to(device=x.device, dtype=torch.uint8).contiguous()
    if lut.numel() != 256:
        raise ValueError("lut must have 256 entries")
    out = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    N.call("mdseg_lut_remap", _ptr(x), _DT[x.dtype], _ptr(out), _DT[out_dtype], _ptr(lut), int(oob), x.numel(),
           _stream())
    return out


# ---- a12 / a13: confusion matrix, mIoU ---------------------------------------------
def multihot_remap(labels, table):
    """bool [..., C_uni]: out[p, :] = table[labels[p], :] with a uint8 [256, C_uni] 0/1 table
    (ClassRemapOneHotLabel.SegRemapping / SingleSegRemappingOneHot, lib/class_remap.py:239-276)."""
    _require_cuda(labels)
    lab = _labels(labels)
    table = torch.as_tensor(table).to(device=lab.device, dtype=torch.uint8).contiguous()
    if table.dim() != 2 or table.shape[0] != 256:
        raise ValueError("table must be [256, C_uni]")
    Cu = table.shape[1]
    out = torch.empty(tuple(lab.shape) + (Cu,), dtype=torch.bool, device=lab.device)
    N.call("mdseg_multihot_remap", _ptr(lab), _DT[lab.dtype], _ptr(table), Cu, lab.numel(), _ptr(out), _stream())
    return out


def confusion(label, pred, n_a, n_b=None, lut=None, ignore=255, hist=None):
    """hist[l, p] += 1 for label != ignore (evaluate.py:89-93).  int64 [n_a, n_b], accumulated in place."""
    _require_cuda(label, pred)
    n_b = n_b or n_a
    label = _labels(label)
    pred = _labels(pred)
    if label.numel() != pred.numel():
        raise ValueError("label / pred size mismatch")
    if hist is None:
        hist = torch.zeros(n_a, n_b, dtype=torch.int64, device=label.device)
    if lut is not None:
        lut = torch.as_tensor(lut).to(device=label.device, dtype=torch.uint8).contiguous()
    N.call("mdseg_confusion", _ptr(label), _DT[label.dtype], _ptr(pred), _DT[pred.dtype], _ptr(lut), _ptr(hist),
           int(n_a), int(n_b), int(ignore), label.numel(), _ptr(err_flag(label.device)), _stream())
    return hist


def miou(hist):
    """(iou[C], miou) from an int64 [C, C] histogram, on the device (evaluate.py:94-98)."""
    _require_cuda(hist)
    Cn = hist.shape[0]
    iou = torch.empty(Cn, dtype=torch.float32, device=hist.device)
    m = torch.empty((), dtype=torch.float32, device=hist.device)
    N.call("mdseg_miou", _ptr(hist.contiguous()), Cn, _ptr(iou), _ptr(m), _stream())
    return iou, m


# ---- a1 / a12 / a13 for a whole multi-dataset batch: one launch each ---------------------------------------
def lut_remap_images(x, luts, lut_ids, out_dtype=None, oob=255):
    """out[b] = luts[lut_ids[b]][x[b]] for a batch [B, H, W] holding images of several datasets
    (one lb_map per dataset, lib/base_dataset.py:81-82).  luts: uint8 [n_luts, 256]."""
    _require_cuda(x)
    x = x.contiguous()
    if x.dtype not in (torch.uint8, torch.int32, torch.int64):
        raise TypeError(f"lut_remap_images: unsupported input dtype {x.dtype}")
    out_dtype = out_dtype or x.dtype
    luts = torch.as_tensor(luts).to(device=x.device, dtype=torch.uint8).contiguous()
    if luts.dim() != 2 or luts.shape[1] != 256:
        raise ValueError("luts must be [n_luts, 256]")
    B = x.shape[0]
    ids = _ids32(lut_ids, B, x.device)
    out = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    N.call("mdseg_lut_remap_images", _ptr(x), _DT[x.dtype], _ptr(out), _DT[out_dtype], _ptr(luts), luts.shape[0],
           _ptr(ids), int(oob), B, x[0].numel() if B else 0, _ptr(err_flag(x.device)), _stream())
    return out


def _hist_table(n_cats):
    tab = N.HistTable()
    tab.n_datasets = len(n_cats)
    off = 0
    for i, c in enumerate(n_cats):
        tab.C[i], tab.offset[i] = int(c), off
        off += int(c) * int(c)
    return tab, off


def confusion_images(label, pred, dataset_ids, n_cats, luts=None, ignore=255, hist=None):
    """Per-dataset square confusion matrices of a multi-dataset batch in ONE launch.  Returns (flat int64
    accumulator, [views [C_d, C_d]]); `hist` (flat) is accumulated into when given (evaluate.py:89-93)."""
    _require_cuda(label, pred)
    label, pred = _labels(label), _labels(pred)
    if label.shape != pred.shape:
        raise ValueError("label / pred shape mismatch")
    tab, total = _hist_table(n_cats)
    if hist is None:
        hist = torch.zeros(total, dtype=torch.int64, device=label.device)
    B = label.shape[0]
    ppi = label[0].numel() if B else 0
    if luts is not None:
        luts = torch.as_tensor(luts).to(device=label.device, dtype=torch.uint8).contiguous()
    if ppi % 16 or label.data_ptr() % 16 or pred.data_ptr() % 16:  # ragged images: one call per image
        ids = [int(v) for v in torch.as_tensor(dataset_ids).tolist()]
        for b, d in enumerate(ids):
            confusion(label[b], pred[b], n_cats[d], lut=None if luts is None else luts[d], ignore=ignore,
                      hist=hist[tab.offset[d]:tab.offset[d] + n_cats[d] ** 2].view(n_cats[d], n_cats[d]))
    else:
        ids = _ids32(dataset_ids, B, label.device)
        N.call("mdseg_confusion_images", _ptr(label), _DT[label.dtype], _ptr(pred), _DT[pred.dtype], _ptr(luts),
               _ptr(ids), B, ppi, _ptr(hist), C.byref(tab), int(ignore), _ptr(err_flag(label.device)), _stream())
    views = [hist[tab.offset[i]:tab.offset[i] + c * c].view(c, c) for i, c in enumerate(n_cats)]
    return hist, views


def miou_images(hist, n_cats):
    """(iou [n_datasets, max C] (NaN padded), miou [n_datasets]) from the flat accumulator of confusion_images."""
    _require_cuda(hist)
    tab, total = _hist_table(n_cats)
    if hist.numel() != total or hist.dtype != torch.int64:
        raise ValueError("hist must be the flat int64 accumulator of confusion_images")
    cm = max(n_cats)
    iou = torch.full((len(n_cats), cm), float("nan"), dtype=torch.float32, device=hist.device)
    m = torch.empty(len(n_cats), dtype=torch.float32, device=hist.device)
    N.call("mdseg_miou_images", _ptr(hist.contiguous()), C.byref(tab), _ptr(iou), cm, _ptr(m), _stream())
    return iou, m


# ---- OHEM state helpers ----------------------------------------------------------------
def _new_states(n, thresh, device):
    st = torch.empty(n * STATE_BYTES, dtype=torch.uint8, device=device)
    N.call("mdseg_ohem_begin", _ptr(st), n, float(thresh), _stream())
    return st


def _select(loss_px, n_images, px_per_image, image_seg, states, n_seg):
    ws = torch.empty(N.lib.mdseg_select_workspace_bytes(n_seg), dtype=torch.uint8, device=loss_px.device)
    out = torch.empty(n_seg, dtype=torch.float32, device=loss_px.device)
    N.call("mdseg_ohem_select", _ptr(loss_px), n_images, px_per_image, _ptr(image_seg), _ptr(states), n_seg, _ptr(ws),
           _ptr(out), _ptr(err_flag(loss_px.device)), _stream())
    return out


def _grad_scalar(g, n=1):
    g = g.detach().to(torch.float32).reshape(-1).contiguous()
    assert g.numel() == n
    return g


# ---- a7-a9: OhemCELoss on full-resolution logits -------------------------------------------
class _OhemCE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, labels, thresh, ignore):
        _require_cuda(logits, labels)
        if logits.dim() != 4:
            raise ValueError("logits must be [N, C, H, W]")
        Nn, Cc, H, W = logits.shape
        if logits.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            logits = logits.float()
        if logits.is_contiguous():
            layout = N.NCHW
        elif logits.is_contiguous(memory_format=torch.channels_last):
            layout = N.NHWC
        else:
            logits, layout = logits.contiguous(), N.NCHW
        labels = _labels(labels)
        if labels.numel() != Nn * H * W:
            raise ValueError(f"labels {tuple(labels.shape)} do not match logits {tuple(logits.shape)}")
        dev = logits.device
        P = Nn * H * W
        loss_px = torch.empty(P, dtype=torch.float32, device=dev)
        lse_px = torch.empty(P, dtype=torch.float32, device=dev)
        st = _new_states(1, thresh, dev)
        N.call("mdseg_ohem_ce_fwd", _ptr(logits), _DT[logits.dtype], layout, _ptr(labels), _DT[labels.dtype], Nn, Cc,
               H, W, int(ignore), _ptr(loss_px), _ptr(lse_px), _ptr(st), _ptr(err_flag(dev)), _stream())
        out = _select(loss_px, Nn, H * W, None, st, 1)
        ctx.save_for_backward(logits, labels, loss_px, lse_px, st)
        ctx.meta = (layout, int(ignore))
        ctx.states = st
        return out[0]

    @staticmethod
    def backward(ctx, grad_out):
        logits, labels, loss_px, lse_px, st = ctx.saved_tensors
        layout, ignore = ctx.meta
        Nn, Cc, H, W = logits.shape
        g = _grad_scalar(grad_out)
        dl = torch.empty_like(logits)  # preserves the memory format
        N.call("mdseg_ohem_ce_bwd", _ptr(logits), _DT[logits.dtype], layout, _ptr(labels), _DT[labels.dtype], Nn, Cc,
               H, W, ignore, _ptr(loss_px), _ptr(lse_px), _ptr(st), _ptr(g), 1.0, _ptr(dl), _stream())
        return dl, None, None, None


def ohem_ce(logits, labels, thresh, ignore=255):
    """mean over the OHEM set of CE(logits, labels); `thresh` is already -log(p) (ohem_ce_loss.py:17,21-34)."""
    return _OhemCE.apply(logits, labels, float(thresh), int(ignore))


def ohem_ce_with_state(logits, labels, thresh, ignore=255):
    """Forward only; returns (loss, loss_px, OhemState) — for tests and logging (host sync)."""
    with torch.no_grad():
        class _Ctx:
            def save_for_backward(self, *a):
                self.saved = a
        ctx = _Ctx()
        loss = _OhemCE.forward(ctx, logits, labels, float(thresh), int(ignore))
        return loss, ctx.saved[2], read_states(ctx.saved[4])[0]


# ---- MdsOhemCELoss on full-resolution per-dataset logits (the reference module's own call form) ---------------
class _MdsOhemCEFull(torch.autograd.Function):
    """One OHEM selection over the concatenation of per-dataset CE vectors (lib/loss/ohem_ce_loss.py:48-90).
    logits[k]: [B_k, C_k, H, W]; labels[k]: [B_k, H, W], in the same (ascending dataset id) order."""

    @staticmethod
    def forward(ctx, thresh, ignore, n, *tensors):
        logits, labels = list(tensors[:n]), [_labels(t) for t in tensors[n:]]
        _require_cuda(*logits, *labels)
        dev = logits[0].device
        H, W = logits[0].shape[2:]
        metas, offs, P = [], [], 0
        for k in range(n):
            lg = logits[k]
            if lg.dtype not in (torch.float32, torch.bfloat16, torch.float16):
                lg = lg.float()
            if lg.is_contiguous():
                layout = N.NCHW
            elif lg.is_contiguous(memory_format=torch.channels_last):
                layout = N.NHWC
            else:
                lg, layout = lg.contiguous(), N.NCHW
            if tuple(lg.shape[2:]) != (H, W) or labels[k].numel() != lg.shape[0] * H * W:
                raise ValueError("every dataset's logits / labels must share H x W")
            logits[k] = lg
            metas.append(layout)
            offs.append(P)
            P += lg.shape[0] * H * W
        loss_px = torch.empty(P, dtype=torch.float32, device=dev)
        lse_px = torch.empty(P, dtype=torch.float32, device=dev)
        st = _new_states(1, thresh, dev)
        for k in range(n):
            lg = logits[k]
            N.call("mdseg_ohem_ce_fwd", _ptr(lg), _DT[lg.dtype], metas[k], _ptr(labels[k]), _DT[labels[k].dtype],
                   lg.shape[0], lg.shape[1], H, W, int(ignore), loss_px.data_ptr() + 4 * offs[k],
                   lse_px.data_ptr() + 4 * offs[k], _ptr(st), _ptr(err_flag(dev)), _stream())
        out = _select(loss_px, P // (H * W), H * W, None, st, 1)
        ctx.save_for_backward(loss_px, lse_px, st, *logits, *labels)
        ctx.meta = (n, metas, offs, int(ignore), H, W)
        ctx.states = st
        return out[0]

    @staticmethod
    def backward(ctx, grad_out):
        n, metas, offs, ignore, H, W = ctx.meta
        loss_px, lse_px, st = ctx.saved_tensors[:3]
        logits, labels = ctx.saved_tensors[3:3 + n], ctx.saved_tensors[3 + n:]
        g = _grad_scalar(grad_out)
        grads = []
        for k in range(n):
            lg = logits[k]
            dl = torch.empty_like(lg)
            N.call("mdseg_ohem_ce_bwd", _ptr(lg), _DT[lg.dtype], metas[k], _ptr(labels[k]), _DT[labels[k].dtype],
                   lg.shape[0], lg.shape[1], H, W, ignore, loss_px.data_ptr() + 4 * offs[k],
                   lse_px.data_ptr() + 4 * offs[k], _ptr(st), _ptr(g), 1.0, _ptr(dl), _stream())
            grads.append(dl)
        return (None, None, None, *grads, *([None] * n))


def mds_ohem_ce_full(logits, labels, thresh, ignore=255):
    """logits: list of [B_k, C_k, H, W]; labels: list of [B_k, H, W] — one OHEM selection over all of them."""
    if not logits:
        return torch.tensor(float("nan"))
    return _MdsOhemCEFull.apply(float(thresh), int(ignore), len(logits), *logits, *labels)


# ---- bipartite graphs: host-side cache of the CSR / CSC device images -------------------------
class BipartiteGraphs:
    """Device descriptors of bi_graphs[i] ([C_ds_i, C_uni]) for mdseg_proj_*.

    A graph is stored sparse (CSR + CSC) when at most `dense_frac` of its
    entries are non-zero and it does not require grad (SEG stage: 0/1 graphs
    from UOT / pretrain, lib/models/ltbgnn_direct_learn.py:426-439, or
    ClassRemap.getRemapMatrix, lib/class_remap.py:176-183); otherwise dense (GNN
    stage).  Rebuilding needs one D2H copy and happens only when the tensor
    object, its version counter or its storage changed.  The cache keeps a
    reference to the tensor it was built from, so a recycled allocation can never
    alias a stale entry; writes that bypass autograd's version counter
    (``g.data[...] = ``) need an explicit ``invalidate()``.
    """

    def __init__(self, dense_frac=0.25, assume_dense=False, assume_onehot01=False):
        self.dense_frac = dense_frac
        self.assume_dense = assume_dense  # every graph is a real matrix (folded prototypes): never copied to the host
        # every non-trainable graph is 0/1 with at most one 1 per column (SEG-stage graphs, single-label remap matrices):
        # its index lists are built on the device (mdseg_graph_build_onehot), no host copy; a graph that is not of that
        # kind raises at the next check_errors()
        self.assume_onehot01 = assume_onehot01
        self._cache = {}

    def invalidate(self):
        self._cache.clear()

    def _entry(self, i, g):
        key = (id(g), g.data_ptr(), g._version, tuple(g.shape), g.requires_grad, str(g.device))
        hit = self._cache.get(i)
        if hit is not None and hit["key"] == key:
            return hit
        if g.dim() != 2:
            raise ValueError("bi_graph must be [C_ds, C_uni]")
        dev = g.device
        ent = {"key": key, "tensor": g, "C_ds": g.shape[0], "C_uni": g.shape[1]}
        if g.requires_grad or self.assume_dense:
            # trainable graph (GNN stage): dense by definition, decided without copying it to the host —
            # it changes every iteration and a D2H copy per graph per step would serialise the stream
            ent["dense"], ent["nnz"] = True, g.shape[0] * g.shape[1]
            self._cache[i] = ent
            return ent
        if self.assume_onehot01:
            c_ds, c_uni = g.shape
            r4 = lambda k: (k + 3) & ~3
            buf = torch.empty(N.lib.mdseg_graph_build_onehot_ints(c_ds, c_uni), dtype=torch.int32, device=dev)
            g32 = g.detach().to(torch.float32).contiguous()
            N.call("mdseg_graph_build_onehot", _ptr(g32), c_ds, c_uni, _ptr(buf), _ptr(err_flag(dev)), _stream())
            o = 0
            for name, n in (("csr_ptr", c_ds + 1), ("csc_ptr", c_uni + 1), ("csr4_ptr", c_ds + 1), ("csr_col", c_uni),
                            ("csc_row", c_uni), ("csr4_col", c_uni + 3 * c_ds)):
                ent[name] = buf[o:o + n]
                o += r4(n)
            ent.update(dense=False, nnz=c_uni, csr_val=None, csc_val=None, col_onehot=1, buf=buf)  # nnz: upper bound
            self._cache[i] = ent
            return ent
        m = g.detach().to(torch.float32).cpu().numpy()
        nz = m != 0
        nnz = int(nz.sum())
        if g.requires_grad or nnz > self.dense_frac * m.size:
            ent["dense"] = True
            ent["nnz"] = nnz
        else:
            ent["dense"] = False
            ent["nnz"] = nnz
            rows, cols = np.nonzero(nz)  # row-major order: ascending col within a row
            vals = m[rows, cols]
            csr_ptr = np.zeros(m.shape[0] + 1, dtype=np.int32)
            np.cumsum(np.bincount(rows, minlength=m.shape[0]), out=csr_ptr[1:])
            order = np.lexsort((rows, cols))  # by column, then row
            csc_ptr = np.zeros(m.shape[1] + 1, dtype=np.int32)
            np.cumsum(np.bincount(cols, minlength=m.shape[1]), out=csc_ptr[1:])
            all_ones = bool(np.all(vals == 1.0))
            t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a.astype(dt))).to(dev)
            ent["csr_ptr"] = t(csr_ptr, np.int32)
            ent["csr_col"] = t(cols, np.int32)
            ent["csc_ptr"] = t(csc_ptr, np.int32)
            ent["csc_row"] = t(rows[order], np.int32)
            ent["csr_val"] = None if all_ones else t(vals, np.float32)
            ent["csc_val"] = None if all_ones else t(vals[order], np.float32)
            ent["col_onehot"] = int(np.all(np.diff(csc_ptr) <= 1))
            # rows padded to quads (last entry repeated) for the fused backward's channel broadcast
            nq = (np.diff(csr_ptr) + 3) // 4
            csr4_ptr = np.zeros(m.shape[0] + 1, dtype=np.int32)
            np.cumsum(nq, out=csr4_ptr[1:])
            csr4_col = np.zeros(4 * int(csr4_ptr[-1]), dtype=np.int32)
            for r in range(m.shape[0]):
                seg = cols[csr_ptr[r]:csr_ptr[r + 1]]
                if len(seg):
                    dst = csr4_col[4 * csr4_ptr[r]:4 * csr4_ptr[r + 1]]
                    dst[:len(seg)] = seg
                    dst[len(seg):] = seg[-1]
            ent["csr4_ptr"] = t(csr4_ptr, np.int32)
            ent["csr4_col"] = t(csr4_col, np.int32) if csr4_col.size else torch.zeros(4, dtype=torch.int32, device=dev)
        self._cache[i] = ent
        return ent

    def table(self, graphs):
        """(GraphTable, keepalive list) for a list of graph tensors."""
        if len(graphs) > N.MAX_DATASETS:
            raise ValueError("too many datasets")
        tab = N.GraphTable()
        tab.n_datasets = len(graphs)
        keep = []
        c_uni = None
        for i, g in enumerate(graphs):
            _require_cuda(g)
            e = self._entry(i, g)
            c_uni = e["C_uni"] if c_uni is None else c_uni
            if e["C_uni"] != c_uni:
                raise ValueError("all graphs must share C_uni")
            sg = tab.g[i]
            sg.C_ds, sg.nnz = e["C_ds"], e["nnz"]
            if e["dense"]:
                d = g.detach().to(torch.float32).contiguous()
                keep.append(d)
                sg.dense = d.data_ptr()
            else:
                sg.csr_ptr, sg.csr_col = e["csr_ptr"].data_ptr(), e["csr_col"].data_ptr()
                sg.csc_ptr, sg.csc_row = e["csc_ptr"].data_ptr(), e["csc_row"].data_ptr()
                sg.csr_val = _ptr(e["csr_val"])
                sg.csc_val = _ptr(e["csc_val"])
                sg.col_onehot = e["col_onehot"]
                sg.csr4_ptr, sg.csr4_col = e["csr4_ptr"].data_ptr(), e["csr4_col"].data_ptr()
                keep.append(e)
        tab.C_uni = c_uni
        return tab, keep


_default_graphs = BipartiteGraphs()


def _ids32(dataset_ids, n, device):
    if dataset_ids is None:
        return None
    ids = torch.as_tensor(dataset_ids, device=device)
    if ids.numel() != n:
        raise ValueError("dataset_ids must have one entry per image")
    return ids.to(torch.int32).contiguous()


def _src_table(bases, strides, Cs, dtype, seg_per_dataset, c_alloc=None, cmax=None, cmax_ready=False):
    t = N.SrcTable()
    t.n_datasets = len(bases)
    t.dtype = dtype
    t.seg_per_dataset = int(seg_per_dataset)
    t.cmax = _ptr(cmax)
    t.cmax_ready = int(cmax_ready)
    for i, (b, s, c) in enumerate(zip(bases, strides, Cs)):
        t.base[i] = b
        t.image_stride[i] = s
        t.C[i] = c
        ca = c_alloc[i] if isinstance(c_alloc, (list, tuple)) else c_alloc
        t.C_alloc[i] = ca if ca else c
    return t


def _channels_last(x):
    """A 4-D tensor that is channels_last-contiguous and not NCHW-contiguous (the layout decision of ohem_ce: shapes that
    are both, C = 1 or h * w = 1, count as NCHW)."""
    return x.dim() == 4 and not x.is_contiguous() and x.is_contiguous(memory_format=torch.channels_last)


def _nhwc_proj_ok(x, tab):
    """channels_last logits with sparse graphs inside the limits of mdseg_proj_fwd_nhwc / mdseg_proj_bwd_nhwc: the
    projection reads x as it is.  Anything else (dense graphs included) takes the NCHW kernels on x.contiguous()."""
    return (_channels_last(x) and tab.C_uni <= N.NHWC_MAX_CUNI
            and all(not tab.g[i].dense and tab.g[i].C_ds <= N.NHWC_MAX_CDS for i in range(tab.n_datasets)))


def _tc16_layout(x):
    """The layout (N.NCHW / N.NHWC) in which the TMA-fed tcgen05 kernels (mdseg_proj_*_tc16) read 16-bit x as it lies,
    or None: bf16 / fp16, h * w a multiple of 8 (the planar y / dy), a 16-byte-aligned base, and NCHW-contiguous or
    channels_last with a channel count that is a multiple of 8 (16-byte TMA pixel stride)."""
    if x.dtype not in (torch.bfloat16, torch.float16) or (x.shape[2] * x.shape[3]) % 8 or x.data_ptr() % 16:
        return None
    if _channels_last(x):
        return N.NHWC if x.shape[1] % 8 == 0 else None
    return N.NCHW if x.is_contiguous() else None


def _tc16_envelope(c_uni, c_ds, n_heads=1):
    """Graph sizes the projection runs on the tc16 kernels for: C_uni >= 32 and, per dataset, C_ds >= 8 and
    n_heads * C_ds <= 1024 (the dataset's graphs of n_heads sets stacked into one operand)."""
    return c_uni >= 32 and all(8 <= c and n_heads * c <= 1024 for c in c_ds)


def _dense_tc16(tab):
    """Every graph of the table dense and inside _tc16_envelope."""
    n = tab.n_datasets
    return all(tab.g[i].dense for i in range(n)) and _tc16_envelope(tab.C_uni, [tab.g[i].C_ds for i in range(n)])


def _tc16_operands(mats, dtype, transpose=False):
    """The B operands of the mdseg_proj_*_tc16 kernels for matrices M_d (or M_d^T with `transpose`) in one zero-filled
    buffer: each in `dtype`, its rows padded to whole N tiles (mdseg_head_tc16_tile), its columns to ldb (the widest
    matrix rounded up to a multiple of 8).  -> (buffer, host array of the operands' pointers, ldb)"""
    mats = [m.detach().t() if transpose else m.detach() for m in mats]
    ldb = (max(m.shape[1] for m in mats) + 7) // 8 * 8
    rows = []
    for m in mats:
        nt = N.lib.mdseg_head_tc16_tile(m.shape[0])
        rows.append((m.shape[0] + nt - 1) // nt * nt)
    buf = torch.zeros(sum(rows), ldb, dtype=dtype, device=mats[0].device)
    ptrs = (C.c_void_p * len(mats))()
    o = 0
    for i, m in enumerate(mats):
        buf[o:o + m.shape[0], :m.shape[1]] = m.to(dtype)
        ptrs[i] = buf.data_ptr() + o * ldb * buf.element_size()
        o += rows[i]
    return buf, ptrs, ldb


# ---- a5 projection alone (model-side eval einsum, semseg.py:342-345) --------------------------------
def project(logits_uni, graphs, dataset_ids=None, cache=None):
    """fp32 [B, max C_ds, h, w]: einsum('bchw,nc->bnhw') with the graph of each image's dataset.  channels_last logits
    with sparse graphs are read as they are (no layout copy)."""
    _require_cuda(logits_uni)
    graphs = list(graphs)
    tab, keep = (cache or _default_graphs).table(graphs)
    x = logits_uni if _nhwc_proj_ok(logits_uni, tab) else logits_uni.contiguous()
    B, Cu, h, w = x.shape
    if tab.C_uni != Cu:
        raise ValueError(f"graphs have C_uni={tab.C_uni}, logits have {Cu}")
    cmax = max(g.shape[0] for g in graphs)
    ids = _ids32(dataset_ids, B, x.device)
    y = torch.empty(B, cmax, h, w, dtype=torch.float32, device=x.device)
    _proj_fwd(x, tab, graphs, ids, y, None, err_flag(x.device), _tc16_layout(x) is not None and _dense_tc16(tab))
    return y


def _proj_fwd(x, tab, graphs, ids, y, ymax, ef, tc16):
    """y[b] = G_d x[b], d = ids[b], into fp32 planes y [B, cmax, h, w] (and, unless tc16, their channel maximum into
    ymax when given).  tc16 (the caller's route: 16-bit x with _tc16_layout, graphs that the backward will take the same
    way): mdseg_proj_fwd_tc16 in x's layout.  Otherwise mdseg_proj_fwd_nhwc (channels_last x, which callers pass only
    with sparse graphs inside _nhwc_proj_ok), mdseg_proj_fwd_tc (a dense graph, on the tensor cores) or mdseg_proj_fwd."""
    B, _, h, w = x.shape
    cmax = y.shape[1]
    if tc16:
        n = len(graphs)
        buf, ptrs, ldb = _tc16_operands(graphs, x.dtype)
        N.call("mdseg_proj_fwd_tc16", _ptr(x), _DT[x.dtype], _tc16_layout(x), B, x.shape[1], h * w, ptrs, ldb,
               (C.c_int * n)(*[g.shape[0] for g in graphs]), n, _ptr(ids), _ptr(y), cmax, _stream())
    elif _channels_last(x):
        N.call("mdseg_proj_fwd_nhwc", _ptr(x), _DT[x.dtype], C.byref(tab), _ptr(ids), B, h, w, _ptr(y), cmax, _ptr(ymax),
               _ptr(ef), _stream())
    elif any(tab.g[i].dense for i in range(tab.n_datasets)):
        nbytes = N.lib.mdseg_proj_fwd_tc_workspace_bytes(C.byref(tab), _DT[x.dtype])
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        N.call("mdseg_proj_fwd_tc", _ptr(x), _DT[x.dtype], C.byref(tab), _ptr(ids), B, h, w, _ptr(y), cmax, _ptr(ymax),
               _ptr(ws), nbytes, _ptr(ef), _stream())
    else:
        N.call("mdseg_proj_fwd", _ptr(x), _DT[x.dtype], C.byref(tab), _ptr(ids), B, h, w, _ptr(y), cmax, _ptr(ymax),
               _ptr(ef), _stream())


def _proj_bwd(dy, dyB, graphs, tab, ids, dx):
    """The adjoint of _proj_fwd: dx[b] = G_d^T (dy[b] + dyB[b]), d = ids[b], into dx (its layout and dtype).  16-bit dy
    (the dtype of x, from a backward that took the tc16 route; dyB None): mdseg_proj_bwd_tc16.  fp32 planes:
    mdseg_proj_bwd_nhwc (channels_last dx, sparse graphs), mdseg_proj_bwd_tc (a dense graph) or mdseg_proj_bwd."""
    B, Cu, h, w = dx.shape
    cmax = dy.shape[1]
    if dy.dtype != torch.float32:
        buf, ptrs, ldb = _tc16_operands(graphs, dy.dtype, transpose=True)
        N.call("mdseg_proj_bwd_tc16", _ptr(dy), _DT[dy.dtype], N.NHWC if _channels_last(dx) else N.NCHW, B, cmax, h * w,
               ptrs, ldb, Cu, len(graphs), _ptr(ids), _ptr(dx), _DT[dx.dtype], _stream())
    elif _channels_last(dx):
        N.call("mdseg_proj_bwd_nhwc", _ptr(dy), _ptr(dyB), cmax, C.byref(tab), _ptr(ids), B, h, w, _ptr(dx),
               _DT[dx.dtype], _stream())
    elif any(tab.g[i].dense for i in range(tab.n_datasets)):
        nb = N.lib.mdseg_proj_bwd_tc_workspace_bytes(C.byref(tab), _DT[dx.dtype])
        ws = torch.empty(nb, dtype=torch.uint8, device=dx.device)
        N.call("mdseg_proj_bwd_tc", _ptr(dy), _ptr(dyB), cmax, C.byref(tab), _ptr(ids), B, h, w, _ptr(dx), _DT[dx.dtype],
               _ptr(ws), nb, _stream())
    else:
        N.call("mdseg_proj_bwd", _ptr(dy), _ptr(dyB), cmax, C.byref(tab), _ptr(ids), B, h, w, _ptr(dx), _DT[dx.dtype],
               _stream())


def _proj_bwd_graph(x, dy, dyB, graphs, tab, ids):
    """The graph gradients of _proj_fwd: dG[d] = sum over the images of dataset d of (dy + dyB) x^T, fp32
    [n_datasets, cmax, C_uni].  16-bit dy (see _proj_bwd): mdseg_proj_bwd_graph_tc16 with x in its layout.  fp32
    planes: mdseg_proj_bwd_graph_tc (a dense graph) or mdseg_proj_bwd_graph."""
    B, Cu, h, w = x.shape
    n, cmax = len(graphs), dy.shape[1]
    if dy.dtype != torch.float32:
        if ids is None and n > 1:  # every image belongs to dataset 0; the other datasets get zeros
            ids = torch.zeros(B, dtype=torch.int32, device=x.device)
        dG = torch.empty(n, cmax, Cu, dtype=torch.float32, device=x.device)
        nb = N.lib.mdseg_proj_bwd_graph_tc16_workspace_bytes(B, Cu, h * w, cmax)
        ws = torch.empty(nb, dtype=torch.uint8, device=x.device)
        N.call("mdseg_proj_bwd_graph_tc16", _ptr(dy), _ptr(x), _DT[x.dtype], _tc16_layout(x), B, Cu, h * w, cmax,
               _ptr(ids), n, _ptr(dG), _ptr(ws), nb, _stream())
        return dG
    stride = cmax * Cu
    dG = torch.zeros(n, stride, dtype=torch.float32, device=x.device)
    if any(tab.g[i].dense for i in range(tab.n_datasets)):  # dense graphs: split-K GEMM on the tensor cores
        nb = N.lib.mdseg_proj_bwd_graph_tc_workspace_bytes(C.byref(tab), B, h, w)
        ws = torch.empty(nb, dtype=torch.uint8, device=x.device)
        N.call("mdseg_proj_bwd_graph_tc", _ptr(x), _DT[x.dtype], _ptr(dy), _ptr(dyB), cmax, C.byref(tab), _ptr(ids), B,
               h, w, _ptr(dG), stride, _ptr(ws), nb, _stream())
    else:
        N.call("mdseg_proj_bwd_graph", _ptr(x), _DT[x.dtype], _ptr(dy), _ptr(dyB), cmax, C.byref(tab), _ptr(ids), B, h,
               w, _ptr(dG), stride, _stream())
    return dG.view(n, cmax, Cu)


# ---- f2: the prototype head (producer of the unified logits) on the tcgen05 tensor cores ---------------------------
def _dense_table(weight):
    """GraphTable holding one dense matrix [n_rows, K] (no host copy, no density test)."""
    tab = N.GraphTable()
    tab.n_datasets = 1
    tab.C_uni = weight.shape[1]
    tab.g[0].C_ds, tab.g[0].nnz = weight.shape[0], weight.shape[0] * weight.shape[1]
    tab.g[0].dense = weight.data_ptr()
    return tab


class _PrototypeHead(torch.autograd.Function):
    """logits[b, n, y, x] = sum_c feats[b, c, y, x] * proto[n, c]: torch.einsum('bchw,nc->bnhw', feats, unify_prototype)
    of lib/models/semseg.py:325-333,342-343 and lib/loss/loss_cross_datasets.py:950,961,971: the projection with the
    prototypes as the one dense graph.  bf16 / fp16 features that _tc16_layout reads as they lie (NCHW or channels_last)
    take the TMA-fed tcgen05 kernels (mdseg_proj_*_tc16, one product in their own type, like autocast; d feats in the
    layout of feats, bit-identical between the two layouts); other features are made NCHW-contiguous and take
    mdseg_proj_*_tc (fp32: three bf16 terms per operand, 1e-5 bar).  Backward: d feats = proto^T dlogits, d proto =
    dlogits feats^T as a split-K GEMM over the pixels.  Output fp32 NCHW."""

    @staticmethod
    def forward(ctx, feats, proto):
        _require_cuda(feats, proto)
        x = feats
        if x.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            x = x.float()
        if _tc16_layout(x) is None:
            x = x.contiguous()
        B, K, h, w = x.shape
        if proto.dim() != 2 or proto.shape[1] != K:
            raise ValueError(f"prototypes must be [N, {K}]")
        wgt = proto.detach().to(torch.float32).contiguous()
        y = torch.empty(B, wgt.shape[0], h, w, dtype=torch.float32, device=x.device)
        ctx.save_for_backward(x, wgt)
        ctx.proto_dtype = proto.dtype
        _proj_fwd(x, _dense_table(wgt), [wgt], None, y, None, err_flag(x.device), _tc16_layout(x) is not None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, wgt = ctx.saved_tensors
        tab = _dense_table(wgt)
        dy = dy.to(torch.float32).contiguous()
        if _tc16_layout(x) is not None:  # rounded to the feature dtype, as the reference's autocast backward does
            dy = dy.to(x.dtype)
        dx = dw = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)  # the layout of x
            _proj_bwd(dy, None, [wgt], tab, None, dx)
        if ctx.needs_input_grad[1]:
            dw = _proj_bwd_graph(x, dy, None, [wgt], tab, None)[0].to(ctx.proto_dtype)
        return dx, dw


def prototype_head(feats, proto):
    """einsum('bchw,nc->bnhw', feats [B, K, h, w], proto [N, K]) -> fp32 [B, N, h, w] (NCHW) on the tensor cores.
    channels_last bf16 / fp16 features with K % 8 == 0 are read without a layout copy."""
    return _PrototypeHead.apply(feats, proto)


# ---- a5+a6+a7+a8+a9: the fused multi-dataset loss ------------------------------------------------------
class _MdsProjOhemCE(torch.autograd.Function):
    """MdsOhemCELoss(project -> upsample -> CE) of loss_cross_datasets.py:1006-1007,1074 in four kernels.  channels_last
    logits with sparse graphs are projected as they are and get a channels_last gradient (mdseg_proj_*_nhwc); so are
    channels_last 16-bit logits / features with dense graphs (folded prototypes, trainable graphs) when the backward takes
    the tc16 route (mdseg_proj_*_tc16 with layout NHWC)."""

    @staticmethod
    def forward(ctx, logits_uni, labels, dataset_ids, thresh, ignore, cache, per_dataset, *graphs):
        _require_cuda(logits_uni, labels)
        x = logits_uni
        if x.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            x = x.float()
        B, Cu, h, w = x.shape
        labels = _labels(labels)
        if labels.dim() != 3 or labels.shape[0] != B:
            raise ValueError("labels must be [B, H, W]")
        H, W = labels.shape[1:]
        dev = x.device
        labels = _compact_labels(labels, max(g.shape[0] for g in graphs), ignore)
        tab, keep = cache.table(list(graphs))
        if tab.C_uni != Cu:
            raise ValueError(f"graphs have C_uni={tab.C_uni}, logits have {Cu}")
        Cs = [g.shape[0] for g in graphs]
        cmax = max(Cs)
        ids = _ids32(dataset_ids, B, dev)
        ef = err_flag(dev)
        y = torch.empty(B, cmax, h, w, dtype=torch.float32, device=dev)
        ymax = torch.empty(B, h, w, dtype=torch.float32, device=dev)  # channel maximum of y: the softmax shift
        all_sparse = all(not tab.g[i].dense for i in range(len(Cs)))
        n_seg = len(Cs) if per_dataset else 1
        src = _src_table([y.data_ptr()] * len(Cs), [cmax * h * w] * len(Cs), Cs, N.F32, per_dataset, c_alloc=cmax,
                         cmax=ymax, cmax_ready=all_sparse)
        tc16 = _dense_tc16(tab)
        if not (_nhwc_proj_ok(x, tab)
                or (tc16 and _tc16_layout(x) == N.NHWC and _tc16_bwd_nhwc_ok(ctx, len(Cs), src, h, w, H, W))):
            x = x.contiguous()
        _proj_fwd(x, tab, graphs, ids, y, ymax, ef, tc16 and _tc16_layout(x) is not None)
        P = B * H * W
        loss_px = torch.empty(P, dtype=torch.float32, device=dev)
        lse_px = torch.empty(P, dtype=torch.float32, device=dev)
        st = _new_states(n_seg, thresh, dev)
        N.call("mdseg_up_ce_fwd", C.byref(src), _ptr(ids), _ptr(labels), _DT[labels.dtype], B, h, w, H, W, int(ignore),
               _ptr(loss_px), _ptr(lse_px), _ptr(st), _ptr(ef), _stream())
        out = _select(loss_px, B, H * W, ids if per_dataset else None, st, n_seg)
        ctx.save_for_backward(x, labels, ids, y, loss_px, lse_px, st, *graphs)
        ctx.meta = (int(ignore), cache, Cs, cmax, (h, w, H, W), bool(per_dataset))
        ctx.states = st
        ctx.mark_non_differentiable(st)
        return (out if per_dataset else out[0]), st

    @staticmethod
    def backward(ctx, grad_out, _grad_states=None):
        x, labels, ids, y, loss_px, lse_px, st, *graphs = ctx.saved_tensors
        ignore, cache, Cs, cmax, (h, w, H, W), per_dataset = ctx.meta
        B = x.shape[0]
        dev = x.device
        n = len(Cs)
        g = _grad_scalar(grad_out, n if per_dataset else 1)
        tab, keep = cache.table(list(graphs))
        scratch = torch.empty(1, dtype=torch.float32, device=dev)  # non-NULL cmax selects the TMA kernels
        src = _src_table([y.data_ptr()] * n, [cmax * h * w] * n, Cs, N.F32, per_dataset, c_alloc=cmax, cmax=scratch,
                         cmax_ready=True)
        adj = (src, ids, labels, (B, h, w, H, W), ignore, loss_px, lse_px, st, g)
        want_dg = any(ctx.needs_input_grad[7 + i] for i in range(n))
        dx = None
        if not want_dg:
            if ctx.needs_input_grad[0] and _channels_last(x):
                # channels_last logits (sparse graphs, see forward): d loss / d y from the upsample + CE adjoint, then the
                # broadcast through G^T written pixel-major
                dx = torch.empty_like(x)  # channels_last
                _proj_bwd(*_mds_dy(*adj, y, Cs, cmax), graphs, tab, ids, dx)
            elif ctx.needs_input_grad[0]:
                # one call: softmax recompute + adjoint of the upsample + broadcast through G^T (fused when it applies)
                nbytes = N.lib.mdseg_mds_bwd_workspace_bytes(C.byref(src), C.byref(tab), B, h, w, H, W)
                ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
                dx = torch.empty_like(x)
                N.call("mdseg_mds_bwd", C.byref(src), C.byref(tab), _ptr(ids), _ptr(labels), _DT[labels.dtype], B, h,
                       w, H, W, ignore, _ptr(loss_px), _ptr(lse_px), _ptr(st), _ptr(g), 1.0, _ptr(dx), _DT[x.dtype],
                       _ptr(ws), nbytes, _stream())
            return (dx, None, None, None, None, None, None, *([None] * n))
        if (N.lib.mdseg_up_ce_bwd_direct_is_fused(C.byref(src), h, w, H, W) and _tc16_layout(x) is not None
                and _dense_tc16(tab)):
            # 16-bit logits / features with dense graphs (AMP GNN stage, folded prototypes): d loss / d y leaves the fused
            # kernel in the dtype of x (what autocast's backward rounds it to) and both adjoints of the projection run
            # on the TMA-fed tcgen05 kernels — no register-staged conversion, one launch for all datasets each.
            dy, dyB = torch.zeros(B, cmax, h, w, dtype=x.dtype, device=dev), None  # planes >= C_ds of an image stay 0
            _up_ce_adjoint(*adj, _src_table([dy.data_ptr()] * n, [cmax * h * w] * n, Cs, _DT[x.dtype], False))
        else:
            dy, dyB = _mds_dy(*adj, y, Cs, cmax)
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            _proj_bwd(dy, dyB, graphs, tab, ids, dx)
        dG = _proj_bwd_graph(x, dy, dyB, graphs, tab, ids)
        dgs = [dG[i, :Cs[i]].to(graphs[i].dtype) if ctx.needs_input_grad[7 + i] else None for i in range(n)]
        return (dx, None, None, None, None, None, None, *dgs)


def _tc16_bwd_nhwc_ok(ctx, n, src, h, w, H, W):
    """_MdsProjOhemCE with channels_last x in the tc16 route of the forward: the backward reads x only on its tc16 branch — taken
    when a graph wants a gradient and the upsample + CE adjoint is the fused kernel — or never runs (no input wants a
    gradient).  A d x without d graphs goes through mdseg_mds_bwd, which writes dx planar, so x is copied then."""
    want_dg = any(ctx.needs_input_grad[7 + i] for i in range(n))
    if not want_dg:
        return not ctx.needs_input_grad[0]
    return bool(N.lib.mdseg_up_ce_bwd_direct_is_fused(C.byref(src), h, w, H, W))


def _up_ce_adjoint(src, ids, labels, shape, ignore, loss_px, lse_px, st, g, dst):
    """mdseg_up_ce_bwd_direct: d loss / d (the low-resolution rows src describes) of the fused upsample + CE under the
    selection in st, into the rows dst describes."""
    B, h, w, H, W = shape
    nbytes = N.lib.mdseg_up_ce_bwd_direct_workspace_bytes(C.byref(src), B, h, w, H, W)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=labels.device)
    N.call("mdseg_up_ce_bwd_direct", C.byref(src), _ptr(ids), _ptr(labels), _DT[labels.dtype], B, h, w, H, W, ignore,
           _ptr(loss_px), _ptr(lse_px), _ptr(st), _ptr(g), 1.0, C.byref(dst), _ptr(ws), nbytes, _stream())


def _mds_dy(src, ids, labels, shape, ignore, loss_px, lse_px, st, g, y, Cs, cmax):
    """d loss / d y of the fused loss as fp32 planes shaped like y: (dyA, None) from the fused single-pass kernel with
    the identity in place of G^T when it applies, else the two planes (dyA, dyB) of mdseg_up_ce_bwd, whose sum it is."""
    B, h, w, H, W = shape
    n = len(Cs)
    if N.lib.mdseg_up_ce_bwd_direct_is_fused(C.byref(src), h, w, H, W):
        dyA, dyB = torch.empty_like(y), None  # only the first C_ds planes of an image are written — and read
        _up_ce_adjoint(src, ids, labels, shape, ignore, loss_px, lse_px, st, g,
                       _src_table([dyA.data_ptr()] * n, [cmax * h * w] * n, Cs, N.F32, False))
    else:
        dyA = torch.empty_like(y)
        dyB = torch.empty_like(y)
        dA = _src_table([dyA.data_ptr()] * n, [cmax * h * w] * n, Cs, N.F32, False)
        dB = _src_table([dyB.data_ptr()] * n, [cmax * h * w] * n, Cs, N.F32, False)
        N.call("mdseg_up_ce_bwd", C.byref(src), _ptr(ids), _ptr(labels), _DT[labels.dtype], B, h, w, H, W, ignore,
               _ptr(loss_px), _ptr(lse_px), _ptr(st), _ptr(g), 1.0, C.byref(dA), C.byref(dB), _stream())
    return dyA, dyB


def mds_proj_ohem_ce(logits_uni, labels, dataset_ids, graphs, thresh, ignore=255, cache=None, per_dataset=False):
    """CE(upsample(project(logits_uni, graph[dataset]))) under OHEM.  No host synchronisation in the loss itself
    (counting, branch decision and selection stay on the device); the ONE exception is the descriptor cache of
    non-trainable graphs (`BipartiteGraphs`): a graph tensor it has not seen (new object, new version or new storage)
    is copied to the host once to build its CSR / CSC lists and to pick the sparse or the dense kernels — once per
    run for the SEG stage's fixed 0/1 graphs, every call if the caller rebuilds the tensors.  Trainable graphs and
    folded prototypes (`assume_dense`) are never copied.  One selection over all images
    (0-dim result, MdsOhemCELoss) or, with `per_dataset`, one selection per dataset (vector [n_datasets], NaN for a
    dataset without images: OhemCELoss per dataset, lib/loss/loss_cross_datasets.py:701-708)."""
    return _MdsProjOhemCE.apply(logits_uni, labels, dataset_ids, float(thresh), int(ignore), cache or _default_graphs,
                                bool(per_dataset), *graphs)[0]


class _MdsProjOhemCEHeads(torch.autograd.Function):
    """H losses MdsOhemCELoss(upsample(project(x, graphs_k[dataset]))), k < H, that share x (the GNN stage's hard / soft
    graph pair, lib/loss/loss_cross_datasets.py:996-1004,1063-1071): ONE projection with the graphs of a dataset
    stacked to [H * C_ds, C_uni], H fused CE / OHEM passes on the slices of y, and in the backward one adjoint and one
    d-graph GEMM over the stacked gradient planes — x is read once per direction instead of H times and its gradient
    is written once instead of H times and added.  Dense graphs only (tensor-core routes); `graphs` is head-major.
    16-bit x that _tc16_layout reads as it lies takes the tc16 kernels in both directions when the stacked graphs are in
    _tc16_envelope; channels_last x is then read as it is and gets a channels_last gradient."""

    @staticmethod
    def forward(ctx, x, labels, dataset_ids, thresh, ignore, n_heads, *graphs):
        _require_cuda(x, labels)
        if x.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            x = x.float()
        B, Cu, h, w = x.shape
        labels = _labels(labels)
        H, W = labels.shape[1:]
        dev = x.device
        n = len(graphs) // n_heads
        Cs = [graphs[d].shape[0] for d in range(n)]
        labels = _compact_labels(labels, max(Cs), ignore)
        cmax2 = n_heads * max(Cs)
        stacked = [torch.cat([graphs[k * n + d].detach().to(torch.float32) for k in range(n_heads)], 0) for d in range(n)]
        cache = BipartiteGraphs(assume_dense=True)
        tab, keep = cache.table(stacked)
        tc16 = _dense_tc16(tab)
        if not (tc16 and _tc16_layout(x) == N.NHWC):
            x = x.contiguous()
        tc16 = tc16 and _tc16_layout(x) is not None  # the route of both directions
        ids = _ids32(dataset_ids, B, dev)
        ef = err_flag(dev)
        y = torch.empty(B, cmax2, h, w, dtype=torch.float32, device=dev)
        _proj_fwd(x, tab, stacked, ids, y, None, ef, tc16)
        P = B * H * W
        outs, saved = [], []
        for k in range(n_heads):
            ymax = torch.empty(B, h, w, dtype=torch.float32, device=dev)
            src = _src_table([y.data_ptr() + k * c * h * w * 4 for c in Cs], [cmax2 * h * w] * n, Cs, N.F32, False,
                             c_alloc=[cmax2 - k * c for c in Cs], cmax=ymax, cmax_ready=False)
            loss_px = torch.empty(P, dtype=torch.float32, device=dev)
            lse_px = torch.empty(P, dtype=torch.float32, device=dev)
            st = _new_states(1, thresh, dev)
            N.call("mdseg_up_ce_fwd", C.byref(src), _ptr(ids), _ptr(labels), _DT[labels.dtype], B, h, w, H, W, int(ignore),
                   _ptr(loss_px), _ptr(lse_px), _ptr(st), _ptr(ef), _stream())
            outs.append(_select(loss_px, B, H * W, None, st, 1)[0])
            saved += [loss_px, lse_px, st]
        ctx.save_for_backward(x, labels, ids, y, *saved, *stacked)
        ctx.meta = (int(ignore), Cs, cmax2, (h, w, H, W), n_heads, [g.dtype for g in graphs], tc16)
        return torch.stack(outs)

    @staticmethod
    def backward(ctx, grad_out):
        ignore, Cs, cmax2, (h, w, H, W), n_heads, gdt, tc16 = ctx.meta
        n = len(Cs)
        x, labels, ids, y = ctx.saved_tensors[:4]
        saved = ctx.saved_tensors[4:4 + 3 * n_heads]
        stacked = ctx.saved_tensors[4 + 3 * n_heads:]
        B = x.shape[0]
        dev = x.device
        g = _grad_scalar(grad_out, n_heads)
        ddt = x.dtype if tc16 else torch.float32
        esz = 2 if tc16 else 4
        dy = torch.zeros(B, cmax2, h, w, dtype=ddt, device=dev)  # planes past the heads of an image's dataset stay zero
        scratch = torch.empty(1, dtype=torch.float32, device=dev)
        for k in range(n_heads):
            loss_px, lse_px, st = saved[3 * k:3 * k + 3]
            src = _src_table([y.data_ptr() + k * c * h * w * 4 for c in Cs], [cmax2 * h * w] * n, Cs, N.F32, False,
                             c_alloc=[cmax2 - k * c for c in Cs], cmax=scratch, cmax_ready=True)
            dst = _src_table([dy.data_ptr() + k * c * h * w * esz for c in Cs], [cmax2 * h * w] * n, Cs, _DT[ddt], False)
            _up_ce_adjoint(src, ids, labels, (B, h, w, H, W), ignore, loss_px, lse_px, st, g[k:k + 1], dst)
        tab, keep = (None, None) if tc16 else BipartiteGraphs(assume_dense=True).table(list(stacked))
        dx = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            _proj_bwd(dy, None, stacked, tab, ids, dx)
        dG = _proj_bwd_graph(x, dy, None, stacked, tab, ids)
        dgs = []
        for k in range(n_heads):
            for d in range(n):
                if ctx.needs_input_grad[6 + k * n + d]:
                    dgs.append(dG[d, k * Cs[d]:(k + 1) * Cs[d]].to(gdt[k * n + d]))
                else:
                    dgs.append(None)
        return (dx, None, None, None, None, None, *dgs)


def mds_proj_ohem_ce_heads(x, labels, dataset_ids, graph_sets, thresh, ignore=255):
    """Vector [H] of MdsOhemCELoss values, one per graph set, sharing ONE pass over x per direction (see
    _MdsProjOhemCEHeads).  graph_sets: H lists of n_datasets dense [C_ds, C_uni] matrices (the same C_ds in every set).
    Falls back to H independent fused losses when the stacked route does not apply (graphs that are not all in the
    tensor-core envelope, geometry outside the fused backward).  channels_last 16-bit x inside _tc16_layout is read
    without a layout copy on both routes (the fallback's losses pick their layout one by one)."""
    sets = [list(gs) for gs in graph_sets]
    n = len(sets[0])
    B, Cu, h, w = x.shape
    Hh, Ww = labels.shape[1:]
    Cs = [g.shape[0] for g in sets[0]]
    ok = (len(sets) > 1 and all(len(gs) == n and [g.shape[0] for g in gs] == Cs for gs in sets)
          and _tc16_envelope(Cu, Cs, len(sets)) and x.is_cuda)
    if ok:
        probe = _src_table([x.data_ptr() & ~15] * n, [4 * h * w] * n, Cs, N.F32, False, cmax=x)
        ok = bool(N.lib.mdseg_up_ce_bwd_direct_is_fused(C.byref(probe), h, w, Hh, Ww))
    if not ok:
        return torch.stack([mds_proj_ohem_ce(x, labels, dataset_ids, gs, thresh, ignore,
                                             BipartiteGraphs(assume_dense=all(g.requires_grad for g in gs)))
                            for gs in sets])
    flat = [g for gs in sets for g in gs]
    return _MdsProjOhemCEHeads.apply(x, labels, dataset_ids, float(thresh), int(ignore), len(sets), *flat)


def fold_prototypes(graphs, proto):
    """W_d = bi_graphs[d] @ unify_prototype, fp32 [C_ds, K] per dataset (tiny torch matmuls; autograd carries
    d bi_graph = dW_d proto^T and d proto = sum_d G_d^T dW_d).

    The reference forms the unified logits first and projects them afterwards (lib/loss/loss_cross_datasets.py:971
    then :996-1006; :747 then :759; :692 then :701): y_d = G_d (P f).  The product is associative, so y_d = (G_d P) f:
    the [B, C_uni, h, w] unified logits (3 GB at cfg3) and their gradient are never formed, and the per-pixel
    contraction shrinks from K x C_uni + C_uni x C_ds to K x C_ds multiply-adds (512 x 358 + 358 x 61 -> 512 x 61)."""
    p32 = proto.to(torch.float32)
    graphs = list(graphs)
    if len(graphs) > 1 and all(g.shape[1] == graphs[0].shape[1] for g in graphs):
        # one matmul for all datasets (and one per operand in the backward) instead of one per dataset: the rows of the
        # stacked product are the per-dataset products, handed out as views
        stacked = torch.cat([g.to(torch.float32) for g in graphs], 0) @ p32
        return list(torch.split(stacked, [g.shape[0] for g in graphs], 0))
    return [g.to(torch.float32) @ p32 for g in graphs]


_folded_graphs = None


def _folded_cache():
    global _folded_graphs
    if _folded_graphs is None:
        _folded_graphs = BipartiteGraphs(assume_dense=True)
    return _folded_graphs


def mds_head_proj_ohem_ce(feats, proto, labels, dataset_ids, graphs, thresh, ignore=255, cache=None, per_dataset=False):
    """MdsOhemCELoss(upsample(einsum(einsum(feats, proto), graph[dataset]))) with the two contractions folded into one
    (see fold_prototypes): the fused loss runs on the features [B, K, h, w] with W_d in the role of the dense graph —
    forward, d feats and d W_d on the tcgen05 kernels, no unified-logits tensor."""
    return mds_proj_ohem_ce(feats, labels, dataset_ids, fold_prototypes(graphs, proto), thresh, ignore,
                            cache or _folded_cache(), per_dataset)


def mds_head_proj_ohem_ce_heads(feats, proto, labels, dataset_ids, graph_sets, thresh, ignore=255):
    """mds_proj_ohem_ce_heads on the features with every graph set folded into the prototypes: the GNN stage's hard and
    soft losses (loss_cross_datasets.py:971,996-1004,1063-1071) from ONE pass over the features per direction."""
    return mds_proj_ohem_ce_heads(feats, labels, dataset_ids, [fold_prototypes(gs, proto) for gs in graph_sets], thresh,
                                  ignore)


def mds_head_proj_ce_mean(feats, proto, labels, dataset_ids, graphs, ignore=255, cache=None):
    """mds_proj_ce_mean on the features with folded prototypes (see fold_prototypes)."""
    return mds_proj_ce_mean(feats, labels, dataset_ids, fold_prototypes(graphs, proto), ignore, cache or _folded_cache())


def mds_proj_ce_mean(logits_uni, labels, dataset_ids, graphs, ignore=255, cache=None):
    """Per-dataset plain cross-entropy means, vector [n_datasets]: nn.CrossEntropyLoss(ignore_index)(upsample(project(
    logits[ids == d], G_d)), labels[ids == d]) (lib/loss/loss_cross_datasets.py:341-345, :753-768).  Runs as the fused
    OHEM loss with a threshold below every loss (every pixel selected, ignored ones contribute 0 and get no gradient)
    and is rescaled from the mean over all pixels to the mean over the valid ones on the device."""
    out, st = _MdsProjOhemCE.apply(logits_uni, labels, dataset_ids, -1.0, int(ignore), cache or _default_graphs, True,
                                   *graphs)
    counts = st.view(torch.int64).view(-1, STATE_BYTES // 8)
    n_valid, n_px = counts[:, 0].to(torch.float32), counts[:, 2].to(torch.float32)
    return out * (n_px / n_valid)


# ---- f4: MdsOhemNLLPlusLoss (softmax -> project probabilities -> upsample -> -log, one OHEM selection) ------------
class _MdsNLLPlus(torch.autograd.Function):
    """AdjNLLPlusLoss (lib/loss/loss_helper.py:647-668) under the selection of MdsOhemNLLPlusLoss
    (lib/loss/ohem_ce_loss.py:92-146).  The reference's loss vector holds the valid pixels only; here ignored pixels
    stay in the vector with loss 0 — never above a positive threshold, and never inside the top n_min (= n_valid // 16)
    unless every remaining candidate is 0 as well, which leaves the mean and the gradient unchanged."""

    @staticmethod
    def forward(ctx, logits_uni, labels, dataset_ids, thresh, ignore, cache, *graphs):
        _require_cuda(logits_uni, labels)
        x = logits_uni
        if x.dtype not in (torch.float32, torch.bfloat16, torch.float16):
            x = x.float()
        x = x.contiguous()
        B, Cu, h, w = x.shape
        labels = _labels(labels)
        if labels.dim() != 3 or labels.shape[0] != B:
            raise ValueError("labels must be [B, H, W]")
        H, W = labels.shape[1:]
        dev = x.device
        tab, keep = cache.table(list(graphs))
        if tab.C_uni != Cu:
            raise ValueError(f"graphs have C_uni={tab.C_uni}, logits have {Cu}")
        Cs = [g.shape[0] for g in graphs]
        cmax = max(Cs)
        ids = _ids32(dataset_ids, B, dev)
        ef = err_flag(dev)
        pred = torch.empty(B, Cu, h, w, dtype=torch.float32, device=dev)
        N.call("mdseg_softmax_nchw", _ptr(x), _DT[x.dtype], B, Cu, h * w, _ptr(pred), _stream())
        q = torch.empty(B, cmax, h, w, dtype=torch.float32, device=dev)
        _proj_fwd(pred, tab, graphs, ids, q, None, ef, False)
        src = _src_table([q.data_ptr()] * len(Cs), [cmax * h * w] * len(Cs), Cs, N.F32, False, c_alloc=cmax)
        loss_px = torch.empty(B * H * W, dtype=torch.float32, device=dev)
        st = _new_states(1, thresh, dev)
        N.call("mdseg_up_nll_fwd", C.byref(src), _ptr(ids), _ptr(labels), _DT[labels.dtype], B, h, w, H, W, int(ignore),
               _ptr(loss_px), _ptr(st), _ptr(ef), _stream())
        out = _select(loss_px, B, H * W, None, st, 1)
        ctx.save_for_backward(pred, labels, ids, q, loss_px, st, *graphs)
        ctx.meta = (int(ignore), cache, Cs, cmax, (h, w, H, W), x.dtype)
        ctx.states = st
        return out[0]

    @staticmethod
    def backward(ctx, grad_out):
        pred, labels, ids, q, loss_px, st, *graphs = ctx.saved_tensors
        ignore, cache, Cs, cmax, (h, w, H, W), xdt = ctx.meta
        B, Cu = pred.shape[:2]
        dev = pred.device
        n = len(Cs)
        g = _grad_scalar(grad_out)
        tab, keep = cache.table(list(graphs))
        src = _src_table([q.data_ptr()] * n, [cmax * h * w] * n, Cs, N.F32, False, c_alloc=cmax)
        dq = torch.zeros_like(q)
        dst = _src_table([dq.data_ptr()] * n, [cmax * h * w] * n, Cs, N.F32, False, c_alloc=cmax)
        N.call("mdseg_up_nll_bwd", C.byref(src), _ptr(ids), _ptr(labels), _DT[labels.dtype], B, h, w, H, W, ignore,
               _ptr(loss_px), _ptr(st), _ptr(g), 1.0, C.byref(dst), _stream())
        dx = None
        if ctx.needs_input_grad[0]:
            dpred = torch.empty_like(pred)
            _proj_bwd(dq, None, graphs, tab, ids, dpred)
            dx = dpred if xdt == torch.float32 else torch.empty(pred.shape, dtype=xdt, device=dev)
            N.call("mdseg_softmax_bwd_nchw", _ptr(pred), _ptr(dpred), B, Cu, h * w, _ptr(dx), _DT[xdt], _stream())
        dgs = [None] * n
        if any(ctx.needs_input_grad[6 + i] for i in range(n)):
            dG = _proj_bwd_graph(pred, dq, None, graphs, tab, ids)
            for i in range(n):
                if ctx.needs_input_grad[6 + i]:
                    dgs[i] = dG[i, :Cs[i]].to(graphs[i].dtype)
        return (dx, None, None, None, None, None, *dgs)


def mds_nll_plus(logits_uni, labels, dataset_ids, graphs, thresh, ignore=255, cache=None):
    """mean over the OHEM set of -log(upsample(G_d softmax(logits_uni)))[label]: MdsOhemNLLPlusLoss.forward
    (lib/loss/ohem_ce_loss.py:104-146) for a whole multi-dataset batch; host synchronisation only on a miss of the
    graph-descriptor cache (see mds_proj_ohem_ce)."""
    return _MdsNLLPlus.apply(logits_uni, labels, dataset_ids, float(thresh), int(ignore), cache or _default_graphs,
                             *graphs)


# ---- a10: per-dataset aux heads (upsample + OhemCE, one selection per dataset) ---------------------------
class _UpOhemCE(torch.autograd.Function):
    """channels_last sources (all of them) are not copied: the rows of each head's own images are gathered into one
    planar buffer [B, max C_i, h, w] (mdseg_nhwc_to_planar) and the gradients come back channels_last
    (mdseg_planar_to_nhwc)."""

    @staticmethod
    def forward(ctx, labels, dataset_ids, thresh, ignore, seg_per_dataset, *srcs):
        labels = _labels(labels)
        _require_cuda(labels, *srcs)
        labels = _compact_labels(labels, max(s.shape[1] for s in srcs), ignore)
        B, H, W = labels.shape
        dev = labels.device
        n = len(srcs)
        dt = srcs[0].dtype
        if dt not in (torch.float32, torch.bfloat16, torch.float16):
            dt = torch.float32
        srcs = [s.to(dt) for s in srcs]
        nhwc = all(_channels_last(s) for s in srcs)
        if not nhwc:
            srcs = [s.contiguous() for s in srcs]
        h, w = srcs[0].shape[2:]
        for s in srcs:
            if s.shape[0] != B or tuple(s.shape[2:]) != (h, w):
                raise ValueError("every source must be [B, C_i, h, w] over all B images")
        Cs = [s.shape[1] for s in srcs]
        ids = _ids32(dataset_ids, B, dev) if n > 1 else None
        smax = torch.empty(B, h, w, dtype=torch.float32, device=dev) if dt == torch.float32 else None
        if nhwc:
            cm = max(Cs)
            planar = torch.empty(B, cm, h, w, dtype=dt, device=dev)
            src = _src_table([planar.data_ptr()] * n, [cm * h * w] * n, Cs, _DT[dt], seg_per_dataset, c_alloc=cm,
                             cmax=smax)
            nt = _src_table([s.data_ptr() for s in srcs], [s.stride(0) for s in srcs], Cs, _DT[dt], seg_per_dataset)
            N.call("mdseg_nhwc_to_planar", C.byref(nt), _ptr(ids), B, h, w, C.byref(src), _stream())
            srcs = [planar]
        else:
            src = _src_table([s.data_ptr() for s in srcs], [c * h * w for c in Cs], Cs, _DT[dt], seg_per_dataset,
                             cmax=smax)
        n_seg = n if seg_per_dataset else 1
        P = B * H * W
        loss_px = torch.empty(P, dtype=torch.float32, device=dev)
        lse_px = torch.empty(P, dtype=torch.float32, device=dev)
        st = _new_states(n_seg, thresh, dev)
        N.call("mdseg_up_ce_fwd", C.byref(src), _ptr(ids), _ptr(labels), _DT[labels.dtype], B, h, w, H, W, int(ignore),
               _ptr(loss_px), _ptr(lse_px), _ptr(st), _ptr(err_flag(dev)), _stream())
        out = _select(loss_px, B, H * W, ids if seg_per_dataset else None, st, n_seg)
        ctx.save_for_backward(labels, ids, loss_px, lse_px, st, *srcs)
        ctx.meta = (int(ignore), bool(seg_per_dataset), Cs, dt, (h, w, H, W), nhwc)
        ctx.states = st
        return out

    @staticmethod
    def backward(ctx, grad_out):
        labels, ids, loss_px, lse_px, st, *srcs = ctx.saved_tensors
        ignore, seg_per_dataset, Cs, dt, (h, w, H, W), nhwc = ctx.meta
        B = labels.shape[0]
        n = len(Cs)
        n_seg = n if seg_per_dataset else 1
        g = _grad_scalar(grad_out, n_seg)
        scratch = torch.empty(1, dtype=torch.float32, device=labels.device) if dt == torch.float32 else None
        if nhwc:
            return (None, None, None, None, None,
                    *_up_ohem_ce_bwd_nhwc(srcs[0], labels, ids, loss_px, lse_px, st, g, scratch, ignore, seg_per_dataset,
                                          Cs, dt, (h, w, H, W)))
        src = _src_table([s.data_ptr() for s in srcs], [c * h * w for c in Cs], Cs, _DT[dt], seg_per_dataset,
                         cmax=scratch, cmax_ready=True)
        # images of other datasets get a zero gradient (their rows are never selected, :1051): zero-initialised
        # outputs, the kernel writes only the rows of a head's own images
        grads = [torch.zeros_like(s) for s in srcs]
        dst = _src_table([t.data_ptr() for t in grads], [c * h * w for c in Cs], Cs, _DT[dt], seg_per_dataset)
        _up_ce_adjoint(src, ids, labels, (B, h, w, H, W), ignore, loss_px, lse_px, st, g, dst)
        return (None, None, None, None, None, *grads)


def _up_ohem_ce_bwd_nhwc(planar, labels, ids, loss_px, lse_px, st, g, scratch, ignore, seg_per_dataset, Cs, dt, shape):
    """Gradients of _UpOhemCE's channels_last sources: d loss / d (planar rows) from mdseg_up_ce_bwd_direct, scattered
    into channels_last tensors (zeros for the images of other datasets)."""
    h, w, H, W = shape
    B, cm = planar.shape[:2]
    n = len(Cs)
    dev = planar.device
    src = _src_table([planar.data_ptr()] * n, [cm * h * w] * n, Cs, _DT[dt], seg_per_dataset, c_alloc=cm, cmax=scratch,
                     cmax_ready=True)
    if N.lib.mdseg_up_ce_bwd_direct_is_fused(C.byref(src), h, w, H, W):
        dp = torch.empty_like(planar)  # the rows of image b's own head are written — and read
        dst = _src_table([dp.data_ptr()] * n, [cm * h * w] * n, Cs, _DT[dt], seg_per_dataset, c_alloc=cm)
    else:  # the generic route adds two planes per head: dense [B, C_d, h, w] destinations
        dp = [torch.empty(B, c, h, w, dtype=dt, device=dev) for c in Cs]
        dst = _src_table([t.data_ptr() for t in dp], [c * h * w for c in Cs], Cs, _DT[dt], seg_per_dataset)
    _up_ce_adjoint(src, ids, labels, (B, h, w, H, W), ignore, loss_px, lse_px, st, g, dst)
    grads = [torch.empty((B, c, h, w), dtype=dt, device=dev, memory_format=torch.channels_last) for c in Cs]
    gt = _src_table([t.data_ptr() for t in grads], [t.stride(0) for t in grads], Cs, _DT[dt], seg_per_dataset)
    N.call("mdseg_planar_to_nhwc", C.byref(dst), _ptr(ids), B, h, w, C.byref(gt), _stream())
    return grads


def up_ohem_ce(srcs, labels, dataset_ids, thresh, ignore=255, seg_per_dataset=True):
    """Per-dataset OhemCE(upsample(srcs[d][ids==d]), labels[ids==d]) as a vector [n_datasets]
    (seg_per_dataset) or one selection over all images ([1]).  srcs[d]: [B, C_d, h, w] over ALL images; channels_last
    sources are read without a layout copy and get channels_last gradients."""
    return _UpOhemCE.apply(labels, dataset_ids, float(thresh), int(ignore), bool(seg_per_dataset), *srcs)


# ---- a11: evaluator accumulation --------------------------------------------------------------------------
def eval_accum(logits, probs, flip=False, first=False):
    """probs[C,H,W] (+)= softmax(upsample_bilinear_ac(logits[C,h,w] (flipped along W if flip)))  (evaluate.py:149-171)."""
    _require_cuda(logits, probs)
    if logits.dim() == 4:
        if logits.shape[0] != 1:
            raise ValueError("eval_accum takes one image")
        logits = logits[0]
    if probs.dim() == 4:
        probs = probs[0]
    logits = logits.contiguous()
    if logits.dtype not in _DT or _DT[logits.dtype] > N.F16:
        logits = logits.float()
    Cc, h, w = logits.shape
    if probs.dtype != torch.float32 or not probs.is_contiguous() or probs.shape[0] != Cc:
        raise ValueError("probs must be a contiguous fp32 [C, H, W]")
    H, W = probs.shape[1:]
    N.call("mdseg_eval_accum", _ptr(logits), _DT[logits.dtype], Cc, h, w, _ptr(probs), H, W, int(flip), int(first),
           _stream())
    return probs


def eval_fused(passes, size, label=None, hist=None, lut=None, ignore=255, want_pred=True):
    """All (scale, flip) passes of one image in one kernel (evaluate.py:136-181): pred = argmax_c of the summed
    soft-max of every up-sampled pass, hist[label, pred] += 1.  passes: [(logits [C, h, w], flip), ...] of one
    float dtype; size = (H, W) of the label.  Returns (pred or None, hist or None).  At most 16 passes (see
    eval_fused_fits)."""
    H, W = int(size[0]), int(size[1])
    tab = N.EvalPasses()
    keep = []
    dt = None
    for i, (lg, flip) in enumerate(passes):
        _require_cuda(lg)
        if lg.dim() == 4:
            if lg.shape[0] != 1:
                raise ValueError("eval_fused takes one image")
            lg = lg[0]
        if lg.dtype not in _DT or _DT[lg.dtype] > N.F16:
            lg = lg.float()
        lg = lg.contiguous()
        dt = lg.dtype if dt is None else dt
        if lg.dtype != dt:
            raise TypeError("eval_fused: all passes must share one dtype")
        if i == 0:
            Cc = lg.shape[0]
        elif lg.shape[0] != Cc:
            raise ValueError("eval_fused: all passes must share the class count")
        keep.append(lg)
        tab.p[i].logits, tab.p[i].h, tab.p[i].w, tab.p[i].flip = lg.data_ptr(), lg.shape[1], lg.shape[2], int(bool(flip))
    if not keep:
        raise ValueError("eval_fused: no passes")
    tab.n_passes, tab.dtype = len(keep), _DT[dt]
    dev = keep[0].device
    pred = torch.empty(H, W, dtype=torch.int64, device=dev) if want_pred else None
    lab = None
    if label is not None:
        lab = _labels(label)
        if lab.numel() != H * W:
            raise ValueError("label size mismatch")
        if hist is None:
            hist = torch.zeros(Cc, Cc, dtype=torch.int64, device=dev)
    if lut is not None:
        lut = torch.as_tensor(lut).to(device=dev, dtype=torch.uint8).contiguous()
    nbytes = N.lib.mdseg_eval_fused_workspace_bytes(len(keep), H, W)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    N.call("mdseg_eval_fused", C.byref(tab), Cc, H, W, _ptr(pred), _ptr(lab), _DT[lab.dtype] if lab is not None else N.U8,
           _ptr(lut), _ptr(hist) if lab is not None else None, int(ignore), _ptr(ws), nbytes, _ptr(err_flag(dev)),
           _stream())
    return pred, hist


def eval_fused_fits(n_classes, n_passes):
    return 0 < n_passes <= N.MAX_EVAL_PASSES


def argmax_hist(probs, label=None, hist=None, lut=None, ignore=255, want_pred=True):
    """pred = argmax_c probs; optionally hist[label, pred] += 1 in the same pass (evaluate.py:172-181)."""
    _require_cuda(probs)
    if probs.dim() == 4:
        probs = probs[0]
    probs = probs.contiguous()
    Cc = probs.shape[0]
    n_px = probs[0].numel()
    pred = torch.empty(probs.shape[1:], dtype=torch.int64, device=probs.device) if want_pred else None
    lab = None
    if hist is not None:
        lab = _labels(label)
        if lab.numel() != n_px:
            raise ValueError("label size mismatch")
        if lut is not None:
            lut = torch.as_tensor(lut).to(device=probs.device, dtype=torch.uint8).contiguous()
    N.call("mdseg_argmax_hist", _ptr(probs), Cc, n_px, _ptr(pred), _ptr(lab), _DT[lab.dtype] if lab is not None else 0,
           _ptr(lut), _ptr(hist), int(ignore), _ptr(err_flag(probs.device)), _stream())
    return pred


def eval_chip_accum(logits, probs, y0, x0, logits_flip=None, exp_after=False):
    """probs[:, y0:y0+ch, x0:x0+cw] += softmax(logits) (+ softmax(un-flipped logits_flip)), exp() of the sum when
    `exp_after` (MscEvalCrop.eval_chip + the window add of crop_eval, evaluate.py:684-710).  logits [C, ch, cw]."""
    _require_cuda(logits, probs)
    logits = logits.contiguous()
    if logits.dtype not in _DT or _DT[logits.dtype] > N.F16:
        logits = logits.float()
    if logits_flip is not None:
        logits_flip = logits_flip.to(logits.dtype).contiguous()
    Cc, ch, cw = logits.shape
    if probs.dtype != torch.float32 or not probs.is_contiguous() or probs.shape[0] != Cc:
        raise ValueError("probs must be a contiguous fp32 [C, PH, PW]")
    N.call("mdseg_eval_chip_accum", _ptr(logits), _ptr(logits_flip), _DT[logits.dtype], Cc, ch, cw, _ptr(probs),
           probs.shape[1], probs.shape[2], int(y0), int(x0), int(bool(exp_after)), _stream())
    return probs


def prob_resize_accum(src, window, dst, first=False):
    """dst (+)= bilinear(align_corners=True) resize of src[:, y0:y1, x0:x1] to dst's size (evaluate.py:722-724)."""
    _require_cuda(src, dst)
    y0, y1, x0, x1 = [int(v) for v in window]
    if src.dtype != torch.float32 or dst.dtype != torch.float32 or not src.is_contiguous() or not dst.is_contiguous():
        raise ValueError("probability maps are contiguous fp32 [C, H, W]")
    N.call("mdseg_prob_resize_accum", _ptr(src), src.shape[0], src.shape[1], src.shape[2], y0, x0, y1 - y0, x1 - x0,
           _ptr(dst), dst.shape[1], dst.shape[2], int(bool(first)), _stream())
    return dst


def label_nearest(label, size):
    """Legacy 'nearest' resize of an integer label map [N,H,W] -> [N,h,w] (evaluate.py:156-157)."""
    _require_cuda(label)
    label = _labels(label)
    Nn, Hin, Win = label.shape
    Ho, Wo = size
    out = torch.empty(Nn, Ho, Wo, dtype=label.dtype, device=label.device)
    N.call("mdseg_label_nearest", _ptr(label), _DT[label.dtype], Hin, Win, _ptr(out), Ho, Wo, Nn, _stream())
    return out


# ---- f3: label branch of the data pipeline (LUT -> nearest resize -> pad -> crop -> flip) in one gather ----------
def label_pipeline(srcs, plans, out_size, luts=None, lut_ids=None, out_dtype=torch.int64, pad_value=255):
    """out[b] = flip(crop(pad(cv2_nearest_resize(lut[srcs[b]])))) for a batch of raw uint8 label images
    (lib/base_dataset.py:81-82 + lib/transform_cv2.py:43-61,71-77,300) without materialising any intermediate.

    srcs: list of uint8 CUDA tensors [H_b, W_b] (any row stride); plans: one dict per image with the integers
    ``im_h, im_w, pad_top, pad_left, crop_y, crop_x, flip`` (see dropin.label_transform.plan_random_resized_crop);
    out_size = (crop_h, crop_w), crop_w % 16 == 0; luts: uint8 [n_luts, 256] (or None), lut_ids[b] selects the row
    (-1 / None: identity).  Returns [B, crop_h, crop_w] of `out_dtype` (torch.int64 like the reference, or uint8)."""
    import numpy as np
    _require_cuda(*srcs)
    if len(srcs) != len(plans) or not srcs:
        raise ValueError("label_pipeline: one plan per source image")
    dev = srcs[0].device
    views = (N.LabelView * len(srcs))()
    for b, (t, pl) in enumerate(zip(srcs, plans)):
        if t.dtype != torch.uint8 or t.dim() != 2 or t.stride(1) != 1:
            raise TypeError("label_pipeline: sources must be uint8 [H, W] with unit column stride")
        v = views[b]
        v.src, v.src_row_stride, v.src_h, v.src_w = t.data_ptr(), t.stride(0), t.shape[0], t.shape[1]
        v.im_h, v.im_w = int(pl["im_h"]), int(pl["im_w"])
        v.pad_top, v.pad_left = int(pl.get("pad_top", 0)), int(pl.get("pad_left", 0))
        v.crop_y, v.crop_x, v.flip = int(pl.get("crop_y", 0)), int(pl.get("crop_x", 0)), int(bool(pl.get("flip", False)))
        v.lut = int(lut_ids[b]) if lut_ids is not None else (0 if luts is not None else -1)
        if v.im_h <= 0 or v.im_w <= 0:
            raise ValueError("label_pipeline: empty resized image")
    table = torch.from_numpy(np.frombuffer(bytes(views), dtype=np.uint8).copy()).to(dev, non_blocking=True)
    n_luts = 0
    if luts is not None:
        luts = torch.as_tensor(luts).to(device=dev, dtype=torch.uint8).reshape(-1, 256).contiguous()
        n_luts = luts.shape[0]
    Ho, Wo = int(out_size[0]), int(out_size[1])
    if out_dtype not in (torch.int64, torch.uint8):
        raise TypeError("label_pipeline: out_dtype must be torch.int64 or torch.uint8")
    out = torch.empty(len(srcs), Ho, Wo, dtype=out_dtype, device=dev)
    N.call("mdseg_label_pipeline", _ptr(table), len(srcs), _ptr(luts), n_luts, _ptr(out), _DT[out_dtype], Ho, Wo,
           int(pad_value), _stream())
    return out


# ---- f3: image branch of the data pipeline (resize -> pad -> crop -> flip -> ColorJitter -> ToTensor) in one gather
def to_tensor_tables(mean_std, device):
    """ToTensor(mean, std) (lib/transform_cv2.py) as fp32 [n, 3, 256] tables on `device`, one per (mean, std) pair:
    table[k, c, v] is what the reference's `torch.from_numpy(im.astype(np.float32)).div_(255).sub_(mean).div_(std)`
    gives a byte v in channel c — built with exactly those torch ops, so the lookup is bit-exact by construction."""
    rows = []
    for mean, std in mean_std:
        t = torch.arange(256, dtype=torch.float32).repeat(3, 1)[:, None, :].div_(255)   # [3, 1, 256] like [3, H, W]
        m = torch.as_tensor(mean, dtype=t.dtype)[:, None, None]
        s = torch.as_tensor(std, dtype=t.dtype)[:, None, None]
        rows.append(t.sub_(m).div_(s)[:, 0, :])
    return torch.stack(rows).to(device)


_DEFAULT_TABLES = {}


def image_pipeline(srcs, plans, out_size, jitter=None, norms=None, norm_ids=None, bgr=True,
                   memory_format=torch.contiguous_format):
    """out[b] = ToTensor(ColorJitter(flip(crop(pad(cv2.resize(srcs[b], INTER_LINEAR)))))) for a batch of decoded
    uint8 images (lib/transform_cv2.py: RandomResizedCrop, RandomHorizontalFlip, ColorJitter, ToTensor) without
    materialising any intermediate.

    srcs: list of uint8 CUDA tensors [H_b, W_b, 3] (any row stride, pixel stride 3), BGR as cv2.imread returns them
    when `bgr` (the reference's [:, :, ::-1] view is folded into the gather), RGB otherwise; plans: one dict per image
    with ``im_h, im_w, pad_top, pad_left, crop_y, crop_x, flip`` (the same plans ``label_pipeline`` takes);
    out_size = (crop_h, crop_w), crop_w % 16 == 0; jitter: None, or one entry per image — None or a dict with
    ``lut`` (uint8[256], brightness then contrast) and ``sat`` (None or float32 (1 + 2r, 1 - r)) as
    ``dropin.label_transform.ColorJitterPlan`` draws them; norms: fp32 [n, 3, 256] from ``to_tensor_tables`` (None:
    ToTensor's default mean 0 / std 1), norm_ids[b] selects the row (None: row 0).
    Returns fp32 [B, 3, crop_h, crop_w], NCHW-contiguous or channels_last (`memory_format`)."""
    _require_cuda(*srcs)
    if len(srcs) != len(plans) or not srcs:
        raise ValueError("image_pipeline: one plan per source image")
    if jitter is not None and len(jitter) != len(srcs):
        raise ValueError("image_pipeline: one jitter entry per source image")
    if memory_format not in (torch.contiguous_format, torch.channels_last):
        raise ValueError("image_pipeline: memory_format must be torch.contiguous_format or torch.channels_last")
    dev = srcs[0].device
    if norms is None:
        if dev not in _DEFAULT_TABLES:
            _DEFAULT_TABLES[dev] = to_tensor_tables([((0., 0., 0.), (1., 1., 1.))], dev)
        norms = _DEFAULT_TABLES[dev]
    if not (isinstance(norms, torch.Tensor) and norms.dtype == torch.float32 and norms.device == dev
            and norms.dim() == 3 and norms.shape[1:] == (3, 256) and norms.shape[0] > 0 and norms.is_contiguous()):
        raise TypeError("image_pipeline: norms must be a contiguous fp32 [n, 3, 256] tensor on the sources' device")
    table = image_views(srcs, plans, jitter, norm_ids, norms.shape[0], bgr)
    Ho, Wo = int(out_size[0]), int(out_size[1])
    out = torch.empty(len(srcs), 3, Ho, Wo, dtype=torch.float32, device=dev, memory_format=memory_format)
    layout = N.NHWC if memory_format == torch.channels_last else N.NCHW
    N.call("mdseg_image_pipeline", _ptr(table), len(srcs), _ptr(norms), norms.shape[0], _ptr(out), layout, Ho, Wo,
           _stream())
    return out


def image_views(srcs, plans, jitter, norm_ids, n_norm, bgr):
    """The device array of mdseg_image_view that ``image_pipeline`` passes to the kernel, LUTs inside, uploaded in
    one host-to-device copy; validates the sources, plans, jitter entries and norm indices."""
    views = (N.ImageView * len(srcs))()
    for b, (t, pl) in enumerate(zip(srcs, plans)):
        if t.dtype != torch.uint8 or t.dim() != 3 or t.shape[2] != 3 or t.stride(2) != 1 or t.stride(1) != 3:
            raise TypeError("image_pipeline: sources must be uint8 [H, W, 3] with pixel stride 3")
        v = views[b]
        v.src, v.src_row_stride, v.src_h, v.src_w = t.data_ptr(), t.stride(0), t.shape[0], t.shape[1]
        v.im_h, v.im_w = int(pl["im_h"]), int(pl["im_w"])
        v.pad_top, v.pad_left = int(pl.get("pad_top", 0)), int(pl.get("pad_left", 0))
        v.crop_y, v.crop_x, v.flip = int(pl.get("crop_y", 0)), int(pl.get("crop_x", 0)), int(bool(pl.get("flip", False)))
        if v.im_h <= 0 or v.im_w <= 0 or v.src_h <= 0 or v.src_w <= 0:
            raise ValueError("image_pipeline: empty source or resized image")
        v.swap_rb = int(bool(bgr))
        v.norm = int(norm_ids[b]) if norm_ids is not None else 0
        if not 0 <= v.norm < n_norm:
            raise ValueError(f"image_pipeline: norm_ids[{b}] = {v.norm} outside [0, {n_norm})")
        jt = jitter[b] if jitter is not None else None
        lut = np.arange(256, dtype=np.uint8) if jt is None or jt.get("lut") is None else np.ascontiguousarray(jt["lut"])
        if lut.dtype != np.uint8 or lut.shape != (256,):
            raise TypeError("image_pipeline: a jitter lut must be uint8[256]")
        C.memmove(v.lut, lut.ctypes.data, 256)
        sat = None if jt is None else jt.get("sat")
        v.saturate = int(sat is not None)
        v.sat_diag, v.sat_off = (float(sat[0]), float(sat[1])) if sat is not None else (0.0, 0.0)
    return torch.from_numpy(np.frombuffer(bytes(views), dtype=np.uint8).copy()).to(srcs[0].device, non_blocking=True)


def neg_log(p):
    """-log(p) in fp32, as torch computes OhemCELoss.thresh (ohem_ce_loss.py:17)."""
    return float(-torch.log(torch.tensor(p, dtype=torch.float)))
