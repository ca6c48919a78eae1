"""Float64 reference of the align_corners=False bilinear up-sampling at the BiSeNet heads' power-of-two factors,
and of OhemCELoss on its output (test infrastructure, next to oracle/f64.py and built on its CE and selection).

The geometry follows ATen's fp32 index / weight arithmetic (area_pixel_compute_source_index with
align_corners=False), so the same output pixels use the same corners and weights; everything else is float64."""
import numpy as np

from oracle.f64 import IGNORE, ohem_ce


def axis_weights_ac0(n_in, n_out, scale=None):
    """ATen area_pixel_compute_source_index(align_corners=False), fp32: scale = n_in / n_out (the size= form) or
    1 / scale_factor; s = max(scale * (o + 0.5) - 0.5, 0); i0 = int(s); i1 = i0 + (i0 < n_in - 1); l1 = s - i0."""
    sc = np.float32(scale) if scale is not None else np.float32(n_in) / np.float32(n_out)
    o = np.arange(n_out, dtype=np.float32)
    s = np.maximum(sc * (o + np.float32(0.5)) - np.float32(0.5), np.float32(0)).astype(np.float32)
    i0 = np.minimum(s.astype(np.int64), n_in - 1)
    i1 = i0 + (i0 < n_in - 1)
    l1 = (s - i0.astype(np.float32)).astype(np.float32)
    l0 = (np.float32(1) - l1).astype(np.float32)
    return i0, i1, l0.astype(np.float64), l1.astype(np.float64)


def upsample_ac0(x, H, W):
    """F.interpolate(x, size=(H, W), mode='bilinear', align_corners=False) in float64 on ATen's fp32 weights."""
    x = np.asarray(x, dtype=np.float64)
    y0, y1, l0h, l1h = axis_weights_ac0(x.shape[-2], H)
    x0, x1, l0w, l1w = axis_weights_ac0(x.shape[-1], W)
    top = x[..., y0, :][..., :, x0] * l0w + x[..., y0, :][..., :, x1] * l1w
    bot = x[..., y1, :][..., :, x0] * l0w + x[..., y1, :][..., :, x1] * l1w
    return top * l0h[:, None] + bot * l1h[:, None]


def upsample_ac0_adjoint(g, h, w):
    """Adjoint of `upsample_ac0`: g [..., H, W] -> [..., h, w]."""
    g = np.asarray(g, dtype=np.float64)
    H, W = g.shape[-2:]
    y0, y1, l0h, l1h = axis_weights_ac0(h, H)
    x0, x1, l0w, l1w = axis_weights_ac0(w, W)
    lead = g.shape[:-2]
    tmp = np.zeros(lead + (H, w))
    np.add.at(tmp, (..., slice(None), x0), g * l0w)
    np.add.at(tmp, (..., slice(None), x1), g * l1w)
    out = np.zeros(lead + (h, w))
    np.add.at(out, (..., y0, slice(None)), tmp * l0h[:, None])
    np.add.at(out, (..., y1, slice(None)), tmp * l1h[:, None])
    return out


def up_ohem_ce_ac0(src, labels, thresh, ignore=IGNORE):
    """OhemCE(upsample_ac0(src), labels) with gradient w.r.t. the low-res src (a BiSeNet head + OhemCELoss)."""
    H, W = labels.shape[1:]
    z = upsample_ac0(src, H, W)
    mean, dz, loss_px, mask = ohem_ce(z, labels, thresh, ignore)
    return mean, upsample_ac0_adjoint(dz, src.shape[-2], src.shape[-1]), loss_px, mask
