"""The C ABI refuses dtype codes outside the set an entry point dispatches on: return code 2 and an error message that
names the entry point and says "unsupported".

Every case passes at least one image or element (the n == 0 early returns would hide the check) and non-NULL
placeholder pointers, with arguments for which the refusal comes before any CUDA runtime call: the up_ce fast paths
are not tried (no channel-maximum buffer, cmax = NULL) and mdseg_mds_bwd's label dtype goes down its generic route
(dense graphs), where mdseg_up_ce_bwd refuses it.

Covered: mdseg_lut_remap, mdseg_lut_remap_images, mdseg_multihot_remap, mdseg_confusion, mdseg_confusion_images,
mdseg_ohem_ce_fwd / _bwd, mdseg_proj_fwd / _bwd / _bwd_graph, mdseg_proj_fwd_tc / _bwd_tc / _bwd_graph_tc,
mdseg_proj_fwd_nhwc / _bwd_nhwc, mdseg_nhwc_to_planar, mdseg_planar_to_nhwc, mdseg_up_ce_fwd / _bwd,
mdseg_up_ce_fwd_ac0 / _bwd_ac0, mdseg_mds_bwd, mdseg_argmax_hist, mdseg_eval_fused (logits dtype),
mdseg_softmax_nchw / _bwd_nchw, mdseg_up_nll_fwd / _bwd.

Left out, because the refusal comes after a CUDA runtime call:
- mdseg_add_planes, mdseg_eval_accum, mdseg_label_nearest, mdseg_eval_chip_accum: after sm_count()'s device query;
- mdseg_up_ce_bwd_direct's label dtype: after the planes' memset (generic route) or the tensor-map encode (fused
  route); its destination dtype is refused by the table check, as a bad table;
- mdseg_eval_fused's label dtype: after the statistics kernel.
mdseg_label_pipeline and the tc16 entry points take a part of a set under their own rules, not one of these refusals.

The placeholders are not device memory, so none of this may reach a GPU: the module is skipped wherever CUDA is
available.
"""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.skipif(torch.cuda.is_available(),
                                reason="placeholder pointers are not device memory: run only where no GPU is present")

P = 1 << 20  # placeholder device pointer: non-NULL, 256-byte aligned, never dereferenced on the host
N_IMG, C_CLS, C_UNI, h, w = 1, 4, 8, 4, 4
hw = h * w
BAD_FLOAT = (7, 99, 10)  # 10 = MDSEG_U8: an int code in a float slot
BAD_INT = (7, 99, 0)     # 0 = MDSEG_F32: a float code in an int slot


def _N():
    from mdseg_b200 import native
    return native


def _src(dtype, stride=C_CLS * hw):
    N = _N()
    t = N.SrcTable()
    t.n_datasets, t.dtype, t.C[0], t.C_alloc[0], t.base[0], t.image_stride[0] = 1, dtype, C_CLS, C_CLS, P, stride
    t.cmax = None  # no channel-maximum buffer: the up_ce fast paths are not tried
    return t


def _graphs(dense):
    N = _N()
    g = N.GraphTable()
    g.n_datasets, g.C_uni = 1, C_UNI
    g.g[0].C_ds, g.g[0].nnz = C_CLS, 0
    if dense:
        g.g[0].dense = P
    else:
        g.g[0].csr_ptr, g.g[0].csc_ptr = P, P
    return g


def _up_ce_fwd(label_dtype, dtype):
    N = _N()
    return N.lib.mdseg_up_ce_fwd(C.byref(_src(dtype)), None, P, label_dtype, N_IMG, h, w, 2 * h, 2 * w, 255, P, P, P,
                                 P, None)


def _up_ce_bwd(label_dtype, dtype):
    N = _N()
    dA, dB = _src(N.F32), _src(N.F32)
    return N.lib.mdseg_up_ce_bwd(C.byref(_src(dtype)), None, P, label_dtype, N_IMG, h, w, 2 * h, 2 * w, 255, P, P, P,
                                 P, 1.0, C.byref(dA), C.byref(dB), None)


def _ac0_fwd(label_dtype, dtype):
    N = _N()
    return N.lib.mdseg_up_ce_fwd_ac0(C.byref(_src(dtype)), None, P, label_dtype, N_IMG, h, w, 2 * h, 2 * w, 255, P,
                                     P, P, P, None)


def _ac0_bwd(label_dtype, dtype):
    N = _N()
    src, dst = _src(dtype), _src(N.F32)
    ws = N.lib.mdseg_up_ce_bwd_ac0_workspace_bytes(C.byref(src), N_IMG, h, w, 2 * h, 2 * w)
    # one dataset and no dataset ids: the planes are not zeroed before the dispatch
    return N.lib.mdseg_up_ce_bwd_ac0(C.byref(src), None, P, label_dtype, N_IMG, h, w, 2 * h, 2 * w, 255, P, P, P, P,
                                     1.0, C.byref(dst), P, ws, None)


def _mds_bwd(label_dtype, dx_dtype):
    N = _N()
    src, g = _src(N.F32), _graphs(dense=True)  # a dense graph takes the generic route
    ws = N.lib.mdseg_mds_bwd_workspace_bytes(C.byref(src), C.byref(g), N_IMG, h, w, 2 * h, 2 * w)
    return N.lib.mdseg_mds_bwd(C.byref(src), C.byref(g), None, P, label_dtype, N_IMG, h, w, 2 * h, 2 * w, 255, P, P,
                               P, P, 1.0, P, dx_dtype, P, ws, None)


def _confusion_images(label_dtype, pred_dtype):
    N = _N()
    tab = N.HistTable()
    tab.n_datasets, tab.C[0], tab.offset[0] = 1, C_CLS, 0
    return N.lib.mdseg_confusion_images(P, label_dtype, P, pred_dtype, P, None, N_IMG, hw, P, C.byref(tab), 255, P,
                                        None)


def _nhwc_move(name, dtype):
    N = _N()
    a, b = _src(dtype), _src(dtype)
    return getattr(N.lib, name)(C.byref(a), None, N_IMG, h, w, C.byref(b), None)


def _eval_fused(dtype):
    N = _N()
    ps = N.EvalPasses()
    ps.n_passes, ps.dtype = 1, dtype
    ps.p[0].logits, ps.p[0].h, ps.p[0].w = P, h, w
    return N.lib.mdseg_eval_fused(C.byref(ps), C_CLS, 2 * h, 2 * w, P, P, N.U8, P, P, 255, P, 1 << 20, P, None)


def _lib(name):
    return getattr(_N().lib, name)


# (entry point named in the message, kind of code, call(code) -> rc)
CASES = {
    "lut_remap.in": ("mdseg_lut_remap", BAD_INT, lambda c: _lib("mdseg_lut_remap")(P, c, P, _N().U8, P, 255, hw, None)),
    "lut_remap.out": ("mdseg_lut_remap", BAD_INT,
                      lambda c: _lib("mdseg_lut_remap")(P, _N().U8, P, c, P, 255, hw, None)),
    "lut_remap_images.in": ("mdseg_lut_remap_images", BAD_INT,
                            lambda c: _lib("mdseg_lut_remap_images")(P, c, P, _N().U8, P, 1, None, 255, N_IMG, hw, P,
                                                                     None)),
    # the out_dtype refusal of both remaps may name their common prefix
    "lut_remap_images.out": ("mdseg_lut_remap", BAD_INT,
                             lambda c: _lib("mdseg_lut_remap_images")(P, _N().U8, P, c, P, 1, None, 255, N_IMG, hw, P,
                                                                      None)),
    "multihot_remap": ("mdseg_multihot_remap", BAD_INT,
                       lambda c: _lib("mdseg_multihot_remap")(P, c, P, C_UNI, hw, P, None)),
    "confusion.label": ("mdseg_confusion", BAD_INT,
                        lambda c: _lib("mdseg_confusion")(P, c, P, _N().I64, None, P, C_CLS, C_CLS, 255, hw, P, None)),
    "confusion.pred": ("mdseg_confusion", BAD_INT,
                       lambda c: _lib("mdseg_confusion")(P, _N().U8, P, c, None, P, C_CLS, C_CLS, 255, hw, P, None)),
    "confusion_images.label": ("mdseg_confusion_images", BAD_INT, lambda c: _confusion_images(c, _N().I64)),
    "confusion_images.pred": ("mdseg_confusion_images", BAD_INT, lambda c: _confusion_images(_N().U8, c)),
    "ohem_ce_fwd.dtype": ("mdseg_ohem_ce_fwd", BAD_FLOAT,
                          lambda c: _lib("mdseg_ohem_ce_fwd")(P, c, _N().NCHW, P, _N().I64, N_IMG, C_CLS, h, w, 255, P,
                                                              P, P, P, None)),
    "ohem_ce_fwd.label": ("mdseg_ohem_ce_fwd", BAD_INT,
                          lambda c: _lib("mdseg_ohem_ce_fwd")(P, _N().F32, _N().NCHW, P, c, N_IMG, C_CLS, h, w, 255, P,
                                                              P, P, P, None)),
    "ohem_ce_bwd.dtype": ("mdseg_ohem_ce_bwd", BAD_FLOAT,
                          lambda c: _lib("mdseg_ohem_ce_bwd")(P, c, _N().NCHW, P, _N().I64, N_IMG, C_CLS, h, w, 255, P,
                                                              P, P, P, 1.0, P, None)),
    "ohem_ce_bwd.label": ("mdseg_ohem_ce_bwd", BAD_INT,
                          lambda c: _lib("mdseg_ohem_ce_bwd")(P, _N().F32, _N().NCHW, P, c, N_IMG, C_CLS, h, w, 255, P,
                                                              P, P, P, 1.0, P, None)),
    "proj_fwd": ("mdseg_proj_fwd", BAD_FLOAT,
                 lambda c: _lib("mdseg_proj_fwd")(P, c, C.byref(_graphs(True)), None, N_IMG, h, w, P, C_CLS, None,
                                                  None, None)),
    "proj_bwd": ("mdseg_proj_bwd", BAD_FLOAT,
                 lambda c: _lib("mdseg_proj_bwd")(P, P, C_CLS, C.byref(_graphs(True)), None, N_IMG, h, w, P, c, None)),
    "proj_bwd_graph": ("mdseg_proj_bwd_graph", BAD_FLOAT,
                       lambda c: _lib("mdseg_proj_bwd_graph")(P, c, P, P, C_CLS, C.byref(_graphs(True)), None, N_IMG, h,
                                                              w, P, C_CLS * C_UNI, None)),
    "proj_fwd_tc": ("mdseg_proj_fwd_tc", BAD_FLOAT,
                    lambda c: _lib("mdseg_proj_fwd_tc")(P, c, C.byref(_graphs(True)), None, N_IMG, h, w, P, C_CLS, None,
                                                        P, 1 << 20, None, None)),
    "proj_bwd_tc": ("mdseg_proj_bwd_tc", BAD_FLOAT,
                    lambda c: _lib("mdseg_proj_bwd_tc")(P, P, C_CLS, C.byref(_graphs(True)), None, N_IMG, h, w, P, c, P,
                                                        1 << 20, None)),
    "proj_bwd_graph_tc": ("mdseg_proj_bwd_graph_tc", BAD_FLOAT,
                          lambda c: _lib("mdseg_proj_bwd_graph_tc")(P, c, P, P, C_CLS, C.byref(_graphs(True)), None,
                                                                    N_IMG, h, w, P, C_CLS * C_UNI, P, 1 << 20, None)),
    "proj_fwd_nhwc": ("mdseg_proj_fwd_nhwc", BAD_FLOAT,
                      lambda c: _lib("mdseg_proj_fwd_nhwc")(P, c, C.byref(_graphs(False)), None, N_IMG, h, w, P, C_CLS,
                                                            None, None, None)),
    "proj_bwd_nhwc": ("mdseg_proj_bwd_nhwc", BAD_FLOAT,
                      lambda c: _lib("mdseg_proj_bwd_nhwc")(P, P, C_CLS, C.byref(_graphs(False)), None, N_IMG, h, w, P,
                                                            c, None)),
    "nhwc_to_planar": ("mdseg_nhwc_to_planar", BAD_FLOAT, lambda c: _nhwc_move("mdseg_nhwc_to_planar", c)),
    "planar_to_nhwc": ("mdseg_planar_to_nhwc", BAD_FLOAT, lambda c: _nhwc_move("mdseg_planar_to_nhwc", c)),
    "up_ce_fwd.dtype": ("mdseg_up_ce_fwd", BAD_FLOAT, lambda c: _up_ce_fwd(_N().I64, c)),
    "up_ce_fwd.label": ("mdseg_up_ce_fwd", BAD_INT, lambda c: _up_ce_fwd(c, _N().F32)),
    "up_ce_bwd.dtype": ("mdseg_up_ce_bwd", BAD_FLOAT, lambda c: _up_ce_bwd(_N().I64, c)),
    "up_ce_bwd.label": ("mdseg_up_ce_bwd", BAD_INT, lambda c: _up_ce_bwd(c, _N().F32)),
    "up_ce_fwd_ac0.dtype": ("mdseg_up_ce_fwd_ac0", BAD_FLOAT, lambda c: _ac0_fwd(_N().I64, c)),
    "up_ce_fwd_ac0.label": ("mdseg_up_ce_fwd_ac0", BAD_INT, lambda c: _ac0_fwd(c, _N().F32)),
    "up_ce_bwd_ac0.dtype": ("mdseg_up_ce_bwd_ac0", BAD_FLOAT, lambda c: _ac0_bwd(_N().I64, c)),
    "up_ce_bwd_ac0.label": ("mdseg_up_ce_bwd_ac0", BAD_INT, lambda c: _ac0_bwd(c, _N().F32)),
    "mds_bwd.dx": ("mdseg_mds_bwd", BAD_FLOAT, lambda c: _mds_bwd(_N().I64, c)),
    # the generic route passes the labels to mdseg_up_ce_bwd, which refuses them under its own name
    "mds_bwd.label": ("mdseg_up_ce_bwd", BAD_INT, lambda c: _mds_bwd(c, _N().F32)),
    "argmax_hist": ("mdseg_argmax_hist", BAD_INT,
                    lambda c: _lib("mdseg_argmax_hist")(P, C_CLS, hw, P, P, c, None, P, 255, P, None)),
    "eval_fused.dtype": ("mdseg_eval_fused", BAD_FLOAT, _eval_fused),
    "softmax_nchw": ("mdseg_softmax_nchw", BAD_FLOAT,
                     lambda c: _lib("mdseg_softmax_nchw")(P, c, N_IMG, C_CLS, hw, P, None)),
    "softmax_bwd_nchw": ("mdseg_softmax_bwd_nchw", BAD_FLOAT,
                         lambda c: _lib("mdseg_softmax_bwd_nchw")(P, P, N_IMG, C_CLS, hw, P, c, None)),
    "up_nll_fwd": ("mdseg_up_nll_fwd", BAD_INT,
                   lambda c: _lib("mdseg_up_nll_fwd")(C.byref(_src(_N().F32)), None, P, c, N_IMG, h, w, 2 * h, 2 * w,
                                                      255, P, P, P, None)),
    "up_nll_bwd": ("mdseg_up_nll_bwd", BAD_INT,
                   lambda c: _lib("mdseg_up_nll_bwd")(C.byref(_src(_N().F32)), None, P, c, N_IMG, h, w, 2 * h, 2 * w,
                                                      255, P, P, P, 1.0, C.byref(_src(_N().F32)), None)),
}


@pytest.mark.parametrize("code_index", range(3))
@pytest.mark.parametrize("case", sorted(CASES))
def test_unsupported_dtype_code_is_refused(case, code_index):
    who, codes, call = CASES[case]
    code = codes[code_index]
    rc = call(code)
    msg = _N().lib.mdseg_last_error().decode()
    assert rc == 2, (case, code, rc, msg)
    assert who in msg and "unsupported" in msg, (case, code, msg)
