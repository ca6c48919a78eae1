"""ctypes binding of libmdseg_b200.so (the C ABI declared in include/mdseg.h).

No torch here: plain integers for device pointers and streams.  The library is
built in-tree by ``build.py`` (``__graft_entry__.build()``); importing this
module when the shared object is missing raises — there is no CPU fallback.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmdseg_b200.so")

# --- enums (mirror include/mdseg.h) -------------------------------------------
F32, BF16, F16 = 0, 1, 2
U8, I32, I64 = 10, 11, 12
NCHW, NHWC = 0, 1
ERR_LABEL_RANGE, ERR_PRED_RANGE, ERR_TOPK_RANGE, ERR_DATASET_ID, ERR_GRAPH_KIND = 1, 2, 4, 8, 16
MAX_DATASETS = 32
NHWC_MAX_CUNI, NHWC_MAX_CDS = 1536, 768  # graph limits of mdseg_proj_fwd_nhwc / mdseg_proj_bwd_nhwc


class OhemState(C.Structure):
    _fields_ = [
        ("n_valid", C.c_ulonglong), ("n_hard", C.c_ulonglong), ("n_px", C.c_ulonglong),
        ("n_min", C.c_ulonglong), ("n_sel", C.c_ulonglong), ("n_gt", C.c_ulonglong),
        ("sum_hard", C.c_double), ("sum_sel", C.c_double),
        ("thresh", C.c_float), ("kth", C.c_float), ("inv_n_sel", C.c_float), ("loss", C.c_float),
        ("mode", C.c_uint), ("tie_quota", C.c_uint), ("tie_taken", C.c_uint), ("n_ties", C.c_uint),
        ("reserved", C.c_uint * 8),
    ]


class SrcTable(C.Structure):
    _fields_ = [
        ("base", C.c_void_p * MAX_DATASETS),
        ("image_stride", C.c_longlong * MAX_DATASETS),
        ("C", C.c_int * MAX_DATASETS),
        ("C_alloc", C.c_int * MAX_DATASETS),
        ("n_datasets", C.c_int), ("dtype", C.c_int), ("seg_per_dataset", C.c_int), ("cmax_ready", C.c_int),
        ("cmax", C.c_void_p),
    ]


class SparseGraph(C.Structure):
    _fields_ = [
        ("csr_ptr", C.c_void_p), ("csr_col", C.c_void_p), ("csr_val", C.c_void_p),
        ("csc_ptr", C.c_void_p), ("csc_row", C.c_void_p), ("csc_val", C.c_void_p),
        ("dense", C.c_void_p),
        ("C_ds", C.c_int), ("nnz", C.c_int), ("col_onehot", C.c_int), ("reserved", C.c_int),
        ("csr4_ptr", C.c_void_p), ("csr4_col", C.c_void_p),
    ]


class HistTable(C.Structure):
    _fields_ = [("n_datasets", C.c_int), ("C", C.c_int * MAX_DATASETS), ("offset", C.c_longlong * MAX_DATASETS)]


MAX_EVAL_PASSES = 16


class EvalPass(C.Structure):
    _fields_ = [("logits", C.c_void_p), ("h", C.c_int), ("w", C.c_int), ("flip", C.c_int), ("reserved", C.c_int)]


class EvalPasses(C.Structure):
    _fields_ = [("p", EvalPass * MAX_EVAL_PASSES), ("n_passes", C.c_int), ("dtype", C.c_int)]


class LabelView(C.Structure):
    _fields_ = [("src", C.c_void_p), ("src_row_stride", C.c_longlong), ("src_h", C.c_int), ("src_w", C.c_int),
                ("im_h", C.c_int), ("im_w", C.c_int), ("pad_top", C.c_int), ("pad_left", C.c_int),
                ("crop_y", C.c_int), ("crop_x", C.c_int), ("flip", C.c_int), ("lut", C.c_int)]


class ImageView(C.Structure):
    _fields_ = [("src", C.c_void_p), ("src_row_stride", C.c_longlong), ("src_h", C.c_int), ("src_w", C.c_int),
                ("im_h", C.c_int), ("im_w", C.c_int), ("pad_top", C.c_int), ("pad_left", C.c_int),
                ("crop_y", C.c_int), ("crop_x", C.c_int), ("flip", C.c_int), ("swap_rb", C.c_int),
                ("norm", C.c_int), ("saturate", C.c_int), ("sat_diag", C.c_float), ("sat_off", C.c_float),
                ("lut", C.c_uint8 * 256)]


class GraphTable(C.Structure):
    _fields_ = [("g", SparseGraph * MAX_DATASETS), ("n_datasets", C.c_int), ("C_uni", C.c_int)]


_P, _I, _L, _F = C.c_void_p, C.c_int, C.c_int64, C.c_float

# name -> (restype, argtypes); every symbol of include/mdseg.h
SIGNATURES = {
    "mdseg_version": (_I, []),
    "mdseg_last_error": (C.c_char_p, []),
    "mdseg_sm_count": (_I, []),
    "mdseg_lut_remap": (_I, [_P, _I, _P, _I, _P, _I, _L, _P]),
    "mdseg_multihot_remap": (_I, [_P, _I, _P, _I, _L, _P, _P]),
    "mdseg_confusion": (_I, [_P, _I, _P, _I, _P, _P, _I, _I, _I, _L, _P, _P]),
    "mdseg_miou": (_I, [_P, _I, _P, _P, _P]),
    "mdseg_lut_remap_images": (_I, [_P, _I, _P, _I, _P, _I, _P, _I, _I, _L, _P, _P]),
    "mdseg_confusion_images": (_I, [_P, _I, _P, _I, _P, _P, _I, _L, _P, C.POINTER(HistTable), _I, _P, _P]),
    "mdseg_miou_images": (_I, [_P, C.POINTER(HistTable), _P, _I, _P, _P]),
    "mdseg_ohem_state_bytes": (C.c_size_t, []),
    "mdseg_select_workspace_bytes": (C.c_size_t, [_I]),
    "mdseg_ohem_begin": (_I, [_P, _I, _F, _P]),
    "mdseg_ohem_ce_fwd": (_I, [_P, _I, _I, _P, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "mdseg_ohem_select": (_I, [_P, _I, _L, _P, _P, _I, _P, _P, _P, _P]),
    "mdseg_ohem_ce_bwd": (_I, [_P, _I, _I, _P, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _F, _P, _P]),
    "mdseg_proj_fwd": (_I, [_P, _I, C.POINTER(GraphTable), _P, _I, _I, _I, _P, _I, _P, _P, _P]),
    "mdseg_proj_fwd_tc_workspace_bytes": (C.c_size_t, [C.POINTER(GraphTable), _I]),
    "mdseg_proj_fwd_tc": (_I, [_P, _I, C.POINTER(GraphTable), _P, _I, _I, _I, _P, _I, _P, _P, C.c_size_t, _P, _P]),
    "mdseg_proj_bwd": (_I, [_P, _P, _I, C.POINTER(GraphTable), _P, _I, _I, _I, _P, _I, _P]),
    "mdseg_proj_bwd_tc_workspace_bytes": (C.c_size_t, [C.POINTER(GraphTable), _I]),
    "mdseg_proj_bwd_tc": (_I, [_P, _P, _I, C.POINTER(GraphTable), _P, _I, _I, _I, _P, _I, _P, C.c_size_t, _P]),
    "mdseg_proj_bwd_graph": (_I, [_P, _I, _P, _P, _I, C.POINTER(GraphTable), _P, _I, _I, _I, _P, C.c_longlong, _P]),
    "mdseg_proj_bwd_graph_tc_workspace_bytes": (C.c_size_t, [C.POINTER(GraphTable), _I, _I, _I]),
    "mdseg_proj_bwd_graph_tc": (_I, [_P, _I, _P, _P, _I, C.POINTER(GraphTable), _P, _I, _I, _I, _P, C.c_longlong, _P,
                                     C.c_size_t, _P]),
    "mdseg_proj_fwd_nhwc": (_I, [_P, _I, C.POINTER(GraphTable), _P, _I, _I, _I, _P, _I, _P, _P, _P]),
    "mdseg_proj_bwd_nhwc": (_I, [_P, _P, _I, C.POINTER(GraphTable), _P, _I, _I, _I, _P, _I, _P]),
    "mdseg_nhwc_to_planar": (_I, [C.POINTER(SrcTable), _P, _I, _I, _I, C.POINTER(SrcTable), _P]),
    "mdseg_planar_to_nhwc": (_I, [C.POINTER(SrcTable), _P, _I, _I, _I, C.POINTER(SrcTable), _P]),
    "mdseg_up_ce_fwd": (_I, [C.POINTER(SrcTable), _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "mdseg_up_ce_bwd": (_I, [C.POINTER(SrcTable), _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _F,
                             C.POINTER(SrcTable), C.POINTER(SrcTable), _P]),
    "mdseg_mds_bwd_workspace_bytes": (C.c_size_t, [C.POINTER(SrcTable), C.POINTER(GraphTable), _I, _I, _I, _I, _I]),
    "mdseg_mds_bwd": (_I, [C.POINTER(SrcTable), C.POINTER(GraphTable), _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P,
                           _P, _F, _P, _I, _P, C.c_size_t, _P]),
    "mdseg_up_ce_bwd_direct_workspace_bytes": (C.c_size_t, [C.POINTER(SrcTable), _I, _I, _I, _I, _I]),
    "mdseg_up_ce_bwd_direct_is_fused": (_I, [C.POINTER(SrcTable), _I, _I, _I, _I]),
    "mdseg_up_ce_bwd_direct": (_I, [C.POINTER(SrcTable), _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _F,
                                    C.POINTER(SrcTable), _P, C.c_size_t, _P]),
    "mdseg_add_planes": (_I, [_P, _P, _P, _I, _L, _P]),
    "mdseg_eval_accum": (_I, [_P, _I, _I, _I, _I, _P, _I, _I, _I, _I, _P]),
    "mdseg_eval_fused_workspace_bytes": (C.c_size_t, [_I, _I, _I]),
    "mdseg_eval_fused": (_I, [C.POINTER(EvalPasses), _I, _I, _I, _P, _P, _I, _P, _P, _I, _P, C.c_size_t, _P, _P]),
    "mdseg_argmax_hist": (_I, [_P, _I, _L, _P, _P, _I, _P, _P, _I, _P, _P]),
    "mdseg_label_nearest": (_I, [_P, _I, _I, _I, _P, _I, _I, _I, _P]),
    "mdseg_label_pipeline": (_I, [_P, _I, _P, _I, _P, _I, _I, _I, _I, _P]),
    "mdseg_image_pipeline": (_I, [_P, _I, _P, _I, _P, _I, _I, _I, _P]),
    "mdseg_graph_build_onehot_ints": (C.c_size_t, [_I, _I]),
    "mdseg_graph_build_onehot": (_I, [_P, _I, _I, _P, _P, _P]),
    "mdseg_head_tc16_tile": (_I, [_I]),
    "mdseg_proj_fwd_tc16": (_I, [_P, _I, _I, _I, _I, _L, C.POINTER(C.c_void_p), _I, C.POINTER(C.c_int), _I, _P, _P, _I,
                                 _P]),
    "mdseg_proj_bwd_tc16": (_I, [_P, _I, _I, _I, _I, _L, C.POINTER(C.c_void_p), _I, _I, _I, _P, _P, _I, _P]),
    "mdseg_proj_bwd_graph_tc16_workspace_bytes": (C.c_size_t, [_I, _I, _L, _I]),
    "mdseg_proj_bwd_graph_tc16": (_I, [_P, _P, _I, _I, _I, _I, _L, _I, _P, _I, _P, _P, C.c_size_t, _P]),
    "mdseg_eval_chip_accum": (_I, [_P, _P, _I, _I, _I, _I, _P, _I, _I, _I, _I, _I, _P]),
    "mdseg_prob_resize_accum": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _P, _I, _I, _I, _P]),
    "mdseg_softmax_nchw": (_I, [_P, _I, _I, _I, _L, _P, _P]),
    "mdseg_softmax_bwd_nchw": (_I, [_P, _P, _I, _I, _L, _P, _I, _P]),
    "mdseg_up_nll_fwd": (_I, [C.POINTER(SrcTable), _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P]),
    "mdseg_up_nll_bwd": (_I, [C.POINTER(SrcTable), _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _F,
                              C.POINTER(SrcTable), _P]),
}


class MdsegError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback for the mdseg hot path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def call(name, *args):
    """Call an int-returning entry point; raise MdsegError with the library's message on failure."""
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise MdsegError(f"{name} failed ({rc}): {lib.mdseg_last_error().decode(errors='replace')}")


def version():
    return lib.mdseg_version()
