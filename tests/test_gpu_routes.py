"""GPU: the native entry points each loss runs, forward and backward, and the memory format of every gradient it
returns, for every dtype, layout, graph kind, gradient set and backward geometry the host-side routing distinguishes.
The table is what the routing chose when it was written; a change of route shows up here before it shows up as a
changed number or time.  `python tests/test_gpu_routes.py` prints the table of the current tree."""
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CL = torch.channels_last
N_CATS, C_UNI, IDS = [8, 12, 10], 40, [0, 2, 1, 2]
# (h, w, H, W): the fused backward's geometry, and one with W % 16 != 0 (the two-plane adjoint)
GEOMS = {"fused": (8, 32, 32, 128), "w16": (8, 32, 32, 120)}
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16}
GRADS = ["dx", "dx_dg", "dg", "none"]


def _fmt(t):
    if t.dim() == 4 and not t.is_contiguous() and t.is_contiguous(memory_format=CL):
        return "cl"
    return "contig" if t.is_contiguous() else "strided"


def _record(ops, fn, leaves):
    """(the forward's entry points, the backward's entry points, the memory format of each gradient) of fn(), each a
    space-separated string, entry points without their mdseg_ prefix."""
    names, raw = [], ops.N.call

    def call(name, *a):
        names.append(name)
        return raw(name, *a)

    ops.N.call = call
    try:
        out = fn()
        fwd, names[:] = tuple(names), []
        grads = torch.autograd.grad(out.float().sum(), leaves) if leaves else ()
        torch.cuda.synchronize()
    finally:
        ops.N.call = raw
    short = lambda ns: " ".join(n.removeprefix("mdseg_") for n in ns)
    return short(fwd), short(names), " ".join(_fmt(g) for g in grads)


def _labels(gen, H, W, n_cats=N_CATS, ids=IDS):
    lb = torch.stack([torch.randint(0, n_cats[d], (H, W), generator=gen) for d in ids])
    lb[torch.rand(len(ids), H, W, generator=gen) < 0.05] = 255
    return lb.to(DEV), torch.tensor(ids, dtype=torch.int32, device=DEV)


def _graphs(gen, kind, n_cats=N_CATS, c_uni=C_UNI):
    out = []
    for c in n_cats:
        if kind == "sparse":  # 0/1, one 1 per column
            idx = torch.randint(0, c, (c_uni,), generator=gen)
            idx[:c] = torch.arange(c)
            m = torch.zeros(c, c_uni)
            m[idx, torch.arange(c_uni)] = 1
        else:
            m = torch.randn(c, c_uni, generator=gen) * 0.3
        out.append(m.to(DEV))
    return out


def _x(gen, dtype, layout, shape):
    x = torch.randn(*shape, generator=gen).to(DEV, dtype)
    return x.contiguous(memory_format=CL) if layout == "cl" else x


def _mds_case(ops, dtype, layout, kind, grads, geom, per_dataset=False):
    gen = torch.Generator().manual_seed(1)
    h, w, H, W = GEOMS[geom]
    x = _x(gen, DTYPES[dtype], layout, (len(IDS), C_UNI, h, w))
    graphs = _graphs(gen, kind)
    labels, ids = _labels(gen, H, W)
    leaves = []
    if grads in ("dx", "dx_dg"):
        leaves.append(x.requires_grad_(True))
    if grads in ("dx_dg", "dg"):
        leaves += [g.requires_grad_(True) for g in graphs]
    cache = ops.BipartiteGraphs(assume_dense=kind == "dense_assumed")
    return _record(ops, lambda: ops.mds_proj_ohem_ce(x, labels, ids, graphs, 0.7, cache=cache, per_dataset=per_dataset),
                   leaves)


def _head_case(ops, fn, dtype, layout):
    gen = torch.Generator().manual_seed(2)
    h, w, H, W = GEOMS["fused"]
    feats = _x(gen, DTYPES[dtype], layout, (len(IDS), 32, h, w)).requires_grad_(True)
    proto = (torch.randn(C_UNI, 32, generator=gen) * 0.2).to(DEV).requires_grad_(True)
    graphs = [g.requires_grad_(True) for g in _graphs(gen, "dense")]
    labels, ids = _labels(gen, H, W)
    leaves = [feats, proto, *graphs]
    if fn == "ce_mean":
        return _record(ops, lambda: ops.mds_head_proj_ce_mean(feats, proto, labels, ids, graphs), leaves)
    return _record(ops, lambda: ops.mds_head_proj_ohem_ce(feats, proto, labels, ids, graphs, 0.7), leaves)


def _heads_case(ops, dtype, layout, geom):
    gen = torch.Generator().manual_seed(3)
    h, w, H, W = GEOMS[geom]
    x = _x(gen, DTYPES[dtype], layout, (len(IDS), C_UNI, h, w)).requires_grad_(True)
    sets = [[g.requires_grad_(True) for g in _graphs(gen, "dense")] for _ in range(2)]
    labels, ids = _labels(gen, H, W)
    return _record(ops, lambda: ops.mds_proj_ohem_ce_heads(x, labels, ids, sets, 0.7),
                   [x, *[g for s in sets for g in s]])


def _up_case(ops, dtype, layout, ac, seg, geom):
    gen = torch.Generator().manual_seed(4)
    h, w, H, W = GEOMS[geom]
    srcs = [_x(gen, DTYPES[dtype], layout, (len(IDS), c, h, w)).requires_grad_(True) for c in N_CATS]
    labels, ids = _labels(gen, H, W)
    return _record(ops, lambda: ops.up_ohem_ce(srcs, labels, ids, 0.7, seg_per_dataset=seg, align_corners=ac), srcs)


def _ohem_case(ops, fn, dtype, layout):
    gen = torch.Generator().manual_seed(5)
    _, _, H, W = GEOMS["fused"]
    lgs = [_x(gen, DTYPES[dtype], layout, (2, c, H // 2, W // 2)).requires_grad_(True) for c in N_CATS[:2]]
    lbs = [torch.randint(0, c, (2, H // 2, W // 2), generator=gen).to(DEV) for c in N_CATS[:2]]
    if fn == "ohem_ce":
        return _record(ops, lambda: ops.ohem_ce(lgs[0], lbs[0], 0.7), lgs[:1])
    return _record(ops, lambda: ops.mds_ohem_ce_full(lgs, lbs, 0.7), lgs)


def _nll_case(ops, kind):
    gen = torch.Generator().manual_seed(6)
    h, w, H, W = GEOMS["fused"]
    x = _x(gen, torch.float32, "nchw", (len(IDS), C_UNI, h, w)).requires_grad_(True)
    graphs = _graphs(gen, kind)
    labels, ids = _labels(gen, H, W)
    leaves = [x] + ([g.requires_grad_(True) for g in graphs] if kind == "dense" else [])
    return _record(ops, lambda: ops.mds_nll_plus(x, labels, ids, graphs, 0.7, cache=ops.BipartiteGraphs()), leaves)


def _proto_case(ops, dtype, layout):
    gen = torch.Generator().manual_seed(7)
    h, w, _, _ = GEOMS["fused"]
    feats = _x(gen, DTYPES[dtype], layout, (2, 32, h, w)).requires_grad_(True)
    proto = torch.randn(C_UNI, 32, generator=gen).to(DEV).requires_grad_(True)
    return _record(ops, lambda: ops.prototype_head(feats, proto), [feats, proto])


def _cases():
    cases = {}
    for dt in DTYPES:
        for lay in ("nchw", "cl"):
            for kind in ("sparse", "dense", "dense_assumed"):
                for gr in GRADS:
                    for geom in GEOMS:
                        cases[f"mds-{dt}-{lay}-{kind}-{gr}-{geom}"] = (_mds_case, dt, lay, kind, gr, geom)
            cases[f"mds_per_dataset-{dt}-{lay}"] = (_mds_case, dt, lay, "sparse", "dx", "fused", True)
            for fn in ("ohem", "ce_mean"):
                cases[f"head_{fn}-{dt}-{lay}"] = (_head_case, fn, dt, lay)
            for geom in GEOMS:
                cases[f"heads-{dt}-{lay}-{geom}"] = (_heads_case, dt, lay, geom)
            for ac in (True, False):
                for seg in (True, False):
                    for geom in (GEOMS if ac else ["fused"]):
                        cases[f"up-{dt}-{lay}-ac{int(ac)}-seg{int(seg)}-{geom}"] = (_up_case, dt, lay, ac, seg, geom)
            for fn in ("ohem_ce", "mds_ohem_ce_full"):
                cases[f"{fn}-{dt}-{lay}"] = (_ohem_case, fn, dt, lay)
            cases[f"prototype_head-{dt}-{lay}"] = (_proto_case, dt, lay)
    for kind in ("sparse", "dense"):
        cases[f"nll_plus-{kind}"] = (_nll_case, kind)
    return cases


CASES = _cases()


def run_case(ops, name):
    """The case's record, or ("raises", exception type) for an input the op rejects."""
    fn, *args = CASES[name]
    try:
        return fn(ops, *args)
    except (ValueError, TypeError, RuntimeError) as e:
        return ("raises", type(e).__name__)


# written by `python tests/test_gpu_routes.py` on a B200
EXPECTED = {
    'mds-f32-nchw-sparse-dx-fused': ('lut_remap proj_fwd ohem_begin up_ce_fwd ohem_select', 'mds_bwd', 'contig'),
    'mds-f32-nchw-sparse-dx-w16': ('lut_remap proj_fwd ohem_begin up_ce_fwd ohem_select', 'mds_bwd', 'contig'),
    'mds-f32-nchw-sparse-dx_dg-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-f32-nchw-sparse-dx_dg-w16': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-f32-nchw-sparse-dg-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-f32-nchw-sparse-dg-w16': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-f32-nchw-sparse-none-fused': ('lut_remap proj_fwd ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-f32-nchw-sparse-none-w16': ('lut_remap proj_fwd ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-f32-nchw-dense-dx-fused': ('lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select', 'mds_bwd', 'contig'),
    'mds-f32-nchw-dense-dx-w16': ('lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select', 'mds_bwd', 'contig'),
    'mds-f32-nchw-dense-dx_dg-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-f32-nchw-dense-dx_dg-w16': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-f32-nchw-dense-dg-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-f32-nchw-dense-dg-w16': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-f32-nchw-dense-none-fused': ('lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-f32-nchw-dense-none-w16': ('lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-f32-nchw-dense_assumed-dx-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'mds_bwd',
        'contig',
    ),
    'mds-f32-nchw-dense_assumed-dx-w16': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'mds_bwd',
        'contig',
    ),
    'mds-f32-nchw-dense_assumed-dx_dg-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-f32-nchw-dense_assumed-dx_dg-w16': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-f32-nchw-dense_assumed-dg-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-f32-nchw-dense_assumed-dg-w16': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-f32-nchw-dense_assumed-none-fused': ('lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-f32-nchw-dense_assumed-none-w16': ('lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds_per_dataset-f32-nchw': ('lut_remap proj_fwd ohem_begin up_ce_fwd ohem_select', 'mds_bwd', 'contig'),
    'head_ohem-f32-nchw': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig contig',
    ),
    'head_ce_mean-f32-nchw': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig contig',
    ),
    'heads-f32-nchw-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct up_ce_bwd_direct proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig contig contig contig',
    ),
    'heads-f32-nchw-w16': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig contig contig contig',
    ),
    'up-f32-nchw-ac1-seg1-fused': (
        'lut_remap ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct',
        'contig contig contig',
    ),
    'up-f32-nchw-ac1-seg1-w16': (
        'lut_remap ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct',
        'contig contig contig',
    ),
    'up-f32-nchw-ac1-seg0-fused': (
        'lut_remap ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct',
        'contig contig contig',
    ),
    'up-f32-nchw-ac1-seg0-w16': (
        'lut_remap ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct',
        'contig contig contig',
    ),
    'up-f32-nchw-ac0-seg1-fused': (
        'lut_remap ohem_begin up_ce_fwd_ac0 ohem_select',
        'up_ce_bwd_ac0',
        'contig contig contig',
    ),
    'up-f32-nchw-ac0-seg0-fused': (
        'lut_remap ohem_begin up_ce_fwd_ac0 ohem_select',
        'up_ce_bwd_ac0',
        'contig contig contig',
    ),
    'ohem_ce-f32-nchw': ('ohem_begin ohem_ce_fwd ohem_select', 'ohem_ce_bwd', 'contig'),
    'mds_ohem_ce_full-f32-nchw': (
        'ohem_begin ohem_ce_fwd ohem_ce_fwd ohem_select',
        'ohem_ce_bwd ohem_ce_bwd',
        'contig contig',
    ),
    'prototype_head-f32-nchw': ('proj_fwd_tc', 'proj_bwd_tc proj_bwd_graph_tc', 'contig contig'),
    'mds-f32-cl-sparse-dx-fused': (
        'lut_remap proj_fwd_nhwc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_nhwc',
        'cl',
    ),
    'mds-f32-cl-sparse-dx-w16': (
        'lut_remap proj_fwd_nhwc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_nhwc',
        'cl',
    ),
    'mds-f32-cl-sparse-dx_dg-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-f32-cl-sparse-dx_dg-w16': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-f32-cl-sparse-dg-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-f32-cl-sparse-dg-w16': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-f32-cl-sparse-none-fused': ('lut_remap proj_fwd_nhwc ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-f32-cl-sparse-none-w16': ('lut_remap proj_fwd_nhwc ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-f32-cl-dense-dx-fused': ('lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select', 'mds_bwd', 'contig'),
    'mds-f32-cl-dense-dx-w16': ('lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select', 'mds_bwd', 'contig'),
    'mds-f32-cl-dense-dx_dg-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-f32-cl-dense-dx_dg-w16': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-f32-cl-dense-dg-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-f32-cl-dense-dg-w16': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-f32-cl-dense-none-fused': ('lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-f32-cl-dense-none-w16': ('lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-f32-cl-dense_assumed-dx-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'mds_bwd',
        'contig',
    ),
    'mds-f32-cl-dense_assumed-dx-w16': ('lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select', 'mds_bwd', 'contig'),
    'mds-f32-cl-dense_assumed-dx_dg-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-f32-cl-dense_assumed-dx_dg-w16': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-f32-cl-dense_assumed-dg-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-f32-cl-dense_assumed-dg-w16': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-f32-cl-dense_assumed-none-fused': ('lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-f32-cl-dense_assumed-none-w16': ('lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds_per_dataset-f32-cl': (
        'lut_remap proj_fwd_nhwc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_nhwc',
        'cl',
    ),
    'head_ohem-f32-cl': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig contig',
    ),
    'head_ce_mean-f32-cl': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig contig',
    ),
    'heads-f32-cl-fused': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct up_ce_bwd_direct proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig contig contig contig',
    ),
    'heads-f32-cl-w16': (
        'lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select lut_remap proj_fwd_tc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig contig contig contig',
    ),
    'up-f32-cl-ac1-seg1-fused': (
        'lut_remap nhwc_to_planar ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct planar_to_nhwc',
        'cl cl cl',
    ),
    'up-f32-cl-ac1-seg1-w16': (
        'lut_remap nhwc_to_planar ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct planar_to_nhwc',
        'cl cl cl',
    ),
    'up-f32-cl-ac1-seg0-fused': (
        'lut_remap nhwc_to_planar ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct planar_to_nhwc',
        'cl cl cl',
    ),
    'up-f32-cl-ac1-seg0-w16': (
        'lut_remap nhwc_to_planar ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct planar_to_nhwc',
        'cl cl cl',
    ),
    'up-f32-cl-ac0-seg1-fused': (
        'lut_remap nhwc_to_planar ohem_begin up_ce_fwd_ac0 ohem_select',
        'up_ce_bwd_ac0 planar_to_nhwc',
        'cl cl cl',
    ),
    'up-f32-cl-ac0-seg0-fused': (
        'lut_remap nhwc_to_planar ohem_begin up_ce_fwd_ac0 ohem_select',
        'up_ce_bwd_ac0 planar_to_nhwc',
        'cl cl cl',
    ),
    'ohem_ce-f32-cl': ('ohem_begin ohem_ce_fwd ohem_select', 'ohem_ce_bwd', 'cl'),
    'mds_ohem_ce_full-f32-cl': ('ohem_begin ohem_ce_fwd ohem_ce_fwd ohem_select', 'ohem_ce_bwd ohem_ce_bwd', 'cl cl'),
    'prototype_head-f32-cl': ('proj_fwd_tc', 'proj_bwd_tc proj_bwd_graph_tc', 'contig contig'),
    'mds-bf16-nchw-sparse-dx-fused': ('lut_remap proj_fwd ohem_begin up_ce_fwd ohem_select', 'mds_bwd', 'contig'),
    'mds-bf16-nchw-sparse-dx-w16': ('lut_remap proj_fwd ohem_begin up_ce_fwd ohem_select', 'mds_bwd', 'contig'),
    'mds-bf16-nchw-sparse-dx_dg-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc16 proj_bwd_graph_tc16',
        'contig contig contig contig',
    ),
    'mds-bf16-nchw-sparse-dx_dg-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-bf16-nchw-sparse-dg-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_graph_tc16',
        'contig contig contig',
    ),
    'mds-bf16-nchw-sparse-dg-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-bf16-nchw-sparse-none-fused': ('lut_remap proj_fwd ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-bf16-nchw-sparse-none-w16': ('lut_remap proj_fwd ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-bf16-nchw-dense-dx-fused': ('lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select', 'mds_bwd', 'contig'),
    'mds-bf16-nchw-dense-dx-w16': ('lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select', 'mds_bwd', 'contig'),
    'mds-bf16-nchw-dense-dx_dg-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc16 proj_bwd_graph_tc16',
        'contig contig contig contig',
    ),
    'mds-bf16-nchw-dense-dx_dg-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-bf16-nchw-dense-dg-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_graph_tc16',
        'contig contig contig',
    ),
    'mds-bf16-nchw-dense-dg-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-bf16-nchw-dense-none-fused': ('lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-bf16-nchw-dense-none-w16': ('lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-bf16-nchw-dense_assumed-dx-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'mds_bwd',
        'contig',
    ),
    'mds-bf16-nchw-dense_assumed-dx-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'mds_bwd',
        'contig',
    ),
    'mds-bf16-nchw-dense_assumed-dx_dg-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc16 proj_bwd_graph_tc16',
        'contig contig contig contig',
    ),
    'mds-bf16-nchw-dense_assumed-dx_dg-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-bf16-nchw-dense_assumed-dg-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_graph_tc16',
        'contig contig contig',
    ),
    'mds-bf16-nchw-dense_assumed-dg-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-bf16-nchw-dense_assumed-none-fused': ('lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-bf16-nchw-dense_assumed-none-w16': ('lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds_per_dataset-bf16-nchw': ('lut_remap proj_fwd ohem_begin up_ce_fwd ohem_select', 'mds_bwd', 'contig'),
    'head_ohem-bf16-nchw': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc16 proj_bwd_graph_tc16',
        'contig contig contig contig contig',
    ),
    'head_ce_mean-bf16-nchw': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc16 proj_bwd_graph_tc16',
        'contig contig contig contig contig',
    ),
    'heads-bf16-nchw-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct up_ce_bwd_direct proj_bwd_tc16 proj_bwd_graph_tc16',
        'contig contig contig contig contig contig contig',
    ),
    'heads-bf16-nchw-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig contig contig contig',
    ),
    'up-bf16-nchw-ac1-seg1-fused': (
        'lut_remap ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct',
        'contig contig contig',
    ),
    'up-bf16-nchw-ac1-seg1-w16': (
        'lut_remap ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct',
        'contig contig contig',
    ),
    'up-bf16-nchw-ac1-seg0-fused': (
        'lut_remap ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct',
        'contig contig contig',
    ),
    'up-bf16-nchw-ac1-seg0-w16': (
        'lut_remap ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct',
        'contig contig contig',
    ),
    'up-bf16-nchw-ac0-seg1-fused': (
        'lut_remap ohem_begin up_ce_fwd_ac0 ohem_select',
        'up_ce_bwd_ac0',
        'contig contig contig',
    ),
    'up-bf16-nchw-ac0-seg0-fused': (
        'lut_remap ohem_begin up_ce_fwd_ac0 ohem_select',
        'up_ce_bwd_ac0',
        'contig contig contig',
    ),
    'ohem_ce-bf16-nchw': ('ohem_begin ohem_ce_fwd ohem_select', 'ohem_ce_bwd', 'contig'),
    'mds_ohem_ce_full-bf16-nchw': (
        'ohem_begin ohem_ce_fwd ohem_ce_fwd ohem_select',
        'ohem_ce_bwd ohem_ce_bwd',
        'contig contig',
    ),
    'prototype_head-bf16-nchw': ('proj_fwd_tc16', 'proj_bwd_tc16 proj_bwd_graph_tc16', 'contig contig'),
    'mds-bf16-cl-sparse-dx-fused': (
        'lut_remap proj_fwd_nhwc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_nhwc',
        'cl',
    ),
    'mds-bf16-cl-sparse-dx-w16': (
        'lut_remap proj_fwd_nhwc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_nhwc',
        'cl',
    ),
    'mds-bf16-cl-sparse-dx_dg-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc16 proj_bwd_graph_tc16',
        'cl contig contig contig',
    ),
    'mds-bf16-cl-sparse-dx_dg-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-bf16-cl-sparse-dg-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_graph_tc16',
        'contig contig contig',
    ),
    'mds-bf16-cl-sparse-dg-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-bf16-cl-sparse-none-fused': ('lut_remap proj_fwd_nhwc ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-bf16-cl-sparse-none-w16': ('lut_remap proj_fwd_nhwc ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-bf16-cl-dense-dx-fused': ('lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select', 'mds_bwd', 'contig'),
    'mds-bf16-cl-dense-dx-w16': ('lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select', 'mds_bwd', 'contig'),
    'mds-bf16-cl-dense-dx_dg-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc16 proj_bwd_graph_tc16',
        'cl contig contig contig',
    ),
    'mds-bf16-cl-dense-dx_dg-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-bf16-cl-dense-dg-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_graph_tc16',
        'contig contig contig',
    ),
    'mds-bf16-cl-dense-dg-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-bf16-cl-dense-none-fused': ('lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-bf16-cl-dense-none-w16': ('lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-bf16-cl-dense_assumed-dx-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'mds_bwd',
        'contig',
    ),
    'mds-bf16-cl-dense_assumed-dx-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'mds_bwd',
        'contig',
    ),
    'mds-bf16-cl-dense_assumed-dx_dg-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc16 proj_bwd_graph_tc16',
        'cl contig contig contig',
    ),
    'mds-bf16-cl-dense_assumed-dx_dg-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
    'mds-bf16-cl-dense_assumed-dg-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_graph_tc16',
        'contig contig contig',
    ),
    'mds-bf16-cl-dense_assumed-dg-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_graph_tc',
        'contig contig contig',
    ),
    'mds-bf16-cl-dense_assumed-none-fused': ('lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds-bf16-cl-dense_assumed-none-w16': ('lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select', '', ''),
    'mds_per_dataset-bf16-cl': (
        'lut_remap proj_fwd_nhwc ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_nhwc',
        'cl',
    ),
    'head_ohem-bf16-cl': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc16 proj_bwd_graph_tc16',
        'cl contig contig contig contig',
    ),
    'head_ce_mean-bf16-cl': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct proj_bwd_tc16 proj_bwd_graph_tc16',
        'cl contig contig contig contig',
    ),
    'heads-bf16-cl-fused': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct up_ce_bwd_direct proj_bwd_tc16 proj_bwd_graph_tc16',
        'cl contig contig contig contig contig contig',
    ),
    'heads-bf16-cl-w16': (
        'lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select lut_remap proj_fwd_tc16 ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd proj_bwd_tc proj_bwd_graph_tc up_ce_bwd proj_bwd_tc proj_bwd_graph_tc',
        'contig contig contig contig contig contig contig',
    ),
    'up-bf16-cl-ac1-seg1-fused': (
        'lut_remap nhwc_to_planar ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct planar_to_nhwc',
        'cl cl cl',
    ),
    'up-bf16-cl-ac1-seg1-w16': (
        'lut_remap nhwc_to_planar ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct planar_to_nhwc',
        'cl cl cl',
    ),
    'up-bf16-cl-ac1-seg0-fused': (
        'lut_remap nhwc_to_planar ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct planar_to_nhwc',
        'cl cl cl',
    ),
    'up-bf16-cl-ac1-seg0-w16': (
        'lut_remap nhwc_to_planar ohem_begin up_ce_fwd ohem_select',
        'up_ce_bwd_direct planar_to_nhwc',
        'cl cl cl',
    ),
    'up-bf16-cl-ac0-seg1-fused': (
        'lut_remap nhwc_to_planar ohem_begin up_ce_fwd_ac0 ohem_select',
        'up_ce_bwd_ac0 planar_to_nhwc',
        'cl cl cl',
    ),
    'up-bf16-cl-ac0-seg0-fused': (
        'lut_remap nhwc_to_planar ohem_begin up_ce_fwd_ac0 ohem_select',
        'up_ce_bwd_ac0 planar_to_nhwc',
        'cl cl cl',
    ),
    'ohem_ce-bf16-cl': ('ohem_begin ohem_ce_fwd ohem_select', 'ohem_ce_bwd', 'cl'),
    'mds_ohem_ce_full-bf16-cl': ('ohem_begin ohem_ce_fwd ohem_ce_fwd ohem_select', 'ohem_ce_bwd ohem_ce_bwd', 'cl cl'),
    'prototype_head-bf16-cl': ('proj_fwd_tc16', 'proj_bwd_tc16 proj_bwd_graph_tc16', 'cl contig'),
    'nll_plus-sparse': (
        'softmax_nchw proj_fwd ohem_begin up_nll_fwd ohem_select',
        'up_nll_bwd proj_bwd softmax_bwd_nchw',
        'contig',
    ),
    'nll_plus-dense': (
        'softmax_nchw proj_fwd_tc ohem_begin up_nll_fwd ohem_select',
        'up_nll_bwd proj_bwd_tc softmax_bwd_nchw proj_bwd_graph_tc',
        'contig contig contig contig',
    ),
}


@pytest.fixture(scope="module")
def ops():
    from mdseg_b200 import ops
    return ops


@pytest.mark.parametrize("name", list(CASES))
def test_route(ops, name):
    assert run_case(ops, name) == EXPECTED[name]


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import __graft_entry__
    __graft_entry__.build(quiet=True)
    from mdseg_b200 import ops as _ops
    print("EXPECTED = {")
    for _name in CASES:
        _rec = run_case(_ops, _name)
        _one = f"    {_name!r}: {_rec!r},"
        print(_one if len(_one) <= 120 else f"    {_name!r}: (\n" + "".join(f"        {x!r},\n" for x in _rec) + "    ),")
    print("}")
