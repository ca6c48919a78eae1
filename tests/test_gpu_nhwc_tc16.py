"""GPU: channels_last 16-bit features / logits on the TMA-fed tcgen05 kernels — mdseg_proj_fwd_tc16,
mdseg_proj_bwd_tc16 and mdseg_proj_bwd_graph_tc16 with layout NHWC — and the operators that route through them (the
prototype head, the folded and dense-graph fused losses, the stacked hard / soft pair).  Every output is compared bit
for bit with layout NCHW / NCHW input on the same values."""
import ctypes as C

import pytest
import torch

from test_host_cpu import DictConfiger

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CL = torch.channels_last
DTYPES = [torch.bfloat16, torch.float16]
DT_IDS = ["bf16", "f16"]


@pytest.fixture(scope="module")
def ops():
    from mdseg_b200 import ops
    return ops


@pytest.fixture(scope="module")
def native():
    from mdseg_b200 import native
    return native


def stream():
    return torch.cuda.current_stream().cuda_stream


def offset_channels_last(x):
    """The values of x as a channels_last view that starts one element into its storage (not 16-byte aligned)."""
    B, Cu, h, w = x.shape
    buf = torch.empty(B * h * w * Cu + 1, dtype=x.dtype, device=x.device)
    v = buf[1:].view(B, h, w, Cu).permute(0, 3, 1, 2)
    v.copy_(x)
    assert v.is_contiguous(memory_format=CL) and v.storage_offset() == 1
    return v


# ---- 1. the entry points against the planar ones ------------------------------------------------------------------
# (K, C_ds of three datasets, h, w): K-tail zero fill (48, 96, 600), several N tiles and the N tail (358, 600),
# pixel tiles that are not a multiple of 128
SHAPES = [(512, [19, 150, 64], 12, 20), (48, [19, 150, 64], 12, 20), (96, [19, 150, 64], 20, 36),
          (600, [358, 600, 19], 12, 20)]
IDS = {"sorted": [0, 0, 1, 2, 2], "shuffled": [2, 0, 1, 2, 0], "absent": [2, 0, 7, 1, 0]}  # 7: no such dataset


@pytest.mark.parametrize("ids_name", list(IDS))
@pytest.mark.parametrize("shape", SHAPES, ids=[f"K{s[0]}_N{max(s[1])}" for s in SHAPES])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_layout_entry_points_bit_identical(ops, native, dtype, shape, ids_name):
    K, Cs, h, w = shape
    ids = IDS[ids_name]
    B, hw, n, cmax = len(ids), h * w, len(Cs), max(Cs)
    gen = torch.Generator(device=DEV).manual_seed(K * 7 + len(ids_name))
    x = torch.randn(B, K, h, w, generator=gen, device=DEV).to(dtype)
    xl = x.contiguous(memory_format=CL)
    mats = [torch.randn(c, K, generator=gen, device=DEV) * 0.2 for c in Cs]
    ids_t = torch.tensor(ids, dtype=torch.int32, device=DEV)
    dt = ops._DT[dtype]

    # forward: y = G_d x, planar fp32
    keep, ptrs, ldb = ops._tc16_operands(mats, dtype)
    cds = (C.c_int * n)(*Cs)
    y0 = torch.full((B, cmax, h, w), 3.0, device=DEV)
    y1 = torch.full((B, cmax, h, w), 3.0, device=DEV)
    native.call("mdseg_proj_fwd_tc16", x.data_ptr(), dt, native.NCHW, B, K, hw, ptrs, ldb, cds, n, ids_t.data_ptr(),
                y0.data_ptr(), cmax, stream())
    native.call("mdseg_proj_fwd_tc16", xl.data_ptr(), dt, native.NHWC, B, K, hw, ptrs, ldb, cds, n, ids_t.data_ptr(),
                y1.data_ptr(), cmax, stream())
    torch.cuda.synchronize()
    assert torch.equal(y0, y1)

    # d x = G_d^T dy16, pixel-major, in fp32 and in the input dtype
    dy = torch.zeros(B, cmax, h, w, dtype=dtype, device=DEV)
    for b, d in enumerate(ids):
        if d < n:
            dy[b, :Cs[d]] = torch.randn(Cs[d], h, w, generator=gen, device=DEV).to(dtype)
    keep_t, ptrs_t, ldb_t = ops._tc16_operands(mats, dtype, transpose=True)
    for dx_dt in (dtype, torch.float32):
        dx0 = torch.full((B, K, h, w), 7.0, dtype=dx_dt, device=DEV)
        dx1 = torch.full((B, K, h, w), 7.0, dtype=dx_dt, device=DEV).contiguous(memory_format=CL)
        native.call("mdseg_proj_bwd_tc16", dy.data_ptr(), dt, native.NCHW, B, cmax, hw, ptrs_t, ldb_t, K, n,
                    ids_t.data_ptr(), dx0.data_ptr(), ops._DT[dx_dt], stream())
        native.call("mdseg_proj_bwd_tc16", dy.data_ptr(), dt, native.NHWC, B, cmax, hw, ptrs_t, ldb_t, K, n,
                    ids_t.data_ptr(), dx1.data_ptr(), ops._DT[dx_dt], stream())
        torch.cuda.synchronize()
        assert torch.equal(dx0, dx1.contiguous()), dx_dt
        for b, d in enumerate(ids):
            if d >= n:
                assert not dx1[b].any()  # zero rows for an image of no dataset

    # d G_d = dy16 x^T per dataset, and the one-sum form (dataset_ids NULL), each in both layouts
    nb = native.lib.mdseg_proj_bwd_graph_tc16_workspace_bytes(B, K, hw, cmax)
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    dG0 = torch.empty(n, cmax, K, device=DEV)
    dG1 = torch.empty(n, cmax, K, device=DEV)
    native.call("mdseg_proj_bwd_graph_tc16", dy.data_ptr(), x.data_ptr(), dt, native.NCHW, B, K, hw, cmax,
                ids_t.data_ptr(), n, dG0.data_ptr(), ws.data_ptr(), nb, stream())
    native.call("mdseg_proj_bwd_graph_tc16", dy.data_ptr(), xl.data_ptr(), dt, native.NHWC, B, K, hw, cmax,
                ids_t.data_ptr(), n, dG1.data_ptr(), ws.data_ptr(), nb, stream())
    dW0 = torch.empty(cmax, K, device=DEV)
    dW1 = torch.empty(cmax, K, device=DEV)
    native.call("mdseg_proj_bwd_graph_tc16", dy.data_ptr(), x.data_ptr(), dt, native.NCHW, B, K, hw, cmax, None, 1,
                dW0.data_ptr(), ws.data_ptr(), nb, stream())
    native.call("mdseg_proj_bwd_graph_tc16", dy.data_ptr(), xl.data_ptr(), dt, native.NHWC, B, K, hw, cmax, None, 1,
                dW1.data_ptr(), ws.data_ptr(), nb, stream())
    torch.cuda.synchronize()
    assert torch.equal(dG0, dG1)
    assert torch.equal(dW0, dW1)
    assert dG1.abs().sum() > 0 and dW1.abs().sum() > 0
    ops.check_errors(DEV)


def test_layout_entry_points_reject_bad_inputs(ops, native):
    x = torch.zeros(2, 60, 8, 8, dtype=torch.bfloat16, device=DEV).contiguous(memory_format=CL)
    keep, ptrs, ldb = ops._tc16_operands([torch.zeros(16, 60, device=DEV)], torch.bfloat16)
    y = torch.empty(2, 16, 8, 8, device=DEV)
    with pytest.raises(native.MdsegError, match="multiple of 8"):  # K % 8 != 0
        native.call("mdseg_proj_fwd_tc16", x.data_ptr(), native.BF16, native.NHWC, 2, 60, 64, ptrs, ldb,
                    (C.c_int * 1)(16), 1, None, y.data_ptr(), 16, stream())
    x32 = torch.zeros(2, 64, 8, 8, device=DEV)
    with pytest.raises(native.MdsegError, match="bf16 or fp16"):
        native.call("mdseg_proj_fwd_tc16", x32.data_ptr(), native.F32, native.NHWC, 2, 64, 64, ptrs, 64,
                    (C.c_int * 1)(16), 1, None, y.data_ptr(), 16, stream())
    dy = torch.zeros(2, 16, 8, 8, dtype=torch.bfloat16, device=DEV)
    with pytest.raises(native.MdsegError, match="dataset ids"):
        native.call("mdseg_proj_bwd_graph_tc16", dy.data_ptr(), x.data_ptr(), native.BF16, native.NHWC, 2, 64, 64, 16,
                    None, 2, y.data_ptr(), y.data_ptr(), 1 << 20, stream())


# ---- 2. the prototype head ------------------------------------------------------------------------------------------
def _head_run(ops, feats, proto, dy):
    f = feats.detach().requires_grad_(True)
    p = proto.detach().requires_grad_(True)
    y = ops.prototype_head(f, p)
    y.backward(dy)
    return y.detach(), f.grad, p.grad


@pytest.mark.parametrize("K,Nn", [(512, 358), (64, 600), (48, 19)])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_prototype_head_channels_last(ops, dtype, K, Nn):
    gen = torch.Generator(device=DEV).manual_seed(K + Nn)
    B, h, w = 3, 12, 20
    feats = torch.randn(B, K, h, w, generator=gen, device=DEV).to(dtype)
    proto = torch.randn(Nn, K, generator=gen, device=DEV) * 0.1
    dy = torch.randn(B, Nn, h, w, generator=gen, device=DEV)
    y0, df0, dp0 = _head_run(ops, feats, proto, dy)
    y1, df1, dp1 = _head_run(ops, feats.contiguous(memory_format=CL), proto, dy)
    assert y1.is_contiguous()
    assert torch.equal(y0, y1)
    assert df1.is_contiguous(memory_format=CL) and not df1.is_contiguous()
    assert torch.equal(df0, df1)
    assert torch.equal(dp0, dp1)
    ops.check_errors(DEV)


# ---- 3. the fused losses with dense graphs ---------------------------------------------------------------------------
N_CATS = [19, 150, 64]
C_UNI = 100


def _loss_case(seed, dtype, K, ids, h=16, w=32, H=64, W=128, scale=1.0):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    feats = (torch.randn(len(ids), K, h, w, generator=gen, device=DEV) * scale).to(dtype)
    proto = torch.randn(C_UNI, K, generator=gen, device=DEV) * 0.1
    graphs = [torch.rand(c, C_UNI, generator=gen, device=DEV) for c in N_CATS]
    soft = [torch.rand(c, C_UNI, generator=gen, device=DEV) for c in N_CATS]
    labels = torch.stack([torch.randint(0, N_CATS[d], (H, W), generator=gen, device=DEV) for d in ids])
    labels[torch.rand(labels.shape, generator=gen, device=DEV) < 0.05] = 255
    return feats, proto, graphs, soft, labels.to(torch.uint8), torch.tensor(ids, dtype=torch.int32, device=DEV)


def _run(fn, feats, leaves):
    f = feats.detach().requires_grad_(True)
    ls = [t.detach().requires_grad_(True) for t in leaves]
    loss = fn(f, ls)
    torch.nansum(loss).backward()
    return loss.detach(), f.grad, [t.grad for t in ls]


def _assert_same(ops, fn, feats, leaves, feats_cl=None, want_cl=True):
    l0, g0, gl0 = _run(fn, feats, leaves)
    l1, g1, gl1 = _run(fn, feats.contiguous(memory_format=CL) if feats_cl is None else feats_cl, leaves)
    ops.check_errors(DEV)
    assert torch.equal(l0, l1) or torch.equal(l0.view(torch.int32), l1.view(torch.int32))
    if want_cl:
        assert g1.is_contiguous(memory_format=CL) and not g1.is_contiguous()
    assert torch.equal(g0, g1)
    for a, b in zip(gl0, gl1):
        assert (a is None and b is None) or torch.equal(a, b)
    assert g0.abs().sum() > 0


THRESH = {"threshold": None, "topk": 60.0}  # None: -log(0.4); 60: above every loss, the top-k branch


@pytest.mark.parametrize("branch", list(THRESH))
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("ids", [[0, 0, 1, 2, 2], [2, 0, 1, 2, 0]], ids=["sorted", "shuffled"])
def test_folded_losses_channels_last(ops, dtype, ids, branch):
    feats, proto, graphs, soft, labels, ids_t = _loss_case(31, dtype, 64, ids)
    th = THRESH[branch] or ops.neg_log(0.4)
    n = len(N_CATS)
    _assert_same(ops, lambda f, ls: ops.mds_head_proj_ohem_ce(f, ls[0], labels, ids_t, ls[1:], th),
                 feats, [proto, *graphs])
    _assert_same(ops, lambda f, ls: ops.mds_head_proj_ohem_ce_heads(f, ls[0], labels, ids_t,
                                                                    [ls[1:1 + n], ls[1 + n:]], th),
                 feats, [proto, *graphs, *soft])
    _assert_same(ops, lambda f, ls: ops.mds_head_proj_ce_mean(f, ls[0], labels, ids_t, ls[1:]),
                 feats, [proto, *graphs])


@pytest.mark.parametrize("branch", list(THRESH))
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_dense_trainable_graphs_channels_last(ops, dtype, branch):
    """16-bit unified logits (K = C_uni = 64 channels) with trainable dense graphs: mds_proj_ohem_ce and the pair."""
    ids = [2, 0, 1, 2, 0]
    x, _, _, _, labels, ids_t = _loss_case(5, dtype, 64, ids)
    gen = torch.Generator(device=DEV).manual_seed(6)
    graphs = [torch.rand(c, 64, generator=gen, device=DEV) for c in N_CATS]
    soft = [torch.rand(c, 64, generator=gen, device=DEV) for c in N_CATS]
    th = THRESH[branch] or ops.neg_log(0.4)
    from mdseg_b200.ops import BipartiteGraphs
    _assert_same(ops, lambda f, ls: ops.mds_proj_ohem_ce(f, labels, ids_t, ls, th,
                                                         cache=BipartiteGraphs(assume_dense=True)), x, graphs)
    _assert_same(ops, lambda f, ls: ops.mds_proj_ohem_ce_heads(f, labels, ids_t, [ls[:3], ls[3:]], th),
                 x, [*graphs, *soft])


# ---- 4. inputs that keep the copy route ------------------------------------------------------------------------------
def test_fallbacks_unchanged(ops):
    ids = [2, 0, 1, 2, 0]
    th = ops.neg_log(0.4)
    cases = [("fp32", torch.float32, 64, None), ("K%8", torch.bfloat16, 60, None), ("offset", torch.bfloat16, 64, "off")]
    for name, dtype, K, how in cases:
        feats, proto, graphs, soft, labels, ids_t = _loss_case(41, dtype, K, ids)
        fcl = offset_channels_last(feats) if how == "off" else None
        _assert_same(ops, lambda f, ls: ops.mds_head_proj_ohem_ce(f, ls[0], labels, ids_t, ls[1:], th),
                     feats, [proto, *graphs], feats_cl=fcl, want_cl=False)
        _assert_same(ops, lambda f, ls: ops.mds_head_proj_ohem_ce_heads(f, ls[0], labels, ids_t, [ls[1:4], ls[4:]], th),
                     feats, [proto, *graphs, *soft], feats_cl=fcl, want_cl=False)
        dy = torch.randn(len(ids), C_UNI, 16, 32, device=DEV)
        y0, df0, dp0 = _head_run(ops, feats, proto, dy)
        y1, df1, dp1 = _head_run(ops, feats.contiguous(memory_format=CL) if fcl is None else fcl, proto, dy)
        assert torch.equal(y0, y1) and torch.equal(df0, df1) and torch.equal(dp0, dp1), name


def test_no_backward_or_frozen_graphs(ops):
    """Dense graphs that want no gradient while the features do: the backward writes d x planar, so the features are
    copied; forward-only calls read them as they are.  Both agree with NCHW input."""
    ids = [2, 0, 1, 2, 0]
    feats, proto, graphs, _, labels, ids_t = _loss_case(43, torch.bfloat16, 64, ids)
    th = ops.neg_log(0.4)
    l0, g0, _ = _run(lambda f, ls: ops.mds_head_proj_ohem_ce(f, proto, labels, ids_t, graphs, th), feats, [])
    l1, g1, _ = _run(lambda f, ls: ops.mds_head_proj_ohem_ce(f, proto, labels, ids_t, graphs, th),
                     feats.contiguous(memory_format=CL), [])
    assert torch.equal(l0, l1) and torch.equal(g0, g1)
    with torch.no_grad():
        a = ops.mds_head_proj_ohem_ce(feats, proto, labels, ids_t, graphs, th)
        b = ops.mds_head_proj_ohem_ce(feats.contiguous(memory_format=CL), proto, labels, ids_t, graphs, th)
    assert torch.equal(a, b)
    ops.check_errors(DEV)


# ---- 5. the drop-in loss and the evaluator head ---------------------------------------------------------------------
@pytest.fixture(scope="module")
def dropin():
    import mdseg_b200.dropin as d
    d.install()
    yield d
    d.uninstall()


GNN_CATS = [19, 64, 37, 19, 26, 150, 133]


def _gnn_cfg():
    cfg = {"n_datasets": 7, "iter": 12345,
           "loss": {"with_datasets_aux": True, "aux_weight": 0.2, "ignore_index": 255, "with_spa": False,
                    "spa_loss_weight": 0.1, "with_max_enc": False, "max_enc_weight": 1, "adv_loss_weight": 1,
                    "GridSplit": False, "adj_loss_weight": 1},
           "GNN": {"unify_ratio": 0.8, "output_max_adj": True, "output_softmax_and_max_adj": True, "with_orth": True,
                   "orth_weight": 1, "mse_or_adv": "None"},
           "contrast": {"temperature": 0.07}, "train": {"seg_iters": 200000, "gnn_iters": 60000}}
    for i, c in enumerate(GNN_CATS):
        cfg[f"dataset{i + 1}"] = {"n_cats": c}
    return DictConfiger(cfg)


@pytest.mark.parametrize("fold", [True, False], ids=["folded", "unfolded"])
def test_advgnn_gnn_stage_channels_last(dropin, fold, monkeypatch):
    import mdseg_b200.dropin.loss_cross_datasets as m
    from lib.loss.loss_cross_datasets import CrossDatasetsCELoss_AdvGNN
    from mdseg_b200 import ops
    monkeypatch.setattr(m, "FOLD_PROTOTYPES", fold)
    crit = CrossDatasetsCELoss_AdvGNN(_gnn_cfg())
    ids = [3, 0, 6, 1, 5, 2, 4, 5]
    K, h, w, H, W = 64, 16, 32, 64, 128
    c_uni = int(0.8 * sum(GNN_CATS))
    gen = torch.Generator(device=DEV).manual_seed(17)
    feats = torch.randn(len(ids), K, h, w, generator=gen, device=DEV).to(torch.bfloat16)
    proto = torch.randn(sum(GNN_CATS) + c_uni, K, generator=gen, device=DEV) * 0.1
    graphs = [torch.rand(GNN_CATS[i // 2], c_uni, generator=gen, device=DEV) for i in range(14)]
    labels = torch.stack([torch.randint(0, GNN_CATS[d], (H, W), generator=gen, device=DEV) for d in ids])
    ids_t = torch.tensor(ids, device=DEV)
    runs = []
    for fmt in (torch.contiguous_format, CL):
        f = feats.detach().contiguous(memory_format=fmt).requires_grad_(True)
        p = proto.clone().requires_grad_(True)
        gs = [g.clone().requires_grad_(True) for g in graphs]
        preds = {"seg": f, "unify_prototype": p, "bi_graphs": gs, "adv_out": None}
        loss, orth, aux, adj = crit(preds, labels, ids_t, True, False)
        loss.backward()
        ops.check_errors(DEV)
        runs.append((loss.detach(), aux.detach(), f.grad, p.grad, [g.grad for g in gs]))
    (l0, a0, f0, p0, g0), (l1, a1, f1, p1, g1) = runs
    assert torch.equal(l0, l1) and torch.equal(a0, a1)
    assert f1.is_contiguous(memory_format=CL)
    assert torch.equal(f0, f1)
    assert torch.equal(p0, p1)
    for i in range(14):
        assert torch.equal(g0[i], g1[i]), i


def test_evaluator_head_channels_last(ops):
    """prototype_head + eval_fused (the evaluators' route) on a channels_last embedding: the same histogram."""
    gen = torch.Generator(device=DEV).manual_seed(23)
    B, K, Cc, h, w, H, W = 3, 64, 40, 16, 24, 64, 96
    emb = torch.randn(B, K, h, w, generator=gen, device=DEV).to(torch.bfloat16)
    proto = torch.randn(Cc, K, generator=gen, device=DEV)
    label = torch.randint(0, Cc, (B, H, W), generator=gen, device=DEV).to(torch.uint8)
    hists = []
    for e in (emb, emb.contiguous(memory_format=CL)):
        logits = ops.prototype_head(e, proto)
        hist = torch.zeros(Cc, Cc, dtype=torch.int64, device=DEV)
        for b in range(B):
            ops.eval_fused([(logits[b], False)], (H, W), label=label[b], hist=hist, want_pred=False)
        hists.append(hist)
    assert torch.equal(hists[0], hists[1]) and int(hists[0].sum()) == B * H * W


# ---- 6. no layout copy, 7. CUDA graph ---------------------------------------------------------------------------------
def _peak_growth(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def _pair_step(ops, f, p, gs, labels, ids_t, copy=False):
    f.grad = None
    x = f.contiguous() if copy else f
    loss = ops.mds_head_proj_ohem_ce_heads(x, p, labels, ids_t, [gs[:3], gs[3:]], ops.neg_log(0.4))
    loss.sum().backward()
    return loss.detach()


def test_no_layout_copy(ops):
    ids = [0, 2, 1, 2]
    feats, proto, graphs, soft, labels, ids_t = _loss_case(51, torch.bfloat16, 512, ids, 128, 256, 512, 1024)
    p = proto.requires_grad_(True)
    gs = [g.requires_grad_(True) for g in (*graphs, *soft)]
    fn = feats.requires_grad_(True)
    fl = feats.detach().contiguous(memory_format=CL).requires_grad_(True)
    nbytes = fn.nbytes
    for f, copy in ((fn, False), (fl, False), (fl, True)):  # warm-up
        _pair_step(ops, f, p, gs, labels, ids_t, copy)
    peak = {}
    for key, f, copy in (("nchw", fn, False), ("cl", fl, False), ("copy", fl, True)):
        f.grad = None
        p.grad = None
        for g in gs:
            g.grad = None
        peak[key] = _peak_growth(lambda: _pair_step(ops, f, p, gs, labels, ids_t, copy))
    assert fl.grad.is_contiguous(memory_format=CL)
    assert peak["cl"] <= peak["nchw"] + 0.1 * nbytes, (peak, nbytes)
    assert peak["copy"] >= peak["cl"] + 0.9 * nbytes, (peak, nbytes)  # the copy route would show up


def test_cuda_graph_capture(ops):
    ids = [2, 0, 1, 2]
    feats, proto, graphs, soft, labels, ids_t = _loss_case(61, torch.bfloat16, 64, ids)
    fl = feats.contiguous(memory_format=CL).requires_grad_(True)
    p = proto.requires_grad_(True)
    gs = [g.requires_grad_(True) for g in (*graphs, *soft)]
    leaves = (fl, p, *gs)

    def step():
        for t in leaves:
            t.grad = None
        return _pair_step(ops, fl, p, gs, labels, ids_t)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            eager = step()
    torch.cuda.current_stream().wait_stream(side)
    eager = eager.clone()
    eager_grads = [t.grad.clone() for t in leaves]
    graph = torch.cuda.CUDAGraph()
    for t in leaves:
        t.grad = None
    with torch.cuda.graph(graph):
        captured = step()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, eager)
    for t, g in zip(leaves, eager_grads):
        assert torch.equal(t.grad, g)
    ops.check_errors(DEV)


# ---- 8. at size ---------------------------------------------------------------------------------------------------
def test_cfg3_gnn_stage_pair_channels_last_at_size(ops):
    """16 x 512 x 256 x 512 bf16 features, 1024 x 2048 labels, 7 datasets, C_uni = 358, trainable hard / soft pairs:
    the folded pair step with channels_last features equals the NCHW step."""
    ids = [0, 0, 0, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6]
    gen = torch.Generator(device=DEV).manual_seed(71)
    feats = torch.randn(len(ids), 512, 256, 512, generator=gen, device=DEV).to(torch.bfloat16)
    proto = (torch.randn(358, 512, generator=gen, device=DEV) * 0.05).requires_grad_(True)
    gs = [torch.rand(GNN_CATS[i % 7], 358, generator=gen, device=DEV).requires_grad_(True) for i in range(14)]
    labels = torch.stack([torch.randint(0, GNN_CATS[d], (1024, 2048), generator=gen, device=DEV) for d in ids])
    labels[torch.rand(labels.shape, generator=gen, device=DEV) < 0.05] = 255
    labels = labels.to(torch.uint8)
    ids_t = torch.tensor(ids, dtype=torch.int32, device=DEV)
    sample = torch.randint(0, feats.numel(), (1 << 20,), generator=gen, device=DEV)

    def run(f):
        f = f.requires_grad_(True)
        for t in (proto, *gs):
            t.grad = None
        loss = ops.mds_head_proj_ohem_ce_heads(f, proto, labels, ids_t, [gs[:7], gs[7:]], ops.neg_log(0.4))
        loss.sum().backward()
        ops.check_errors(DEV)
        g = f.grad.permute(0, 2, 3, 1).reshape(-1)[sample]  # sampled in NHWC order for either layout
        layout_cl = f.grad.is_contiguous(memory_format=CL) and not f.grad.is_contiguous()
        return loss.detach(), g, proto.grad.clone(), [t.grad.clone() for t in gs], layout_cl

    l0, s0, p0, g0, _ = run(feats)
    fl = feats.detach().contiguous(memory_format=CL)
    del feats
    l1, s1, p1, g1, cl = run(fl)
    assert cl
    assert torch.equal(l0, l1)
    assert torch.equal(s0, s1)
    assert torch.equal(p0, p1)
    for i in range(14):
        assert torch.equal(g0[i], g1[i]), i
