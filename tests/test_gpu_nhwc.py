"""GPU: channels_last (NHWC) logits in the SEG-stage loss path — the sparse projection and its adjoint
(mdseg_proj_fwd_nhwc / mdseg_proj_bwd_nhwc) and the aux heads (mdseg_nhwc_to_planar / mdseg_planar_to_nhwc) — against
the NCHW kernels on the same values, the reference goldens, memory use and CUDA-graph capture."""
import ctypes as C

import numpy as np
import pytest
import torch

from test_host_cpu import DictConfiger

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL32 = 1e-5
CL = torch.channels_last
IDS = {"sorted": [0, 0, 1, 2, 2], "shuffled": [2, 0, 1, 2, 0], "absent": [0, 2, 2, 0, 2]}


@pytest.fixture(scope="module")
def ops():
    from mdseg_b200 import ops
    return ops


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def graphs_for(gen, kind, n_cats, c_uni):
    out = []
    for c in n_cats:
        if kind == "onehot":
            idx = torch.randint(0, c, (c_uni,), generator=gen)
            idx[:c] = torch.arange(c)
            m = torch.zeros(c, c_uni)
            m[idx, torch.arange(c_uni)] = 1
        else:  # general 0/1 remap matrix: a unified id may serve several dataset classes, some serve none
            m = (torch.rand(c, c_uni, generator=gen) < 0.15).float()
        out.append(m.to(DEV))
    return out


def make_case(seed, kind, n_cats, c_uni, ids, h, w, H, W, dtype=torch.float32, scale=2.5):
    gen = torch.Generator().manual_seed(seed)
    x = (torch.randn(len(ids), c_uni, h, w, generator=gen) * scale).to(dtype).to(DEV)
    graphs = graphs_for(gen, kind, n_cats, c_uni)
    labels = torch.full((len(ids), H, W), 255, dtype=torch.uint8)
    for b, d in enumerate(ids):
        labels[b] = torch.randint(0, n_cats[d], (H, W), generator=gen).to(torch.uint8)
    labels[torch.rand(len(ids), H, W, generator=gen) < 0.05] = 255
    return x, graphs, labels.to(DEV), torch.tensor(ids, dtype=torch.int32, device=DEV)


def offset_channels_last(x):
    """The values of x as a channels_last view that starts one element into its storage (not 16-byte aligned)."""
    B, Cu, h, w = x.shape
    buf = torch.empty(B * h * w * Cu + 1, dtype=x.dtype, device=x.device)
    v = buf[1:].view(B, h, w, Cu).permute(0, 3, 1, 2)
    v.copy_(x)
    assert v.is_contiguous(memory_format=CL) and v.storage_offset() == 1
    return v


def same_bits(a, b):
    return torch.equal(a.view(torch.int32), b.view(torch.int32))  # NaN (a dataset without images) included


def loss_and_grad(ops, x, labels, ids, graphs, thresh, per_dataset=False):
    xd = x.detach().requires_grad_(True)  # same storage, offset and strides
    loss = ops.mds_proj_ohem_ce(xd, labels, ids, graphs, thresh, per_dataset=per_dataset)
    torch.nansum(loss).backward()
    ops.check_errors(DEV)
    return loss.detach(), xd.grad


# ---- 1. reference goldens ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["sorted", "shuffled", "absent"])
def test_golden_reference_outputs_channels_last(ops, golden, name):
    z = golden("mds.npz")
    x = torch.from_numpy(z[f"mds_{name}_x"]).to(DEV).contiguous(memory_format=CL).requires_grad_(True)
    graphs = [torch.from_numpy(z[f"mds_{name}_graph{i}"]).to(DEV) for i in range(3)]
    loss = ops.mds_proj_ohem_ce(x, torch.from_numpy(z[f"mds_{name}_labels"]).to(DEV),
                                torch.from_numpy(z[f"mds_{name}_ids"]).to(DEV), graphs, ops.neg_log(0.4))
    (loss * 2.0).backward()
    ops.check_errors(DEV)
    want = float(z[f"mds_{name}_loss"])
    assert abs(float(loss) - want) <= RTOL32 * abs(want)
    assert x.grad.is_contiguous(memory_format=CL) and not x.grad.is_contiguous()
    assert rel_err(x.grad.cpu().numpy(), z[f"mds_{name}_dx"]) <= RTOL32


# ---- 2. + 3. bit-identity of the forward, the adjoint against mdseg_proj_bwd --------------------------------------
GEOM = {358: (12, 20, 45, 80), 67: (9, 13, 35, 50), 19: (7, 11, 26, 41)}  # h * w never a multiple of the tile
N_CATS = {358: [61, 19, 150], 67: [13, 5, 30], 19: [7, 3, 12]}


@pytest.mark.parametrize("c_uni", [358, 67, 19])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16], ids=["f32", "bf16", "f16"])
@pytest.mark.parametrize("kind", ["onehot", "sparse01"])
def test_forward_bit_identical_to_nchw(ops, kind, dtype, c_uni):
    h, w, H, W = GEOM[c_uni]
    n_cats = N_CATS[c_uni]
    tol = RTOL32 if dtype == torch.float32 else 2e-2
    for k, (case, ids) in enumerate(IDS.items()):
        x, graphs, labels, ids_t = make_case(c_uni * 7 + k, kind, n_cats, c_uni, ids, h, w, H, W, dtype)
        xl = x.contiguous(memory_format=CL)
        assert not xl.is_contiguous()
        y0 = ops.project(x, graphs, ids_t)
        for xv in (xl, offset_channels_last(x)):
            y1 = ops.project(xv, graphs, ids_t)
            for b, d in enumerate(ids):  # planes past C_ds of an image are not written
                assert torch.equal(y0[b, :n_cats[d]], y1[b, :n_cats[d]]), case
        # threshold branch, and a threshold above every loss (the top-k branch)
        for thresh, per_dataset in ((ops.neg_log(0.4), False), (60.0, False), (ops.neg_log(0.4), True), (60.0, True)):
            l0, g0 = loss_and_grad(ops, x, labels, ids_t, graphs, thresh, per_dataset)
            l1, g1 = loss_and_grad(ops, xl, labels, ids_t, graphs, thresh, per_dataset)
            assert same_bits(l0, l1), (case, thresh, per_dataset)
            assert g1.is_contiguous(memory_format=CL)
            assert rel_err(g1.float().cpu().numpy(), g0.float().cpu().numpy()) <= tol, (case, thresh, per_dataset)
        l0, g0 = loss_and_grad(ops, x, labels, ids_t, graphs, ops.neg_log(0.4))
        l2, g2 = loss_and_grad(ops, offset_channels_last(x), labels, ids_t, graphs, ops.neg_log(0.4))
        assert same_bits(l0, l2), case
        assert rel_err(g2.float().cpu().numpy(), g0.float().cpu().numpy()) <= tol, case


@pytest.mark.parametrize("two_planes", [False, True], ids=["dyA", "dyA+dyB"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16], ids=["f32", "bf16", "f16"])
@pytest.mark.parametrize("kind", ["onehot", "sparse01"])
def test_adjoint_bit_identical_to_proj_bwd(ops, kind, dtype, two_planes):
    from mdseg_b200 import native as N
    c_uni, (h, w, _, _) = 358, GEOM[358]
    n_cats = N_CATS[358]
    ids = [2, 0, 1, 7, 2]  # 7: no such dataset, a zero gradient
    gen = torch.Generator().manual_seed(11)
    graphs = graphs_for(gen, kind, n_cats, c_uni)
    cmax = max(n_cats)
    dyA = torch.randn(len(ids), cmax, h, w, generator=gen).to(DEV)
    dyB = torch.randn(len(ids), cmax, h, w, generator=gen).to(DEV) if two_planes else None
    ids_t = torch.tensor(ids, dtype=torch.int32, device=DEV)
    tab, keep = ops._default_graphs.table(graphs)
    dx0 = torch.full((len(ids), c_uni, h, w), 7.0, dtype=dtype, device=DEV)
    dx1 = torch.full((len(ids), c_uni, h, w), 7.0, dtype=dtype, device=DEV).contiguous(memory_format=CL)
    stream = torch.cuda.current_stream().cuda_stream
    N.call("mdseg_proj_bwd", dyA.data_ptr(), dyB.data_ptr() if two_planes else None, cmax, C.byref(tab),
           ids_t.data_ptr(), len(ids), h, w, dx0.data_ptr(), ops._DT[dtype], stream)
    N.call("mdseg_proj_bwd_nhwc", dyA.data_ptr(), dyB.data_ptr() if two_planes else None, cmax, C.byref(tab),
           ids_t.data_ptr(), len(ids), h, w, dx1.data_ptr(), ops._DT[dtype], stream)
    torch.cuda.synchronize()
    assert torch.equal(dx0, dx1)
    assert not dx1[3].any()


# ---- 4. aux heads ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("geom", [(12, 20, 45, 80), (9, 13, 35, 50)], ids=["fused", "generic"])
@pytest.mark.parametrize("seg_per_dataset", [True, False])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16], ids=["f32", "bf16", "f16"])
def test_aux_heads_channels_last(ops, dtype, seg_per_dataset, geom):
    h, w, H, W = geom
    n_cats, ids = [5, 19, 7], [2, 0, 1, 2, 0, 1]
    B = len(ids)
    gen = torch.Generator().manual_seed(h * 31 + W)
    aux = [(torch.randn(B, c, h, w, generator=gen) * 2.0).to(dtype).to(DEV) for c in n_cats]
    labels = torch.stack([torch.randint(0, n_cats[d], (H, W), generator=gen) for d in ids]).to(DEV)
    ids_t = torch.tensor(ids, device=DEV)
    outs = []
    for fmt in (torch.contiguous_format, CL):
        src = [a.detach().contiguous(memory_format=fmt).requires_grad_(True) for a in aux]
        loss = ops.up_ohem_ce(src, labels, ids_t, ops.neg_log(0.7), seg_per_dataset=seg_per_dataset)
        (loss * torch.arange(1, loss.numel() + 1, device=DEV)).sum().backward()
        ops.check_errors(DEV)
        outs.append((loss.detach(), [s.grad for s in src]))
    (l0, g0), (l1, g1) = outs
    assert same_bits(l0, l1)
    ids_np = np.array(ids)
    for d in range(len(n_cats)):
        assert g1[d].is_contiguous(memory_format=CL) and g1[d].dtype == dtype
        assert torch.equal(g0[d], g1[d]), d
        assert not g1[d][torch.from_numpy(ids_np != d)].any(), d  # rows of other datasets' images are zero
        assert g1[d][torch.from_numpy(ids_np == d)].any(), d


# ---- 5. no layout copy ------------------------------------------------------------------------------------------
def _peak_growth(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = fn()
    torch.cuda.synchronize()
    return out, torch.cuda.max_memory_allocated() - base


def test_no_layout_copy(ops):
    n_cats, ids = [19, 61, 37], [0, 1, 2, 1]
    x, graphs, labels, ids_t = make_case(5, "onehot", n_cats, 358, ids, 64, 128, 256, 512)
    xl = x.contiguous(memory_format=CL).requires_grad_(True)
    del x
    ops.mds_proj_ohem_ce(xl, labels, ids_t, graphs, ops.neg_log(0.4)).backward()  # warm the graph cache
    xl.grad = None
    loss, fwd = _peak_growth(lambda: ops.mds_proj_ohem_ce(xl, labels, ids_t, graphs, ops.neg_log(0.4)))
    assert fwd < 0.5 * xl.nbytes, (fwd, xl.nbytes)
    _, bwd = _peak_growth(lambda: loss.backward())
    assert xl.nbytes <= bwd < 1.5 * xl.nbytes, (bwd, xl.nbytes)
    assert xl.grad.is_contiguous(memory_format=CL)


def test_no_layout_copy_aux(ops):
    n_cats, ids = [19, 64, 37, 19, 26, 150, 133], [5, 6, 1, 0]
    B, h, w, H, W = len(ids), 64, 128, 256, 512
    gen = torch.Generator(device=DEV).manual_seed(3)
    aux = [torch.randn(B, c, h, w, generator=gen, device=DEV).contiguous(memory_format=CL).requires_grad_(True)
           for c in n_cats]
    labels = torch.stack([torch.randint(0, n_cats[d], (H, W), generator=gen, device=DEV) for d in ids]).to(torch.uint8)
    ids_t = torch.tensor(ids, dtype=torch.int32, device=DEV)
    nbytes = sum(a.nbytes for a in aux)
    loss, fwd = _peak_growth(lambda: ops.up_ohem_ce(aux, labels, ids_t, ops.neg_log(0.7)))
    assert fwd < 0.5 * nbytes, (fwd, nbytes)
    _, bwd = _peak_growth(lambda: torch.nansum(loss).backward())
    assert nbytes <= bwd < 2 * nbytes, (bwd, nbytes)  # the gradients, the planar dy rows and the kernel's workspace
    assert all(a.grad.is_contiguous(memory_format=CL) for a in aux)


# ---- 6. CUDA graph capture ---------------------------------------------------------------------------------------
def test_cuda_graph_capture(ops):
    n_cats, ids = [61, 19, 150], [2, 0, 1, 2]
    x, graphs, labels, ids_t = make_case(9, "onehot", n_cats, 358, ids, 16, 32, 64, 128)
    xl = x.contiguous(memory_format=CL).requires_grad_(True)
    aux = [torch.randn(len(ids), c, 16, 32, device=DEV).contiguous(memory_format=CL).requires_grad_(True)
           for c in n_cats]

    def step():
        for t in (xl, *aux):
            t.grad = None
        loss = ops.mds_proj_ohem_ce(xl, labels, ids_t, graphs, ops.neg_log(0.4))
        loss = loss + ops.up_ohem_ce(aux, labels, ids_t, ops.neg_log(0.7)).sum()
        loss.backward()
        return loss.detach()

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            eager = step()
    torch.cuda.current_stream().wait_stream(side)
    eager = eager.clone()
    eager_grads = [t.grad.clone() for t in (xl, *aux)]
    graph = torch.cuda.CUDAGraph()
    for t in (xl, *aux):
        t.grad = None
    with torch.cuda.graph(graph):
        captured = step()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, eager)
    for t, g in zip((xl, *aux), eager_grads):
        assert torch.equal(t.grad, g)
    ops.check_errors(DEV)


# ---- 7. drop-in loss with a channels_last model ---------------------------------------------------------------------
@pytest.fixture(scope="module")
def dropin():
    import mdseg_b200.dropin as d
    d.install()
    yield d
    d.uninstall()


def test_cross_datasets_celoss_advgnn_seg_stage_channels_last(dropin, golden):
    from lib.loss.loss_cross_datasets import CrossDatasetsCELoss_AdvGNN
    from mdseg_b200 import ops
    z = golden("advgnn_seg_stage.npz")
    n_cats = [int(c) for c in z["n_cats"]]
    n = len(n_cats)
    cfg = {"n_datasets": n, "loss": {"with_datasets_aux": True, "aux_weight": float(z["aux_weight"])},
           "GNN": {"unify_ratio": float(z["c_uni"]) / sum(n_cats) + 1e-9}}
    for i, c in enumerate(n_cats):
        cfg[f"dataset{i + 1}"] = {"n_cats": c}
    crit = CrossDatasetsCELoss_AdvGNN(DictConfiger(cfg))
    runs = []
    for fmt in (torch.contiguous_format, CL):
        x = torch.from_numpy(z["x"]).to(DEV).contiguous(memory_format=fmt).requires_grad_(True)
        aux = [torch.from_numpy(z[f"aux{i}"]).to(DEV).contiguous(memory_format=fmt).requires_grad_(True)
               for i in range(n)]
        preds = {"seg": x, "aux": aux, "unify_prototype": None,
                 "bi_graphs": [torch.from_numpy(z[f"graph{i}"]).to(DEV) for i in range(n)], "adv_out": None}
        loss, orth, aux_loss, adj = crit(preds, torch.from_numpy(z["labels"]).to(DEV),
                                         torch.from_numpy(z["ids"]).to(DEV), False, False)
        loss.backward()
        ops.check_errors(DEV)
        runs.append((loss.detach(), aux_loss.detach(), x.grad, [a.grad for a in aux]))
    (_, _, dx0, daux0), (loss, aux_loss, dx, daux) = runs
    assert abs(float(loss) - float(z["loss"])) <= RTOL32 * abs(float(z["loss"]))
    assert abs(float(aux_loss) - float(z["aux_loss"])) <= RTOL32 * abs(float(z["aux_loss"]))
    assert dx.is_contiguous(memory_format=CL)
    assert rel_err(dx.cpu().numpy(), z["dx"]) <= RTOL32
    assert rel_err(dx.cpu().numpy(), dx0.cpu().numpy()) <= RTOL32
    for i in range(n):
        assert daux[i].is_contiguous(memory_format=CL)
        assert rel_err(daux[i].cpu().numpy(), z[f"daux{i}"]) <= RTOL32, i
        assert torch.equal(daux[i], daux0[i]), i


# ---- 8. at size -------------------------------------------------------------------------------------------------
def test_cfg3_channels_last_at_size(ops):
    """16 x 358 x 256 x 512 fp32 logits, 1024 x 2048 labels, 7 datasets (BASELINE config 3)."""
    n_cats = [19, 64, 37, 19, 26, 150, 133]
    ids = [0, 0, 0, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6]
    gen = torch.Generator().manual_seed(7)
    graphs = graphs_for(gen, "onehot", n_cats, 358)
    dgen = torch.Generator(device=DEV).manual_seed(7)
    x = torch.randn(len(ids), 358, 256, 512, generator=dgen, device=DEV)
    labels = torch.stack([torch.randint(0, n_cats[d], (1024, 2048), generator=dgen, device=DEV) for d in ids])
    labels[torch.rand(labels.shape, generator=dgen, device=DEV) < 0.05] = 255
    labels = labels.to(torch.uint8)
    ids_t = torch.tensor(ids, dtype=torch.int32, device=DEV)
    l0, g0 = loss_and_grad(ops, x, labels, ids_t, graphs, ops.neg_log(0.4))
    xl = x.contiguous(memory_format=CL)
    del x
    l1, g1 = loss_and_grad(ops, xl, labels, ids_t, graphs, ops.neg_log(0.4))
    assert torch.equal(l0, l1)
    assert g1.is_contiguous(memory_format=CL)
    assert float((g1 - g0).abs().max()) <= RTOL32 * float(g0.abs().max())
