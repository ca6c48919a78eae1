"""SURVEY 8 row f2: the prototype head einsum('bchw,nc->bnhw', feats, unify_prototype) (lib/models/semseg.py:325-333,
lib/loss/loss_cross_datasets.py:940-969) on the tcgen05 tensor cores, forward and both gradients, against a float64
einsum.  Bars: 1e-5 relative (fp32 inputs, three bf16 terms per operand), 2e-2 (bf16 / fp16 inputs)."""
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def ops():
    from mdseg_b200 import ops
    return ops


def rel(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max())


@pytest.mark.parametrize("B,K,N,h,w", [(2, 512, 358, 24, 40), (1, 64, 19, 16, 16), (3, 96, 600, 9, 13), (2, 512, 150, 32, 32),
                                      (1, 40, 5, 8, 8)])
@pytest.mark.parametrize("dt,tol", [(torch.float32, 1e-5), (torch.bfloat16, 2e-2), (torch.float16, 2e-2)])
def test_prototype_head_forward_and_gradients(ops, B, K, N, h, w, dt, tol):
    g = torch.Generator(device=DEV).manual_seed(B * 1000 + N)
    feats = (torch.randn(B, K, h, w, generator=g, device=DEV)).to(dt).requires_grad_(True)
    proto = (torch.randn(N, K, generator=g, device=DEV) * 0.2).requires_grad_(True)
    dy = torch.randn(B, N, h, w, generator=g, device=DEV)
    y = ops.prototype_head(feats, proto)
    assert y.dtype == torch.float32 and tuple(y.shape) == (B, N, h, w)
    y.backward(dy)
    f64, p64 = feats.detach().double(), proto.detach().double()
    if dt != torch.float32:  # what autocast does to the reference einsum: the weights rounded to the input type
        p64 = proto.detach().to(dt).double()
    want = torch.einsum("bchw,nc->bnhw", f64, p64)
    assert rel(y, want) <= tol
    assert rel(feats.grad, torch.einsum("bnhw,nc->bchw", dy.double(), p64)) <= tol
    assert rel(proto.grad, torch.einsum("bnhw,bchw->nc", dy.double(), f64)) <= tol
    ops.check_errors(DEV)


def _mds_case(g, n_cats, ids, K, Cu, h, w, f, dt):
    feats = torch.randn(len(ids), K, h, w, generator=g, device=DEV).to(dt).requires_grad_(True)
    proto = (torch.randn(Cu, K, generator=g, device=DEV) * 0.2).requires_grad_(True)
    graphs = [torch.softmax(torch.randn(c, Cu, generator=g, device=DEV) * 3, dim=0).requires_grad_(True) for c in n_cats]
    labels = torch.stack([torch.randint(0, n_cats[d], (h * f, w * f), generator=g, device=DEV) for d in ids])
    labels[torch.rand(labels.shape, generator=g, device=DEV) < 0.05] = 255
    return feats, proto, graphs, labels


@pytest.mark.parametrize("dt,tol", [(torch.float32, 1e-5), (torch.bfloat16, 2e-2), (torch.float16, 2e-2)])
@pytest.mark.parametrize("ids", [[0, 0, 1, 2, 2], [2, 0, 1, 0]], ids=["sorted", "shuffled"])
def test_folded_head_loss_matches_float64_reference_order(ops, dt, tol, ids):
    """einsum(feats, bi_graph @ unify_prototype) -> up-sample -> OHEM CE (ops.mds_head_proj_ohem_ce) against the
    reference's order einsum(einsum(feats, prototypes), bi_graph) evaluated by torch in float64: loss and the gradients
    to the features, the prototypes and every graph.  16-bit features take mdseg_proj_fwd_tc16 / mdseg_proj_bwd_tc16 /
    mdseg_proj_bwd_graph_tc16."""
    import torch.nn.functional as F
    n_cats, K, Cu, h, w, f = [19, 9, 33], 64, 48, 8, 16, 4
    g = torch.Generator(device=DEV).manual_seed(len(ids))
    feats, proto, graphs, labels = _mds_case(g, n_cats, ids, K, Cu, h, w, f, dt)
    ids_t = torch.tensor(ids, dtype=torch.int32, device=DEV)
    # 16-bit operands move every loss by ~1e-3: a pixel that close to the threshold changes sides and takes its whole
    # gradient with it (seen: one pixel, 2.5 % of the largest gradient).  The selection rule is tested in fp32; the
    # 16-bit cases put the threshold below every loss so that the comparison measures the arithmetic.
    thresh = ops.neg_log(0.4 if dt == torch.float32 else 0.999)
    loss = ops.mds_head_proj_ohem_ce(feats, proto, labels, ids_t, graphs, thresh)
    scale = 4096.0  # what amp.GradScaler does: the per-pixel gradients (~1 / |S|) are subnormal in fp16 otherwise
    (loss * scale).backward()
    ops.check_errors(DEV)

    f64 = feats.detach().double().requires_grad_(True)
    p64 = proto.detach().double().requires_grad_(True)
    g64 = [m.detach().double().requires_grad_(True) for m in graphs]
    logits = torch.einsum("bchw,nc->bnhw", f64, p64)
    per_px = []
    for b, d in enumerate(ids):
        y = torch.einsum("chw,nc->nhw", logits[b], g64[d])[None]
        y = F.interpolate(y, size=(h * f, w * f), mode="bilinear", align_corners=True)
        per_px.append(F.cross_entropy(y, labels[b][None], ignore_index=255, reduction="none").view(-1))
    per_px = torch.cat(per_px)
    n_min = int((labels != 255).sum()) // 16
    hard = per_px[per_px > thresh]
    assert hard.numel() >= n_min  # the threshold branch (soft graphs keep every loss high)
    want = hard.mean()
    (want * scale).backward()
    assert abs(float(loss) - float(want)) <= tol * float(want)
    assert rel(feats.grad, f64.grad) <= tol
    assert rel(proto.grad, p64.grad) <= tol
    for i in range(len(n_cats)):
        if i in ids:
            assert rel(graphs[i].grad, g64[i].grad) <= tol, i


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("B,Cu,cmax,Cs,h,w", [(5, 512, 150, [19, 150, 64], 16, 24), (3, 48, 40, [40, 8], 8, 8),
                                              (4, 358, 133, [133, 26, 37, 19], 12, 20)])
def test_proj_bwd_tc16_nchw_entry_points_match_float64(ops, dt, B, Cu, cmax, Cs, h, w):
    """mdseg_proj_bwd_tc16 (d x = G_d^T dy) and mdseg_proj_bwd_graph_tc16 (d G_d = sum over the dataset's images of
    dy x^T) through the C ABI, including an image whose dataset id is out of range (zero rows in d x, no contribution
    to any d G)."""
    from mdseg_b200 import native as N
    g = torch.Generator(device=DEV).manual_seed(B * 100 + Cu)
    n = len(Cs)
    ids = [(b % n) for b in range(B)]
    ids[-1] = 99 if B > 3 else ids[-1]  # one image of no dataset
    ids_t = torch.tensor(ids, dtype=torch.int32, device=DEV)
    x = torch.randn(B, Cu, h, w, generator=g, device=DEV).to(dt)
    graphs = [torch.randn(c, Cu, generator=g, device=DEV) * 0.3 for c in Cs]
    dy = torch.zeros(B, cmax, h, w, device=DEV)
    for b, d in enumerate(ids):
        if d < n:
            dy[b, :Cs[d]] = torch.randn(Cs[d], h, w, generator=g, device=DEV)
    dy16 = dy.to(dt)
    dtc = {torch.bfloat16: N.BF16, torch.float16: N.F16}[dt]
    keep, ptrs, ldb = ops._tc16_operands(graphs, dt, transpose=True)
    dx = torch.full((B, Cu, h, w), float("nan"), dtype=dt, device=DEV)
    stream = torch.cuda.current_stream().cuda_stream
    N.call("mdseg_proj_bwd_tc16", dy16.data_ptr(), dtc, N.NCHW, B, cmax, h * w, ptrs, ldb, Cu, n, ids_t.data_ptr(),
           dx.data_ptr(), dtc, stream)
    dG = torch.full((n, cmax, Cu), float("nan"), dtype=torch.float32, device=DEV)
    nb = N.lib.mdseg_proj_bwd_graph_tc16_workspace_bytes(B, Cu, h * w, cmax)
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    N.call("mdseg_proj_bwd_graph_tc16", dy16.data_ptr(), x.data_ptr(), dtc, N.NCHW, B, Cu, h * w, cmax, ids_t.data_ptr(),
           n, dG.data_ptr(), ws.data_ptr(), nb, stream)
    torch.cuda.synchronize()
    want_dx = torch.zeros(B, Cu, h, w, dtype=torch.float64, device=DEV)
    want_dG = torch.zeros(n, cmax, Cu, dtype=torch.float64, device=DEV)
    for b, d in enumerate(ids):
        if d >= n:
            continue
        g16 = graphs[d].to(dt).double()
        want_dx[b] = torch.einsum("nhw,nc->chw", dy16[b, :Cs[d]].double(), g16)
        want_dG[d, :Cs[d]] += torch.einsum("nhw,chw->nc", dy16[b, :Cs[d]].double(), x[b].double())
    assert torch.isfinite(dx.float()).all() and torch.isfinite(dG).all()
    assert rel(dx, want_dx) <= 2e-2
    assert rel(dG, want_dG) <= 1e-3  # fp32 accumulation of exact 16-bit products
    if B > 3:
        assert float(dx[-1].float().abs().max()) == 0.0
    for d in range(n):
        assert float(dG[d, Cs[d]:].abs().max()) == 0.0 if Cs[d] < cmax else True


@pytest.mark.parametrize("dt,tol", [(torch.float32, 1e-5), (torch.bfloat16, 2e-2)])
@pytest.mark.parametrize("ids", [[0, 0, 1, 2, 2], [2, 0, 1, 0]], ids=["sorted", "shuffled"])
def test_stacked_heads_equal_independent_losses(ops, dt, tol, ids):
    """The GNN stage's (hard, soft) graph pair as ONE stacked projection (ops.mds_head_proj_ohem_ce_heads) against two
    independent folded losses: both loss values, and the gradients of a blend to the features, the prototypes and all
    graphs of both sets."""
    n_cats, K, Cu, h, w, f = [19, 9, 33], 64, 48, 8, 16, 4
    g = torch.Generator(device=DEV).manual_seed(7 + len(ids))
    feats, proto, hard, labels = _mds_case(g, n_cats, ids, K, Cu, h, w, f, dt)
    soft = [torch.softmax(torch.randn(c, Cu, generator=g, device=DEV), dim=0).requires_grad_(True) for c in n_cats]
    ids_t = torch.tensor(ids, dtype=torch.int32, device=DEV)
    thresh = ops.neg_log(0.4 if dt == torch.float32 else 0.999)  # see test_folded_head_loss_matches_float64_reference_order
    scale = 4096.0
    pair = ops.mds_head_proj_ohem_ce_heads(feats, proto, labels, ids_t, [hard, soft], thresh)
    assert tuple(pair.shape) == (2,)
    ((0.3 * pair[0] + 0.7 * pair[1]) * scale).backward()
    ops.check_errors(DEV)
    f2 = feats.detach().clone().requires_grad_(True)
    p2 = proto.detach().clone().requires_grad_(True)
    h2 = [m.detach().clone().requires_grad_(True) for m in hard]
    s2 = [m.detach().clone().requires_grad_(True) for m in soft]
    a = ops.mds_head_proj_ohem_ce(f2, p2, labels, ids_t, h2, thresh)
    b = ops.mds_head_proj_ohem_ce(f2, p2, labels, ids_t, s2, thresh)
    ((0.3 * a + 0.7 * b) * scale).backward()
    assert abs(float(pair[0]) - float(a)) <= tol * float(a) and abs(float(pair[1]) - float(b)) <= tol * float(b)
    assert rel(feats.grad, f2.grad) <= tol
    assert rel(proto.grad, p2.grad) <= tol
    for i in range(len(n_cats)):
        if i in ids:
            assert rel(hard[i].grad, h2[i].grad) <= tol, i
            assert rel(soft[i].grad, s2[i].grad) <= tol, i
