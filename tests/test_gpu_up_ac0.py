"""GPU: the BiSeNet heads' align_corners=False up-sampling fused into OhemCELoss (ops.up_ohem_ce(...,
align_corners=False), OhemCELoss.forward_fused) against the float64 oracle and against the composition
F.interpolate(align_corners=False) + ops.ohem_ce on the GPU.  Tolerances: 1e-5 relative (fp32), 2e-2 (bf16 / fp16);
the selected set is exact outside the near-threshold band."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

import oracle_ac0 as ac0  # tests/oracle_ac0.py
from oracle import f64

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL32 = 1e-5
RTOL16 = 2e-2


@pytest.fixture(scope="module")
def ops():
    from mdseg_b200 import ops
    return ops


def close(a, b, rtol):
    a, b = float(a), float(b)
    return (np.isnan(a) and np.isnan(b)) or abs(a - b) <= rtol * abs(b)


def rel_err(a, b):
    return np.abs(np.asarray(a, dtype=np.float64) - b).max() / max(np.abs(b).max(), 1e-30)


def make_case(seed, N, C, h, w, fy, fx, scale=3.0, conf=0.0, p_ign=0.05):
    g = torch.Generator().manual_seed(seed)
    src = torch.randn(N, C, h, w, generator=g) * scale
    labels = torch.randint(0, C, (N, h * fy, w * fx), generator=g)
    if conf:  # one class per image with a few odd low-res cells, leading at its corners: the top-k branch is taken
        lab0 = torch.randint(0, C, (N, 1, 1), generator=g).expand(N, h, w).clone()
        odd = torch.rand(N, h, w, generator=g) < 0.01
        lab0[odd] = torch.randint(0, C, (int(odd.sum()),), generator=g)
        src = src + torch.zeros_like(src).scatter_(1, lab0[:, None], conf)
        labels = lab0.repeat_interleave(fy, 1).repeat_interleave(fx, 2)
    labels[torch.rand(labels.shape, generator=g) < p_ign] = 255
    return src, labels


def composition(ops, src, labels, thresh):
    """Route the fused call replaces: the head's nn.Upsample, then OhemCELoss on the full-resolution logits."""
    x = src.detach().clone().requires_grad_(True)
    up = F.interpolate(x, size=labels.shape[-2:], mode="bilinear", align_corners=False)
    loss = ops.ohem_ce(up, labels, thresh)
    loss.backward()
    return loss.detach(), x.grad


def fused(ops, src, labels, thresh, grad_scale=1.0):
    x = src.detach().clone().requires_grad_(True)
    loss = ops.up_ohem_ce([x], labels, None, thresh, align_corners=False)[0]
    (loss * grad_scale).backward()
    return loss.detach(), x.grad


def fused_loss_px(ops, src, labels, thresh):
    """The forward entry point and the selection alone: (per-pixel loss after the selection, state)."""
    from mdseg_b200 import native as N
    src = src.contiguous()
    B, Cc, h, w = src.shape
    H, W = labels.shape[1:]
    lab = labels.to(DEV).contiguous()
    tab = ops._src_table([src.data_ptr()], [Cc * h * w], [Cc], ops._DT[src.dtype], True)
    loss_px = torch.empty(B * H * W, dtype=torch.float32, device=DEV)
    lse_px = torch.empty_like(loss_px)
    st = ops._new_states(1, thresh, DEV)
    N.call("mdseg_up_ce_fwd_ac0", C.byref(tab), None, lab.data_ptr(), ops._DT[lab.dtype], B, h, w, H, W, 255,
           loss_px.data_ptr(), lse_px.data_ptr(), st.data_ptr(), ops.err_flag(DEV).data_ptr(), ops._stream())
    ops._select(loss_px, B, H * W, None, st, 1)
    return loss_px.view(B, H, W).cpu().numpy(), ops.read_states(st)[0]


SHAPES = [  # (N, C, h, w, fy, fx)
    (2, 19, 8, 12, 8, 8),     # cfg1-like main head
    (1, 171, 5, 5, 16, 16),   # cfg4-like x16 aux head
    (2, 19, 6, 10, 2, 2),
    (1, 7, 9, 7, 4, 4),       # w not a multiple of 4
    (1, 5, 1, 37, 8, 2),      # h = 1, w not a multiple of 32, different factors per axis
    (2, 2, 3, 33, 2, 16),     # C = 2
    (1, 11, 4, 3, 16, 4),
    (1, 3, 1, 1, 2, 2),       # one low-res pixel
]


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("mode", ["thresh", "topk"])
def test_fp32_against_oracle_and_composition(ops, shape, mode):
    N_, Cc, h, w, fy, fx = shape
    if mode == "topk" and N_ * h * fy * w * fx < 16 * 16:
        pytest.skip("n_min = 0: the top-k branch is not reachable")
    # top-k: the label class leads the log-sum-exp of the others by about 3.5 (losses near 0.03, few above the
    # threshold); far larger leads make losses so small that no fp32 CE holds them to 1e-5
    conf, scale = (0.0, 3.0) if mode == "thresh" else (float(np.log(max(Cc - 1, 1))) + 4.0, 1.0)
    src, labels = make_case(1 + Cc + h + w, N_, Cc, h, w, fy, fx, scale=scale, conf=conf)
    thresh = ops.neg_log(0.7)
    ref_loss, ref_dsrc, ref_px, ref_mask = ac0.up_ohem_ce_ac0(src.numpy(), labels.numpy(), thresh)
    loss, dsrc = fused(ops, src.to(DEV), labels.to(DEV), thresh)
    ops.check_errors(DEV)
    assert close(loss, ref_loss, RTOL32), (float(loss), ref_loss)
    assert rel_err(dsrc.cpu().numpy(), ref_dsrc) <= RTOL32
    closs, cdsrc = composition(ops, src.to(DEV), labels.to(DEV), thresh)
    assert close(loss, closs, RTOL32)
    assert rel_err(dsrc.cpu().numpy(), cdsrc.cpu().numpy().astype(np.float64)) <= RTOL32
    # the selected set, exact outside the band where an fp32 evaluation order may decide either way
    loss_px, st = fused_loss_px(ops, src.to(DEV), labels, thresh)
    valid = labels.numpy() != 255
    assert np.abs(loss_px - ref_px)[valid].max() <= RTOL32 * max(1.0, np.abs(ref_px).max())
    n_min = int(valid.sum()) // 16
    assert st.mode == (0 if int((ref_px > thresh).sum()) >= n_min else 1)
    assert st.mode == (0 if mode == "thresh" else 1) or N_ * h * w < 4  # both branches are reached
    if st.mode == 0:
        sel, cut = loss_px > st.thresh, thresh
    else:
        sel, cut = loss_px >= st.kth, ref_px.reshape(-1)[ref_mask.reshape(-1)].min()
    keep = ~f64.threshold_band(ref_px, cut)
    assert np.array_equal(sel[keep], ref_mask[keep])


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("shape", [(2, 19, 8, 12, 8, 8), (1, 171, 5, 5, 16, 16), (1, 5, 1, 37, 8, 2)])
def test_16bit_against_oracle(ops, dtype, shape):
    N_, Cc, h, w, fy, fx = shape
    src, labels = make_case(7 + Cc, N_, Cc, h, w, fy, fx)
    src = src.to(dtype)
    thresh = ops.neg_log(0.7)
    ref_loss, ref_dsrc, _, _ = ac0.up_ohem_ce_ac0(src.float().numpy(), labels.numpy(), thresh)
    loss, dsrc = fused(ops, src.to(DEV), labels.to(DEV), thresh)
    assert dsrc.dtype == dtype
    assert abs(float(loss) - ref_loss) <= RTOL16 * abs(ref_loss)
    assert rel_err(dsrc.float().cpu().numpy(), ref_dsrc) <= RTOL16


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", [(2, 19, 8, 12, 8, 8), (2, 24, 5, 9, 4, 16)])
def test_channels_last_bit_identical(ops, dtype, shape):
    N_, Cc, h, w, fy, fx = shape
    src, labels = make_case(3, N_, Cc, h, w, fy, fx)
    src = src.to(dtype).to(DEV)
    labels = labels.to(DEV)
    thresh = ops.neg_log(0.7)
    loss_a, g_a = fused(ops, src, labels, thresh)
    loss_b, g_b = fused(ops, src.to(memory_format=torch.channels_last), labels, thresh)
    assert g_b.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(loss_a, loss_b) and torch.equal(g_a, g_b.contiguous())


@pytest.mark.parametrize("seg_per_dataset", [True, False])
def test_multi_source_dataset_ids(ops, seg_per_dataset):
    g = torch.Generator().manual_seed(11)
    ids = [0, 1, 1, 0, 2]
    Cs, h, w, f = [5, 9, 3], 6, 10, 8
    srcs = [torch.randn(len(ids), c, h, w, generator=g) * 3 for c in Cs]
    labels = torch.stack([torch.randint(0, Cs[d], (h * f, w * f), generator=g) for d in ids])
    labels[torch.rand(labels.shape, generator=g) < 0.05] = 255
    thresh = ops.neg_log(0.7)
    xs = [s.to(DEV).requires_grad_(True) for s in srcs]
    out = ops.up_ohem_ce(xs, labels.to(DEV), torch.tensor(ids, device=DEV), thresh, seg_per_dataset=seg_per_dataset,
                         align_corners=False)
    out.sum().backward()
    ops.check_errors(DEV)
    ids_np = np.array(ids)
    if seg_per_dataset:
        for d in range(len(Cs)):
            sel = ids_np == d
            ref_loss, ref_dsrc, _, _ = ac0.up_ohem_ce_ac0(srcs[d].numpy()[sel], labels.numpy()[sel], thresh)
            assert close(out[d].detach(), ref_loss, RTOL32)
            grad = xs[d].grad.cpu().numpy()
            assert rel_err(grad[sel], ref_dsrc) <= RTOL32
            assert (grad[~sel] == 0).all()  # rows of other datasets' images: exactly zero
    else:
        # one selection over the whole batch, each image through its own head
        z = [ac0.upsample_ac0(srcs[d].numpy()[b], h * f, w * f) for b, d in enumerate(ids)]
        loss_px = np.stack([f64.ce_per_pixel(zb[None], labels.numpy()[b:b + 1])[0][0] for b, zb in enumerate(z)])
        ref_loss, _, _, _ = f64.ohem_select(loss_px.reshape(-1), int((labels.numpy() != 255).sum()), thresh)
        assert close(out[0].detach(), ref_loss, RTOL32)
        for d in range(len(Cs)):
            assert (xs[d].grad.cpu().numpy()[ids_np != d] == 0).all()


def test_backward_is_bit_reproducible(ops):
    src, labels = make_case(5, 2, 171, 10, 10, 8, 8)
    src, labels = src.to(DEV), labels.to(DEV)
    thresh = ops.neg_log(0.7)
    _, g1 = fused(ops, src, labels, thresh)
    _, g2 = fused(ops, src, labels, thresh)
    assert torch.equal(g1, g2)


def test_all_ignored_nan_and_zero_grad(ops):
    src, labels = make_case(9, 1, 7, 4, 6, 4, 4)
    labels[:] = 255
    loss, dsrc = fused(ops, src.to(DEV), labels.to(DEV), ops.neg_log(0.7))
    assert torch.isnan(loss)
    assert float(dsrc.abs().max()) == 0.0


def test_bad_label_flagged(ops):
    src, labels = make_case(9, 1, 7, 4, 6, 4, 4)
    labels[0, 3, 5] = 9
    ops.check_errors(DEV)
    fused(ops, src.to(DEV), labels.to(DEV), ops.neg_log(0.7))
    with pytest.raises(RuntimeError, match="label out of range"):
        ops.check_errors(DEV)


def test_grad_scaling_as_under_amp(ops):
    """A scaled loss (GradScaler) scales the gradient and nothing else."""
    src, labels = make_case(13, 2, 19, 6, 8, 8, 8)
    src, labels = src.to(DEV), labels.to(DEV)
    thresh = ops.neg_log(0.7)
    l1, g1 = fused(ops, src, labels, thresh)
    l2, g2 = fused(ops, src, labels, thresh, grad_scale=65536.0)
    assert torch.equal(l1, l2)
    assert rel_err((g2 / 65536.0).cpu().numpy(), g1.cpu().numpy().astype(np.float64)) <= 1e-6


def test_cuda_graph_capture_replay(ops):
    src, labels = make_case(17, 2, 19, 8, 12, 8, 8)
    src, labels = src.to(DEV), labels.to(DEV)
    thresh = ops.neg_log(0.7)
    want_loss, want_grad = fused(ops, src, labels, thresh)
    x = src.clone().requires_grad_(True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):  # warm-up on the capture stream
        for _ in range(2):
            x.grad = None
            ops.up_ohem_ce([x], labels, None, thresh, align_corners=False)[0].backward()
    torch.cuda.current_stream().wait_stream(s)
    x.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loss = ops.up_ohem_ce([x], labels, None, thresh, align_corners=False)[0]
        loss.backward()
    for _ in range(2):
        x.grad.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(loss, want_loss)
        assert torch.equal(x.grad, want_grad)


@pytest.mark.parametrize("shape", [(2, 19, 8, 16, 8, 8), (2, 171, 5, 5, 16, 16), (1, 19, 20, 20, 2, 2)])
def test_dropin_forward_fused_matches_forward(ops, shape):
    from mdseg_b200.dropin.ohem_ce_loss import OhemCELoss
    N_, Cc, h, w, fy, fx = shape
    src, labels = make_case(21, N_, Cc, h, w, fy, fx)
    src, labels = src.to(DEV), labels.to(DEV)
    crit = OhemCELoss(0.7)
    x1 = src.clone().requires_grad_(True)
    l1 = crit.forward(F.interpolate(x1, size=labels.shape[-2:], mode="bilinear", align_corners=False), labels)
    l1.backward()
    x2 = src.clone().requires_grad_(True)
    l2 = crit.forward_fused(x2, labels)
    l2.backward()
    assert l2.dim() == 0
    assert abs(float(l2) - float(l1)) <= RTOL32 * abs(float(l1))
    assert rel_err(x2.grad.cpu().numpy(), x1.grad.cpu().numpy().astype(np.float64)) <= RTOL32


def test_head_parameter_gradients(ops):
    """A small head ending in nn.Upsample(scale_factor=8, bilinear, align_corners=False): training through
    forward_fused on the logits before the up-sample gives the parameter gradients of forward on its output."""
    from mdseg_b200.dropin.ohem_ce_loss import OhemCELoss
    torch.manual_seed(0)
    # (no bias ahead of the BatchNorm: its gradient is zero up to rounding on both routes)
    head = nn.Sequential(nn.Conv2d(16, 32, 3, padding=1, bias=False), nn.BatchNorm2d(32), nn.ReLU(), nn.Conv2d(32, 19, 1),
                         nn.Upsample(scale_factor=8, mode="bilinear", align_corners=False)).to(DEV)
    feats = torch.randn(2, 16, 12, 20, device=DEV)
    labels = torch.randint(0, 19, (2, 96, 160), device=DEV)
    labels[torch.rand(labels.shape, device=DEV) < 0.05] = 255
    crit = OhemCELoss(0.7)

    def grads(loss):
        head.zero_grad()
        loss.backward()
        return [p.grad.detach().clone() for p in head.parameters()]

    g_ref = grads(crit.forward(head(feats), labels))
    g_fused = grads(crit.forward_fused(head[:-1](feats), labels))
    for a, b in zip(g_fused, g_ref):
        assert rel_err(a.cpu().numpy(), b.cpu().numpy().astype(np.float64)) <= 1e-4
