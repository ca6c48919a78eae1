"""CPU checks of the align_corners=False geometry the fused BiSeNet-head loss relies on: the float64 reference's weights
and adjoint against CPU F.interpolate (size= and scale_factor= forms), the cell structure the kernels assume for
power-of-two factors, and the refusals of unsupported inputs by ops.up_ohem_ce and the C ABI."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import oracle_ac0 as ac0  # tests/oracle_ac0.py

FACTORS = (2, 4, 8, 16)
SIZES = (1, 2, 3, 5, 40, 80, 161, 320)


def _weight_matrix(n_in, n_out):
    i0, i1, l0, l1 = ac0.axis_weights_ac0(n_in, n_out)
    m = np.zeros((n_out, n_in))
    np.add.at(m, (np.arange(n_out), i0), l0)
    np.add.at(m, (np.arange(n_out), i1), l1)
    return m


def _torch_matrix(n_in, n_out, **kw):
    """Column j = F.interpolate of the j-th unit row: ATen's weights themselves (products with 0 / 1 are exact)."""
    eye = torch.eye(n_in, dtype=torch.float32).reshape(n_in, 1, 1, n_in)
    y = F.interpolate(eye, mode="bilinear", align_corners=False, **kw)[:, 0, 0, :]  # [n_in, n_out]
    return y.T.double().numpy()


@pytest.mark.parametrize("f", FACTORS)
@pytest.mark.parametrize("n", SIZES)
def test_weights_match_aten_exactly(f, n):
    want = _weight_matrix(n, f * n)
    assert np.array_equal(_torch_matrix(n, f * n, size=(1, f * n)), want)
    assert np.array_equal(_torch_matrix(n, f * n, scale_factor=(1, f)), want)
    # the scale ATen derives from scale_factor is the same fp32 value as in / out
    i0a, _, _, l1a = ac0.axis_weights_ac0(n, f * n, scale=1.0 / f)
    i0b, _, _, l1b = ac0.axis_weights_ac0(n, f * n)
    assert np.array_equal(i0a, i0b) and np.array_equal(l1a, l1b)


@pytest.mark.parametrize("f", FACTORS)
@pytest.mark.parametrize("n", SIZES)
def test_cell_structure(f, n):
    """o = f i + f/2 + k has i0 = i and l1 = (k + 0.5) / f for i in [0, n-1]; the first f/2 outputs have i0 = 0 and
    l1 = 0; the last input's outputs have i1 = i0."""
    i0, i1, _, l1 = ac0.axis_weights_ac0(n, f * n)
    assert (i0[:f // 2] == 0).all() and (l1[:f // 2] == 0).all()
    o = np.arange(f // 2, f * n)
    k = (o - f // 2) % f
    assert np.array_equal(i0[o], (o - f // 2) // f)
    assert np.array_equal(l1[o], (k + 0.5) / f)
    assert (i1[i0 == n - 1] == n - 1).all() and (i1[i0 < n - 1] == i0[i0 < n - 1] + 1).all()
    cnt = np.bincount(i0, minlength=n)
    if n >= 2:
        assert cnt[0] == f + f // 2 and cnt[-1] == f // 2 and (cnt[1:-1] == f).all()


def _ulp32(v):
    return np.spacing(np.abs(v).astype(np.float32)).astype(np.float64)


@pytest.mark.parametrize("fy,fx", [(2, 2), (4, 4), (8, 8), (16, 16), (8, 2), (2, 16), (16, 4)])
def test_values_and_adjoint_against_interpolate(fy, fx):
    g = torch.Generator().manual_seed(fy * 100 + fx)
    h, w = 5, 7
    x = torch.randn(2, 3, h, w, generator=g) * 4
    want = ac0.upsample_ac0(x.numpy(), fy * h, fx * w)
    scale = ac0.upsample_ac0(np.abs(x.numpy()), fy * h, fx * w)  # magnitude of the fp32 terms that are summed
    for kw in (dict(size=(fy * h, fx * w)), dict(scale_factor=(fy, fx))):
        y = F.interpolate(x, mode="bilinear", align_corners=False, **kw).double().numpy()
        assert (np.abs(y - want) <= 2 * _ulp32(scale)).all()
    # adjoint: autograd of the float64 interpolation
    xd = x.double().requires_grad_(True)
    gy = torch.randn(2, 3, fy * h, fx * w, generator=g, dtype=torch.float64)
    for kw in (dict(size=(fy * h, fx * w)), dict(scale_factor=(fy, fx))):
        xd.grad = None
        F.interpolate(xd, mode="bilinear", align_corners=False, **kw).backward(gy)
        ref = ac0.upsample_ac0_adjoint(gy.numpy(), h, w)
        assert np.abs(xd.grad.numpy() - ref).max() <= 1e-12 * np.abs(ref).max()


@pytest.fixture(scope="module")
def ops():
    from mdseg_b200 import ops
    return ops


@pytest.mark.parametrize("src_hw,lab_hw", [((10, 10), (30, 30)), ((10, 10), (50, 80)), ((10, 10), (320, 20)),
                                            ((10, 10), (10, 10)), ((10, 10), (20, 25)), ((10, 10), (15, 20))])
def test_ops_rejects_other_geometries(ops, src_hw, lab_hw):
    src = torch.zeros(1, 3, *src_hw)
    labels = torch.zeros(1, *lab_hw, dtype=torch.long)
    with pytest.raises(ValueError, match=r"\(1, 3, 10, 10\).*\(1, %d, %d\)" % lab_hw):
        ops.up_ohem_ce([src], labels, None, 0.5, align_corners=False)


def test_ops_rejects_cpu_tensors(ops):
    src = torch.zeros(1, 3, 10, 10)
    labels = torch.zeros(1, 80, 40, dtype=torch.long)
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.up_ohem_ce([src], labels, None, 0.5, align_corners=False)


def test_dropin_forward_fused_rejects_other_geometries():
    from mdseg_b200.dropin.ohem_ce_loss import OhemCELoss
    crit = OhemCELoss(0.7)
    with pytest.raises(ValueError):
        crit.forward_fused(torch.zeros(1, 3, 10, 10), torch.zeros(1, 30, 30, dtype=torch.long))


@pytest.mark.parametrize("h,w,H,W,ok", [(10, 10, 80, 80, True), (10, 10, 20, 160, True), (10, 10, 30, 30, False),
                                        (10, 10, 80, 81, False), (10, 10, 320, 320, False), (10, 10, 10, 10, False)])
def test_c_abi_rejects_other_geometries(h, w, H, W, ok):
    """The geometry is checked before anything touches the device: with n_images = 0 a good geometry returns 0."""
    from mdseg_b200 import native as N
    src = N.SrcTable()
    src.n_datasets, src.dtype, src.C[0], src.base[0] = 1, N.F32, 3, 256
    dst = N.SrcTable()
    dst.n_datasets, dst.dtype, dst.C[0], dst.base[0], dst.image_stride[0] = 1, N.F32, 3, 256, 3 * h * w
    rc = N.lib.mdseg_up_ce_fwd_ac0(C.byref(src), None, None, N.U8, 0, h, w, H, W, 255, None, None, None, None, None)
    rcb = N.lib.mdseg_up_ce_bwd_ac0(C.byref(src), None, None, N.U8, 0, h, w, H, W, 255, None, None, None, None, 1.0,
                                    C.byref(dst), None, 0, None)
    if ok:
        assert rc == 0 and rcb == 0
    else:
        assert rc != 0 and rcb != 0
        assert b"factors 2, 4, 8 or 16" in N.lib.mdseg_last_error()
