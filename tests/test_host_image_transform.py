"""Host side of the image branch of the training transforms (SURVEY §8 f3): the numpy restatement in
oracle/image_space.py against real cv2 / numpy / torch, and the random draws of dropin.label_transform.TrainPipeline
against LabelPipeline.  No GPU needed."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import image_space as ims

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE = os.environ.get("MDSEG_REFERENCE_ROOT", "")


def _geometries():
    rng = np.random.RandomState(0)
    out = [((1, 1), (7, 5)), ((1, 40), (3, 17)), ((40, 1), (17, 3)), ((9, 13), (9, 13)), ((64, 96), (32, 48)),
           ((63, 97), (127, 193)), ((5, 5), (1, 1)), ((300, 200), (60, 40))]
    for i in range(120):
        H, W = int(rng.randint(1, 300)), int(rng.randint(1, 300))
        s = rng.uniform(0.2, 3.0)
        out.append(((H, W), (max(1, int(np.ceil(H * s))), max(1, int(np.ceil(W * s * rng.uniform(0.8, 1.25)))))))
    return out


def test_linear_resize_equals_cv2():
    """Up, down, the exact halving cv2 routes to INTER_AREA, identity, 1-pixel-wide / -high sources, odd sizes;
    3-channel and 1-channel."""
    cv2 = pytest.importorskip("cv2")
    cv2.setNumThreads(1)
    rng = np.random.RandomState(1)
    for (H, W), (h, w) in _geometries():
        img = rng.randint(0, 256, (H, W, 3)).astype(np.uint8)
        want = cv2.resize(img, (w, h))
        want = want.reshape(h, w, -1)
        assert np.array_equal(ims.cv2_linear_resize_u8(img, (h, w)), want), ((H, W), (h, w))
        assert np.array_equal(ims.cv2_linear_resize_u8(img[:, :, 0], (h, w)), cv2.resize(img[:, :, 0].copy(), (w, h)))


def test_linear_resize_at_size_equals_cv2():
    """A 1024 x 2048 source at the scales of the ltbgnn crop (0.5 .. 2.0 after the 1080 rescale)."""
    cv2 = pytest.importorskip("cv2")
    cv2.setNumThreads(1)
    img = np.random.RandomState(2).randint(0, 256, (1024, 2048, 3)).astype(np.uint8)
    for s in (0.5 * 1080 / 1024, 1.3, 2.0 * 1080 / 1024):
        h, w = int(np.ceil(1024 * s)), int(np.ceil(2048 * s))
        assert np.array_equal(ims.cv2_linear_resize_u8(img, (h, w)), cv2.resize(img, (w, h))), s


def _all_colours():
    v = np.arange(1 << 24)
    return np.stack([v >> 16, (v >> 8) & 255, v & 255], -1).astype(np.uint8)


@pytest.mark.parametrize("rate", [0.6, 0.8731, 1.0, 1.2345, 1.4])
def test_saturate_fma_on_every_colour(rate):
    """saturate_fma is the explicit chain fmaf(x2, m2, fmaf(x1, m1, x0 * m0)) / 3 on all 2^24 colours: for these rates
    x1 * m1 + p (and x2 * m2 + q) are exact in float64, so one rounding to float32 is the fma.  np.matmul takes
    whatever order the host's BLAS takes; it stays within 1 everywhere."""
    im = _all_colours()
    got = ims.saturate_fma(im, rate)
    diag, off = ims.saturation_coeffs(rate)
    x = im.astype(np.float32)
    want = np.empty_like(x)
    for c in range(3):
        m = [np.float64(diag if k == c else off) for k in range(3)]
        acc = (x[:, 0] * np.float32(m[0])).astype(np.float32)
        for k in (1, 2):
            p = x[:, k].astype(np.float64) * m[k]
            s = p + acc.astype(np.float64)
            bb = s - p
            assert not np.any((p - (s - bb)) + (acc.astype(np.float64) - bb))  # TwoSum error 0: the sum is exact
            acc = s.astype(np.float32)
        want[:, c] = acc
    want = np.clip(want / np.float32(3), 0, 255).astype(np.uint8)
    assert np.array_equal(got, want)
    M = np.float32([[1 + 2 * rate, 1 - rate, 1 - rate], [1 - rate, 1 + 2 * rate, 1 - rate],
                    [1 - rate, 1 - rate, 1 + 2 * rate]])
    ref = np.clip(np.matmul(im, M) / 3, 0, 255).astype(np.uint8)
    assert np.abs(ref.astype(np.int16) - got).max() <= 1


def test_jitter_lut_is_the_reference_tables_composed():
    rng = np.random.RandomState(3)
    im = rng.randint(0, 256, (50, 60, 3)).astype(np.uint8)
    for rb, rc in [(0.6, 1.4), (1.4, 0.6), (1.0, 1.0), (0.8731, 1.2345)]:
        tb = np.array([i * rb for i in range(256)]).clip(0, 255).astype(np.uint8)
        tc = np.array([74 + (i - 74) * rc for i in range(256)]).clip(0, 255).astype(np.uint8)
        assert np.array_equal(ims.jitter_lut(rb, rc)[im], tc[tb[im]])


@pytest.mark.parametrize("mean_std", [((0., 0., 0.), (1., 1., 1.)), ((0.3257, 0.3690, 0.3223), (0.2112, 0.2148, 0.2115)),
                                      ((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))])
def test_to_tensor_table_equals_the_torch_ops(mean_std):
    import torch
    im = np.random.RandomState(4).randint(0, 256, (97, 131, 3)).astype(np.uint8)
    mean, std = mean_std
    t = torch.from_numpy(im.transpose(2, 0, 1).astype(np.float32)).div_(255)
    want = t.sub_(torch.as_tensor(mean)[:, None, None]).div_(torch.as_tensor(std)[:, None, None]).numpy()
    table = ims.to_tensor_table(mean, std)
    got = np.stack([table[c][im[:, :, c]] for c in range(3)])
    assert np.array_equal(got, want)
    from mdseg_b200 import ops
    assert np.array_equal(ops.to_tensor_tables([mean_std], "cpu")[0].numpy(), table)


def test_train_pipeline_plans_match_label_pipeline():
    """Same seed: TrainPipeline draws crop, flip and the three ColorJitter rates per sample; LabelPipeline draws and
    drops the rates.  Crop and flip plans are identical, the rates lie in [0.6, 1.4], and the lut / saturation entries
    are the reference's expressions of those rates."""
    from mdseg_b200.dropin.label_transform import LabelPipeline, TrainPipeline
    rng = np.random.RandomState(5)
    shapes = [(int(rng.randint(200, 1300)), int(rng.randint(200, 2100))) for _ in range(200)]
    for scales, size in [((0.5, 2.0), (768, 768)), ((0.03, 0.06), (64, 96))]:
        a = TrainPipeline(scales, size).plans(shapes, np.random.RandomState(17))
        b = LabelPipeline(scales, size).plans(shapes, np.random.RandomState(17))
        for pa, pb in zip(a, b):
            jt = pa.pop("jitter")
            assert pa == pb
            rb, rc, rs = jt["brightness"], jt["contrast"], jt["saturation"]
            assert all(0.6 <= r <= 1.4 for r in (rb, rc, rs))
            assert np.array_equal(jt["lut"], ims.jitter_lut(rb, rc))
            assert (jt["sat"][0], jt["sat"][1]) == ims.saturation_coeffs(rs)
        c = TrainPipeline(scales, size, jitter=None).plans(shapes[:20], np.random.RandomState(17))
        d = LabelPipeline(scales, size, image_draws=0).plans(shapes[:20], np.random.RandomState(17))
        assert [dict(p, jitter=None) for p in d] == c


def test_image_transform_chain_steps():
    """The chain on a hand-checkable case: identity geometry, no jitter, default ToTensor = byte / 255 with the
    channels reversed for BGR input; a pad-only geometry gives the contrast table's value of 0 in the padding."""
    im = np.random.RandomState(6).randint(0, 256, (16, 32, 3)).astype(np.uint8)
    plan = dict(im_h=16, im_w=32, pad_top=0, pad_left=0, crop_y=0, crop_x=0, flip=False)
    out = ims.image_transform_chain(im, plan, None, size=(16, 32), bgr=True)
    assert np.array_equal(out, (im[:, :, ::-1].transpose(2, 0, 1).astype(np.float32) / np.float32(255)))
    plan = dict(im_h=16, im_w=32, pad_top=3, pad_left=2, crop_y=0, crop_x=0, flip=True)
    jt = dict(brightness=None, contrast=0.7, saturation=None)
    out = ims.image_transform_chain(im, plan, jt, size=(16, 32), bgr=False)
    pad = np.float32(np.uint8(74 + (0 - 74) * 0.7)) / np.float32(255)
    assert np.all(out[:, :3, :] == pad) and np.all(out[:, :, -2:] == pad)


@pytest.mark.skipif(not REFERENCE or not os.path.isfile(os.path.join(REFERENCE, "lib", "transform_cv2.py")),
                    reason="needs a checkout of the reference project under $MDSEG_REFERENCE_ROOT")
def test_image_chain_against_the_real_transform_cv2(tmp_path):
    """The reference's own Compose([RandomResizedCrop, RandomHorizontalFlip, ColorJitter(.4, .4, .4)]) + ToTensor
    (lib/transform_cv2.py, real cv2) on a seeded np.random stream, against image_transform_chain driven by
    TrainPipeline.plans on the same seed: this pins the image arithmetic on the real file."""
    pytest.importorskip("cv2")
    code = f"""
import sys, numpy as np
sys.dont_write_bytecode = True
sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {REFERENCE!r})
import lib.transform_cv2 as T
from oracle import image_space as ims
from mdseg_b200.dropin.label_transform import TrainPipeline
gen = np.random.default_rng(8)
cases = [([(96, 160), (120, 200), (1100, 1200)], (0.5, 1.0), (64, 96)),
         ([(1090, 1100), (1200, 1085)], (0.03, 0.06), (64, 96)),
         ([(300, 700), (250, 650)], (0.75, 2.0), (256, 512))]
mean, std = (0.3257, 0.3690, 0.3223), (0.2112, 0.2148, 0.2115)
for ci, (shapes, scales, size) in enumerate(cases):
    trans = T.Compose([T.RandomResizedCrop(scales, size), T.RandomHorizontalFlip(),
                       T.ColorJitter(brightness=0.4, contrast=0.4, saturation=0.4)])
    to_tensor = T.ToTensor(mean=mean, std=std)
    ims_bgr = [gen.integers(0, 256, (H, W, 3)).astype(np.uint8) for H, W in shapes]
    np.random.seed(100 + ci)
    refs = [to_tensor(trans(dict(im=im[:, :, ::-1], lb=np.zeros(im.shape[:2], np.uint8))))['im'].numpy()
            for im in ims_bgr]
    plans = TrainPipeline(scales, size).plans(shapes, np.random.RandomState(100 + ci))
    for im, pl, ref in zip(ims_bgr, plans, refs):
        got = ims.image_transform_chain(im, pl, pl['jitter'], mean, std, size, bgr=True)
        assert np.array_equal(got, ref), (ci, pl)
print('ok')
"""
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stderr[-2000:]
