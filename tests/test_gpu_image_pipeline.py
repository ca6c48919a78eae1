"""GPU parity: the image branch of the training transforms in one gather (SURVEY §8 f3) — cv2 INTER_LINEAR resize,
zero padding, crop, flip, ColorJitter and ToTensor — bit for bit (torch.equal) against oracle/image_space.py, whose
resize is checked against the real cv2 in tests/test_host_image_transform.py."""
import numpy as np
import pytest
import torch

from oracle import image_space as ims
from oracle import label_space as ls

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
NORMS = [((0., 0., 0.), (1., 1., 1.)), ((0.3257, 0.3690, 0.3223), (0.2112, 0.2148, 0.2115)),
         ((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))]


@pytest.fixture(scope="module")
def ops():
    from mdseg_b200 import ops
    return ops


def _want(img, plan, jt, norm, size, bgr):
    mean, std = NORMS[norm]
    return torch.from_numpy(ims.image_transform_chain(img, plan, jt, mean, std, size, bgr))


def _random_case(rng, b, size):
    """Source H, W in 1 .. 200 (every sixth a 1-pixel-high or -wide one), resized by 0.2 .. 3x, padded on whichever
    axis ends up smaller than the crop, crop origin at either border or inside."""
    H, W = int(rng.randint(1, 200)), int(rng.randint(1, 200))
    if b % 6 == 4:
        H = 1
    if b % 6 == 5:
        W = 1
    im_h = max(1, int(np.ceil(H * rng.uniform(0.2, 3.0)))) if H > 1 else int(rng.randint(1, 120))
    im_w = max(1, int(np.ceil(W * rng.uniform(0.2, 3.0)))) if W > 1 else int(rng.randint(1, 160))
    pad_h = (size[0] - im_h) // 2 + 1 if im_h < size[0] else 0
    pad_w = (size[1] - im_w) // 2 + 1 if im_w < size[1] else 0
    hh, ww = im_h + 2 * pad_h - size[0], im_w + 2 * pad_w - size[1]
    edge = b % 3
    plan = dict(im_h=im_h, im_w=im_w, pad_top=pad_h, pad_left=pad_w, flip=bool(b & 1),
                crop_y=[0, hh, int(rng.randint(0, hh + 1))][edge], crop_x=[0, ww, int(rng.randint(0, ww + 1))][edge])
    return H, W, plan


@pytest.mark.parametrize("bgr", [True, False])
def test_image_pipeline_random_geometry(ops, bgr):
    """Up- and down-scaling, padding on either axis, crops at every border, flips, 1-pixel sources, row-strided views
    into a larger buffer, jitter on every image, three ToTensor tables."""
    from mdseg_b200.dropin.label_transform import ColorJitterPlan
    rng = np.random.RandomState(21 + bgr)
    size = (48, 80)
    jp = ColorJitterPlan(0.4, 0.4, 0.4)
    srcs, plans, jts, ids, wants = [], [], [], [], []
    for b in range(36):
        H, W, plan = _random_case(rng, b, size)
        big = rng.randint(0, 256, (H + 4, W + 7, 3)).astype(np.uint8)
        t = torch.from_numpy(big).to(DEV)
        view = t[2:2 + H, 5:5 + W, :] if b % 2 == 0 else t[:H, :W, :].contiguous()
        jt = jp.plan(rng)
        srcs.append(view)
        plans.append(plan)
        jts.append(jt)
        ids.append(b % 3)
        wants.append(_want(view.cpu().numpy(), plan, jt, b % 3, size, bgr))
    norms = ops.to_tensor_tables(NORMS, DEV)
    out = ops.image_pipeline(srcs, plans, size, jitter=jts, norms=norms, norm_ids=ids, bgr=bgr)
    assert out.dtype == torch.float32 and tuple(out.shape) == (len(srcs), 3) + size and out.is_contiguous()
    for b in range(len(srcs)):
        assert torch.equal(out[b].cpu(), wants[b]), (b, plans[b])


@pytest.mark.parametrize("jitter", [None, (0.4, 0.4, 0.4), (0.4, None, None), (None, 0.4, None), (None, None, 0.4),
                                    (0.4, None, 0.4)])
def test_image_pipeline_jitter_off_on_and_partly_on(ops, jitter):
    from mdseg_b200.dropin.label_transform import ColorJitterPlan
    rng = np.random.RandomState(31)
    size = (64, 96)
    jp = ColorJitterPlan(*jitter) if jitter is not None else None
    srcs, plans, jts = [], [], []
    for b in range(8):
        H, W, plan = _random_case(rng, b, size)
        srcs.append(torch.from_numpy(rng.randint(0, 256, (H, W, 3)).astype(np.uint8)).to(DEV))
        plans.append(plan)
        jts.append(jp.plan(rng) if jp is not None else None)
    out = ops.image_pipeline(srcs, plans, size, jitter=jts if jp is not None else None)
    for b in range(len(srcs)):
        assert torch.equal(out[b].cpu(), _want(srcs[b].cpu().numpy(), plans[b], jts[b], 0, size, True)), b


def test_image_pipeline_every_colour_through_saturation(ops):
    """All 2^24 colours as one 4096 x 4096 image at identity geometry: the saturation matrix at several rates equals
    the oracle's fma chain on every colour and stays within 1 of this host's np.matmul."""
    v = np.arange(1 << 24)
    rgb = np.stack([v >> 16, (v >> 8) & 255, v & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)
    src = torch.from_numpy(rgb).to(DEV)
    plan = dict(im_h=4096, im_w=4096, pad_top=0, pad_left=0, crop_y=0, crop_x=0, flip=False)
    table = torch.from_numpy(ims.to_tensor_table()).to(DEV)
    for rate in (0.6, 0.8731, 1.2345, 1.4):
        jt = dict(lut=np.arange(256, dtype=np.uint8), sat=ims.saturation_coeffs(rate))
        out = ops.image_pipeline([src], [plan], (4096, 4096), jitter=[jt], bgr=False)[0]
        want = torch.from_numpy(ims.saturate_fma(rgb, rate)).to(DEV).long()
        want_f = torch.stack([table[c][want[:, :, c]] for c in range(3)])
        assert torch.equal(out, want_f), rate
        got_u8 = torch.round(out * 255).to(torch.int16).permute(1, 2, 0).cpu().numpy()
        M = np.float32([[1 + 2 * rate, 1 - rate, 1 - rate], [1 - rate, 1 + 2 * rate, 1 - rate],
                        [1 - rate, 1 - rate, 1 + 2 * rate]])
        ref = np.clip(np.matmul(rgb.reshape(-1, 3), M).reshape(rgb.shape) / 3, 0, 255).astype(np.uint8)
        assert np.abs(got_u8 - ref).max() <= 1, rate


def test_image_pipeline_norm_ids_and_channels_last(ops):
    """Per-image ToTensor tables; the channels_last output equals the NCHW one bit for bit and has channels_last
    strides."""
    from mdseg_b200.dropin.label_transform import ColorJitterPlan
    rng = np.random.RandomState(41)
    size = (96, 128)
    jp = ColorJitterPlan(0.4, 0.4, 0.4)
    srcs, plans, jts, ids = [], [], [], []
    for b in range(9):
        H, W, plan = _random_case(rng, b, size)
        srcs.append(torch.from_numpy(rng.randint(0, 256, (H, W, 3)).astype(np.uint8)).to(DEV))
        plans.append(plan)
        jts.append(jp.plan(rng))
        ids.append(int(rng.randint(0, 3)))
    norms = ops.to_tensor_tables(NORMS, DEV)
    a = ops.image_pipeline(srcs, plans, size, jitter=jts, norms=norms, norm_ids=ids)
    c = ops.image_pipeline(srcs, plans, size, jitter=jts, norms=norms, norm_ids=ids, memory_format=torch.channels_last)
    assert c.is_contiguous(memory_format=torch.channels_last) and not c.is_contiguous()
    assert torch.equal(a, c)
    for b in range(len(srcs)):
        assert torch.equal(a[b].cpu(), _want(srcs[b].cpu().numpy(), plans[b], jts[b], ids[b], size, True)), b


def test_image_pipeline_errors(ops):
    from mdseg_b200.native import MdsegError
    src = torch.zeros(20, 30, 3, dtype=torch.uint8, device=DEV)
    plan = dict(im_h=40, im_w=60, pad_top=0, pad_left=0, crop_y=0, crop_x=0, flip=False)
    with pytest.raises(MdsegError):
        ops.image_pipeline([src], [plan], (32, 40))                       # out_w not a multiple of 16
    with pytest.raises(TypeError):
        ops.image_pipeline([src.float()], [plan], (32, 48))               # not uint8
    with pytest.raises(TypeError):
        ops.image_pipeline([src[:, :, :2]], [plan], (32, 48))             # two channels
    with pytest.raises(TypeError):
        ops.image_pipeline([torch.zeros(20, 30, 4, dtype=torch.uint8, device=DEV)[:, :, :3]], [plan], (32, 48))
    with pytest.raises(TypeError):
        ops.image_pipeline([src[:, :, 0]], [plan], (32, 48))              # a label image
    norms = ops.to_tensor_tables(NORMS[:2], DEV)
    with pytest.raises(ValueError):
        ops.image_pipeline([src], [plan], (32, 48), norms=norms, norm_ids=[2])
    with pytest.raises(ValueError):
        ops.image_pipeline([src], [plan], (32, 48), norms=norms, norm_ids=[-1])
    with pytest.raises(ValueError):
        ops.image_pipeline([src], [plan, plan], (32, 48))
    with pytest.raises(ValueError):
        ops.image_pipeline([src], [dict(plan, im_w=0)], (32, 48))
    with pytest.raises(ValueError):
        ops.image_pipeline([src], [plan], (32, 48), memory_format=torch.preserve_format)
    with pytest.raises(RuntimeError):
        ops.image_pipeline([src.cpu()], [plan], (32, 48))


def test_train_pipeline_on_a_seeded_stream(ops):
    """TrainPipeline draws crop, flip and jitter per sample from one stream; each image equals the oracle chain with
    that sample's draws, and the labels equal LabelPipeline's on the same seed."""
    from mdseg_b200.dropin.label_transform import LabelPipeline, TrainPipeline
    rng = np.random.RandomState(51)
    luts = rng.randint(0, 256, (3, 256)).astype(np.uint8)
    shapes = [(120, 200), (1100, 1200), (300, 700), (1090, 1100), (96, 160), (250, 650)]
    imgs = [rng.randint(0, 256, (H, W, 3)).astype(np.uint8) for H, W in shapes]
    lbs = [rng.randint(0, 256, (H, W)).astype(np.uint8) for H, W in shapes]
    ids = [0, 2, 1, 1, 0, 2]
    for scales, size in [((0.5, 1.0), (64, 96)), ((0.75, 2.0), (256, 512)), ((0.03, 0.06), (64, 96))]:
        for fmt in (torch.contiguous_format, torch.channels_last):
            pipe = TrainPipeline(scales, size, luts=torch.from_numpy(luts).to(DEV), norms=NORMS, memory_format=fmt)
            im, lb = pipe([torch.from_numpy(x).to(DEV) for x in imgs], [torch.from_numpy(x).to(DEV) for x in lbs], ids,
                          rng=np.random.RandomState(7))
            assert im.is_contiguous(memory_format=fmt) and lb.dtype == torch.int64
            plans = pipe.plans(shapes, np.random.RandomState(7))
            for b in range(len(imgs)):
                assert torch.equal(im[b].cpu(), _want(imgs[b], plans[b], plans[b]["jitter"], ids[b], size, True)), b
                assert np.array_equal(lb[b].cpu().numpy(), ls.label_transform_chain(lbs[b], luts[ids[b]], plans[b], size))
            lpipe = LabelPipeline(scales, size, luts=torch.from_numpy(luts).to(DEV))
            assert torch.equal(lb, lpipe([torch.from_numpy(x).to(DEV) for x in lbs], ids, rng=np.random.RandomState(7)))


@pytest.mark.parametrize("fmt", [torch.contiguous_format, torch.channels_last])
def test_train_pipeline_full_ltbgnn_batch(ops, fmt):
    """28 sources of 1024 x 2048 x 3 -> 768 x 768 (the ltbgnn_7_datasets_snp crop, 4 images per dataset): two images
    in full against the oracle, every value finite and inside the range of its image's ToTensor table."""
    from mdseg_b200.dropin.label_transform import TrainPipeline
    rng = np.random.RandomState(61)
    raws = [rng.randint(0, 256, (1024, 2048, 3)).astype(np.uint8) for _ in range(4)]
    srcs = [torch.from_numpy(raws[b % 4]).to(DEV) for b in range(28)]
    lbs = [torch.zeros(1024, 2048, dtype=torch.uint8, device=DEV) for _ in range(28)]
    ids = [b // 4 for b in range(28)]
    norms = [NORMS[d % 3] for d in range(7)]
    pipe = TrainPipeline((0.5, 2.0), (768, 768), norms=norms, memory_format=fmt)
    plans = pipe.plans([(1024, 2048)] * 28, np.random.RandomState(9))
    im, lb = pipe(srcs, lbs, ids, plans=plans)
    assert tuple(im.shape) == (28, 3, 768, 768) and im.is_contiguous(memory_format=fmt)
    assert torch.isfinite(im).all()
    tables = ops.to_tensor_tables(norms, DEV)
    lo, hi = tables.amin(dim=2), tables.amax(dim=2)                  # [7, 3]
    idt = torch.tensor(ids, device=DEV)
    assert (im >= lo[idt][:, :, None, None]).all() and (im <= hi[idt][:, :, None, None]).all()
    for b in (0, 27):
        want = _want(raws[b % 4], plans[b], plans[b]["jitter"], ids[b] % 3, (768, 768), True)
        assert torch.equal(im[b].cpu(), want), b
