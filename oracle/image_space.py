"""numpy restatement of the image branch of the training transforms (test infrastructure, see oracle/__init__.py).

The reference's `lib/transform_cv2.py` is not part of this tree.  The arithmetic below follows the upstream BiSeNet
`lib/transform_cv2.py` the fork derives from (RandomResizedCrop, RandomHorizontalFlip, ColorJitter, ToTensor) and
OpenCV 4.x `imgproc/resize.cpp` for `cv2.resize(..., INTER_LINEAR)` on uint8.  The resize is checked against the real
cv2 in tests/test_host_image_transform.py; the chain as a whole is pinned on the real file only through
`$MDSEG_REFERENCE_ROOT` (same file).  No cv2 import here.
"""
import numpy as np

COEF = 2048  # INTER_RESIZE_COEF_SCALE: OpenCV's fixed-point weights have 11 fractional bits


def _linear_taps(dst, src, zero_border):
    """OpenCV's per-output-index source taps and weights for one axis of INTER_LINEAR.
    scale = 1 / ((double)dst / src); f = (float)((d + 0.5) * scale - 0.5); s = floor(f); f -= s.  On the column axis
    (zero_border) f is zeroed where s < 0 or s >= src - 1 and s clamped; on the row axis only the two indices are
    clamped.  Weights rint((1 - f) * 2048), rint(f * 2048) in fp32, half to even."""
    scale = 1.0 / (float(dst) / float(src))
    f = ((np.arange(dst, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int64)
    f = (f - s.astype(np.float32)).astype(np.float32)
    if zero_border:
        lo, hi = s < 0, s >= src - 1
        f[lo | hi] = 0
        s[lo] = 0
        s[hi] = src - 1
    w0 = np.rint((np.float32(1) - f) * np.float32(COEF)).astype(np.int64)
    w1 = np.rint(f * np.float32(COEF)).astype(np.int64)
    return np.clip(s, 0, src - 1), np.clip(s + 1, 0, src - 1), w0, w1


def cv2_linear_resize_u8(img, size):
    """cv2.resize(img, (w, h)) with INTER_LINEAR on uint8 [H, W] or [H, W, C] (lib/transform_cv2.py RandomResizedCrop).
    Horizontal pass h = S[sx0] * a0 + S[sx1] * a1 (int32), vertical pass
    ((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2, OpenCV's VResizeLinear<uchar> arithmetic.  The
    exact 2x down-scale cv2 routes to INTER_AREA gives the same numbers under these rules."""
    img = np.asarray(img)
    H, W = img.shape[:2]
    h, w = size
    sx0, sx1, a0, a1 = _linear_taps(w, W, True)
    sy0, sy1, b0, b1 = _linear_taps(h, H, False)
    s = img.astype(np.int64)
    ex = (slice(None),) + (None,) * (img.ndim - 2)            # weights along w, broadcast over channels
    ey = (slice(None), None) + (None,) * (img.ndim - 2)       # weights along h, broadcast over w and channels
    hx = s[:, sx0] * a0[ex] + s[:, sx1] * a1[ex]              # [H, w(, C)]
    top = (b0[ey] * (hx[sy0] >> 4)) >> 16
    bot = (b1[ey] * (hx[sy1] >> 4)) >> 16
    return np.clip((top + bot + 2) >> 2, 0, 255).astype(np.uint8)


def jitter_lut(brightness=None, contrast=None):
    """ColorJitter.adj_brightness then adj_contrast as one uint8[256] table: each is the reference's own expression,
    `np.array([...]).clip(0, 255).astype(np.uint8)`, and the second is applied to the first (table[im])."""
    lut = np.arange(256).astype(np.uint8)
    if brightness is not None:
        lut = np.array([i * brightness for i in range(256)]).clip(0, 255).astype(np.uint8)[lut]
    if contrast is not None:
        lut = np.array([74 + (i - 74) * contrast for i in range(256)]).clip(0, 255).astype(np.uint8)[lut]
    return lut


def saturation_coeffs(rate):
    """The two distinct entries of ColorJitter.adj_saturation's np.float32 matrix: (1 + 2r, 1 - r)."""
    m = np.float32([[1 + 2 * rate, 1 - rate, 1 - rate]])
    return m[0, 0], m[0, 1]


def _fmaf(a, b, c):
    """Correctly rounded float32 fma(a, b, c) for float32 arrays.  a * b is exact in float64 here (a holds byte
    values); the float64 sum is made round-to-odd with its exact error term so that the final rounding to float32 is
    a single correct rounding."""
    p = a.astype(np.float64) * b.astype(np.float64)
    c = c.astype(np.float64)
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)                           # TwoSum: s + err == p + c exactly
    bits = s.view(np.int64)
    fix = (err != 0) & ((bits & 1) == 0)
    step = np.where((err > 0) == (s > 0), 1, -1)              # move |s| toward the exact value
    s = np.where(fix, (bits + step).view(np.float64), s)
    return s.astype(np.float32)


def saturate_fma(im, rate):
    """ColorJitter.adj_saturation on uint8 [..., 3]:
    np.clip(np.matmul(im.reshape(-1, 3), M).reshape(shape) / 3, 0, 255).astype(np.uint8), with the product of each
    output channel c taken as fmaf(x2, M[2][c], fmaf(x1, M[1][c], x0 * M[0][c])) — the order x86-64 numpy's matmul
    takes — then fp32 / 3, the clip and truncation."""
    im = np.asarray(im)
    diag, off = saturation_coeffs(rate)
    x = im.reshape(-1, 3).astype(np.float32)
    out = np.empty_like(x)
    for c in range(3):
        m = [diag if k == c else off for k in range(3)]
        acc = (x[:, 0] * m[0]).astype(np.float32)
        acc = _fmaf(x[:, 1], np.float32(m[1]), acc)
        acc = _fmaf(x[:, 2], np.float32(m[2]), acc)
        out[:, c] = acc
    out = out / np.float32(3)
    return np.clip(out, 0, 255).astype(np.uint8).reshape(im.shape)


def to_tensor(im, mean=(0., 0., 0.), std=(1., 1., 1.)):
    """ToTensor(mean, std) of lib/transform_cv2.py on uint8 [H, W, 3]: transpose(2, 0, 1).astype(np.float32), then
    torch .div_(255).sub_(mean).div_(std) in fp32.  Returns float32 [3, H, W]."""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(np.asarray(im).transpose(2, 0, 1).astype(np.float32))).div_(255)
    m = torch.as_tensor(mean, dtype=t.dtype)[:, None, None]
    s = torch.as_tensor(std, dtype=t.dtype)[:, None, None]
    return t.sub_(m).div_(s).numpy()


def to_tensor_table(mean=(0., 0., 0.), std=(1., 1., 1.)):
    """ToTensor as a float32 [3, 256] table: table[c, v] is what to_tensor gives a byte v in channel c."""
    return to_tensor(np.tile(np.arange(256, dtype=np.uint8)[None, :, None], (1, 1, 3)), mean, std)[:, 0, :]


def image_transform_chain(img, plan, jitter=None, mean=(0., 0., 0.), std=(1., 1., 1.), size=None, bgr=True):
    """One sample's image through lib/transform_cv2.py, step by step as the reference does: BGR -> RGB view ->
    RandomResizedCrop (INTER_LINEAR resize, zero pad, crop) -> RandomHorizontalFlip -> ColorJitter (brightness,
    contrast, saturation in that order; `jitter` holds the drawn rates, None for a disabled term) -> ToTensor.
    Mirrors label_space.label_transform_chain; returns float32 [3, crop_h, crop_w]."""
    im = np.asarray(img)
    if bgr:
        im = im[:, :, ::-1]
    im = cv2_linear_resize_u8(im, (plan["im_h"], plan["im_w"]))
    ph, pw = plan.get("pad_top", 0), plan.get("pad_left", 0)
    if ph > 0 or pw > 0:
        im = np.pad(im, ((ph, ph), (pw, pw), (0, 0)))
    sh, sw = plan.get("crop_y", 0), plan.get("crop_x", 0)
    im = im[sh:sh + size[0], sw:sw + size[1], :]
    if plan.get("flip", False):
        im = im[:, ::-1, :]
    if jitter is not None:
        if jitter.get("brightness") is not None:
            im = jitter_lut(brightness=jitter["brightness"])[im]
        if jitter.get("contrast") is not None:
            im = jitter_lut(contrast=jitter["contrast"])[im]
        if jitter.get("saturation") is not None:
            im = saturate_fma(im, jitter["saturation"])
    return to_tensor(im, mean, std)
