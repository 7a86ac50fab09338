"""numpy restatement of the multi-scale resize contract (DESIGN.md §2 deviation 7): OpenCV's portable fixed-point
INTER_CUBIC arithmetic for 8-bit images, the arithmetic cv2.resize(img, None, fx=rate, fy=rate, interpolation=INTER_CUBIC)
uses without a HAL.  Test infrastructure: the device producer (csrc/tiles.cu) is checked against it, and
tests/golden/gen_golden_multiscale.py substitutes it for cv2.resize inside the reference's own splitter.

Everything after the tables is integer arithmetic, so the result does not depend on platform or summation order.
"""
import numpy as np

A = np.float32(-0.75)
_ONE = np.float32(1.0)


def dst_size(n, rate):
    """saturate_cast<int>(n * rate): round half to even; an empty result is an error (cv2 asserts !dsize.empty())"""
    if not rate > 0:
        raise ValueError("rate must be > 0, got %r" % (rate,))
    m = int(np.rint(np.float64(n) * np.float64(rate)))
    if m < 1:
        raise ValueError("%d px at rate %r resize to an empty image" % (n, rate))
    return m


def table(n_src, rate):
    """one axis: (idx int64 [n_dst, 4] clamped source taps, w int16 [n_dst, 4] weights in units of 1/2048)"""
    n_dst = dst_size(n_src, rate)
    scale = 1.0 / np.float64(rate)
    f = ((np.arange(n_dst, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f)
    f = (f - s).astype(np.float32)
    x1 = f + _ONE
    g = _ONE - f
    c0 = ((A * x1 - np.float32(5) * A) * x1 + np.float32(8) * A) * x1 - np.float32(4) * A
    c1 = ((A + np.float32(2)) * f - (A + np.float32(3))) * f * f + _ONE
    c2 = ((A + np.float32(2)) * g - (A + np.float32(3))) * g * g + _ONE
    c3 = _ONE - c0 - c1 - c2
    c = np.stack([c0, c1, c2, c3], 1).astype(np.float32)
    assert c.dtype == np.float32
    w = np.rint(c * np.float32(2048)).astype(np.int16)
    idx = np.clip(s.astype(np.int64)[:, None] + np.arange(-1, 3)[None, :], 0, n_src - 1)
    return idx, w


def resize(img, rate):
    """uint8 [H, W] or [H, W, C] -> the image resized by the fixed-point arithmetic above (rate 1 returns the input unchanged)"""
    img = np.asarray(img)
    if img.dtype != np.uint8:
        raise TypeError("uint8 image expected")
    if rate == 1:
        return img
    squeeze = img.ndim == 2
    src = img[:, :, None] if squeeze else img
    h, w, c = src.shape
    xi, xw = table(w, rate)
    yi, yw = table(h, rate)
    hor = np.zeros((h, xi.shape[0], c), np.int64)
    for j in range(4):
        hor += xw[:, j].astype(np.int64)[None, :, None] * src[:, xi[:, j], :]
    out = np.empty((yi.shape[0], xi.shape[0], c), np.uint8)
    for r0 in range(0, yi.shape[0], 512):                     # row chunks keep the int64 accumulator small
        r1 = min(r0 + 512, yi.shape[0])
        v = np.zeros((r1 - r0, xi.shape[0], c), np.int64)
        for k in range(4):
            v += yw[r0:r1, k].astype(np.int64)[:, None, None] * hor[yi[r0:r1, k]]
        out[r0:r1] = np.clip((v + (1 << 21)) >> 22, 0, 255)
    return out[:, :, 0] if squeeze else out
