"""Photometric pixel operations (oracle, NumPy).

Restates, in the reference's float32 order, what ``ssdk_photometric`` computes for each ``ssdk_pixel_op``:
  * ``ConvertDataType``  data_generator/object_detection_2d_photometric_ops.py:62-86 (``np.round`` half to even, then uint8)
  * ``ConvertColor``     :23-60, i.e. ``cv2.cvtColor`` on uint8 between RGB and HSV, restated from OpenCV's 8-bit arithmetic
  * ``Hue`` :110-133, ``Saturation`` :166-189, ``Brightness`` :225-246, ``Contrast`` :281-304 on float32 images, the Python-float
    parameter rounded to float32 first (NumPy 2 / NEP 50)
  * ``ChannelSwap``      :438-455

The colour conversions are vectorised so that their whole domains (2^24 RGB colours, 181 x 256 x 256 HSV triples) run in a few
seconds; tests/golden/make_photometric_golden.py stores ``cv2.cvtColor``'s digests over those domains.  ``cv2`` itself is never
imported here.

Operations are the ``(op, arg, a0)`` tuples of ``ssd_keras_b200.data_generator.batch_assembly``; see ``include/ssdk.h``.
"""
import numpy as np

END, TO_FLOAT, TO_U8, RGB2HSV, HSV2RGB, BRIGHTNESS, CONTRAST, SATURATION, HUE, CHANNEL_SWAP = range(10)
HSV_SHIFT = 12
_f32 = np.float32


def _hsv_tables():
    """OpenCV's RGB2HSV_b division tables: cvRound((255 << 12) / i) and cvRound((180 << 12) / (6 i))."""
    i = np.arange(1, 256, dtype=np.float64)
    sdiv = np.zeros(256, np.int64)
    hdiv = np.zeros(256, np.int64)
    sdiv[1:] = np.rint((255 << HSV_SHIFT) / i)
    hdiv[1:] = np.rint((180 << HSV_SHIFT) / (6.0 * i))
    return sdiv, hdiv


_SDIV, _HDIV = _hsv_tables()


def rgb2hsv(img):
    """``cv2.cvtColor(img, cv2.COLOR_RGB2HSV)`` on uint8: OpenCV's integer path (hsv_shift = 12, hue range 180)."""
    r, g, b = (img[..., c].astype(np.int64) for c in range(3))
    v = np.maximum(np.maximum(b, g), r)
    diff = v - np.minimum(np.minimum(b, g), r)
    s = (diff * _SDIV[v] + (1 << (HSV_SHIFT - 1))) >> HSV_SHIFT
    h = np.where(v == r, g - b, np.where(v == g, b - r + 2 * diff, r - g + 4 * diff))
    h = (h * _HDIV[diff] + (1 << (HSV_SHIFT - 1))) >> HSV_SHIFT
    h = np.where(h < 0, h + 180, h)
    return np.stack([h, s, v], -1).astype(np.uint8)


def _fma_f32(a, b, c):
    """float32 fused multiply-add.  The float64 product of two float32 values is exact; the sum is rounded twice (float64, then
    float32), which over the HSV domain never differs from one rounding (the full-domain digest pins it)."""
    return (a.astype(np.float64) * b.astype(np.float64) + np.float64(c)).astype(_f32)


# OpenCV's sector_data: (b, g, r) indices into (v, p, q, t) per hue sector
_SECTOR = np.array([[1, 3, 0], [1, 0, 2], [3, 0, 1], [0, 2, 1], [0, 1, 3], [2, 1, 0]])


# OpenCV 4.13's optimised (AVX2) HSV2RGB_b converts 32 pixels per vector iteration; the last (width mod 32) pixels of a row
# take its scalar code, which rounds where the vector code truncates.
CV_VEC_PIXELS = 32


def hsv2rgb(img, optimized=True):
    """``cv2.cvtColor(img, cv2.COLOR_HSV2RGB)`` on a uint8 ``(h, w, 3)`` image (OpenCV's HSV2RGB_b): h * (6 / 180), s / 255,
    v / 255 in float32, the hue sector table, the result * 255.  The default (optimised) build fuses 1 - s*h and 1 - s*(1 - h)
    into one multiply-add each; on whole 32-pixel vectors of a row it truncates the result, on the last (w mod 32) pixels it
    rounds to nearest even.  ``optimized=False`` restates the whole-vector arithmetic of its portable path
    (``cv2.setUseOptimized(False)``): no multiply-add, truncation.  Over all 181 x 256 x 256 triples with H <= 180 in whole
    vectors the two differ by 1 in one channel on 1758 triples."""
    H = img[..., 0].astype(_f32)
    s = img[..., 1].astype(_f32) * _f32(1.0 / 255.0)
    v = img[..., 2].astype(_f32) * _f32(1.0 / 255.0)
    h = np.fmod(H * (_f32(6.0) / _f32(180.0)), _f32(6.0))
    sector = np.floor(h).astype(np.int64)
    h = (h - sector.astype(_f32)).astype(_f32)
    wrap = (sector < 0) | (sector >= 6)
    sector = np.where(wrap, 0, sector)
    h = np.where(wrap, _f32(0), h).astype(_f32)
    one = _f32(1.0)
    if optimized:
        q, t = v * _fma_f32(-s, h, one), v * _fma_f32(-s, one - h, one)
    else:
        q, t = v * (one - s * h), v * (one - s * (one - h))
    tab = np.stack([v, v * (one - s), q, t], -1)
    bgr = np.take_along_axis(tab, _SECTOR[sector], -1) * _f32(255.0)
    out = np.trunc(bgr)
    if optimized:
        w = img.shape[-2]
        tail = np.arange(w) >= w // CV_VEC_PIXELS * CV_VEC_PIXELS
        out = np.where(tail[:, None], np.rint(bgr), out)
    return np.clip(out, 0, 255)[..., ::-1].astype(np.uint8)


def apply(image, ops, optimized=True):
    """One uint8 ``(h, w, 3)`` image through a pixel-op list; returns uint8.  The list is assumed valid (see
    ``batch_assembly._pixel_state``): float32 arithmetic only in float32 state, colour conversions only in uint8 state."""
    x = np.asarray(image)
    for o in ops:
        kind, arg, a0 = int(o[0]), int(o[1]), float(o[2])
        if kind == END:
            break
        if kind == TO_FLOAT:
            x = x.astype(_f32)
        elif kind == TO_U8:
            x = np.round(x, decimals=0).astype(np.uint8)
        elif kind == RGB2HSV:
            x = rgb2hsv(x)
        elif kind == HSV2RGB:
            x = hsv2rgb(x, optimized)
        elif kind == BRIGHTNESS:
            x = np.clip(x + _f32(a0), 0, 255)
        elif kind == CONTRAST:
            x = np.clip(_f32(127.5) + _f32(a0) * (x - _f32(127.5)), 0, 255)
        elif kind == SATURATION:
            x = x.copy()
            x[..., 1] = np.clip(x[..., 1] * _f32(a0), 0, 255)
        elif kind == HUE:
            x = x.copy()
            x[..., 0] = np.remainder(x[..., 0] + _f32(a0), _f32(180.0))
        elif kind == CHANNEL_SWAP:
            x = x[..., [arg & 255, (arg >> 8) & 255, (arg >> 16) & 255]]
        else:
            raise ValueError('unknown pixel operation %d' % kind)
    assert x.dtype == np.uint8, 'the list must end in uint8 state'
    return np.ascontiguousarray(x)


def apply_images(images, pixel_ops, optimized=True):
    return [apply(im, ops, optimized) for im, ops in zip(images, pixel_ops)]


def rgb_domain():
    """All 2^24 RGB colours as one 4096 x 4096 image: pixel i is (i >> 16, (i >> 8) & 255, i & 255)."""
    i = np.arange(1 << 24, dtype=np.uint32)
    return np.stack([i >> 16, (i >> 8) & 255, i & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)


def hsv_domain():
    """All 181 x 256 x 256 HSV triples with H <= 180 as one 2896 x 4096 image: pixel i is (i >> 16, (i >> 8) & 255, i & 255)."""
    i = np.arange(181 << 16, dtype=np.uint32)
    return np.stack([i >> 16, (i >> 8) & 255, i & 255], -1).astype(np.uint8).reshape(2896, 4096, 3)
