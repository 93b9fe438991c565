"""Image half of the geometric augmentation ops (oracle, NumPy).

Restates the pixel arithmetic of
  * ``CropPad.__call__``  data_generator/object_detection_2d_patch_sampling_ops.py:266-313 (``SSDExpand`` / ``SSDRandomCrop``)
  * ``Flip.__call__``     data_generator/object_detection_2d_geometric_ops.py:171-195
  * ``Resize.__call__``   data_generator/object_detection_2d_geometric_ops.py:61-72, i.e. ``cv2.resize`` on 3-channel uint8 for
                          INTER_NEAREST, INTER_LINEAR, INTER_CUBIC, INTER_AREA and INTER_LANCZOS4 (what ``ResizeRandomInterp``
                          draws from, data_augmentation_chain_original_ssd.py:258-266)
as one fused map, the way ``ssdk_assemble_images`` computes it: the resize taps are computed in the frame of the image that
enters the resize, clamped there like OpenCV clamps them, and mapped back through the crop/pad and flip operations in reverse
order; a tap that leaves the input of a crop/pad operation takes that operation's background.

The interpolation rules are OpenCV's fixed-point / float arithmetic for 8-bit images, stated element by element, and pinned bit
for bit to ``cv2.resize`` outputs (tests/golden/make_image_golden.py).  ``cv2`` itself is never imported here.

Operations are the tuples of ``ssd_keras_b200.data_generator.batch_assembly`` (``op, flags, a0, a1, a2, a3``); see
``include/ssdk.h`` for the encoding.
"""
import math

import numpy as np

END, CROP_PAD, FLIP_H, FLIP_V, RESIZE, FILTER = 0, 1, 2, 3, 4, 5
INTER_NEAREST, INTER_LINEAR, INTER_CUBIC, INTER_AREA, INTER_LANCZOS4 = 0, 1, 2, 3, 4
COEF_BITS = 11
COEF_SCALE = 1 << COEF_BITS
# INTER_CUBIC's vertical pass runs in float32 on whole 8-lane vectors of a row (OpenCV's VResizeCubicVec_32s8u); the last
# (row length mod 8) values of a row take the integer form.
CUBIC_VEC_LANES = 8

_f32 = np.float32


def background_rgb(flags):
    """Background colour of a CROP_PAD operation: ``flags`` bits 8-15 R, 16-23 G, 24-31 B."""
    f = int(flags) & 0xffffffff
    return ((f >> 8) & 255, (f >> 16) & 255, (f >> 24) & 255)


def resize_mode(flags):
    return (int(flags) >> 8) & 255


def _floor_f32(v):
    return int(math.floor(float(v)))


# ------------------------------------------------------------------------------------------------------------------------------
# Per-axis taps (OpenCV resize.cpp, cv::resize / resizeGeneric): index of the first tap, float32 fraction
# ------------------------------------------------------------------------------------------------------------------------------

def _cubic_coeffs(x):
    """interpolateCubic, A = -0.75, float32 without contraction."""
    A = _f32(-0.75)
    x = _f32(x)
    one = _f32(1)
    xp1 = x + one
    c0 = ((A * xp1 - _f32(5) * A) * xp1 + _f32(8) * A) * xp1 - _f32(4) * A
    c1 = ((A + _f32(2)) * x - (A + _f32(3))) * x * x + one
    omx = one - x
    c2 = ((A + _f32(2)) * omx - (A + _f32(3))) * omx * omx + one
    c3 = one - c0 - c1 - c2
    return [c0, c1, c2, c3]


_S45 = 0.70710678118654752440084436210485
_CS = ((1, 0), (-_S45, -_S45), (0, 1), (_S45, -_S45), (-1, 0), (_S45, _S45), (0, -1), (-_S45, _S45))


def _lanczos4_coeffs(x):
    """interpolateLanczos4: sin / cos in double, coefficients in float32, normalised by the float32 reciprocal of their sum."""
    x = _f32(x)
    y0 = -float(_f32(x + _f32(3))) * math.pi * 0.25
    s0, c0 = math.sin(y0), math.cos(y0)
    coeffs, total = [], _f32(0)
    for i in range(8):
        y0_ = _f32(_f32(x + _f32(3)) - _f32(i))
        if abs(y0_) >= _f32(1e-6):
            y = -float(y0_) * math.pi * 0.25
            c = _f32((_CS[i][0] * s0 + _CS[i][1] * c0) / (y * y))
        else:
            c = _f32(1e30)
        coeffs.append(c)
        total = _f32(total + c)
    inv = _f32(_f32(1) / total)
    return [_f32(c * inv) for c in coeffs]


def _fixed(c):
    """saturate_cast<short>(c * INTER_RESIZE_COEF_SCALE): float32 product, round half to even."""
    v = float(_f32(_f32(c) * _f32(COEF_SCALE)))
    return int(max(-32768, min(32767, np.rint(v))))


def axis_taps(n_in, n_out, mode):
    """Taps of one axis for the fixed-point modes.  Returns (idx (n_out, K) int64, clamped to [0, n_in-1]; coef (n_out, K) int64).
    INTER_AREA here is OpenCV's up-scaling form (linear taps with area fractions); the down-scaling forms are separate."""
    inv_scale = n_out / n_in
    scale = 1.0 / inv_scale
    K = {INTER_LINEAR: 2, INTER_AREA: 2, INTER_CUBIC: 4, INTER_LANCZOS4: 8}[mode]
    idx = np.zeros((n_out, K), np.int64)
    coef = np.zeros((n_out, K), np.int64)
    for d in range(n_out):
        if mode == INTER_AREA:
            s = int(math.floor(d * scale))
            f = _f32((d + 1) - (s + 1) * inv_scale)
            f = _f32(0) if f <= 0 else _f32(f - _f32(math.floor(f)))
        else:
            f = _f32((d + 0.5) * scale - 0.5)
            s = _floor_f32(f)
            f = _f32(f - _f32(s))
        if mode in (INTER_LINEAR, INTER_AREA):
            if s < 0:
                s, f = 0, _f32(0)
            if s >= n_in - 1:
                s, f = n_in - 1, _f32(0)
            cb = [_f32(1) - f, f]
        elif mode == INTER_CUBIC:
            cb = _cubic_coeffs(f)
        else:
            cb = _lanczos4_coeffs(f)
        first = s - (K // 2 - 1)
        for k in range(K):
            idx[d, k] = min(max(first + k, 0), n_in - 1)
            coef[d, k] = _fixed(cb[k])
    return idx, coef


def axis_taps_linear_rows(n_in, n_out, mode):
    """The vertical axis of INTER_LINEAR / INTER_AREA(up): OpenCV takes the row fraction WITHOUT the border reset of the
    horizontal axis; the two rows are clamp(sy) and clamp(sy + 1)."""
    inv_scale = n_out / n_in
    scale = 1.0 / inv_scale
    idx = np.zeros((n_out, 2), np.int64)
    coef = np.zeros((n_out, 2), np.int64)
    for d in range(n_out):
        if mode == INTER_AREA:
            s = int(math.floor(d * scale))
            f = _f32((d + 1) - (s + 1) * inv_scale)
            f = _f32(0) if f <= 0 else _f32(f - _f32(math.floor(f)))
        else:
            f = _f32((d + 0.5) * scale - 0.5)
            s = _floor_f32(f)
            f = _f32(f - _f32(s))
        idx[d] = (min(max(s, 0), n_in - 1), min(max(s + 1, 0), n_in - 1))
        c0 = _fixed(_f32(1) - f)
        coef[d] = (c0, COEF_SCALE - c0)
    return idx, coef


def area_tab(n_in, n_out):
    """computeResizeAreaTab: for every output index the (source index, float32 weight) list in OpenCV's order."""
    scale = 1.0 / (n_out / n_in)
    tab = []
    for d in range(n_out):
        fs1 = d * scale
        fs2 = fs1 + scale
        cell = min(scale, n_in - fs1)
        s1, s2 = int(math.ceil(fs1)), int(math.floor(fs2))
        s2 = min(s2, n_in - 1)
        s1 = min(s1, s2)
        row = []
        if s1 - fs1 > 1e-3:
            row.append((s1 - 1, _f32((s1 - fs1) / cell)))
        for s in range(s1, s2):
            row.append((s, _f32(1.0 / cell)))
        if fs2 - s2 > 1e-3:
            row.append((s2, _f32(min(min(fs2 - s2, 1.0), cell) / cell)))
        tab.append(row)
    return tab


def resize_kind(in_h, in_w, out_h, out_w, mode):
    """Which of OpenCV's code paths cv::resize takes: 'copy', 'nearest', 'fixed' (separable fixed point), 'area_fast'
    (integer ratio), 'area' (float weights)."""
    if (in_h, in_w) == (out_h, out_w):
        return 'copy'
    if mode == INTER_NEAREST:
        return 'nearest'
    sx, sy = 1.0 / (out_w / in_w), 1.0 / (out_h / in_h)
    isx, isy = int(round(sx)), int(round(sy))
    fast = abs(sx - isx) < np.finfo(np.float64).eps and abs(sy - isy) < np.finfo(np.float64).eps
    if mode == INTER_LINEAR and fast and isx == 2 and isy == 2:
        return 'area_fast'
    if mode == INTER_AREA and sx >= 1 and sy >= 1:
        return 'area_fast' if fast else 'area'
    return 'fixed'


# ------------------------------------------------------------------------------------------------------------------------------
# Resize of an image given as a gather function (rows, cols) -> uint8 (..., 3): the fused map reads through it
# ------------------------------------------------------------------------------------------------------------------------------

def _resize(read, in_h, in_w, out_h, out_w, mode):
    kind = resize_kind(in_h, in_w, out_h, out_w, mode)
    ys, xs = np.arange(out_h), np.arange(out_w)
    if kind == 'copy':
        return read(ys[:, None], xs[None, :])
    if kind == 'nearest':
        sx = np.minimum(np.floor(xs * (1.0 / (out_w / in_w))).astype(np.int64), in_w - 1)
        sy = np.minimum(np.floor(ys * (1.0 / (out_h / in_h))).astype(np.int64), in_h - 1)
        return read(sy[:, None], sx[None, :])
    if kind == 'area_fast':
        fx, fy = int(round(1.0 / (out_w / in_w))), int(round(1.0 / (out_h / in_h)))
        total = np.zeros((out_h, out_w, 3), np.int64)
        for j in range(fy):
            for i in range(fx):
                total += read((ys * fy + j)[:, None], (xs * fx + i)[None, :]).astype(np.int64)
        if fx == 2 and fy == 2:                          # the 2x2 kernel: rounds half up
            return ((total + 2) >> 2).astype(np.uint8)
        v = total.astype(np.float32) * _f32(_f32(1) / _f32(fx * fy))
        return np.clip(np.rint(v), 0, 255).astype(np.uint8)
    if kind == 'area':
        xt, yt = area_tab(in_w, out_w), area_tab(in_h, out_h)
        out = np.zeros((out_h, out_w, 3), np.uint8)
        kx = max(len(r) for r in xt)
        xi = np.array([[r[min(k, len(r) - 1)][0] for k in range(kx)] for r in xt], np.int64)
        xw = np.array([[r[k][1] if k < len(r) else 0 for k in range(kx)] for r in xt], np.float32)
        for dy in range(out_h):
            acc = None
            for sy, beta in yt[dy]:
                row = read(np.full((out_w, kx), sy, np.int64), xi).astype(np.float32)      # (out_w, kx, 3)
                buf = np.zeros((out_w, 3), np.float32)
                for k in range(kx):
                    buf = np.where((xw[:, k] != 0)[:, None], buf + row[:, k] * xw[:, k, None], buf).astype(np.float32)
                acc = (beta * buf).astype(np.float32) if acc is None else (acc + buf * beta).astype(np.float32)
            out[dy] = np.clip(np.rint(acc), 0, 255).astype(np.uint8)
        return out
    # separable fixed point
    xi, xa = axis_taps(in_w, out_w, mode)
    if mode in (INTER_LINEAR, INTER_AREA):
        yi, yb = axis_taps_linear_rows(in_h, out_h, mode)
    else:
        yi, yb = axis_taps(in_h, out_h, mode)
    K = xi.shape[1]
    # h[k] = horizontal pass of row tap k: (out_h, out_w, 3) int64
    h = []
    for k in range(K):
        acc = np.zeros((out_h, out_w, 3), np.int64)
        for t in range(K):
            acc += read(yi[:, k][:, None], xi[:, t][None, :]).astype(np.int64) * xa[None, :, t, None]
        h.append(acc)
    b = [yb[:, k][:, None, None] for k in range(K)]
    if mode in (INTER_LINEAR, INTER_AREA):
        v = (((b[0] * (h[0] >> 4)) >> 16) + ((b[1] * (h[1] >> 4)) >> 16) + 2) >> 2
        return np.clip(v, 0, 255).astype(np.uint8)
    iv = sum(b[k] * h[k] for k in range(K))
    iv = (iv + (1 << (2 * COEF_BITS - 1))) >> (2 * COEF_BITS)
    if mode == INTER_LANCZOS4:
        return np.clip(iv, 0, 255).astype(np.uint8)
    # INTER_CUBIC: float32 vertical pass  round(h0*b0 + (h1*b1 + (h2*b2 + h3*b3))), b_k = beta_k * 2^-22 in float32
    scl = _f32(1.0 / (COEF_SCALE * COEF_SCALE))
    bf = [(yb[:, k].astype(np.float32) * scl)[:, None, None] for k in range(K)]
    hf = [x.astype(np.float32) for x in h]
    fv = hf[3] * bf[3]
    fv = (hf[2] * bf[2]).astype(np.float32) + fv
    fv = (hf[1] * bf[1]).astype(np.float32) + fv
    fv = (hf[0] * bf[0]).astype(np.float32) + fv
    fv = np.clip(np.rint(fv), -32768, 32767)
    fv = np.clip(fv, 0, 255).astype(np.int64)
    row_len = out_w * 3
    vec_end = row_len // CUBIC_VEC_LANES * CUBIC_VEC_LANES
    pos = (np.arange(out_w)[:, None] * 3 + np.arange(3)[None, :])[None]
    return np.where(pos < vec_end, fv, np.clip(iv, 0, 255)).astype(np.uint8)


def resize(image, out_h, out_w, mode=INTER_LINEAR):
    """``cv2.resize(image, (out_w, out_h), interpolation=mode)`` for a uint8 (h, w, 3) image."""
    image = np.asarray(image, np.uint8)
    h, w = image.shape[:2]
    return _resize(lambda r, c: image[r, c], h, w, int(out_h), int(out_w), int(mode))


# ------------------------------------------------------------------------------------------------------------------------------
# The fused map
# ------------------------------------------------------------------------------------------------------------------------------

def image_extents(src_hw, ops):
    """Walk an op list: [(h, w) of the image entering op i for every op] + [final (h, w)].  Raises ValueError for what
    ``ssdk_assemble_images`` refuses."""
    h, w = int(src_hw[0]), int(src_hw[1])
    if h <= 0 or w <= 0:
        raise ValueError('empty source image')
    ext, resized = [], False
    for o in ops:
        kind = int(o[0])
        if kind == END:
            break
        ext.append((h, w))
        if kind == CROP_PAD:
            if resized:
                raise ValueError('crop/pad after the resize')
            py, px, ph, pw = int(o[2]), int(o[3]), int(o[4]), int(o[5])
            if py > h or px > w:
                raise ValueError("The given patch doesn't overlap with the input image.")
            if ph <= 0 or pw <= 0:
                raise ValueError('empty patch')
            h, w = ph, pw
        elif kind in (FLIP_H, FLIP_V):
            if resized:
                raise ValueError('flip after the resize')
        elif kind == RESIZE:
            if resized:
                raise ValueError('more than one resize')
            if resize_mode(o[1]) > INTER_LANCZOS4:
                raise ValueError('interpolation mode %d is not one of 0..4' % resize_mode(o[1]))
            resized = True
            h, w = int(o[4]), int(o[5])
            if h <= 0 or w <= 0:
                raise ValueError('empty resize target')
    ext.append((h, w))
    return ext


def assemble_image(src, ops, out_h, out_w):
    """One image through its op list -> uint8 (out_h, out_w, 3).  The fused map of ``ssdk_assemble_images``."""
    src = np.asarray(src, np.uint8)
    ops = [o for o in ops]
    ops = ops[:next((i for i, o in enumerate(ops) if int(o[0]) == END), len(ops))]
    ext = image_extents(src.shape[:2], ops)
    if ext[-1] != (int(out_h), int(out_w)):
        raise ValueError('final image size %s differs from (%d, %d)' % (ext[-1], out_h, out_w))
    r = next((i for i, o in enumerate(ops) if int(o[0]) == RESIZE), len(ops))

    def read(rows, cols):
        """Pixels of the image that enters op r at (rows, cols) (broadcast), walking ops r-1 .. 0 in reverse."""
        rows, cols = np.broadcast_arrays(np.asarray(rows, np.int64), np.asarray(cols, np.int64))
        rows, cols = rows.copy(), cols.copy()
        bg = np.full(rows.shape, -1, np.int64)          # index of the op whose background a pixel takes, -1 = source
        for i in range(r - 1, -1, -1):
            o = ops[i]
            kind = int(o[0])
            h, w = ext[i]
            if kind == FLIP_H:
                cols = w - 1 - cols
            elif kind == FLIP_V:
                rows = h - 1 - rows
            elif kind == CROP_PAD:
                rows = rows + int(o[2])
                cols = cols + int(o[3])
                outside = (rows < 0) | (rows >= h) | (cols < 0) | (cols >= w)
                bg = np.where((bg < 0) & outside, i, bg)
        inside = bg < 0
        out = np.zeros(rows.shape + (3,), np.uint8)
        out[inside] = src[np.clip(rows, 0, src.shape[0] - 1), np.clip(cols, 0, src.shape[1] - 1)][inside]
        for i in np.unique(bg[~inside]):
            out[bg == i] = np.array(background_rgb(ops[i][1]), np.uint8)
        return out

    if r == len(ops):
        h, w = ext[-1]
        return read(np.arange(h)[:, None], np.arange(w)[None, :])
    o = ops[r]
    h, w = ext[r]
    return _resize(read, h, w, int(o[4]), int(o[5]), resize_mode(o[1]))


def assemble_images(images, ops_per_image, out_h, out_w, dtype=np.float32):
    """B images -> (B, out_h, out_w, 3) in ``dtype`` (float32 holds the uint8 values)."""
    return np.stack([assemble_image(im, ops, out_h, out_w) for im, ops in zip(images, ops_per_image)]).astype(dtype)
