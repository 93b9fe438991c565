"""Batch assembly for the encoder on the device (SURVEY.md section 8f(3)).

In the reference, ``DataGenerator.generate`` (``data_generator/object_detection_2d_data_generator.py:830``) runs the augmentation
chain per image on the host -- image ops and, for every geometric op, the matching arithmetic on the label array -- filters
degenerate boxes (``:1095-1112``) and hands the list of label arrays to ``SSDInputEncoder.__call__`` (``:1146-1151``).
Here the label half runs on the GPU: ``assemble_batch_device`` uploads the ragged labels once (one pinned copy), applies a
per-image list of box operations (``ssdk_assemble_batch``: the label arithmetic of the reference's ``CropPad`` / ``Flip`` /
``Resize`` / ``BoxFilter``, with the parameters the caller's random augmentation logic picked) and leaves the packed
``(sum G_i, 5)`` rows + ``(B+1,)`` offsets on the device, which ``SSDInputEncoder.encode_device_offsets`` consumes without a
host round trip.

The image half runs there too: ``assemble_images_device`` uploads the ragged uint8 source images once (one pinned buffer) and
``ssdk_assemble_images`` applies the same operation lists to the pixels -- ``CropPad``'s canvas, ``Flip`` and ``cv2.resize`` with
any of the five modes ``ResizeRandomInterp`` draws from -- in one fused kernel that writes the ``(B, H, W, 3)`` model input.
``augment_batch_device`` runs both halves from one list per image.

The photometric distortions, which come first in the reference's chains, run there as well: ``pixel_ops=`` takes one list of
pointwise pixel operations per image (built with ``convert_data_type`` / ``convert_color`` / ``brightness`` / ``contrast`` /
``saturation`` / ``hue`` / ``channel_swap``, or drawn like ``SSDPhotometricDistortions`` by ``ssd_photometric_distortions``),
and ``ssdk_photometric`` applies them to the uploaded sources in place before ``ssdk_assemble_images`` reads them, so canvas
backgrounds are never distorted.  Decoding stays with the caller."""
import ctypes as C

import numpy as np

from .. import _ffi


# cv2's interpolation flags (the package does not import cv2)
INTER_NEAREST, INTER_LINEAR, INTER_CUBIC, INTER_AREA, INTER_LANCZOS4 = 0, 1, 2, 3, 4


def _int32(v):
    """An unsigned 32-bit flags word as the C ``int`` it is stored in."""
    v &= 0xffffffff
    return v - (1 << 32) if v >= (1 << 31) else v


def crop_pad(patch_ymin, patch_xmin, patch_height, patch_width, center_point_filter=False, clip_boxes=True, background=(0, 0, 0)):
    """``CropPad`` (patch_sampling_ops.py:266-330).  ``SSDExpand``: negative origin, no filter, no clip, ``background=(123, 117,
    104)``; ``SSDRandomCrop``: ``center_point_filter=True, clip_boxes=True``.  ``background`` is the (R, G, B) fill of the canvas
    (``flags`` bits 8-31); it only matters to the pixels."""
    bg = tuple(int(c) for c in background)
    if len(bg) != 3 or any(c < 0 or c > 255 for c in bg):
        raise ValueError('background must be three values in 0..255')
    flags = (1 if center_point_filter else 0) | (2 if clip_boxes else 0) | (bg[0] << 8) | (bg[1] << 16) | (bg[2] << 24)
    return (_ffi.BOXOP_CROP_PAD, _int32(flags), float(patch_ymin), float(patch_xmin), float(patch_height), float(patch_width))


def flip(img_size, dim='horizontal'):
    """``Flip`` (geometric_ops.py:186,194): ``img_size`` is the image width (horizontal) or height (vertical)."""
    if dim not in ('horizontal', 'vertical'):
        raise ValueError("`dim` can be one of 'horizontal' and 'vertical'.")
    return (_ffi.BOXOP_FLIP_H if dim == 'horizontal' else _ffi.BOXOP_FLIP_V, 0, float(img_size), 0.0, 0.0, 0.0)


def resize(in_height, in_width, out_height, out_width, drop_degenerate=True, interpolation_mode=INTER_LINEAR):
    """``Resize`` (geometric_ops.py:61-100) with its degenerate-box ``BoxFilter``.  ``interpolation_mode`` is one of the
    ``INTER_*`` flags (``flags`` bits 8-15); it only matters to the pixels."""
    mode = int(interpolation_mode)
    if not 0 <= mode <= 255:
        raise ValueError('interpolation_mode must be one of INTER_NEAREST .. INTER_LANCZOS4')
    return (_ffi.BOXOP_RESIZE, (1 if drop_degenerate else 0) | (mode << 8), float(in_height), float(in_width), float(out_height),
            float(out_width))


def box_filter(check_degenerate=True, min_area=None):
    """``BoxFilter`` without the overlap test (validation_utils.py:155-165); also ``degenerate_box_handling='remove'``."""
    return (_ffi.BOXOP_FILTER, (1 if check_degenerate else 0) | (2 if min_area is not None else 0), float(min_area or 0.0), 0.0, 0.0, 0.0)


def assemble_batch_device(labels_list, ops_per_image=None):
    """``labels_list``: B arrays ``(k_i, 5)`` ``[class_id, xmin, ymin, xmax, ymax]`` (any numeric dtype, possibly empty).
    ``ops_per_image``: optional list of B lists of operations built with ``crop_pad`` / ``flip`` / ``resize`` / ``box_filter``.
    Returns ``(gt_dev (N,5) float32, offsets_dev (B+1,) int32, stats_dev int32[2] = (boxes left, largest image), total_upper,
    max_upper)`` -- CUDA tensors; the two upper bounds are host integers (box counts before filtering)."""
    import torch
    rows, offs = [], [0]
    for g in labels_list:
        g = np.asarray(g.detach().cpu().numpy() if hasattr(g, 'detach') else g, dtype=np.float64).reshape(-1, 5) if np.size(g) else np.zeros((0, 5), np.float64)
        rows.append(g)
        offs.append(offs[-1] + g.shape[0])
    B = len(rows)
    total = offs[-1]
    max_g = max([r.shape[0] for r in rows] + [0])
    flat = np.concatenate(rows, axis=0) if total else np.zeros((1, 5), np.float64)      # float64 like the reference's label arrays
    gt_in = torch.from_numpy(np.ascontiguousarray(flat)).pin_memory().cuda(non_blocking=True)
    offs_in = torch.from_numpy(np.asarray(offs, dtype=np.int32)).pin_memory().cuda(non_blocking=True)
    max_ops = max([len(o) for o in ops_per_image] + [0]) if ops_per_image else 0
    ops_dev = None
    if max_ops:
        if len(ops_per_image) != B:
            raise ValueError('ops_per_image must have one list per batch item')
        arr = (_ffi.BoxOp * (B * max_ops))()
        for b, lst in enumerate(ops_per_image):
            for i, o in enumerate(lst):
                e = arr[b * max_ops + i]
                e.op, e.flags, e.a0, e.a1, e.a2, e.a3 = o
        host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
        ops_dev = host.pin_memory().cuda(non_blocking=True)
    gt_out = torch.empty((max(total, 1), 5), dtype=torch.float32, device='cuda')
    offs_out = torch.empty((B + 1,), dtype=torch.int32, device='cuda')
    stats = torch.empty((2,), dtype=torch.int32, device='cuda')
    _ffi.check(_ffi.lib().ssdk_assemble_batch(_ffi.context(), _ffi.dptr(gt_in), 1, _ffi.dptr(offs_in), B, int(total), _ffi.dptr(ops_dev),
                                              int(max_ops), _ffi.dptr(gt_out), _ffi.dptr(offs_out), _ffi.dptr(stats), _ffi.stream_ptr()))
    return gt_out, offs_out, stats, int(total), int(max_g)


def encode_batch_device(encoder, labels_list, ops_per_image=None, out=None):
    """``label_encoder(batch_y)`` of the reference's generator (:1146-1151) without leaving the device: box operations, packing
    and ``SSDInputEncoder`` -> float32 CUDA tensor ``(B, P, C+12)``."""
    gt, offs, _, total, max_g = assemble_batch_device(labels_list, ops_per_image)
    return encoder.encode_device_offsets(gt, offs, total, max_g, out=out)


def convert_data_type(to='uint8'):
    """``ConvertDataType`` (photometric_ops.py:62-86): ``np.round(x).astype(uint8)`` or ``astype(float32)``."""
    if not (to == 'uint8' or to == 'float32'):
        raise ValueError("`to` can be either of 'uint8' or 'float32'.")
    return (_ffi.PIXOP_TO_U8 if to == 'uint8' else _ffi.PIXOP_TO_FLOAT, 0, 0.0)


def convert_color(current='RGB', to='HSV'):
    """``ConvertColor`` (photometric_ops.py:23-60) between RGB and HSV, i.e. ``cv2.cvtColor`` on a uint8 image.  Grayscale
    conversions are not supported (``NotImplementedError``); a conversion to the current space is the identity."""
    if not ((current in {'RGB', 'HSV'}) and (to in {'RGB', 'HSV', 'GRAY'})):
        raise NotImplementedError
    if to == 'GRAY':
        raise NotImplementedError('grayscale conversions are not supported on the device')
    if current == to:
        return channel_swap((0, 1, 2))
    return (_ffi.PIXOP_RGB2HSV if to == 'HSV' else _ffi.PIXOP_HSV2RGB, 0, 0.0)


def brightness(delta):
    """``Brightness`` (photometric_ops.py:225-246) on a float32 RGB image: ``clip(x + delta, 0, 255)``."""
    delta = float(delta)
    if delta != delta:
        raise ValueError('`delta` must not be NaN.')
    return (_ffi.PIXOP_BRIGHTNESS, 0, delta)


def _factor(kind, factor):
    factor = float(factor)
    if factor <= 0.0:
        raise ValueError('It must be `factor > 0`.')
    if not np.isfinite(factor):
        raise ValueError('`factor` must be finite.')
    return (kind, 0, factor)


def contrast(factor):
    """``Contrast`` (photometric_ops.py:281-304) on a float32 RGB image: ``clip(127.5 + factor * (x - 127.5), 0, 255)``."""
    return _factor(_ffi.PIXOP_CONTRAST, factor)


def saturation(factor):
    """``Saturation`` (photometric_ops.py:166-189) on a float32 HSV image: channel 1 = ``clip(x * factor, 0, 255)``."""
    return _factor(_ffi.PIXOP_SATURATION, factor)


def hue(delta):
    """``Hue`` (photometric_ops.py:110-133) on a float32 HSV image: channel 0 = ``(x + delta) % 180.0``."""
    delta = float(delta)
    if not (-180 <= delta <= 180):
        raise ValueError("`delta` must be in the closed interval `[-180, 180]`.")
    return (_ffi.PIXOP_HUE, 0, delta)


def channel_swap(order):
    """``ChannelSwap`` (photometric_ops.py:438-455): ``x[..., order]`` for three indices in 0..2."""
    order = tuple(int(i) for i in order)
    if len(order) != 3 or any(i < 0 or i > 2 for i in order):
        raise ValueError('`order` must be three channel indices in 0..2.')
    return (_ffi.PIXOP_CHANNEL_SWAP, order[0] | (order[1] << 8) | (order[2] << 16), 0.0)


# RandomChannelSwap's permutations (photometric_ops.py:470-472)
CHANNEL_SWAP_PERMUTATIONS = ((0, 2, 1), (1, 0, 2), (1, 2, 0), (2, 0, 1), (2, 1, 0))


def ssd_photometric_distortions():
    """One image's pixel-op list for ``SSDPhotometricDistortions.__call__`` (data_augmentation_chain_original_ssd.py:146-206),
    drawn from ``np.random`` with the same calls in the same order: ``choice(2)`` picks the sequence, then every ``Random*`` step
    draws ``uniform(0, 1)`` and, when it applies, its value.  Afterwards ``np.random`` is in the state the reference's call leaves
    it in.  The list always holds the uint8 HSV round trip, which the reference runs whether or not a distortion applies."""
    def maybe(prob, draw):
        p = np.random.uniform(0, 1)
        return [draw()] if p >= (1.0 - prob) else []

    def bright():
        return maybe(0.5, lambda: brightness(np.random.uniform(-32.0, 32.0)))

    def contr():
        return maybe(0.5, lambda: contrast(np.random.uniform(0.5, 1.5)))

    def hsv_part():
        return ([convert_data_type('uint8'), convert_color('RGB', 'HSV'), convert_data_type('float32')]
                + maybe(0.5, lambda: saturation(np.random.uniform(0.5, 1.5)))
                + maybe(0.5, lambda: hue(np.random.uniform(-18, 18)))
                + [convert_data_type('uint8'), convert_color('HSV', 'RGB')])

    def swap():
        return maybe(0.0, lambda: channel_swap(CHANNEL_SWAP_PERMUTATIONS[np.random.randint(5)]))

    if np.random.choice(2):
        ops = [convert_data_type('float32')] + bright()
        ops += contr()
        ops += hsv_part()
    else:
        ops = [convert_data_type('float32')] + bright()
        ops += hsv_part()
        ops += [convert_data_type('float32')] + contr() + [convert_data_type('uint8')]
    return ops + swap()


def _pixel_state(b, ops):
    """Check image b's pixel-op list like ``ssdk_photometric`` does; raise ValueError for what it refuses."""
    if len(ops) > _ffi.MAX_PIXEL_OPS:
        raise ValueError('image %d: more than %d pixel operations' % (b, _ffi.MAX_PIXEL_OPS))
    u8 = True
    for i, o in enumerate(ops):
        kind, arg, a0 = int(o[0]), int(o[1]), float(o[2])
        if kind == _ffi.PIXOP_END:
            break
        if kind == _ffi.PIXOP_TO_FLOAT:
            u8 = False
        elif kind == _ffi.PIXOP_TO_U8:
            u8 = True
        elif kind in (_ffi.PIXOP_RGB2HSV, _ffi.PIXOP_HSV2RGB):
            if not u8:
                raise ValueError('image %d, op %d: colour conversion of a float32 image (convert it to uint8 first)' % (b, i))
        elif kind in (_ffi.PIXOP_BRIGHTNESS, _ffi.PIXOP_CONTRAST, _ffi.PIXOP_SATURATION, _ffi.PIXOP_HUE):
            if u8:
                raise ValueError('image %d, op %d: photometric arithmetic on a uint8 image (convert it to float32 first)' % (b, i))
            if a0 != a0:
                raise ValueError('image %d, op %d: the parameter is NaN' % (b, i))
            if kind == _ffi.PIXOP_HUE and not -180 <= a0 <= 180:
                raise ValueError('image %d, op %d: `delta` must be in the closed interval `[-180, 180]`.' % (b, i))
            if kind in (_ffi.PIXOP_CONTRAST, _ffi.PIXOP_SATURATION) and not (a0 > 0.0 and np.isfinite(a0)):
                raise ValueError('image %d, op %d: It must be `factor > 0`.' % (b, i))
        elif kind == _ffi.PIXOP_CHANNEL_SWAP:
            if arg < 0 or arg >> 24 or any(((arg >> s) & 255) > 2 for s in (0, 8, 16)):
                raise ValueError('image %d, op %d: channel order %#x has an index outside 0..2' % (b, i, arg))
        else:
            raise ValueError('image %d: unknown pixel operation %d' % (b, kind))
    if not u8:
        raise ValueError('image %d: the pixel operations end in float32 state (end them with convert_data_type(\'uint8\'))' % b)


def _pack_pixel_ops(pixel_ops, B):
    max_ops = max([len(o) for o in pixel_ops] + [0])
    arr = (_ffi.PixelOp * max(B * max_ops, 1))()
    for b, lst in enumerate(pixel_ops):
        for i, o in enumerate(lst):
            e = arr[b * max_ops + i]
            e.op, e.arg, e.a0 = int(o[0]), int(o[1]), float(o[2])
    return bytes(arr)[:B * max_ops * C.sizeof(_ffi.PixelOp)], max_ops


def _image_extents(b, h, w, ops):
    """Walk image b's op list like ``ssdk_assemble_images`` does; raise ValueError for what it refuses.  Returns the final size."""
    resized = False
    for o in ops:
        kind = int(o[0])
        if kind == _ffi.BOXOP_END:
            break
        if kind == _ffi.BOXOP_CROP_PAD:
            if resized:
                raise ValueError('image %d: crop/pad after the resize' % b)
            if any(float(v) != int(v) for v in o[2:]):
                raise ValueError('image %d: crop/pad parameters must be integers' % b)
            if o[2] > h or o[3] > w:
                raise ValueError("image %d: The given patch doesn't overlap with the input image." % b)
            if o[4] <= 0 or o[5] <= 0:
                raise ValueError('image %d: empty patch' % b)
            h, w = int(o[4]), int(o[5])
        elif kind in (_ffi.BOXOP_FLIP_H, _ffi.BOXOP_FLIP_V):
            if resized:
                raise ValueError('image %d: flip after the resize' % b)
            if o[2] != (w if kind == _ffi.BOXOP_FLIP_H else h):
                raise ValueError('image %d: flip size %g is not the image size (%d x %d)' % (b, o[2], h, w))
        elif kind == _ffi.BOXOP_RESIZE:
            if resized:
                raise ValueError('image %d: more than one resize' % b)
            mode = (int(o[1]) >> 8) & 255
            if mode > INTER_LANCZOS4:
                raise ValueError('image %d: interpolation mode %d is not one of INTER_NEAREST .. INTER_LANCZOS4' % (b, mode))
            if (o[2], o[3]) != (h, w):
                raise ValueError('image %d: resize input %g x %g is not the image size %d x %d' % (b, o[2], o[3], h, w))
            if float(o[4]) != int(o[4]) or float(o[5]) != int(o[5]) or o[4] <= 0 or o[5] <= 0:
                raise ValueError('image %d: bad resize target' % b)
            h, w = int(o[4]), int(o[5])
            resized = True
        elif kind != _ffi.BOXOP_FILTER:
            raise ValueError('image %d: unknown operation %d' % (b, kind))
    return h, w


def _pack_ops(ops_per_image, B):
    max_ops = max([len(o) for o in ops_per_image] + [0]) if ops_per_image else 0
    if max_ops and len(ops_per_image) != B:
        raise ValueError('ops_per_image must have one list per batch item')
    arr = (_ffi.BoxOp * max(B * max_ops, 1))()
    for b, lst in enumerate(ops_per_image or []):
        for i, o in enumerate(lst):
            e = arr[b * max_ops + i]
            e.op, e.flags, e.a0, e.a1, e.a2, e.a3 = o
    return bytes(arr)[:B * max_ops * C.sizeof(_ffi.BoxOp)], max_ops


def assemble_images_device(images, ops_per_image, height, width, dtype=None, out=None, pixel_ops=None):
    """The image half of the augmentation chain on the device.  ``images``: B uint8 ``(h_i, w_i, 3)`` arrays;
    ``ops_per_image``: B op lists built with ``crop_pad`` / ``flip`` / ``resize`` / ``box_filter`` (``box_filter`` does not touch
    pixels), each ending at ``(height, width)``.  ``pixel_ops``: optional B lists of photometric pixel operations (see
    ``ssd_photometric_distortions``), applied to the sources before the geometric operations, in one extra launch.  Returns a
    CUDA tensor ``(B, height, width, 3)`` in ``dtype`` (``torch.float32``, the model input, or ``torch.uint8``), written into
    ``out`` if given.  Validation errors are raised as ValueError before anything is uploaded or launched."""
    import torch
    dtype = torch.float32 if dtype is None else dtype
    if dtype not in (torch.float32, torch.uint8):
        raise ValueError('dtype must be torch.float32 or torch.uint8')
    height, width = int(height), int(width)
    if height <= 0 or width <= 0:
        raise ValueError('height and width must be positive')
    arrs = []
    for b, im in enumerate(images):
        a = im.detach().cpu().numpy() if hasattr(im, 'detach') else np.asarray(im)
        if a.dtype != np.uint8:
            raise ValueError('image %d: expected uint8, got %s' % (b, a.dtype))
        if a.ndim != 3 or a.shape[2] != 3:
            raise ValueError('image %d: expected an (h, w, 3) image, got shape %s' % (b, a.shape))
        if a.shape[0] == 0 or a.shape[1] == 0:
            raise ValueError('image %d is empty' % b)
        arrs.append(np.ascontiguousarray(a))
    B = len(arrs)
    if B == 0:
        raise ValueError('no images')
    if ops_per_image is not None and len(ops_per_image) != B:
        raise ValueError('ops_per_image must have one list per batch item')
    for b, a in enumerate(arrs):
        hw = _image_extents(b, a.shape[0], a.shape[1], ops_per_image[b] if ops_per_image is not None else [])
        if hw != (height, width):
            raise ValueError('image %d ends at %d x %d, the batch is %d x %d' % (b, hw[0], hw[1], height, width))
    if pixel_ops is not None:
        if len(pixel_ops) != B:
            raise ValueError('pixel_ops must have one list per batch item')
        for b, lst in enumerate(pixel_ops):
            _pixel_state(b, lst)
    if out is not None and (not out.is_cuda or out.dtype != dtype or tuple(out.shape) != (B, height, width, 3) or not out.is_contiguous()):
        raise ValueError('out must be a contiguous CUDA tensor (%d, %d, %d, 3) of %s' % (B, height, width, dtype))
    ops_bytes, max_ops = _pack_ops(ops_per_image, B)
    # one pinned buffer: [ops | offsets int64 | sizes int32 | pixels], each section 256-byte aligned
    offs = np.cumsum([0] + [a.size for a in arrs[:-1]]).astype(np.int64)
    hw = np.asarray([a.shape[:2] for a in arrs], np.int32).reshape(-1)
    al = lambda n: (n + 255) // 256 * 256                                                       # noqa: E731
    o_offs = al(len(ops_bytes))
    o_hw = o_offs + al(offs.nbytes)
    o_pix = o_hw + al(hw.nbytes)
    total = o_pix + int(sum(a.size for a in arrs))
    if pixel_ops is not None:                                                                   # [... | pixels | pixel ops]
        px_bytes, px_max_ops = _pack_pixel_ops(pixel_ops, B)
        o_px_ops = al(total)
        total = o_px_ops + len(px_bytes)
    host = torch.empty((total,), dtype=torch.uint8, pin_memory=True)
    hv = host.numpy()
    hv[:len(ops_bytes)] = np.frombuffer(ops_bytes, np.uint8)
    hv[o_offs:o_offs + offs.nbytes] = offs.view(np.uint8)
    hv[o_hw:o_hw + hw.nbytes] = hw.view(np.uint8)
    pos = o_pix
    for a in arrs:
        hv[pos:pos + a.size] = a.reshape(-1)
        pos += a.size
    if pixel_ops is not None:
        hv[o_px_ops:o_px_ops + len(px_bytes)] = np.frombuffer(px_bytes, np.uint8)
    dev = host.cuda(non_blocking=True)
    base = dev.data_ptr()
    if out is None:
        out = torch.empty((B, height, width, 3), dtype=dtype, device='cuda')
    if pixel_ops is not None:                                                  # in place on this call's own copy of the sources
        _ffi.check(_ffi.lib().ssdk_photometric(_ffi.context(), C.c_void_p(base + o_pix), C.c_void_p(base + o_pix), C.c_void_p(base + o_offs),
                                               C.c_void_p(base + o_hw), B, C.c_void_p(base + o_px_ops) if px_max_ops else C.c_void_p(0),
                                               int(px_max_ops), _ffi.stream_ptr()))
    _ffi.check(_ffi.lib().ssdk_assemble_images(_ffi.context(), C.c_void_p(base + o_pix), C.c_void_p(base + o_offs), C.c_void_p(base + o_hw), B,
                                               C.c_void_p(base + 0) if max_ops else C.c_void_p(0), int(max_ops), height, width,
                                               0 if dtype == torch.float32 else 1, _ffi.dptr(out), _ffi.stream_ptr()))
    return out


def augment_batch_device(images, labels_list, ops_per_image, height, width, pixel_ops=None):
    """``SSDDataAugmentation`` for a batch, pixels and boxes from ONE op list per image (plus, optionally, one photometric
    ``pixel_ops`` list per image, which only touches pixels): returns ``(images (B, height, width, 3) float32, (gt_dev,
    offsets_dev, stats_dev, total_upper, max_upper))``, the second part being what ``assemble_batch_device`` returns (feed it to
    ``SSDInputEncoder.encode_device_offsets``)."""
    imgs = assemble_images_device(images, ops_per_image, height, width, pixel_ops=pixel_ops)
    return imgs, assemble_batch_device(labels_list, ops_per_image)
