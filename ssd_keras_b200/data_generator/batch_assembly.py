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
``augment_batch_device`` runs both halves from one list per image.  Decoding and photometric distortions stay with the caller:
they come first in the reference's chain, so the images handed in are what enters ``SSDExpand``."""
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


def assemble_images_device(images, ops_per_image, height, width, dtype=None, out=None):
    """The image half of the augmentation chain on the device.  ``images``: B uint8 ``(h_i, w_i, 3)`` arrays (the photometric
    distortions already applied); ``ops_per_image``: B op lists built with ``crop_pad`` / ``flip`` / ``resize`` / ``box_filter``
    (``box_filter`` does not touch pixels), each ending at ``(height, width)``.  Returns a CUDA tensor ``(B, height, width, 3)``
    in ``dtype`` (``torch.float32``, the model input, or ``torch.uint8``), written into ``out`` if given.  Validation errors
    are raised as ValueError before anything is uploaded or launched."""
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
    host = torch.empty((total,), dtype=torch.uint8, pin_memory=True)
    hv = host.numpy()
    hv[:len(ops_bytes)] = np.frombuffer(ops_bytes, np.uint8)
    hv[o_offs:o_offs + offs.nbytes] = offs.view(np.uint8)
    hv[o_hw:o_hw + hw.nbytes] = hw.view(np.uint8)
    pos = o_pix
    for a in arrs:
        hv[pos:pos + a.size] = a.reshape(-1)
        pos += a.size
    dev = host.cuda(non_blocking=True)
    base = dev.data_ptr()
    if out is None:
        out = torch.empty((B, height, width, 3), dtype=dtype, device='cuda')
    _ffi.check(_ffi.lib().ssdk_assemble_images(_ffi.context(), C.c_void_p(base + o_pix), C.c_void_p(base + o_offs), C.c_void_p(base + o_hw), B,
                                               C.c_void_p(base + 0) if max_ops else C.c_void_p(0), int(max_ops), height, width,
                                               0 if dtype == torch.float32 else 1, _ffi.dptr(out), _ffi.stream_ptr()))
    return out


def augment_batch_device(images, labels_list, ops_per_image, height, width):
    """The geometric half of ``SSDDataAugmentation`` for a batch, pixels and boxes from ONE op list per image: returns
    ``(images (B, height, width, 3) float32, (gt_dev, offsets_dev, stats_dev, total_upper, max_upper))``, the second part being
    what ``assemble_batch_device`` returns (feed it to ``SSDInputEncoder.encode_device_offsets``)."""
    imgs = assemble_images_device(images, ops_per_image, height, width)
    return imgs, assemble_batch_device(labels_list, ops_per_image)
