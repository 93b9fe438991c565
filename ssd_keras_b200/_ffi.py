"""ctypes binding of libssdk.so (include/ssdk.h).  PyTorch is used only for device memory and streams."""
import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, '_lib', 'libssdk.so')

SSDK_OK = 0
SSDK_ERR_INVALID = -1
SSDK_ERR_CUDA = -2
SSDK_ERR_UNSUPPORTED = -3
SSDK_ERR_NOMEM = -4
SSDK_ERR_DEGENERATE = -5

COORDS = {'centroids': 0, 'corners': 1, 'minmax': 2}
BORDER_D = {'half': 0, 'include': 1, 'exclude': -1}

c_int_p = C.POINTER(C.c_int)
c_float_p = C.POINTER(C.c_float)
c_double_p = C.POINTER(C.c_double)


class AnchorCfg(C.Structure):
    _fields_ = [('img_height', C.c_int), ('img_width', C.c_int), ('n_layers', C.c_int),
                ('fm_height', c_int_p), ('fm_width', c_int_p), ('scales', c_double_p),
                ('n_aspect_ratios', c_int_p), ('aspect_ratios', c_double_p), ('two_boxes_for_ar1', C.c_int),
                ('steps_h', c_double_p), ('steps_w', c_double_p), ('offsets_h', c_double_p), ('offsets_w', c_double_p),
                ('clip_boxes', C.c_int), ('coords', C.c_int), ('normalize_coords', C.c_int)]


class EncodeCfg(C.Structure):
    _fields_ = [('img_height', C.c_int), ('img_width', C.c_int), ('n_classes_total', C.c_int), ('P', C.c_int),
                ('background_id', C.c_int), ('coords', C.c_int), ('matching_multi', C.c_int),
                ('pos_iou_threshold', C.c_double), ('neg_iou_limit', C.c_double), ('border_d', C.c_int),
                ('normalize_coords', C.c_int), ('variances', C.c_double * 4),
                ('n_layers', C.c_int), ('fm_height', c_int_p), ('fm_width', c_int_p), ('n_boxes', c_int_p)]


class DecodeCfg(C.Structure):
    _fields_ = [('mode', C.c_int), ('layer_semantics', C.c_int), ('n_classes_total', C.c_int), ('P', C.c_int),
                ('confidence_thresh', C.c_double), ('iou_threshold', C.c_double), ('top_k', C.c_int),
                ('nms_max_output', C.c_int), ('coords', C.c_int), ('normalize_coords', C.c_int),
                ('img_height', C.c_int), ('img_width', C.c_int), ('border_d', C.c_int), ('max_out', C.c_int)]


class BoxOp(C.Structure):
    _fields_ = [('op', C.c_int), ('flags', C.c_int), ('a0', C.c_double), ('a1', C.c_double), ('a2', C.c_double), ('a3', C.c_double)]


BOXOP_END, BOXOP_CROP_PAD, BOXOP_FLIP_H, BOXOP_FLIP_V, BOXOP_RESIZE, BOXOP_FILTER = range(6)


class PixelOp(C.Structure):
    _fields_ = [('op', C.c_int), ('arg', C.c_int), ('a0', C.c_double)]


(PIXOP_END, PIXOP_TO_FLOAT, PIXOP_TO_U8, PIXOP_RGB2HSV, PIXOP_HSV2RGB, PIXOP_BRIGHTNESS, PIXOP_CONTRAST, PIXOP_SATURATION, PIXOP_HUE,
 PIXOP_CHANNEL_SWAP) = range(10)
MAX_PIXEL_OPS = 64


class LossWsLayout(C.Structure):
    _fields_ = [('bytes', C.c_longlong), ('counts_offset', C.c_longlong), ('counts_n', C.c_longlong), ('hist1_offset', C.c_longlong),
                ('hist2_offset', C.c_longlong), ('hist_n', C.c_longlong), ('ties_offset', C.c_longlong)]


class LayerDesc(C.Structure):
    _fields_ = [('op', C.c_int), ('input', C.c_int), ('cout', C.c_int), ('kh', C.c_int), ('kw', C.c_int),
                ('stride', C.c_int), ('dilation', C.c_int), ('pad_t', C.c_int), ('pad_l', C.c_int),
                ('pad_b', C.c_int), ('pad_r', C.c_int), ('act', C.c_int), ('n_boxes', C.c_int),
                ('kernel', c_float_p), ('bias', c_float_p), ('bn_scale', c_float_p), ('bn_shift', c_float_p),
                ('kernel2', c_float_p), ('bias2', c_float_p), ('mean', c_float_p), ('stddev', c_float_p),
                ('swap', c_int_p), ('bn_gamma', c_float_p), ('bn_beta', c_float_p), ('bn_mean', c_float_p), ('bn_var', c_float_p),
                ('bn_eps', C.c_float), ('bn_momentum', C.c_float)]


class ModelDesc(C.Structure):
    _fields_ = [('batch', C.c_int), ('img_height', C.c_int), ('img_width', C.c_int), ('img_channels', C.c_int),
                ('n_classes_total', C.c_int), ('n_layers', C.c_int), ('layers', C.POINTER(LayerDesc)),
                ('precision', C.c_int), ('anchors_f32', c_float_p), ('variances', C.c_float * 4), ('training', C.c_int)]


OP_INPUT, OP_CONV, OP_MAXPOOL, OP_L2NORM, OP_HEAD = range(5)
ACT_NONE, ACT_RELU, ACT_ELU = range(3)

_lib = None
_lock = threading.Lock()


class SSDKError(RuntimeError):
    pass


def lib():
    """Load libssdk.so.  There is no fallback: a missing library is a hard error."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(_LIB_PATH):
            raise SSDKError("libssdk.so is not built (%s). Run `python -m ssd_keras_b200.build` "
                            "(or __graft_entry__.build()); there is no CPU/PyTorch fallback." % _LIB_PATH)
        L = C.CDLL(_LIB_PATH)
        vp = C.c_void_p
        L.ssdk_version.restype = C.c_int
        L.ssdk_last_error.restype = C.c_char_p
        L.ssdk_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
        L.ssdk_ctx_destroy.argtypes = [vp]
        L.ssdk_ctx_launch_count.argtypes = [vp]
        L.ssdk_ctx_launch_count.restype = C.c_int64
        L.ssdk_anchors_count.argtypes = [C.POINTER(AnchorCfg), c_int_p, c_int_p]
        L.ssdk_anchors_generate.argtypes = [C.POINTER(AnchorCfg), c_double_p, c_float_p]
        L.ssdk_encoder_create.argtypes = [vp, C.POINTER(EncodeCfg), c_double_p, C.POINTER(vp)]
        L.ssdk_encoder_destroy.argtypes = [vp]
        L.ssdk_encode.argtypes = [vp, vp, c_int_p, C.c_int, vp, vp, vp, vp]
        L.ssdk_encode_f64.argtypes = [vp, vp, c_int_p, C.c_int, vp, vp, vp, vp]
        L.ssdk_encode_dev.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp]
        L.ssdk_iou_matrix.argtypes = [vp, vp, C.c_int, vp, vp]
        L.ssdk_iou.argtypes = [vp, vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
        L.ssdk_decode.argtypes = [vp, C.POINTER(DecodeCfg), vp, C.c_int, vp, vp, vp, vp]
        L.ssdk_nms.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int, vp, vp, vp, vp]
        L.ssdk_ssd_loss_fwd.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, vp, vp, vp]
        L.ssdk_ssd_loss_bwd.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, vp, vp, vp]
        L.ssdk_ssd_loss_fwd_bwd.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, vp, vp, vp, vp, vp]
        L.ssdk_ssd_loss_ws_layout.argtypes = [C.c_int, C.c_int, C.POINTER(LossWsLayout)]
        L.ssdk_ssd_loss_phase.argtypes = [vp, C.c_int, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, vp, C.c_int, vp,
                                          C.c_int, vp, vp, vp, vp, vp]
        for name in ('ssdk_ssd_loss_fwd_bwd', 'ssdk_ssd_loss_ws_layout', 'ssdk_ssd_loss_phase'):
            getattr(L, name).restype = C.c_int
        L.ssdk_eval_match.argtypes = [vp, C.c_int, vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, C.c_double, C.c_int, vp, vp, vp]
        L.ssdk_eval_cumsum.argtypes = [vp, vp, vp, vp, C.c_int, vp, vp, vp]
        L.ssdk_eval_match.restype = C.c_int
        L.ssdk_eval_cumsum.restype = C.c_int
        L.ssdk_assemble_batch.argtypes = [vp, vp, C.c_int, vp, C.c_int, C.c_int, vp, C.c_int, vp, vp, vp, vp]
        L.ssdk_assemble_batch.restype = C.c_int
        L.ssdk_assemble_images.argtypes = [vp, vp, vp, vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
        L.ssdk_assemble_images.restype = C.c_int
        L.ssdk_photometric.argtypes = [vp, vp, vp, vp, vp, C.c_int, vp, C.c_int, vp]
        L.ssdk_photometric.restype = C.c_int
        L.ssdk_l2_normalize.argtypes = [vp, vp, C.c_longlong, C.c_int, vp, vp, vp]
        L.ssdk_l2_normalize.restype = C.c_int
        L.ssdk_conv2d_fwd.argtypes = [vp, vp] + [C.c_int] * 4 + [vp, vp] + [C.c_int] * 11 + [vp, vp]
        L.ssdk_conv2d_fwd.restype = C.c_int
        L.ssdk_maxpool.argtypes = [vp, vp] + [C.c_int] * 11 + [vp, vp]
        L.ssdk_maxpool.restype = C.c_int
        if hasattr(L, 'ssdk_model_create'):
            L.ssdk_model_create.argtypes = [vp, C.POINTER(ModelDesc), C.POINTER(vp)]
            L.ssdk_model_destroy.argtypes = [vp]
            L.ssdk_model_num_priors.argtypes = [vp, c_int_p]
            L.ssdk_model_layer_shape.argtypes = [vp, C.c_int, c_int_p, c_int_p, c_int_p]
            L.ssdk_model_forward.argtypes = [vp, vp, vp, vp]
            L.ssdk_model_read_layer.argtypes = [vp, C.c_int, vp, vp]
            L.ssdk_model_flops.argtypes = [vp, c_double_p, c_double_p]
            L.ssdk_model_set_timing.argtypes = [vp, C.c_int]
            L.ssdk_model_last_conv_ms.argtypes = [vp, c_float_p]
        if hasattr(L, 'ssdk_trainer_create'):
            L.ssdk_trainer_create.argtypes = [vp, vp, C.POINTER(vp)]
            L.ssdk_trainer_destroy.argtypes = [vp]
            L.ssdk_trainer_num_params.argtypes = [vp, C.POINTER(C.c_longlong)]
            L.ssdk_trainer_param_span.argtypes = [vp, C.c_int, C.c_int, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
            L.ssdk_trainer_grad_buffer.argtypes = [vp]
            L.ssdk_trainer_grad_buffer.restype = vp
            L.ssdk_train_backward.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_float, vp, vp]
            L.ssdk_train_apply_adam.argtypes = [vp, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int, vp]
            L.ssdk_train_apply_adam.restype = C.c_int
            L.ssdk_trainer_read_bn_stats.argtypes = [vp, C.c_int, vp, vp, vp]
            L.ssdk_trainer_read_bn_stats.restype = C.c_int
            L.ssdk_train_backward_dy.argtypes = [vp, vp, vp]
            L.ssdk_train_backward_dy.restype = C.c_int
            L.ssdk_train_backward_begin.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_float, vp, vp]
            L.ssdk_train_backward_begin.restype = C.c_int
            L.ssdk_train_backward_layers.argtypes = [vp, vp, C.c_int, C.c_int, vp]
            L.ssdk_train_backward_layers.restype = C.c_int
            L.ssdk_train_apply.argtypes = [vp, C.c_float, C.c_float, C.c_float, C.c_float, vp]
            L.ssdk_trainer_read_params.argtypes = [vp, vp, vp]
            for name in ('ssdk_trainer_create', 'ssdk_trainer_destroy', 'ssdk_trainer_num_params', 'ssdk_trainer_param_span',
                         'ssdk_train_backward', 'ssdk_train_apply', 'ssdk_trainer_read_params'):
                getattr(L, name).restype = C.c_int
        for name in ('ssdk_ctx_create', 'ssdk_ctx_destroy', 'ssdk_anchors_count', 'ssdk_anchors_generate',
                     'ssdk_encoder_create', 'ssdk_encoder_destroy', 'ssdk_encode', 'ssdk_encode_f64', 'ssdk_encode_dev', 'ssdk_iou_matrix', 'ssdk_iou', 'ssdk_decode',
                     'ssdk_nms', 'ssdk_ssd_loss_fwd', 'ssdk_ssd_loss_bwd'):
            getattr(L, name).restype = C.c_int
        _lib = L
    return _lib


def check(rc):
    """Translate a status code into the exception the reference would raise."""
    if rc == SSDK_OK:
        return
    msg = lib().ssdk_last_error().decode('utf-8', 'replace')
    if rc == SSDK_ERR_INVALID:
        raise ValueError(msg)
    if rc == SSDK_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if rc == SSDK_ERR_NOMEM:
        raise MemoryError(msg)
    raise SSDKError('libssdk error %d: %s' % (rc, msg))


def np_ptr(a, ctype):
    return a.ctypes.data_as(C.POINTER(ctype))


_ctx = {}


def context(device=None):
    """One ssdk_ctx per (process, device, thread)."""
    import torch
    if not torch.cuda.is_available():
        raise SSDKError('No CUDA device: ssd_keras_b200 has no CPU fallback')
    if device is None:
        device = torch.cuda.current_device()
    key = (device, threading.get_ident())
    if key not in _ctx:
        h = C.c_void_p()
        check(lib().ssdk_ctx_create(int(device), C.byref(h)))
        _ctx[key] = h
    return _ctx[key]


def launch_count(device=None):
    return int(lib().ssdk_ctx_launch_count(context(device)))


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def dptr(t):
    """Device pointer of a contiguous torch CUDA tensor (or None)."""
    if t is None:
        return C.c_void_p(0)
    assert t.is_cuda and t.is_contiguous()
    return C.c_void_p(t.data_ptr())


# ---------------------------------------------------------------------------------------------
# host-only helper: anchors (works without a GPU)
# ---------------------------------------------------------------------------------------------
def _pair_or_nan(v):
    if v is None:
        return float('nan'), float('nan')
    if isinstance(v, (list, tuple, np.ndarray)) and len(v) == 2:
        return float(v[0]), float(v[1])
    return float(v), float(v)


def generate_anchors(img_height, img_width, predictor_sizes, scales, aspect_ratios_per_layer, two_boxes_for_ar1=True,
                     steps=None, offsets=None, clip_boxes=False, coords='centroids', normalize_coords=True):
    """-> (anchors float64 (P,4), anchors float32 (P,4), n_boxes per layer) via ssdk_anchors_generate."""
    if coords not in COORDS:
        raise ValueError("Unexpected value for `coords`. Supported values are 'minmax', 'corners' and 'centroids'.")
    L = lib()
    ps = np.asarray(predictor_sizes, dtype=np.int32).reshape(-1, 2)
    n = ps.shape[0]
    fm_h = np.ascontiguousarray(ps[:, 0]); fm_w = np.ascontiguousarray(ps[:, 1])
    sc = np.ascontiguousarray(np.asarray(scales, dtype=np.float64))
    n_ar = np.array([len(a) for a in aspect_ratios_per_layer], dtype=np.int32)
    ars = np.ascontiguousarray(np.concatenate([np.asarray(a, dtype=np.float64) for a in aspect_ratios_per_layer]))
    st = np.array([_pair_or_nan(s) for s in (steps if steps is not None else [None] * n)], dtype=np.float64)
    of = np.array([_pair_or_nan(o) for o in (offsets if offsets is not None else [None] * n)], dtype=np.float64)
    st_h, st_w = np.ascontiguousarray(st[:, 0]), np.ascontiguousarray(st[:, 1])
    of_h, of_w = np.ascontiguousarray(of[:, 0]), np.ascontiguousarray(of[:, 1])
    cfg = AnchorCfg(int(img_height), int(img_width), int(n), np_ptr(fm_h, C.c_int), np_ptr(fm_w, C.c_int),
                    np_ptr(sc, C.c_double), np_ptr(n_ar, C.c_int), np_ptr(ars, C.c_double), int(bool(two_boxes_for_ar1)),
                    np_ptr(st_h, C.c_double), np_ptr(st_w, C.c_double), np_ptr(of_h, C.c_double), np_ptr(of_w, C.c_double),
                    int(bool(clip_boxes)), COORDS[coords], int(bool(normalize_coords)))
    P = C.c_int(0)
    nb = np.zeros(n, dtype=np.int32)
    check(L.ssdk_anchors_count(C.byref(cfg), C.byref(P), np_ptr(nb, C.c_int)))
    a64 = np.empty((P.value, 4), dtype=np.float64)
    a32 = np.empty((P.value, 4), dtype=np.float32)
    check(L.ssdk_anchors_generate(C.byref(cfg), np_ptr(a64, C.c_double), np_ptr(a32, C.c_float)))
    return a64, a32, nb.tolist()
