"""Host-side graph description shared by ``ssd_300`` / ``ssd_512`` / ``build_model``.

The builders mirror the reference functions' arguments and produce an ``SSDModel`` whose forward pass
is a static plan of hand-written sm_100a kernels inside libssdk.so (``ssdk_model_*``).  The object offers
the part of the Keras ``Model`` surface that the reference's callers use: ``predict``, ``get_layer(name)
.output_shape``, ``load_weights`` / ``set_weights`` / ``get_weights``.
"""
import ctypes as C

import numpy as np

from .. import _ffi
from ..keras_layers.keras_layer_DecodeDetections import DecodeDetections
from ..keras_layers.keras_layer_DecodeDetectionsFast import DecodeDetectionsFast
from ._keras_api import KerasTrainingMixin


class _LayerInfo:
    def __init__(self, name, output_shape):
        self.name = name
        self.output_shape = output_shape          # (None, H, W, C) like Keras


class Spec:
    """One node of the graph (see ssdk_layer_desc in include/ssdk.h)."""

    def __init__(self, name, op, inp=None, cout=0, k=(1, 1), stride=1, dilation=1, pad=(0, 0, 0, 0), act=_ffi.ACT_NONE,
                 n_boxes=0, bn=None, params=None):
        self.name, self.op, self.inp, self.cout = name, op, inp, cout
        self.kh, self.kw = k
        self.stride, self.dilation, self.pad, self.act, self.n_boxes = stride, dilation, pad, act, n_boxes
        self.bn = bn                               # name of the BatchNormalization layer folded into this conv
        self.params = params or {}


def same_pad(k, dilation=1):
    p = dilation * (k - 1) // 2
    return (p, p, p, p)


def tf_same_pool_pad(size, k, s):
    """TensorFlow 'same' pooling: total pad = max((ceil(n/s)-1)*s + k - n, 0), extra goes to the END."""
    out = -(-size // s)
    total = max((out - 1) * s + k - size, 0)
    return total // 2, total - total // 2


def records_config(name):
    """Decorator of the three builders: remembers the (JSON-able) arguments of the call on the model it returns, for ``save``."""
    import functools
    import inspect

    def plain(v):
        if isinstance(v, np.ndarray):
            return v.tolist()
        if isinstance(v, (np.floating, np.integer)):
            return v.item()
        if isinstance(v, (list, tuple)):
            return [plain(q) for q in v]
        return v

    def deco(fn):
        sig = inspect.signature(fn)

        @functools.wraps(fn)
        def wrapper(*a, **kw):
            out = fn(*a, **kw)
            b = sig.bind(*a, **kw)
            b.apply_defaults()
            args = {k: plain(v) for k, v in b.arguments.items() if k != 'return_predictor_sizes'}
            (out[0] if isinstance(out, tuple) else out)._build_config = (name, args)
            return out
        return wrapper
    return deco


class SSDModel(KerasTrainingMixin):
    def __init__(self, specs, img_height, img_width, img_channels, n_classes_total, anchor_cfg, variances, mode,
                 decode_cfg, l2_reg=0.0, precision='bf16x3', seed=0):
        self.specs = specs
        self.index = {s.name: i for i, s in enumerate(specs)}
        self.img_height, self.img_width, self.img_channels = img_height, img_width, img_channels
        self.n_classes = n_classes_total
        self.anchor_cfg = anchor_cfg
        self.variances = np.asarray(variances, dtype=np.float32)
        self.mode = mode
        self.decode_cfg = decode_cfg
        self.l2_regularization = l2_reg
        self.precision = precision
        self._plans = {}
        self._trainers = []                        # weak references to the SSDTrainer objects attached to this model
        self._shapes = self._infer_shapes()
        self.predictor_sizes = np.array([self._shapes[self.index[s.name]][:2] for s in specs if s.op == _ffi.OP_HEAD])
        a64, a32, nb = _ffi.generate_anchors(img_height, img_width, self.predictor_sizes, **anchor_cfg)
        self.anchors, self.anchors_f32 = a64, a32
        self.n_boxes_total = a64.shape[0]
        self.weights = {}
        self._init_weights(seed)
        if mode == 'inference':
            self.decoder = DecodeDetections(**decode_cfg)
        elif mode == 'inference_fast':
            self.decoder = DecodeDetectionsFast(**decode_cfg)
        else:
            self.decoder = None

    # -- graph bookkeeping -------------------------------------------------------------------
    def _infer_shapes(self):
        shapes = []
        for s in self.specs:
            if s.op == _ffi.OP_INPUT:
                shapes.append((self.img_height, self.img_width, self.img_channels))
                continue
            h, w, c = shapes[self.index[s.inp]]
            pt, pl, pb, pr = s.pad
            if s.op in (_ffi.OP_CONV, _ffi.OP_HEAD):
                ho = (h + pt + pb - s.dilation * (s.kh - 1) - 1) // s.stride + 1
                wo = (w + pl + pr - s.dilation * (s.kw - 1) - 1) // s.stride + 1
                shapes.append((ho, wo, s.cout if s.op == _ffi.OP_CONV else s.n_boxes * (self.n_classes + 4)))
            elif s.op == _ffi.OP_MAXPOOL:
                shapes.append(((h + pt + pb - s.kh) // s.stride + 1, (w + pl + pr - s.kw) // s.stride + 1, c))
            else:
                shapes.append((h, w, c))
        return shapes

    def get_layer(self, name):
        if name in self.index:
            h, w, c = self._shapes[self.index[name]]
            return _LayerInfo(name, (None, h, w, c))
        # reference layer names for the fused predictor heads: '<src>_mbox_conf' / '<src>_mbox_loc', 'classesN' / 'boxesN'
        for s in self.specs:
            if s.op == _ffi.OP_HEAD and name in (s.params.get('conf_name'), s.params.get('loc_name')):
                h, w, _ = self._shapes[self.index[s.name]]
                c = s.n_boxes * (self.n_classes if name == s.params['conf_name'] else 4)
                return _LayerInfo(name, (None, h, w, c))
        raise ValueError('No such layer: ' + name)

    @property
    def layers(self):
        return [self.get_layer(s.name) for s in self.specs]

    @property
    def input_shape(self):
        return (None, self.img_height, self.img_width, self.img_channels)

    @property
    def output_shape(self):
        """(None, P, C+12) in 'training' mode, (None, top_k, 6) with a decoder layer at the end (keras_ssd300.py:421-446)."""
        if self.decoder is None:
            return (None, self.n_boxes_total, self.n_classes + 12)
        return (None, int(self.decode_cfg['top_k']), 6)

    def count_params(self):
        """Keras' ``model.count_params()``: trainable + non-trainable (BatchNormalization moving statistics) parameters."""
        return int(sum(int(np.prod(s)) for s in self.weight_shapes().values()))

    def summary(self, line_length=100, print_fn=print):
        """A ``model.summary()`` in Keras' spirit: one row per layer of the plan (the fused predictor heads show up under both of
        their Keras names), then the parameter totals."""
        shapes = self.weight_shapes()
        rows = []
        for s in self.specs:
            h, w, c = self._shapes[self.index[s.name]]
            if s.op == _ffi.OP_HEAD:
                for nm in (s.params['conf_name'], s.params['loc_name']):
                    n_par = sum(int(np.prod(v)) for k, v in shapes.items() if k.startswith(nm + '/'))
                    rows.append((nm + ' (Conv2D)', str(self.get_layer(nm).output_shape), n_par, s.inp))
                continue
            kind = {_ffi.OP_INPUT: 'InputLayer', _ffi.OP_CONV: 'Conv2D', _ffi.OP_MAXPOOL: 'MaxPooling2D', _ffi.OP_L2NORM: 'L2Normalization'}.get(s.op, '?')
            n_par = sum(int(np.prod(v)) for k, v in shapes.items() if k.split('/')[0] in (s.name, s.bn))
            rows.append(('%s (%s)' % (s.name, kind), str((None, h, w, c)), n_par, s.inp or ''))
        print_fn('_' * line_length)
        print_fn('%-38s%-26s%-12s%s' % ('Layer (type)', 'Output Shape', 'Param #', 'Connected to'))
        print_fn('=' * line_length)
        for r in rows:
            print_fn('%-38s%-26s%-12d%s' % r)
        print_fn('=' * line_length)
        total = self.count_params()
        non_tr = sum(int(np.prod(v)) for k, v in shapes.items() if k.endswith(('/moving_mean', '/moving_variance')))
        print_fn('Output: %s   (mode=%r)' % (self.output_shape, self.mode))
        print_fn('Total params: {:,}'.format(total))
        print_fn('Trainable params: {:,}'.format(total - non_tr))
        print_fn('Non-trainable params: {:,}'.format(non_tr))
        print_fn('_' * line_length)

    # -- weights -----------------------------------------------------------------------------
    def weight_shapes(self):
        out = {}
        for s in self.specs:
            if s.op == _ffi.OP_CONV:
                cin = self._shapes[self.index[s.inp]][2]
                out[s.name + '/kernel'] = (s.kh, s.kw, cin, s.cout); out[s.name + '/bias'] = (s.cout,)
                if s.bn:
                    for p in ('gamma', 'beta', 'moving_mean', 'moving_variance'):
                        out[s.bn + '/' + p] = (s.cout,)
            elif s.op == _ffi.OP_HEAD:
                cin = self._shapes[self.index[s.inp]][2]
                out[s.params['conf_name'] + '/kernel'] = (3, 3, cin, s.n_boxes * self.n_classes)
                out[s.params['conf_name'] + '/bias'] = (s.n_boxes * self.n_classes,)
                out[s.params['loc_name'] + '/kernel'] = (3, 3, cin, s.n_boxes * 4)
                out[s.params['loc_name'] + '/bias'] = (s.n_boxes * 4,)
            elif s.op == _ffi.OP_L2NORM:
                out[s.name + '/gamma'] = (self._shapes[self.index[s.name]][2],)
        return out

    def _init_weights(self, seed):
        """kernel_initializer='he_normal' (truncation ignored), zero biases, gamma_init=20, BN identity."""
        rng = np.random.default_rng(seed)
        for name, shp in sorted(self.weight_shapes().items()):
            if name.endswith('/kernel'):
                fan_in = shp[0] * shp[1] * shp[2]
                self.weights[name] = (rng.standard_normal(shp) * np.sqrt(2.0 / fan_in)).astype(np.float32)
            elif name.endswith('norm/gamma'):
                self.weights[name] = np.full(shp, 20.0, np.float32)
            elif name.endswith(('/gamma', '/moving_variance')):
                self.weights[name] = np.ones(shp, np.float32)
            else:
                self.weights[name] = np.zeros(shp, np.float32)

    def set_weights(self, weights):
        """``weights``: dict name -> array using Keras' names ('conv1_1/kernel', 'conv4_3_norm/gamma', ...)."""
        shapes = self.weight_shapes()
        for k, v in weights.items():
            if k not in shapes:
                continue                                   # by_name semantics: unknown entries are skipped
            v = np.asarray(v, dtype=np.float32)
            if tuple(v.shape) != tuple(shapes[k]):
                raise ValueError('Weight %s has shape %s, expected %s' % (k, v.shape, shapes[k]))
            self.weights[k] = np.ascontiguousarray(v)
        self._release()

    def get_weights(self):
        self._sync_trained()
        return dict(self.weights)

    # -- trained weights: the model owns them ---------------------------------------------------
    def _live_trainers(self):
        out = []
        for r in self._trainers:
            t = r()
            if t is not None:
                out.append(t)
        return out

    def _sync_trained(self):
        """An attached ``SSDTrainer`` updates float32 master weights on the device (its training plan).  Before anything else
        looks at the weights -- ``get_weights`` / ``save_weights``, or a plan for another batch size / mode -- they are copied
        back into ``self.weights`` and the plans built from the old values are dropped (Keras' ``train_on_batch`` mutates the
        model; so does this)."""
        for t in self._live_trainers():
            if t._dirty:
                self.weights.update(t.get_weights())
                t._dirty = False
                keep = t.plan
                for key, h in list(self._plans.items()):
                    if h is not keep:
                        _ffi.lib().ssdk_model_destroy(h['handle'])
                        del self._plans[key]

    def load_weights(self, path, by_name=True):
        """``model.load_weights(path, by_name=True)`` (reference ``ssd300_training.ipynb:162``).  Accepts the Keras HDF5 files the
        reference ships (``README.md:223-239``) -- weights files (``/<layer>/<layer>/kernel:0``) and full-model files
        (``/model_weights/...``), read by ``misc_utils/hdf5_lite.py`` without h5py -- and ``.npz`` files with Keras weight names
        as keys.  Matching is by name like Keras' ``by_name=True``: entries for layers this model does not have are skipped,
        layers without an entry keep their weights; a shape mismatch raises."""
        p = str(path)
        if p.endswith('.npz'):
            with np.load(p) as f:
                self.set_weights({k: f[k] for k in f.files})
            return
        with open(p, 'rb') as f:
            magic = f.read(8)
        if magic != b'\x89HDF\r\n\x1a\n':
            raise ValueError('%s is neither an .npz nor an HDF5 file' % p)
        from ..misc_utils.hdf5_lite import read_keras_weights
        self.set_weights(read_keras_weights(p))

    def save_weights(self, path):
        """``model.save_weights(path)``: a Keras-layout HDF5 weights file for ``*.h5`` / ``*.hdf5`` (what ``load_weights`` of this
        package AND of Keras read), an ``.npz`` with the same names otherwise."""
        self._sync_trained()
        p = str(path)
        if p.endswith(('.h5', '.hdf5')):
            from ..misc_utils.hdf5_lite import write_keras_weights
            write_keras_weights(p, self.weights)
        else:
            np.savez(p, **self.weights)

    def save(self, filepath):
        """``model.save(filepath)`` (reference ``ssd300_training.ipynb:409-413`` via ``ModelCheckpoint``): one HDF5 file with the
        weights below ``/model_weights`` (Keras' layout: ``load_weights(filepath, by_name=True)`` of either library reads it) and,
        as the root attribute ``model_config``, the builder call that made this model -- what ``models.load_model`` rebuilds it
        from.  Optimizer state is not stored."""
        import json
        self._sync_trained()
        if getattr(self, '_build_config', None) is None:
            raise ValueError('this model was not made by ssd_300 / ssd_512 / build_model: save_weights() it instead')
        name, kwargs = self._build_config
        cfg = json.dumps({'class_name': 'SSDModel', 'config': {'builder': name, 'kwargs': kwargs}}).encode()
        from ..misc_utils.hdf5_lite import write_keras_weights
        write_keras_weights(str(filepath), self.weights, full_model=True,
                            root_attrs={'model_config': cfg, 'keras_version': b'2.1.4', 'backend': b'ssd_keras_b200'})

    # -- execution ---------------------------------------------------------------------------
    def _release(self):
        # trainers hold a raw pointer into their training plan: detach them first (they re-attach, with fresh optimiser
        # state, the next time they are used)
        for t in self._live_trainers():
            t._detach()
        for h in self._plans.values():
            _ffi.lib().ssdk_model_destroy(h['handle'])
        self._plans = {}

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    def _plan(self, batch, training=False):
        key = (batch, bool(training))
        if key in self._plans:
            hit = self._plans[key]
            if not any(t._dirty and t.plan is not hit for t in self._live_trainers()):
                return hit
        self._sync_trained()
        if key in self._plans:
            return self._plans[key]
        n = len(self.specs)
        descs = (_ffi.LayerDesc * n)()
        keep = []

        def fptr(a):
            a = np.ascontiguousarray(a, dtype=np.float32)
            keep.append(a)
            return _ffi.np_ptr(a, C.c_float)

        for i, s in enumerate(self.specs):
            d = descs[i]
            d.op = s.op
            d.input = self.index[s.inp] if s.inp is not None else -1
            d.cout, d.kh, d.kw, d.stride, d.dilation = s.cout, s.kh, s.kw, s.stride, s.dilation
            d.pad_t, d.pad_l, d.pad_b, d.pad_r = s.pad
            d.act, d.n_boxes = s.act, s.n_boxes
            if s.op == _ffi.OP_INPUT:
                # the reference broadcasts np.array(subtract_mean) over the channel axis: a scalar is legal
                if s.params.get('mean') is not None:
                    d.mean = fptr(np.broadcast_to(np.asarray(s.params['mean'], dtype=np.float32).reshape(-1), (3,)))
                if s.params.get('stddev') is not None:
                    d.stddev = fptr(np.broadcast_to(np.asarray(s.params['stddev'], dtype=np.float32).reshape(-1), (3,)))
                if s.params.get('swap'):
                    sw = np.ascontiguousarray(s.params['swap'], dtype=np.int32); keep.append(sw)
                    d.swap = _ffi.np_ptr(sw, C.c_int)
            elif s.op == _ffi.OP_CONV:
                d.kernel = fptr(self.weights[s.name + '/kernel']); d.bias = fptr(self.weights[s.name + '/bias'])
                if s.bn:   # inference-mode BatchNormalization(eps=1e-3) folded to scale/shift
                    g, b = self.weights[s.bn + '/gamma'], self.weights[s.bn + '/beta']
                    mu, var = self.weights[s.bn + '/moving_mean'], self.weights[s.bn + '/moving_variance']
                    scale = (g.astype(np.float64) / np.sqrt(var.astype(np.float64) + 1e-3))
                    d.bn_scale = fptr(scale); d.bn_shift = fptr(b - mu * scale)
                    if training:   # Keras' training phase normalises with batch statistics: the plan needs the raw parameters
                        d.bn_gamma, d.bn_beta, d.bn_mean, d.bn_var = fptr(g), fptr(b), fptr(mu), fptr(var)
                        d.bn_eps, d.bn_momentum = 1e-3, 0.99
            elif s.op == _ffi.OP_HEAD:
                d.kernel = fptr(self.weights[s.params['conf_name'] + '/kernel']); d.bias = fptr(self.weights[s.params['conf_name'] + '/bias'])
                d.kernel2 = fptr(self.weights[s.params['loc_name'] + '/kernel']); d.bias2 = fptr(self.weights[s.params['loc_name'] + '/bias'])
            elif s.op == _ffi.OP_L2NORM:
                d.kernel = fptr(self.weights[s.name + '/gamma'])
        anc = np.ascontiguousarray(self.anchors_f32)
        md = _ffi.ModelDesc(int(batch), self.img_height, self.img_width, self.img_channels, self.n_classes, n, descs,
                            0 if self.precision == 'bf16x3' else 1, _ffi.np_ptr(anc, C.c_float),
                            (C.c_float * 4)(*[float(v) for v in self.variances]), 1 if training else 0)
        h = C.c_void_p()
        _ffi.check(_ffi.lib().ssdk_model_create(_ffi.context(), C.byref(md), C.byref(h)))
        P = C.c_int()
        _ffi.check(_ffi.lib().ssdk_model_num_priors(h, C.byref(P)))
        assert P.value == self.n_boxes_total, (P.value, self.n_boxes_total)
        self._plans[key] = {'handle': h}
        return self._plans[key]

    def forward_device(self, images, training=False):
        """images: float32 CUDA tensor (B,H,W,3) -> y_pred float32 CUDA tensor (B,P,C+12) (raw predictions)."""
        import torch
        B = images.shape[0]
        plan = self._plan(B, training)
        images = images.to(dtype=torch.float32).contiguous()
        y = torch.empty((B, self.n_boxes_total, self.n_classes + 12), dtype=torch.float32, device=images.device)
        _ffi.check(_ffi.lib().ssdk_model_forward(plan['handle'], _ffi.dptr(images), _ffi.dptr(y), _ffi.stream_ptr()))
        return y

    def predict_device(self, images):
        y = self.forward_device(images)
        return y if self.decoder is None else self.decoder(y)

    def predict_stream(self, batches, post=None):
        """Generator over HOST batches -> HOST results, in order, software-pipelined: while the kernels of batch i run, batch
        i+1 is already on its way to the device (copy stream) and the host is still reading the result of batch i-1; the host
        only ever waits for the device->host copy of the PREVIOUS batch, so the GPU does not idle between batches (what Keras'
        ``predict_generator`` does with its queue of prefetched batches; the reference drives its models that way in
        eval_utils/average_precision_evaluator.py:373-380).

        batches: iterable of float32 (B,H,W,3) pinned CPU tensors (used as they are) or ndarrays (pinned here, one host copy).
        post:    optional function applied to the device result of each batch before it is downloaded (e.g. an all-gather).
        Yields pinned CPU tensors out of three rotating buffers owned by the model (allocating pinned memory costs milliseconds,
        so it happens once per result shape): a yielded tensor is overwritten when two more batches have gone through this model."""
        import torch
        main = torch.cuda.current_stream()
        if getattr(self, '_up_stream', None) is None:
            self._up_stream = torch.cuda.Stream()
            self._pin_slots = [None, None, None]
            self._pin_next = 0
        up = self._up_stream
        slots = self._pin_slots                         # pinned result buffers, rotated

        def upload(hb):
            if not torch.is_tensor(hb):
                hb = torch.from_numpy(np.ascontiguousarray(hb, dtype=np.float32))
            if not hb.is_pinned():
                hb = hb.pin_memory()
            with torch.cuda.stream(up):
                x = hb.cuda(non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(up)
            return x, ev, hb                            # hb is kept alive until its copy has been consumed

        it = iter(batches)
        nxt = None
        for hb in it:
            nxt = upload(hb)
            break
        pending = None                                  # (pinned buffer, event) of the batch whose result is still in flight
        i = 0
        while nxt is not None:
            x, ev, _keep = nxt
            nxt = None
            for hb in it:                               # issue the NEXT upload before this batch's kernels
                nxt = upload(hb)
                break
            main.wait_event(ev)
            x.record_stream(main)
            out = self.predict_device(x)
            if post is not None:
                out = post(out)
            k = self._pin_next
            self._pin_next = (k + 1) % 3
            buf = slots[k]
            if buf is None or buf.shape != out.shape or buf.dtype != out.dtype:
                buf = slots[k] = torch.empty(out.shape, dtype=out.dtype).pin_memory()
            buf.copy_(out, non_blocking=True)
            done = torch.cuda.Event()
            done.record(main)
            if pending is not None:
                pending[1].synchronize()
                yield pending[0]
            pending = (buf, done)
            i += 1
        if pending is not None:
            pending[1].synchronize()
            yield pending[0]

    def predict_generator(self, generator, steps=None):
        """Keras' ``Model.predict_generator``: pulls ``steps`` batches (all of them if None) from ``generator`` -- each an image
        batch or a tuple whose first element is one -- and returns the concatenated predictions as one ndarray.  The batches are
        pipelined through :meth:`predict_stream`."""
        import itertools

        def images():
            src = generator if steps is None else itertools.islice(generator, int(steps))
            for item in src:
                yield item[0] if isinstance(item, (tuple, list)) else item
        outs = [r.numpy().copy() for r in self.predict_stream(images())]
        if not outs:
            raise ValueError('predict_generator: the generator yielded no batch')
        return np.concatenate(outs, axis=0)

    def predict(self, x, batch_size=None):
        """Keras-style: ndarray (N,H,W,3) -> ndarray ((N,P,C+12) in 'training' mode, (N,top_k,6) otherwise)."""
        x = np.asarray(x, dtype=np.float32)
        bs = batch_size or x.shape[0]
        outs = [r.numpy().copy() for r in self.predict_stream(x[i:i + bs] for i in range(0, x.shape[0], bs))]
        return np.concatenate(outs, axis=0)

    def read_layer(self, name, batch, training=False):
        """Activation of a layer after the last forward with this batch size, float32 ndarray (B,h,w,c).  ``training``: of the
        training plan (``forward_device(..., training=True)``, what ``SSDTrainer`` runs), where a predictor head reads as its
        raw output, per box [class logits | 4 offsets]."""
        import torch
        i = self.index[name]
        h, w, c = self._shapes[i]
        out = torch.empty((batch, h, w, c), dtype=torch.float32, device='cuda')
        _ffi.check(_ffi.lib().ssdk_model_read_layer(self._plan(batch, training)['handle'], i, _ffi.dptr(out), _ffi.stream_ptr()))
        return out.cpu().numpy()

    def flops(self, batch):
        a, b = C.c_double(), C.c_double()
        _ffi.check(_ffi.lib().ssdk_model_flops(self._plan(batch)['handle'], C.byref(a), C.byref(b)))
        return a.value, b.value

    def set_timing(self, batch, enable=True):
        _ffi.check(_ffi.lib().ssdk_model_set_timing(self._plan(batch)['handle'], 1 if enable else 0))

    def last_conv_ms(self, batch):
        v = C.c_float()
        _ffi.check(_ffi.lib().ssdk_model_last_conv_ms(self._plan(batch)['handle'], C.byref(v)))
        return v.value


# ---------------------------------------------------------------------------------------------
# argument handling shared by the three builders (reference: models/keras_ssd300.py:183-240)
# ---------------------------------------------------------------------------------------------
def resolve_box_args(n_predictor_layers, min_scale, max_scale, scales, aspect_ratios_global, aspect_ratios_per_layer,
                     two_boxes_for_ar1, steps, offsets, variances):
    if aspect_ratios_global is None and aspect_ratios_per_layer is None:
        raise ValueError("`aspect_ratios_global` and `aspect_ratios_per_layer` cannot both be None. At least one needs to be specified.")
    if aspect_ratios_per_layer:
        if len(aspect_ratios_per_layer) != n_predictor_layers:
            raise ValueError("It must be either aspect_ratios_per_layer is None or len(aspect_ratios_per_layer) == {}, but "
                             "len(aspect_ratios_per_layer) == {}.".format(n_predictor_layers, len(aspect_ratios_per_layer)))
    if (min_scale is None or max_scale is None) and scales is None:
        raise ValueError("Either `min_scale` and `max_scale` or `scales` need to be specified.")
    if scales:
        if len(scales) != n_predictor_layers + 1:
            raise ValueError("It must be either scales is None or len(scales) == {}, but len(scales) == {}."
                             .format(n_predictor_layers + 1, len(scales)))
    else:
        scales = np.linspace(min_scale, max_scale, n_predictor_layers + 1)
    if len(variances) != 4:
        raise ValueError("4 variance values must be pased, but {} values were received.".format(len(variances)))
    variances = np.array(variances)
    if np.any(variances <= 0):
        raise ValueError("All variances must be >0, but the variances given are {}".format(variances))
    if (steps is not None) and (len(steps) != n_predictor_layers):
        raise ValueError("You must provide at least one step value per predictor layer.")
    if (offsets is not None) and (len(offsets) != n_predictor_layers):
        raise ValueError("You must provide at least one offset value per predictor layer.")
    if aspect_ratios_per_layer:
        aspect_ratios = aspect_ratios_per_layer
    else:
        aspect_ratios = [aspect_ratios_global] * n_predictor_layers
    n_boxes = [len(ar) + (1 if (1 in ar) and two_boxes_for_ar1 else 0) for ar in aspect_ratios]
    return scales, aspect_ratios, n_boxes, variances
