"""Layer-by-layer GPU check of the training step at the benchmarked batch: every layer of the training plan's forward pass and
every parameter gradient of ``ssdk_train_backward_layers`` against a float64 reference that differentiates each layer at the
activations the device stored (oracle/graph.py::backward_teacher_forced, itself pinned to plain float64 autograd by
tests/test_oracle_teacher_forced_cpu.py).  Sharing the device's activations and ReLU masks makes the comparison
well-conditioned at any depth and batch, unlike test_gpu_train.py's full-model autograd (whose own float64 forward can put a
pre-activation near 0 on the other side of a ReLU), so the bar can be tight and max-norm.

Cases (each takes the batch-dependent backward plans the smaller tests do not reach):
  * SSD300, B=32, 21 classes (the benchmark's model and batch): a dense N(0,1)/B upstream gradient in every column of every
    prior, then one forward_backward with the real loss on encoded synthetic ground truth;
  * the same with SSDK_WGRAD_TRANSPOSED=1 (per-tap transposed weight-gradient GEMMs instead of the native kernel);
  * SSD7, B=32, 96x128, BatchNormalization in its training phase (5x5 image-facing conv through wgrad_direct_kernel,
    32/48-channel inputs through the transposed path);
  * SSD512, B=4 (64x64 maps, the 4x4 'valid' conv10_2, seven heads).

Bars: forward layers FWD_TOL of the tensor's max (as test_gpu_model.CONV_TOL); gradients GRAD_TOL of each tensor's max,
max-norm.  A conv bias in front of BatchNormalization has an exactly zero gradient: the device value is compared with the
layer's beta gradient instead.  Sensitivity: two deliberately wrong references -- (a) image 0's upstream gradient zeroed
(a lost split-K chunk or tile), (b) one deep layer's data gradient with its kernel not rotated -- must miss the device
result by at least MISS x GRAD_TOL on every tensor they affect.  Every measured error is recorded with
test_gpu_model._record, beside the forward-pass errors of the inference plans.

Measured on an NVIDIA B200 (1000 W power limit), error / tensor max:
  * forward layers: SSD300 B=32 <= 1.5e-5 (conv4_2), SSD7 B=32 <= 1.2e-5 (conv2), SSD512 B=4 <= 1.4e-5 (fc6);
  * gradients: SSD300 B=32 with the dense dY 1.2e-4 (conv1_2/kernel), 6.1e-5 with SSDK_WGRAD_TRANSPOSED=1 (conv2_1/bias;
    conv1_2/kernel 3.8e-5 from the same gradient planes -- the native kernel sums 461 patches of 64 pixels per split in one
    accumulator there), 1.5e-4 with the loss's dY (fc7_mbox_conf/bias and the layers below it: the loss gradient's 1/p on the
    true class most likely makes the softmax derivative sensitive to the ~1e-5 difference between the device's logits and the
    reference's); SSD7 B=32 7.9e-5 (bn1/beta); SSD512 B=4 6.3e-5 (conv1_2/kernel).  GRAD_TOL is 3x the largest of these.
  * the wrong references miss by at least 8.4e-2 (SSD300), 5.5e-2 (SSD7), 3.1e-1 (SSD512) with image 0 dropped and 4.1e-1
    with conv5_3 / conv5 unrotated: 120x GRAD_TOL or more.
  * runtime of this file 31 s on its own, 20 s inside the whole GPU suite.  One SSD300 B=32 reference walk (cuDNN float64
    convolutions) takes 3.5 s (10.7 s as the process's first cuDNN work) at a peak of 11.3 GB of device memory on top of
    the 3.6 GB of stored activations; SSD512 B=4 0.45 s and 4.1 GB, SSD7 B=32 0.04 s and 1.0 GB.
"""
import time

import numpy as np
import pytest
from test_gpu_model import _record

pytestmark = pytest.mark.gpu

FWD_TOL = 1e-4
GRAD_TOL = 4.5e-4
MISS = 10.0


@pytest.fixture(scope='module', autouse=True)
def _built():
    import __graft_entry__ as entry
    entry.build()
    import torch
    assert torch.cuda.is_available()


def _randomise(w, seed):
    rng = np.random.default_rng(seed)
    for k in w:
        if k.endswith('/bias'):
            w[k] = (rng.standard_normal(w[k].shape) * 0.05).astype(np.float32)
        elif k.endswith('/gamma') and not k.endswith('norm/gamma'):
            w[k] = rng.uniform(0.8, 1.2, w[k].shape).astype(np.float32)
        elif k.endswith('/beta'):
            w[k] = (rng.standard_normal(w[k].shape) * 0.1).astype(np.float32)
    return w


def _read_acts(m, B):
    """Every layer of the training plan after its last forward, as float32 CUDA tensors (B,h,w,c)."""
    import torch
    return {s.name: torch.from_numpy(m.read_layer(s.name, B, training=True)).cuda() for s in m.specs}


def _same_acts(m, B, acts):
    import torch
    return all(torch.equal(torch.from_numpy(m.read_layer(s.name, B, training=True)).cuda(), acts[s.name]) for s in m.specs)


def _dense_dy(seed, B, m):
    return (np.random.default_rng(seed).standard_normal((B, m.n_boxes_total, m.n_classes + 12)) / B).astype(np.float32)


def _walk(m, w, acts, dy, bn_training=False, **kw):
    """The teacher-forced reference on the GPU; -> (gradients, forward errors, seconds, MB of device memory the walk itself
    allocated at its peak, on top of the stored activations)."""
    import torch
    from oracle import graph as og
    fwd = {}
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    t0 = time.perf_counter()
    ref = og.backward_teacher_forced(m.specs, w, acts, dy, m.n_classes, bn_training=bn_training, device='cuda', fwd_err=fwd, **kw)
    torch.cuda.synchronize()
    return ref, fwd, time.perf_counter() - t0, (torch.cuda.max_memory_allocated() - base) / 2**20


def _bn_bias(m, k):
    """The BatchNormalization layer behind conv bias ``k`` (its gradient is exactly zero), or None."""
    name, _, tag = k.partition('/')
    return getattr(m.specs[m.index[name]], 'bn', None) if tag == 'bias' and name in m.index else None


def _grad_errors(m, grads, ref, bn_training):
    errs = {}
    for k in ref:
        bn = _bn_bias(m, k) if bn_training else None
        if bn:
            errs[k] = float(np.abs(grads[k]).max() / np.abs(ref[bn + '/beta']).max())
        elif np.abs(ref[k]).max() > 0:
            errs[k] = float(np.abs(grads[k] - ref[k]).max() / np.abs(ref[k]).max())
        else:                                       # no gradient reaches this tensor (a head whose priors the loss ignores)
            errs[k] = 0.0 if not np.abs(grads[k]).any() else float('inf')
    return errs


def _check(test, m, grads, ref, fwd, bn_training=False):
    errs = _grad_errors(m, grads, ref, bn_training)
    _record(test + ':forward', **fwd)
    _record(test + ':grad', **errs)
    print('%s: forward worst %.2e (%s), gradient worst %.2e (%s)' % (test, max(fwd.values()), max(fwd, key=fwd.get),
                                                                   max(errs.values()), max(errs, key=errs.get)))
    assert set(grads) == set(ref)
    bad = {k: v for k, v in fwd.items() if not v <= FWD_TOL}
    assert not bad, 'forward layers beyond %.1e of their max: %s' % (FWD_TOL, bad)
    bad = {k: v for k, v in errs.items() if not v <= GRAD_TOL}
    assert not bad, 'gradients beyond %.1e of their max: %s' % (GRAD_TOL, bad)


def _below(m, name):
    """Parameter-owning layer names strictly below ``name`` (its producers, transitively)."""
    out, s = set(), m.specs[m.index[name]]
    while s.inp is not None:
        s = m.specs[m.index[s.inp]]
        out |= {s.name} | ({s.bn} if getattr(s, 'bn', None) else set())
    return out


def _perturbed(m, w, acts, dy, layer, bn_training=False):
    """The two deliberately wrong references: (a) image 0's upstream gradient zeroed, (b) ``layer``'s data gradient unrotated."""
    dy_a = dy.copy()
    dy_a[0] = 0.0
    ref_a = _walk(m, w, acts, dy_a, bn_training)[0]
    ref_b = _walk(m, w, acts, dy, bn_training, unrotated=layer)[0]
    return ref_a, ref_b, layer


def _sensitivity(test, m, grads, perturbed, bn_training=False):
    ref_a, ref_b, layer = perturbed
    below = _below(m, layer)
    miss_a = {k: v for k, v in _grad_errors(m, grads, ref_a, bn_training).items() if not (bn_training and _bn_bias(m, k))}
    miss_b = {k: v for k, v in _grad_errors(m, grads, ref_b, bn_training).items()
              if k.split('/')[0] in below and not (bn_training and _bn_bias(m, k))}
    _record(test + ':miss_image0_dropped', **miss_a)
    _record(test + ':miss_unrotated_' + layer, **miss_b)
    print('%s: wrong references miss by >= %.2e (image 0 dropped), %.2e (%s unrotated, %d tensors); bar %.1e'
          % (test, min(miss_a.values()), min(miss_b.values()), layer, len(miss_b), GRAD_TOL))
    assert miss_b, layer
    for name, miss in (('image 0 dropped', miss_a), (layer + ' unrotated', miss_b)):
        weak = {k: v for k, v in miss.items() if not v >= MISS * GRAD_TOL}
        assert not weak, 'the reference with %s is within %.0fx the bar on %s' % (name, MISS, weak)


def _ssd300(B, seed=2):
    from oracle import synth
    from oracle.encoder import OracleEncoder
    from ssd_keras_b200.models.keras_ssd300 import ssd_300
    sc = [0.1, 0.2, 0.37, 0.54, 0.71, 0.88, 1.05]
    m = ssd_300((300, 300, 3), 20, mode='training', scales=sc, divide_by_stddev=[64.0] * 3, weights_seed=seed)
    w = _randomise(m.get_weights(), seed)
    m.set_weights(w)
    enc = OracleEncoder(300, 300, 20, m.predictor_sizes, scales=sc, aspect_ratios_per_layer=m.anchor_cfg['aspect_ratios_per_layer'],
                        steps=[8, 16, 32, 64, 100, 300], variances=[0.1, 0.1, 0.2, 0.2])
    x = synth.synth_images(seed, B, 300, 300)
    y_true = enc(synth.synth_gt(seed + 1, B, 4, 300, 300, 20)).astype(np.float32)
    return m, w, x, y_true


@pytest.fixture(scope='module')
def ssd300_b32():
    """SSD300 at B=32: the device's activations and gradients (dense dY, then the loss) and the float64 references."""
    import torch
    from oracle.loss import ssd_loss_grad
    from ssd_keras_b200.training import SSDTrainer
    B = 32
    m, w, x, y_true = _ssd300(B)
    tr = SSDTrainer(m, B, lr=1e-3, momentum=0.9, l2_regularization=5e-4)
    xd = torch.from_numpy(x).cuda()
    m.forward_device(xd, training=True)
    acts = _read_acts(m, B)
    dy = _dense_dy(12, B, m)
    tr._backward_layers(torch.from_numpy(dy).cuda(), len(m.specs) - 1, 0)
    grads = tr.gradients()
    ref, fwd, secs, peak = _walk(m, w, acts, dy)
    print('ssd300 b32: reference walk %.1f s, peak %.0f MB on top of the stored activations (%.0f MB)'
          % (secs, peak, sum(a.numel() for a in acts.values()) * 4 / 2**20))
    _record('ssd300_b32:walk', seconds=secs, peak_mb=peak)
    perturbed = _perturbed(m, w, acts, dy, 'conv5_3')
    _, y_pred = tr.forward_backward(xd, torch.from_numpy(y_true).cuda())
    torch.cuda.synchronize()
    loss_same_forward = _same_acts(m, B, acts)
    grads_loss = tr.gradients()
    dy_loss = ssd_loss_grad(y_true, y_pred.cpu().numpy())
    ref_loss = _walk(m, w, acts, dy_loss)[0]
    del tr
    return dict(m=m, w=w, x=x, acts=acts, dy=dy, grads=grads, ref=ref, fwd=fwd, perturbed=perturbed,
                loss_same_forward=loss_same_forward, grads_loss=grads_loss, ref_loss=ref_loss)


def test_ssd300_b32_dense_dy(ssd300_b32):
    r = ssd300_b32
    _check('ssd300_b32_dense', r['m'], r['grads'], r['ref'], r['fwd'])
    _sensitivity('ssd300_b32_dense', r['m'], r['grads'], r['perturbed'])


def test_ssd300_b32_loss(ssd300_b32):
    """One forward_backward with the SSD loss: its dY is the loss gradient of the device's own y_pred (the loss kernel is
    checked on identical y_pred in test_gpu_codec.py); the second forward must store bit-identical activations."""
    r = ssd300_b32
    assert r['loss_same_forward']
    errs = _grad_errors(r['m'], r['grads_loss'], r['ref_loss'], False)
    _record('ssd300_b32_loss:grad', **errs)
    print('ssd300_b32_loss: gradient worst %.2e (%s)' % (max(errs.values()), max(errs, key=errs.get)))
    bad = {k: v for k, v in errs.items() if not v <= GRAD_TOL}
    assert not bad, 'gradients beyond %.1e of their max: %s' % (GRAD_TOL, bad)


def test_ssd300_b32_transposed_wgrad(ssd300_b32, monkeypatch):
    """SSDK_WGRAD_TRANSPOSED=1 changes only the backward plans: the forward is bit-identical and the reference is reused."""
    import torch
    from ssd_keras_b200.models.keras_ssd300 import ssd_300
    from ssd_keras_b200.training import SSDTrainer
    monkeypatch.setenv('SSDK_WGRAD_TRANSPOSED', '1')
    r = ssd300_b32
    B = 32
    m = ssd_300((300, 300, 3), 20, mode='training', scales=[0.1, 0.2, 0.37, 0.54, 0.71, 0.88, 1.05], divide_by_stddev=[64.0] * 3)
    m.set_weights(r['w'])
    tr = SSDTrainer(m, B, lr=1e-3, momentum=0.9)
    m.forward_device(torch.from_numpy(r['x']).cuda(), training=True)
    assert _same_acts(m, B, r['acts'])
    tr._backward_layers(torch.from_numpy(r['dy']).cuda(), len(m.specs) - 1, 0)
    grads = tr.gradients()
    _check('ssd300_b32_transposed', m, grads, r['ref'], r['fwd'])
    _sensitivity('ssd300_b32_transposed', m, grads, r['perturbed'])


def test_ssd7_b32_batchnorm():
    import torch
    from oracle import synth
    from ssd_keras_b200.models.keras_ssd7 import build_model
    from ssd_keras_b200.training import SSDTrainer
    B, H, W, ncls = 32, 96, 128, 5
    m = build_model((H, W, 3), ncls, mode='training', l2_regularization=5e-4, scales=[0.08, 0.16, 0.32, 0.64, 0.96],
                    normalize_coords=True, weights_seed=4, subtract_mean=127.5, divide_by_stddev=127.5)
    w = _randomise(m.get_weights(), 3)
    m.set_weights(w)
    tr = SSDTrainer(m, B, lr=1e-3, l2_regularization=5e-4, optimizer='adam')
    m.forward_device(torch.from_numpy(synth.synth_images(7, B, H, W)).cuda(), training=True)
    acts = _read_acts(m, B)
    dy = _dense_dy(13, B, m)
    tr._backward_layers(torch.from_numpy(dy).cuda(), len(m.specs) - 1, 0)
    grads = tr.gradients()
    ref, fwd, secs, peak = _walk(m, w, acts, dy, bn_training=True)
    print('ssd7 b32: reference walk %.1f s, peak %.0f MB on top of the stored activations' % (secs, peak))
    _record('ssd7_b32:walk', seconds=secs, peak_mb=peak)
    _check('ssd7_b32', m, grads, ref, fwd, bn_training=True)
    _sensitivity('ssd7_b32', m, grads, _perturbed(m, w, acts, dy, 'conv5', bn_training=True), bn_training=True)


def test_ssd512_b4():
    import torch
    from oracle import synth
    from ssd_keras_b200.models.keras_ssd512 import ssd_512
    from ssd_keras_b200.training import SSDTrainer
    B = 4
    m = ssd_512((512, 512, 3), 20, mode='training', scales=[0.04, 0.1, 0.26, 0.42, 0.58, 0.74, 0.9, 1.06],
                divide_by_stddev=[64.0] * 3, weights_seed=3)
    w = _randomise(m.get_weights(), 3)
    m.set_weights(w)
    tr = SSDTrainer(m, B, lr=1e-3, momentum=0.9)
    m.forward_device(torch.from_numpy(synth.synth_images(9, B, 512, 512)).cuda(), training=True)
    acts = _read_acts(m, B)
    dy = _dense_dy(14, B, m)
    tr._backward_layers(torch.from_numpy(dy).cuda(), len(m.specs) - 1, 0)
    grads = tr.gradients()
    ref, fwd, secs, peak = _walk(m, w, acts, dy)
    print('ssd512 b4: reference walk %.1f s, peak %.0f MB on top of the stored activations' % (secs, peak))
    _record('ssd512_b4:walk', seconds=secs, peak_mb=peak)
    _check('ssd512_b4', m, grads, ref, fwd)
    _sensitivity('ssd512_b4', m, grads, _perturbed(m, w, acts, dy, 'conv5_3'))
