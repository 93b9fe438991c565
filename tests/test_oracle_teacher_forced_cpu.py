"""CPU self-test of the teacher-forced float64 backward (oracle/graph.py::backward_teacher_forced) that
tests/test_gpu_train_layers.py compares the CUDA backward pass with.  Given the float64 forward's own activations as the
"device" activations, the layer-by-layer walk must reproduce plain float64 autograd of ``forward`` + ``.backward(dy)`` to
rounding (1e-12 of each tensor's max): the same ReLU masks, max-pool routing, L2Norm, softmax, ELU and BatchNormalization
(batch statistics) derivatives, and the same gradient summed over every consumer of a layer."""
import importlib.util
import os

import numpy as np
import pytest
import torch

from oracle import graph as og

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))
TOL = 1e-12


def _train_check():
    spec = importlib.util.spec_from_file_location('train_check', os.path.join(ROOT, 'tools', 'train_check.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _compare(specs, w, x, n_classes, anchors, variances, bn_training=False, seed=0):
    params = og.make_params(specs, w, dtype=torch.float64)
    yp, outs = og.forward(specs, params, x, n_classes, anchors, variances, dtype=torch.float64, bn_training=bn_training)
    dy = np.random.default_rng(seed).standard_normal(yp.shape)          # every column, anchors / variances included
    yp.backward(torch.from_numpy(dy))
    acts = {s.name: outs[s.name].detach().permute(0, 2, 3, 1) for s in specs if s.op != og.OP_HEAD}
    fwd = {}
    got = og.backward_teacher_forced(specs, w, acts, dy, n_classes, bn_training=bn_training, fwd_err=fwd)
    assert fwd and max(fwd.values()) == 0.0, fwd
    trainable = {k for k in w if not k.endswith(('/moving_mean', '/moving_variance'))}
    assert set(got) == trainable
    bn_of = {s.name: s.bn for s in specs if getattr(s, 'bn', None)}
    for k in sorted(trainable):
        ref = params[k].grad.numpy()
        layer = k.split('/')[0]
        if bn_training and k.endswith('/bias') and layer in bn_of:
            # zero in exact arithmetic (the batch mean removes the bias): both sides are rounding noise
            scale = np.abs(params[bn_of[layer] + '/beta'].grad.numpy()).max()
            assert np.abs(got[k]).max() <= TOL * scale and np.abs(ref).max() <= TOL * scale, k
            continue
        err = np.abs(got[k] - ref).max() / np.abs(ref).max()
        assert err <= TOL, '%s: %.3e' % (k, err)


@pytest.mark.parametrize('case', [0, 1, 2, 3])
def test_matches_autograd_on_small_graphs(case):
    """conv / pool (2x2 'same' and 3x3/s1) / 1x1 / L2Norm / two heads / stride 2 / dilation 3 / 'valid' graphs."""
    tc = _train_check()
    m, w, n_cls = tc.build(tc.CASES[case])
    _, hw, B, _ = tc.CASES[case]
    x = np.random.default_rng(11).integers(0, 256, size=(B, hw, hw, 3)).astype(np.float32)
    _compare(m.specs, w, x, n_cls, m.anchors, [0.1, 0.1, 0.2, 0.2], seed=case)


def test_matches_autograd_on_ssd7_with_batchnorm_training_phase():
    """SSD7: 5x5 image-facing conv, conv + BatchNormalization (batch statistics) + ELU stages, four heads."""
    from oracle import synth
    from ssd_keras_b200.models.keras_ssd7 import build_model
    B, H, W, ncls = 2, 64, 96, 5
    m = build_model((H, W, 3), ncls, mode='training', scales=[0.08, 0.16, 0.32, 0.64, 0.96], normalize_coords=True,
                    weights_seed=4, subtract_mean=127.5, divide_by_stddev=127.5)
    w = m.get_weights()
    rng = np.random.default_rng(3)
    for k in w:
        if k.endswith('/bias'):
            w[k] = (rng.standard_normal(w[k].shape) * 0.05).astype(np.float32)
        elif k.endswith('/gamma'):
            w[k] = rng.uniform(0.8, 1.2, w[k].shape).astype(np.float32)
        elif k.endswith('/beta'):
            w[k] = (rng.standard_normal(w[k].shape) * 0.1).astype(np.float32)
    x = synth.synth_images(7, B, H, W)
    _compare(m.specs, w, x, ncls + 1, m.anchors, [1.0] * 4, bn_training=True, seed=5)


def test_unrotated_data_gradient_differs():
    """The deliberately wrong reference (one layer's data gradient with its kernel not rotated) changes every gradient below
    that layer and none above it."""
    tc = _train_check()
    m, w, n_cls = tc.build(tc.CASES[1])
    _, hw, B, _ = tc.CASES[1]
    x = np.random.default_rng(11).integers(0, 256, size=(B, hw, hw, 3)).astype(np.float32)
    params = og.make_params(m.specs, w, dtype=torch.float64, requires_grad=False)
    yp, outs = og.forward(m.specs, params, x, n_cls, m.anchors, [0.1, 0.1, 0.2, 0.2], dtype=torch.float64)
    acts = {s.name: outs[s.name].permute(0, 2, 3, 1) for s in m.specs if s.op != og.OP_HEAD}
    dy = np.random.default_rng(0).standard_normal(yp.shape)
    good = og.backward_teacher_forced(m.specs, w, acts, dy, n_cls)
    bad = og.backward_teacher_forced(m.specs, w, acts, dy, n_cls, unrotated='c3')
    for k in good:
        rel = np.abs(bad[k] - good[k]).max() / np.abs(good[k]).max()
        if k.split('/')[0] in ('c1', 'c2'):
            assert rel > 0.1, (k, rel)
        else:
            assert rel == 0.0, (k, rel)
