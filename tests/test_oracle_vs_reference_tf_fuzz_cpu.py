"""Differential fuzzing of the TensorFlow/Keras half of the oracle against THE REFERENCE'S OWN loss / layer source executed over
tests/golden/tf_shim.py (see that file for what the stand-in assumes), on random inputs, beyond the fixed vectors of
tests/golden/ref_tf_shim_golden.npz.  The inputs are generated here from their seeds; what the reference returned for them is
stored in tests/golden/ref_fuzz_golden.npz.xz (tests/golden/make_fuzz_golden.py)."""
import numpy as np
import pytest

from test_oracle_vs_reference_fuzz_cpu import check_inputs, ref  # noqa: F401  (ref: the golden fixture)


def loss_case(seed):
    from oracle import synth
    rng = np.random.default_rng(4000 + seed)
    B, P, C = int(rng.integers(1, 4)), int(rng.integers(30, 300)), int(rng.integers(2, 8))
    anchors = rng.uniform(0.1, 0.9, (P, 4))
    y_pred = synth.synth_y_pred(seed, B, anchors, C, sharp=float(rng.uniform(0.5, 4)))
    y_true = np.zeros_like(y_pred)
    cls = rng.integers(0, C, (B, P))
    cls[rng.uniform(size=(B, P)) < rng.uniform(0.5, 1.0)] = 0
    y_true[np.arange(B)[:, None], np.arange(P)[None, :], cls] = 1.0
    if rng.integers(0, 2):
        y_true[0, :int(rng.integers(1, 10)), :C] = 0.0                         # neutral boxes
    if rng.integers(0, 4) == 0:
        y_pred[:, :, :C] = 1.0 / C                                             # all losses tie
    y_true[:, :, C:C + 4] = rng.standard_normal((B, P, 4))
    kw = dict(neg_pos_ratio=int(rng.integers(1, 5)), n_neg_min=int(rng.choice([0, 0, 3, 50])), alpha=float(rng.choice([0.5, 1.0, 2.0])))
    return y_true.astype(np.float32), y_pred.astype(np.float32), kw


def decode_layer_case(seed):
    from oracle import synth
    rng = np.random.default_rng(5000 + seed)
    P, C, B = int(rng.integers(20, 150)), int(rng.integers(2, 6)), int(rng.integers(1, 3))
    anchors = np.concatenate([rng.uniform(0.1, 0.9, (P, 2)), rng.uniform(0.05, 0.5, (P, 2))], axis=1)
    y = synth.synth_y_pred(seed, B, anchors, C, sharp=float(rng.uniform(1, 5)), loc_scale=float(rng.uniform(0.3, 1.5)))
    kw = dict(confidence_thresh=float(rng.choice([0.01, 0.2, 0.5])), iou_threshold=float(rng.choice([0.3, 0.45, 0.6])),
              top_k=int(rng.choice([3, 20, 200])), nms_max_output_size=int(rng.choice([2, 10, 400])),
              normalize_coords=bool(rng.integers(0, 2)), img_height=120, img_width=160)
    return y, kw


@pytest.mark.parametrize('seed', range(20))
def test_ssd_loss_fuzz(ref, seed):
    from oracle.loss import ssd_loss
    y_true, y_pred, kw = loss_case(seed)
    check_inputs(ref, 'loss/%d' % seed, kw, y_true, y_pred)
    want = ref['loss/%d/out' % seed]
    got = ssd_loss(y_true, y_pred, kw['neg_pos_ratio'], kw['n_neg_min'], kw['alpha'])
    np.testing.assert_allclose(got, want, rtol=5e-6, atol=1e-6)


@pytest.mark.parametrize('seed', range(20))
def test_decode_layers_fuzz(ref, seed):
    from oracle.decoder import decode_layer, decode_layer_fast
    y, kw = decode_layer_case(seed)
    check_inputs(ref, 'layer/%d' % seed, kw, y)
    for name, fn in (('DecodeDetections', decode_layer), ('DecodeDetectionsFast', decode_layer_fast)):
        want = ref['layer/%d/%s' % (seed, name)]
        got = fn(y, kw['confidence_thresh'], kw['iou_threshold'], kw['top_k'], kw['nms_max_output_size'], kw['normalize_coords'], 120, 160)
        assert got.shape == want.shape
        np.testing.assert_array_equal(got[..., :2], want[..., :2])             # class ids and confidences, row by row
        np.testing.assert_allclose(got[..., 2:], want[..., 2:], rtol=1e-6, atol=1e-4)
