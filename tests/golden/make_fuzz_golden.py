#!/usr/bin/env python
"""Golden outputs for the differential fuzz tests (tests/test_oracle_vs_reference_fuzz_cpu.py and
tests/test_oracle_vs_reference_tf_fuzz_cpu.py): the REAL reference is run on the random inputs those tests generate from their
seeds, and what it returns is written to tests/golden/ref_fuzz_golden.npz.xz together with a digest of the inputs of every case.
The NumPy half is imported directly, the Keras loss and layers run over tests/golden/tf_shim.py (as in make_tf_golden.py).

    SSD_REFERENCE_ROOT=<checkout of the original ssd_keras> python tests/golden/make_fuzz_golden.py
"""
import io
import lzma
import os
import sys

import numpy as np

np.float = float   # noqa  the reference targets NumPy < 1.24 (caller-side aliases, as in make_golden.py)
np.int = int       # noqa

REF = os.environ['SSD_REFERENCE_ROOT']
HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path.insert(0, REF)
sys.path.insert(0, HERE)
sys.path.insert(0, TESTS)
sys.path.insert(0, os.path.dirname(TESTS))

import test_oracle_vs_reference_fuzz_cpu as fz     # noqa: E402  (the input generators of the tests)
import test_oracle_vs_reference_tf_fuzz_cpu as tfz  # noqa: E402


def numpy_half(arrays):
    from bounding_box_utils.bounding_box_utils import convert_coordinates, convert_coordinates2, iou
    from ssd_encoder_decoder.ssd_input_encoder import SSDInputEncoder
    from ssd_encoder_decoder.ssd_output_decoder import decode_detections, decode_detections_fast

    for seed in range(40):
        cfg, gt = fz.encoder_case(seed)
        key = 'enc/%d' % seed
        arrays[key + '/inputs'] = np.array(fz.digest(cfg, *gt))
        r = SSDInputEncoder(**cfg)
        arrays[key + '/anchors'] = r.generate_encoding_template(1)[0][:, -8:-4]
        arrays[key + '/template2'] = r.generate_encoding_template(2)
        arrays[key + '/y'] = r(gt)
        arrays[key + '/n_layers'] = np.array(len(r.boxes_list))
        for i, b in enumerate(r.boxes_list):
            arrays['%s/boxes/%d' % (key, i)] = b

    for seed in range(25):
        y, kw = fz.decoder_case(seed)
        arrays['dec/%d/inputs' % seed] = np.array(fz.digest(kw, y))
        for name, fn in (('decode_detections', decode_detections), ('decode_detections_fast', decode_detections_fast)):
            key = 'dec/%d/%s' % (seed, name)
            want = fn(y, **kw)
            arrays[key + '/n'] = np.array(len(want))
            for i, b in enumerate(want):
                arrays['%s/%d' % (key, i)] = fz.sorted_rows(b)

    for seed in range(10):
        b1, b2, wide = fz.box_case(seed)
        key = 'box/%d' % seed
        arrays[key + '/inputs'] = np.array(fz.digest(b1, b2, wide))
        for conv in ('minmax2centroids', 'centroids2minmax'):
            arrays['%s/cc2/%s' % (key, conv)] = convert_coordinates2(wide, 2, conv)
        for coords in ('minmax', 'centroids'):
            arrays['%s/as/%s/1' % (key, coords)] = convert_coordinates(b1, 0, 'corners2' + coords)
            arrays['%s/as/%s/2' % (key, coords)] = convert_coordinates(b2, 0, 'corners2' + coords)
        k = min(len(b1), len(b2))
        for border in fz.BORDERS:
            for conv in fz.CONVERSIONS:
                arrays['%s/cc/%s/%s' % (key, border, conv)] = convert_coordinates(b1, 0, conv, border)
            for coords in ('corners', 'minmax', 'centroids'):
                c1 = b1 if coords == 'corners' else arrays['%s/as/%s/1' % (key, coords)]
                c2 = b2 if coords == 'corners' else arrays['%s/as/%s/2' % (key, coords)]
                arrays['%s/iou/%s/%s/outer' % (key, border, coords)] = iou(c1, c2, coords, 'outer_product', border)
                arrays['%s/iou/%s/%s/elem' % (key, border, coords)] = iou(c1[:k], c2[:k], coords, 'element-wise', border)


def keras_half(arrays):
    import tf_shim
    tf_shim.install()
    from keras_layers.keras_layer_DecodeDetections import DecodeDetections
    from keras_layers.keras_layer_DecodeDetectionsFast import DecodeDetectionsFast
    from keras_loss_function.keras_ssd_loss import SSDLoss

    for seed in range(20):
        y_true, y_pred, kw = tfz.loss_case(seed)
        arrays['loss/%d/inputs' % seed] = np.array(fz.digest(kw, y_true, y_pred))
        arrays['loss/%d/out' % seed] = np.asarray(SSDLoss(**kw).compute_loss(y_true, y_pred), np.float32)

    for seed in range(20):
        y, kw = tfz.decode_layer_case(seed)
        arrays['layer/%d/inputs' % seed] = np.array(fz.digest(kw, y))
        for name, cls in (('DecodeDetections', DecodeDetections), ('DecodeDetectionsFast', DecodeDetectionsFast)):
            arrays['layer/%d/%s' % (seed, name)] = np.asarray(cls(**kw).call(y.astype(np.float32)), np.float32)


def main():
    arrays = {}
    numpy_half(arrays)
    keras_half(arrays)
    # an .npz inside LZMA: the ~1000 small arrays cost less than in a zip, and the anchors repeated in the encoder outputs compress
    buf = io.BytesIO()
    np.savez(buf, **arrays)
    out = os.path.join(HERE, 'ref_fuzz_golden.npz.xz')
    with open(out, 'wb') as f:
        f.write(lzma.compress(buf.getvalue(), preset=9))
    print('wrote %d arrays, %d bytes' % (len(arrays), os.path.getsize(out)))


if __name__ == '__main__':
    main()
