"""Differential fuzzing of the NumPy half of the oracle against the REAL reference, beyond the fixed golden vectors: random
encoder configurations and ground truth, random prediction tensors for the two NumPy decoders, random box sets for iou /
convert_coordinates.  The inputs are generated here from their seeds; what the reference returned for them is stored in
tests/golden/ref_fuzz_golden.npz.xz (tests/golden/make_fuzz_golden.py), next to a digest of the inputs it was given.
Bit-exact float64 equality is required, as in tests/test_oracle_golden.py."""
import hashlib
import io
import json
import lzma
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ref_fuzz_golden.npz.xz')
BORDERS = ('half', 'include', 'exclude')
CONVERSIONS = ('minmax2centroids', 'centroids2minmax', 'corners2centroids', 'centroids2corners', 'minmax2corners', 'corners2minmax')


@pytest.fixture(scope='module')
def ref():
    with lzma.open(GOLDEN) as f, np.load(io.BytesIO(f.read())) as z:
        return {k: z[k] for k in z.files}


def digest(*parts):
    """SHA-256 of configurations (dicts, as sorted JSON) and arrays (dtype, shape and bytes)."""
    h = hashlib.sha256()
    for p in parts:
        if isinstance(p, dict):
            h.update(json.dumps(p, sort_keys=True).encode())
        else:
            p = np.ascontiguousarray(p)
            h.update(repr((p.dtype.str, p.shape)).encode())
            h.update(p.tobytes())
    return h.hexdigest()


def check_inputs(ref, key, *parts):
    assert digest(*parts) == str(ref[key + '/inputs']), '%s: the inputs differ from those the golden outputs were made from' % key


def _random_encoder_cfg(rng):
    n_layers = int(rng.integers(1, 4))
    H, W = int(rng.integers(60, 200)), int(rng.integers(60, 200))
    sizes = [(int(rng.integers(1, 7)), int(rng.integers(1, 7))) for _ in range(n_layers)]
    scales = sorted(rng.uniform(0.05, 1.0, n_layers + 1).tolist())
    per_layer = bool(rng.integers(0, 2))
    pool = [0.5, 1.0, 2.0, 3.0, 1.0 / 3.0, 1.5]
    ars = [list(rng.choice(pool, size=int(rng.integers(1, 5)), replace=False)) for _ in range(n_layers)]
    cfg = dict(img_height=H, img_width=W, n_classes=int(rng.integers(1, 6)), predictor_sizes=sizes, scales=scales,
               aspect_ratios_global=ars[0] if not per_layer else None, aspect_ratios_per_layer=ars if per_layer else None,
               two_boxes_for_ar1=bool(rng.integers(0, 2)), clip_boxes=bool(rng.integers(0, 2)),
               variances=rng.choice([0.1, 0.2, 1.0], size=4).tolist(), matching_type=str(rng.choice(['multi', 'bipartite'])),
               pos_iou_threshold=float(rng.choice([0.3, 0.5, 0.7])), neg_iou_limit=float(rng.choice([0.2, 0.3, 0.5])),
               border_pixels=str(rng.choice(['half', 'include', 'exclude'])), coords=str(rng.choice(['centroids', 'minmax', 'corners'])),
               normalize_coords=bool(rng.integers(0, 2)))
    cfg['neg_iou_limit'] = min(cfg['neg_iou_limit'], cfg['pos_iou_threshold'])
    if rng.integers(0, 2):
        cfg['steps'] = [(float(rng.uniform(8, 40)), float(rng.uniform(8, 40))) if rng.integers(0, 2) else float(rng.uniform(8, 40))
                        for _ in range(n_layers)]
    if rng.integers(0, 2):
        cfg['offsets'] = [float(rng.uniform(0.2, 0.8)) for _ in range(n_layers)]
    cfg['background_id'] = int(rng.integers(0, cfg['n_classes'] + 1)) if rng.integers(0, 3) == 0 else 0
    return cfg


def _random_gt(rng, cfg, B):
    out = []
    for _ in range(B):
        G = int(rng.integers(0, 6))
        x0 = rng.uniform(0, 0.7 * cfg['img_width'], G); y0 = rng.uniform(0, 0.7 * cfg['img_height'], G)
        w = rng.uniform(5, 0.6 * cfg['img_width'], G); h = rng.uniform(5, 0.6 * cfg['img_height'], G)
        ids = [c for c in range(cfg['n_classes'] + 1) if c != cfg['background_id']]
        g = np.stack([rng.choice(ids, G) if G else np.zeros(0), x0, y0, np.minimum(x0 + w, cfg['img_width'] - 1),
                      np.minimum(y0 + h, cfg['img_height'] - 1)], axis=1) if G else np.zeros((0, 5))
        if G >= 2 and rng.integers(0, 3) == 0:
            g[1] = g[0]                                    # duplicate box: exercises the tie rules
        out.append(g.astype(np.float64))
    return out


def encoder_case(seed):
    rng = np.random.default_rng(1000 + seed)
    cfg = _random_encoder_cfg(rng)
    return cfg, _random_gt(rng, cfg, int(rng.integers(1, 4)))


def decoder_case(seed):
    from oracle import synth
    rng = np.random.default_rng(2000 + seed)
    P, C, B = int(rng.integers(20, 200)), int(rng.integers(2, 7)), int(rng.integers(1, 3))
    anchors = np.concatenate([rng.uniform(0.1, 0.9, (P, 2)), rng.uniform(0.05, 0.5, (P, 2))], axis=1)
    y = synth.synth_y_pred(seed, B, anchors, C, sharp=float(rng.uniform(1, 5)), loc_scale=float(rng.uniform(0.3, 1.5)))
    kw = dict(confidence_thresh=float(rng.choice([0.01, 0.2, 0.5])), iou_threshold=float(rng.choice([0.3, 0.45, 0.6])),
              top_k=int(rng.choice([5, 20, 200])), normalize_coords=bool(rng.integers(0, 2)), img_height=120, img_width=160,
              border_pixels=str(rng.choice(['half', 'include', 'exclude'])))
    return y, kw


def sorted_rows(a):
    """Detections of one image as float64 rows in lexicographic order: top-k of the reference is an unordered argpartition
    set, so results are compared as sorted rows."""
    a = np.asarray(a, np.float64).reshape(-1, 6)
    return a[np.lexsort(a.T[::-1])]


def box_case(seed):
    rng = np.random.default_rng(3000 + seed)
    m, n = int(rng.integers(1, 9)), int(rng.integers(1, 9))

    def boxes(k):
        xy = rng.uniform(0, 80, (k, 2)); wh = rng.uniform(0, 40, (k, 2))
        return np.concatenate([xy, xy + wh], axis=1)
    b1, b2 = boxes(m), boxes(n)
    wide = np.concatenate([rng.standard_normal((m, 2)), b1], axis=1)          # conversion in the middle of a wider row
    return b1, b2, wide


@pytest.mark.parametrize('seed', range(40))
def test_encoder_fuzz(ref, seed):
    from oracle.encoder import OracleEncoder
    cfg, gt = encoder_case(seed)
    key = 'enc/%d' % seed
    check_inputs(ref, key, cfg, *gt)
    o = OracleEncoder(**cfg)
    np.testing.assert_array_equal(o.anchors, ref[key + '/anchors'])
    np.testing.assert_array_equal(o(gt), ref[key + '/y'])


@pytest.mark.parametrize('seed', range(25))
def test_numpy_decoders_fuzz(ref, seed):
    from oracle.decoder import decode_detections, decode_detections_fast
    y, kw = decoder_case(seed)
    check_inputs(ref, 'dec/%d' % seed, kw, y)
    for name, fn in (('decode_detections', decode_detections), ('decode_detections_fast', decode_detections_fast)):
        key = 'dec/%d/%s' % (seed, name)
        got = fn(y, **kw)
        assert len(got) == int(ref[key + '/n'])
        for i, a in enumerate(got):
            a, b = sorted_rows(a), ref['%s/%d' % (key, i)]
            assert a.shape == b.shape
            np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize('seed', range(10))
def test_box_math_fuzz(ref, seed):
    from oracle.boxes import convert_coordinates, iou
    from ssd_keras_b200.bounding_box_utils.bounding_box_utils import convert_coordinates as mirror_cc
    from ssd_keras_b200.bounding_box_utils.bounding_box_utils import convert_coordinates2 as mirror_cc2
    b1, b2, wide = box_case(seed)
    key = 'box/%d' % seed
    check_inputs(ref, key, b1, b2, wide)
    for conv in ('minmax2centroids', 'centroids2minmax'):
        np.testing.assert_array_equal(mirror_cc2(wide, 2, conv), ref['%s/cc2/%s' % (key, conv)])
    for border in BORDERS:
        for conv in CONVERSIONS:
            want = ref['%s/cc/%s/%s' % (key, border, conv)]
            np.testing.assert_array_equal(convert_coordinates(b1, 0, conv, border), want)
            np.testing.assert_array_equal(mirror_cc(b1, 0, conv, border), want)   # product (host side)
        for coords in ('corners', 'minmax', 'centroids'):
            # the reference's own conversions of the two box sets (default border) are the iou inputs
            c1 = b1 if coords == 'corners' else ref['%s/as/%s/1' % (key, coords)]
            c2 = b2 if coords == 'corners' else ref['%s/as/%s/2' % (key, coords)]
            np.testing.assert_array_equal(iou(c1, c2, coords, 'outer_product', border), ref['%s/iou/%s/%s/outer' % (key, border, coords)])
            k = min(len(b1), len(b2))
            np.testing.assert_array_equal(iou(c1[:k], c2[:k], coords, 'element-wise', border),
                                          ref['%s/iou/%s/%s/elem' % (key, border, coords)])


@pytest.mark.parametrize('seed', range(40))
def test_product_anchor_generation_fuzz(ref, seed):
    """PRODUCT code: the library's host-side anchor generator (`ssdk_anchors_generate`, csrc/api.cu) behind the mirror's
    SSDInputEncoder constructor against the real reference on the same random configurations (no GPU needed)."""
    from ssd_keras_b200.ssd_encoder_decoder.ssd_input_encoder import SSDInputEncoder
    cfg, gt = encoder_case(seed)
    key = 'enc/%d' % seed
    check_inputs(ref, key, cfg, *gt)
    m = SSDInputEncoder(**cfg)
    np.testing.assert_array_equal(m.anchors, ref[key + '/anchors'])
    tpl = m.generate_encoding_template(2)
    np.testing.assert_array_equal(tpl, ref[key + '/template2'])
    assert len(m.boxes_list) == int(ref[key + '/n_layers'])
    for i, a in enumerate(m.boxes_list):
        np.testing.assert_array_equal(a, ref['%s/boxes/%d' % (key, i)])
