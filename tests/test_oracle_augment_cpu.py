"""oracle/augment.py (the fused crop/pad + flip + cv2.resize map of ssdk_assemble_images, restated in NumPy) against the REAL
reference's CropPad / Flip / Resize outputs (tests/golden/make_image_golden.py), and the op encoders of
ssd_keras_b200.data_generator.batch_assembly packing background and interpolation mode into ``flags``."""
import hashlib
import io
import itertools
import json
import lzma
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
with lzma.open(os.path.join(HERE, 'golden', 'ref_image_golden.npz.xz')) as _f:
    G = dict(np.load(io.BytesIO(_f.read())))
META = json.load(open(os.path.join(HERE, 'golden', 'ref_image_golden.json')))
CASES = META['cases']


def case_image(seed, h, w):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


def encode_ops(lst):
    from ssd_keras_b200.data_generator import batch_assembly as ba
    out = []
    for o in lst:
        if o[0] == 'crop_pad':
            out.append(ba.crop_pad(o[1], o[2], o[3], o[4], center_point_filter=o[5], clip_boxes=o[6], background=o[7]))
        elif o[0] == 'flip':
            out.append(ba.flip(o[1], o[2]))
        else:
            out.append(ba.resize(o[1], o[2], o[3], o[4], drop_degenerate=o[5], interpolation_mode=o[6]))
    return out


def _uses(case, mode):
    return any(o[0] == 'resize' and o[6] == mode for o in case['ops'])


@pytest.mark.parametrize('i', range(len(CASES)), ids=[c['name'] for c in CASES])
def test_oracle_equals_reference_chain(i):
    from oracle import augment
    c = CASES[i]
    img = case_image(c['seed'], *c['src'])
    assert hashlib.sha256(img.tobytes()).hexdigest()[:16] == c['digest'], 'the synthetic inputs are generated differently now'
    got = augment.assemble_image(img, encode_ops(c['ops']), *c['out'])
    ref = G['img%d' % i]
    if c.get('generic'):
        # INTER_CUBIC: bit-exact to OpenCV's portable implementation; the default optimised cv2.resize is within 1 of it
        assert _uses(c, augment.INTER_CUBIC), c['name']
        np.testing.assert_array_equal(got, G['generic%d' % i])
        assert np.abs(got.astype(np.int32) - ref.astype(np.int32)).max() <= 1
    else:
        np.testing.assert_array_equal(got, ref)


def test_only_cubic_needs_the_portable_golden():
    from oracle import augment
    flagged = [c for c in CASES if c.get('generic')]
    assert flagged and all(_uses(c, augment.INTER_CUBIC) for c in flagged)
    total = sum(G['img%d' % i].size for i, c in enumerate(CASES) if _uses(c, augment.INTER_CUBIC))
    differ = sum(int((G['img%d' % i] != G['generic%d' % i]).sum()) for i, c in enumerate(CASES) if c.get('generic'))
    assert 0 < differ / total < 0.05, differ / total


def test_resize_rules_on_random_sizes():
    """The five rules of oracle.augment.resize through the fused map with identity crops, against the stored reference."""
    from oracle import augment
    c = next(c for c in CASES if c['name'] == 'mode1_down')
    img = case_image(c['seed'], *c['src'])
    h, w = c['src']
    ops = encode_ops([['crop_pad', 0, 0, h, w, False, False, [0, 0, 0]]] + c['ops'])
    np.testing.assert_array_equal(augment.assemble_image(img, ops, *c['out']), G['img%d' % CASES.index(c)])


def test_encoders_pack_background_and_mode():
    from ssd_keras_b200.data_generator import batch_assembly as ba
    from oracle import augment
    op = ba.crop_pad(-3, -4, 10, 12, background=(123, 117, 104))
    assert op[0] == 1 and augment.background_rgb(op[1]) == (123, 117, 104) and op[1] & 3 == 2
    op = ba.crop_pad(0, 0, 5, 5, center_point_filter=True, background=(255, 255, 255))
    assert augment.background_rgb(op[1]) == (255, 255, 255) and op[1] & 3 == 3 and -2 ** 31 <= op[1] < 2 ** 31
    assert ba.crop_pad(1, 2, 3, 4)[1] == 2                                      # default background packs to zero bits
    for m in range(5):
        op = ba.resize(10, 20, 30, 40, interpolation_mode=m)
        assert augment.resize_mode(op[1]) == m and op[1] & 3 == 1
    assert (ba.INTER_NEAREST, ba.INTER_LINEAR, ba.INTER_CUBIC, ba.INTER_AREA, ba.INTER_LANCZOS4) == (0, 1, 2, 3, 4)
    assert ba.resize(1, 2, 3, 4)[1] == 1 | (ba.INTER_LINEAR << 8)
    with pytest.raises(ValueError):
        ba.crop_pad(0, 0, 1, 1, background=(0, 0, 256))


@pytest.mark.parametrize('filt,clip,bg', list(itertools.product([False, True], [False, True], [(0, 0, 0), (123, 117, 104), (255, 0, 255)])))
def test_crop_pad_low_bits_unchanged(filt, clip, bg):
    """Bits 0-1 (what the box kernel reads) are what they were before the background was added."""
    from ssd_keras_b200.data_generator import batch_assembly as ba
    op = ba.crop_pad(-1, 2, 30, 40, center_point_filter=filt, clip_boxes=clip, background=bg)
    assert op[1] & 3 == (1 if filt else 0) | (2 if clip else 0)
    assert op[2:] == (-1.0, 2.0, 30.0, 40.0)


@pytest.mark.parametrize('drop,mode', list(itertools.product([False, True], range(5))))
def test_resize_low_bits_unchanged(drop, mode):
    from ssd_keras_b200.data_generator import batch_assembly as ba
    op = ba.resize(10, 20, 30, 40, drop_degenerate=drop, interpolation_mode=mode)
    assert op[1] & 3 == (1 if drop else 0) and op[2:] == (10.0, 20.0, 30.0, 40.0)


def test_oracle_refuses_what_the_kernel_refuses():
    from ssd_keras_b200.data_generator import batch_assembly as ba
    from oracle import augment
    img = np.zeros((10, 12, 3), np.uint8)
    bad = [
        [ba.resize(10, 12, 5, 5), ba.resize(5, 5, 6, 6)],                       # two resizes
        [ba.resize(10, 12, 5, 5), ba.flip(5)],                                  # flip after the resize
        [ba.resize(10, 12, 5, 5), ba.crop_pad(0, 0, 5, 5)],                     # crop after the resize
        [ba.resize(10, 12, 5, 5, interpolation_mode=7)],                        # unknown mode
        [ba.crop_pad(11, 0, 5, 5), ba.resize(5, 5, 5, 5)],                      # patch past the image
    ]
    for ops in bad:
        with pytest.raises(ValueError):
            augment.assemble_image(img, ops, 5, 5)
    with pytest.raises(ValueError):
        augment.assemble_image(img, [ba.resize(10, 12, 5, 6)], 5, 5)           # final size
    with pytest.raises(ValueError):
        augment.assemble_image(np.zeros((0, 3, 3), np.uint8), [], 0, 3)        # empty source
