"""The photometric oracle (oracle/photometric.py) and the host side of the pixel-op lists, against the REAL reference's outputs
(tests/golden/make_photometric_golden.py): cv2.cvtColor over its whole uint8 domains, the reference classes on seeded images,
SSDPhotometricDistortions' draws and RNG state for every stored seed, and full photometric + geometric chains.  No device."""
import hashlib
import io
import json
import lzma
import os

import numpy as np
import pytest

from oracle import augment, photometric
from ssd_keras_b200 import _ffi
from ssd_keras_b200.data_generator import batch_assembly as ba

HERE = os.path.dirname(os.path.abspath(__file__))
with lzma.open(os.path.join(HERE, 'golden', 'ref_photometric_golden.npz.xz')) as _f:
    G = dict(np.load(io.BytesIO(_f.read())))
META = json.load(open(os.path.join(HERE, 'golden', 'ref_photometric_golden.json')))


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def state_digest():
    st = np.random.get_state()
    return digest(np.concatenate([st[1].view(np.uint8), np.asarray([st[2], st[3]], np.int64).view(np.uint8),
                                  np.asarray([st[4]], np.float64).view(np.uint8)]))


def case_image(seed, h, w):
    img = np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
    g = np.arange(w, dtype=np.int64) * 255 // max(w - 1, 1)
    img[0] = np.stack([g, g, g], -1)
    img[1] = 0
    img[2] = 255
    img[3, :, 0], img[3, :, 1], img[3, :, 2] = 255, g, 0
    return img


def encode(specs):
    out = []
    for s in specs:
        if s[0] == 'convert_data_type':
            out.append(ba.convert_data_type(s[1]))
        elif s[0] == 'convert_color':
            out.append(ba.convert_color(s[1], s[2]))
        else:
            out.append(getattr(ba, s[0])(s[1]))
    return out


def encode_geometric(lst):
    out = []
    for o in lst:
        if o[0] == 'crop_pad':
            out.append(ba.crop_pad(o[1], o[2], o[3], o[4], center_point_filter=o[5], clip_boxes=o[6], background=o[7]))
        elif o[0] == 'flip':
            out.append(ba.flip(o[1], o[2]))
        else:
            out.append(ba.resize(o[1], o[2], o[3], o[4], drop_degenerate=o[5], interpolation_mode=o[6]))
    return out


@pytest.mark.parametrize('name', ['rgb2hsv', 'roundtrip', 'hsv2rgb'])
def test_full_domain_digests(name):
    """RGB2HSV and the round trip over all 2^24 colours, HSV2RGB over all 181 x 256 x 256 triples: bit-exact to the default
    cv2.cvtColor, and the portable restatement bit-exact to cv2's portable path."""
    d = META['domains'][name]
    if name == 'hsv2rgb':
        x = photometric.hsv_domain()
        assert digest(x) == META['domains']['hsv_input']
        opt, port = photometric.hsv2rgb(x, True), photometric.hsv2rgb(x, False)
    else:
        x = photometric.rgb_domain()
        assert digest(x) == META['domains']['rgb_input']
        hsv = photometric.rgb2hsv(x)
        opt = port = hsv
        if name == 'roundtrip':
            opt, port = photometric.hsv2rgb(hsv, True), photometric.hsv2rgb(hsv, False)
    assert digest(opt) == d['optimized']
    assert digest(port) == d['portable']
    diff = (opt != port).any(-1)
    assert int(diff.sum()) == d['n_diff']
    if d['n_diff']:
        np.testing.assert_array_equal(x[diff], G['diff_%s_in' % name])
        np.testing.assert_array_equal(opt[diff], G['diff_%s_opt' % name])
        np.testing.assert_array_equal(port[diff], G['diff_%s_port' % name])
        assert np.abs(opt[diff].astype(int) - port[diff].astype(int)).max() == 1


def test_hsv2rgb_scalar_part_of_rows():
    """The same triples in rows of 16 pixels, all of which cv2's default build converts with its scalar (rounding) code."""
    x = photometric.hsv_domain().reshape(-1, 16, 3)
    assert digest(photometric.hsv2rgb(x)) == META['domains']['hsv2rgb_rows16']['optimized']


def test_hue_never_exceeds_179_and_180_is_reachable():
    assert photometric.rgb2hsv(photometric.rgb_domain())[..., 0].max() == 179
    x = np.zeros((1, 1, 3), np.uint8)
    out = photometric.apply(x, [ba.convert_data_type('float32'), ba.hue(-1e-7), ba.convert_data_type('uint8')])
    assert out[0, 0, 0] == 180
    assert np.float32(-4.7e-7) % 180.0 == 180.0


@pytest.mark.parametrize('i', range(len(META['cases'])), ids=[c['name'] for c in META['cases']])
def test_reference_cases(i):
    c = META['cases'][i]
    img = case_image(c['seed'], *c['src'])
    assert digest(img) == c['digest']
    ops = encode(c['ops'])
    ba._pixel_state(0, ops)
    out = photometric.apply(img, ops)
    if 'out_digest' in c:
        assert digest(out) == c['out_digest']
    else:
        np.testing.assert_array_equal(out, G['case%d' % i])


def test_ssd_photometric_distortions_draws_and_state():
    """ssd_photometric_distortions() makes the reference's np.random calls in its order, leaves the same RNG state, and its list
    reproduces the reference's output image, for every stored seed."""
    names = ('uniform', 'choice', 'randint')
    orig = {n: getattr(np.random, n) for n in names}
    assert len(META['ssd']) >= 64
    for rec in META['ssd']:
        img = case_image(9000 + rec['seed'], *rec['src'])
        assert digest(img) == rec['digest']
        log = []

        def wrap(n):
            def f(*a, **kw):
                r = orig[n](*a, **kw)
                log.append([n, [float(v) for v in a], float(r)])
                return r
            return f

        np.random.seed(rec['seed'])
        for n in names:
            setattr(np.random, n, wrap(n))
        try:
            ops = ba.ssd_photometric_distortions()
        finally:
            for n in names:
                setattr(np.random, n, orig[n])
        assert log == rec['draws'], rec['seed']
        assert state_digest() == rec['state'], rec['seed']
        ba._pixel_state(0, ops)
        out = photometric.apply(img, ops)
        assert digest(out) == rec['out_digest'], rec['seed']
        if 'ssd%d' % rec['seed'] in G:
            np.testing.assert_array_equal(out, G['ssd%d' % rec['seed']])


def test_ssd_photometric_distortions_always_round_trips():
    np.random.seed(0)
    for _ in range(50):
        kinds = [o[0] for o in ba.ssd_photometric_distortions()]
        assert kinds.count(_ffi.PIXOP_RGB2HSV) == 1 and kinds.count(_ffi.PIXOP_HSV2RGB) == 1
        assert kinds.index(_ffi.PIXOP_RGB2HSV) < kinds.index(_ffi.PIXOP_HSV2RGB)
        assert _ffi.PIXOP_CHANNEL_SWAP not in kinds                                   # RandomChannelSwap(prob=0.0)


@pytest.mark.parametrize('i', range(len(META['chains'])), ids=[c['name'] for c in META['chains']])
def test_full_chains(i):
    """Photometric distortions, then expand -> crop -> flip -> resize: oracle/photometric.py followed by oracle/augment.py."""
    c = META['chains'][i]
    img = case_image(c['seed'], *c['src'])
    assert digest(img) == c['digest']
    np.random.seed(c['np_seed'])
    dist = photometric.apply(img, ba.ssd_photometric_distortions())
    assert digest(dist) == c['photometric_digest']
    out = augment.assemble_image(dist, encode_geometric(c['ops']), *c['out'])
    want = G['chain_generic%d' % i] if c.get('generic') else G['chain%d' % i]
    np.testing.assert_array_equal(out, want.astype(out.dtype))
    if c.get('generic'):
        assert np.abs(out.astype(int) - G['chain%d' % i].astype(int)).max() <= 1


def test_builders_refuse_like_the_reference():
    with pytest.raises(ValueError, match="`to` can be either of 'uint8' or 'float32'."):
        ba.convert_data_type('float64')
    for cur, to in (('RGB', 'GRAY'), ('HSV', 'GRAY'), ('BGR', 'HSV'), ('RGB', 'LAB')):
        with pytest.raises(NotImplementedError):
            ba.convert_color(cur, to)
    assert ba.convert_color('RGB', 'RGB') == ba.channel_swap((0, 1, 2))
    for f in (ba.contrast, ba.saturation):
        for v in (0.0, -1.0):
            with pytest.raises(ValueError, match='It must be `factor > 0`.'):
                f(v)
        with pytest.raises(ValueError):
            f(float('inf'))
    for d in (-180.0001, 181, float('nan')):
        with pytest.raises(ValueError, match=r'`delta` must be in the closed interval `\[-180, 180\]`.'):
            ba.hue(d)
    assert ba.hue(-180)[2] == -180.0 and ba.hue(180)[2] == 180.0
    with pytest.raises(ValueError):
        ba.brightness(float('nan'))
    for order in ((0, 1, 3), (0, 1), (-1, 0, 1), (0, 1, 2, 0)):
        with pytest.raises(ValueError):
            ba.channel_swap(order)


REFUSED = [
    ('colour conversion in float state', [(_ffi.PIXOP_TO_FLOAT, 0, 0.0), (_ffi.PIXOP_RGB2HSV, 0, 0.0), (_ffi.PIXOP_TO_U8, 0, 0.0)]),
    ('HSV2RGB in float state', [(_ffi.PIXOP_TO_FLOAT, 0, 0.0), (_ffi.PIXOP_HSV2RGB, 0, 0.0), (_ffi.PIXOP_TO_U8, 0, 0.0)]),
    ('brightness in uint8 state', [(_ffi.PIXOP_BRIGHTNESS, 0, 3.0)]),
    ('contrast in uint8 state', [(_ffi.PIXOP_CONTRAST, 0, 1.1)]),
    ('saturation in uint8 state', [(_ffi.PIXOP_SATURATION, 0, 1.1)]),
    ('hue in uint8 state', [(_ffi.PIXOP_HUE, 0, 1.0)]),
    ('ends in float state', [(_ffi.PIXOP_TO_FLOAT, 0, 0.0)]),
    ('unknown op', [(10, 0, 0.0)]),
    ('negative op', [(-1, 0, 0.0)]),
    ('hue delta out of range', [(_ffi.PIXOP_TO_FLOAT, 0, 0.0), (_ffi.PIXOP_HUE, 0, 180.5), (_ffi.PIXOP_TO_U8, 0, 0.0)]),
    ('zero contrast factor', [(_ffi.PIXOP_TO_FLOAT, 0, 0.0), (_ffi.PIXOP_CONTRAST, 0, 0.0), (_ffi.PIXOP_TO_U8, 0, 0.0)]),
    ('negative saturation factor', [(_ffi.PIXOP_TO_FLOAT, 0, 0.0), (_ffi.PIXOP_SATURATION, 0, -0.5), (_ffi.PIXOP_TO_U8, 0, 0.0)]),
    ('NaN brightness', [(_ffi.PIXOP_TO_FLOAT, 0, 0.0), (_ffi.PIXOP_BRIGHTNESS, 0, float('nan')), (_ffi.PIXOP_TO_U8, 0, 0.0)]),
    ('swap index 3', [(_ffi.PIXOP_CHANNEL_SWAP, 0 | (1 << 8) | (3 << 16), 0.0)]),
    ('swap high bits', [(_ffi.PIXOP_CHANNEL_SWAP, 1 << 24, 0.0)]),
    ('too many ops', [(_ffi.PIXOP_TO_U8, 0, 0.0)] * (_ffi.MAX_PIXEL_OPS + 1)),
]


@pytest.mark.parametrize('name,ops', REFUSED, ids=[r[0] for r in REFUSED])
def test_typed_state_refusals_on_the_host(name, ops):
    with pytest.raises(ValueError):
        ba._pixel_state(0, ops)


def test_valid_lists_pass_the_host_check():
    for ops in ([], [(_ffi.PIXOP_TO_U8, 0, 0.0)], [ba.convert_data_type('float32'), ba.convert_data_type('float32'), ba.convert_data_type('uint8')],
                [ba.channel_swap((2, 2, 0))], [(_ffi.PIXOP_TO_U8, 0, 0.0), (_ffi.PIXOP_END, 0, 0.0), (_ffi.PIXOP_HUE, 0, 999.0)]):
        ba._pixel_state(0, ops)
