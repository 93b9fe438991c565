"""Device-side photometric distortions (ssdk_photometric, assemble_images_device(..., pixel_ops=)): cv2.cvtColor's whole uint8
domains, the REAL reference's photometric classes and SSDPhotometricDistortions (tests/golden/make_photometric_golden.py), and
oracle/photometric.py + oracle/augment.py on VOC-sized batches."""
import ctypes as C
import hashlib
import io
import json
import lzma
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
with lzma.open(os.path.join(HERE, 'golden', 'ref_photometric_golden.npz.xz')) as _f:
    G = dict(np.load(io.BytesIO(_f.read())))
META = json.load(open(os.path.join(HERE, 'golden', 'ref_photometric_golden.json')))
EXPAND_BG = (123, 117, 104)


@pytest.fixture(scope='module', autouse=True)
def _built():
    import __graft_entry__ as entry
    entry.build()


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def case_image(seed, h, w):
    img = np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
    g = np.arange(w, dtype=np.int64) * 255 // max(w - 1, 1)
    img[0] = np.stack([g, g, g], -1)
    img[1] = 0
    img[2] = 255
    img[3, :, 0], img[3, :, 1], img[3, :, 2] = 255, g, 0
    return img


def encode(specs):
    from ssd_keras_b200.data_generator import batch_assembly as ba
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


def pixels(images, pixel_ops, dtype='uint8'):
    """The photometric pass alone: every image keeps its size (no geometric op), one batch per size."""
    import torch
    from ssd_keras_b200.data_generator.batch_assembly import assemble_images_device
    out = [None] * len(images)
    by = {}
    for i, im in enumerate(images):
        by.setdefault(im.shape[:2], []).append(i)
    for (h, w), idx in by.items():
        got = assemble_images_device([images[i] for i in idx], None, h, w, dtype=getattr(torch, dtype),
                                     pixel_ops=[pixel_ops[i] for i in idx]).cpu().numpy()
        for k, i in enumerate(idx):
            out[i] = got[k]
    return out


@pytest.mark.parametrize('name', ['rgb2hsv', 'roundtrip', 'hsv2rgb', 'hsv2rgb_rows16'])
def test_full_domains_equal_cv2_digests(name):
    """All 2^24 RGB colours (4096 x 4096) and all 181 x 256 x 256 HSV triples (2896 x 4096, and as rows of 16 pixels) through the
    device: bit-exact to the default cv2.cvtColor."""
    from oracle import photometric
    from ssd_keras_b200.data_generator import batch_assembly as ba
    if name.startswith('hsv2rgb'):
        x = photometric.hsv_domain()
        if name == 'hsv2rgb_rows16':
            x = x.reshape(-1, 16, 3)
        ops = [ba.convert_color('HSV', 'RGB')]
    else:
        x = photometric.rgb_domain()
        ops = [ba.convert_color('RGB', 'HSV')] + ([ba.convert_color('HSV', 'RGB')] if name == 'roundtrip' else [])
    got = pixels([x], [ops])[0]
    assert digest(got) == META['domains'][name]['optimized']


@pytest.mark.parametrize('dtype', ['float32', 'uint8'])
def test_reference_cases(dtype):
    cases = META['cases']
    images = [case_image(c['seed'], *c['src']) for c in cases]
    got = pixels(images, [encode(c['ops']) for c in cases], dtype)
    for i, c in enumerate(cases):
        g = got[i]
        assert g.dtype == np.dtype(dtype)
        g = g.astype(np.uint8)
        assert np.array_equal(g.astype(dtype), got[i])
        if 'out_digest' in c:
            assert digest(g) == c['out_digest'], c['name']
        else:
            np.testing.assert_array_equal(g, G['case%d' % i], err_msg=c['name'])


def test_ssd_photometric_distortions_seeds():
    from ssd_keras_b200.data_generator.batch_assembly import ssd_photometric_distortions
    images, ops = [], []
    for rec in META['ssd']:
        images.append(case_image(9000 + rec['seed'], *rec['src']))
        np.random.seed(rec['seed'])
        ops.append(ssd_photometric_distortions())
    got = pixels(images, ops)
    for rec, g in zip(META['ssd'], got):
        assert digest(g) == rec['out_digest'], rec['seed']


@pytest.mark.parametrize('dtype', ['float32', 'uint8'])
def test_full_chains(dtype):
    """Photometric -> expand -> crop -> flip -> resize in each mode, one batch: the reference's outputs (INTER_CUBIC: OpenCV's
    portable resize of the same distorted image, within 1 of the default) and its boxes."""
    import torch
    from ssd_keras_b200.data_generator.batch_assembly import augment_batch_device, assemble_images_device, ssd_photometric_distortions
    chains = META['chains']
    images, px = [], []
    for c in chains:
        images.append(case_image(c['seed'], *c['src']))
        np.random.seed(c['np_seed'])
        px.append(ssd_photometric_distortions())
    ops = [encode_geometric(c['ops']) for c in chains]
    h, w = chains[0]['out']
    got = assemble_images_device(images, ops, h, w, dtype=getattr(torch, dtype), pixel_ops=px).cpu().numpy()
    for i, c in enumerate(chains):
        g = got[i].astype(np.int32)
        ref = G['chain%d' % i].astype(np.int32)
        if c.get('generic'):
            np.testing.assert_array_equal(g, G['chain_generic%d' % i].astype(np.int32), err_msg=c['name'])
            assert np.abs(g - ref).max() <= 1
        else:
            np.testing.assert_array_equal(g, ref, err_msg=c['name'])
    _, (gt, offs, _, _, _) = augment_batch_device(images, [G['chain_in%d' % i] for i in range(len(chains))], ops, h, w, pixel_ops=px)
    gt, offs = gt.cpu().numpy(), offs.cpu().numpy()
    for i in range(len(chains)):
        np.testing.assert_array_equal(gt[offs[i]:offs[i + 1]].astype(np.float64), G['chain_out%d' % i].astype(np.float32).astype(np.float64))


def _voc_batch(seed, B=32):
    from ssd_keras_b200.data_generator import batch_assembly as ba
    rng = np.random.default_rng(seed)
    np.random.seed(seed)
    images, ops, px = [], [], []
    for b in range(B):
        h, w = (375, 500) if b % 2 == 0 else (500, 375)
        images.append(rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
        px.append(ba.ssd_photometric_distortions())
        lst = []
        if rng.uniform() < 0.5:
            r = rng.uniform(1, 4)
            ph, pw = int(h * r), int(w * r)
            lst.append(ba.crop_pad(-int(rng.integers(0, ph - h + 1)), -int(rng.integers(0, pw - w + 1)), ph, pw, background=EXPAND_BG))
            h, w = ph, pw
        if rng.uniform() < 0.8:
            ph, pw = int(h * rng.uniform(0.3, 1)), int(w * rng.uniform(0.3, 1))
            lst.append(ba.crop_pad(int(rng.integers(0, h - ph + 1)), int(rng.integers(0, w - pw + 1)), ph, pw, center_point_filter=True))
            h, w = ph, pw
        if rng.uniform() < 0.5:
            lst.append(ba.flip(w, 'horizontal'))
        lst.append(ba.resize(h, w, 300, 300, interpolation_mode=int(rng.integers(0, 5))))
        ops.append(lst)
    return images, ops, px


def test_voc_batch_equals_oracle():
    """B=32 VOC-sized sources with seeded SSD photometric lists plus the geometric chain: oracle/photometric.py then
    oracle/augment.py (INTER_CUBIC is the portable resize there too)."""
    import torch
    from oracle import augment, photometric
    from ssd_keras_b200.data_generator.batch_assembly import assemble_images_device
    images, ops, px = _voc_batch(3)
    got = assemble_images_device(images, ops, 300, 300, pixel_ops=px).cpu().numpy()
    want = augment.assemble_images(photometric.apply_images(images, px), ops, 300, 300)
    bad = np.argwhere((got != want).any(axis=(1, 2, 3))).ravel().tolist()
    assert not bad, bad
    u8 = assemble_images_device(images, ops, 300, 300, dtype=torch.uint8, pixel_ops=px).cpu().numpy()
    np.testing.assert_array_equal(u8.astype(np.float32), want)
    # the photometric pass alone, in place on the ragged upload (arbitrary source offsets: heads, bodies and tails)
    alone = pixels(images, px)
    for b in range(len(images)):
        np.testing.assert_array_equal(alone[b], photometric.apply(images[b], px[b]), err_msg=str(b))


def test_expand_background_is_not_distorted():
    from oracle import photometric
    from ssd_keras_b200.data_generator import batch_assembly as ba
    img = case_image(4, 20, 30)
    px = [ba.convert_data_type('float32'), ba.brightness(40.0), ba.convert_data_type('uint8')]
    out = ba.assemble_images_device([img], [[ba.crop_pad(-10, -12, 50, 60, background=EXPAND_BG)]], 50, 60, pixel_ops=[px]).cpu().numpy()[0]
    inside = np.zeros((50, 60), bool)
    inside[10:30, 12:42] = True
    np.testing.assert_array_equal(out[inside].reshape(20, 30, 3), photometric.apply(img, px).astype(np.float32))
    assert (out[~inside] == np.asarray(EXPAND_BG, np.float32)).all()


def test_separate_destination_any_alignment():
    """The C entry with dst != src at every byte misalignment: the image is the same, whatever path moves the bytes."""
    import torch
    from oracle import photometric
    from ssd_keras_b200 import _ffi
    from ssd_keras_b200.data_generator import batch_assembly as ba
    images = [case_image(11, 37, 53), case_image(12, 64, 64), case_image(13, 5, 7)]
    px = [[ba.convert_data_type('float32'), ba.contrast(1.3), ba.convert_data_type('uint8'), ba.convert_color('RGB', 'HSV'),
           ba.convert_data_type('float32'), ba.hue(-11.5), ba.convert_data_type('uint8'), ba.convert_color('HSV', 'RGB')]] * 3
    raw, max_ops = ba._pack_pixel_ops(px, 3)
    ops_dev = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
    flat = np.concatenate([a.reshape(-1) for a in images])
    offs = torch.from_numpy(np.cumsum([0] + [a.size for a in images[:-1]]).astype(np.int64)).cuda()
    hw = torch.from_numpy(np.asarray([a.shape[:2] for a in images], np.int32).reshape(-1)).cuda()
    want = np.concatenate([photometric.apply(a, p).reshape(-1) for a, p in zip(images, px)])
    for s_off in (0, 1, 5):
        for d_off in (0, 3, 7, 16):
            src = torch.zeros(flat.size + 32, dtype=torch.uint8, device='cuda')
            src[s_off:s_off + flat.size] = torch.from_numpy(flat).cuda()
            dst = torch.zeros(flat.size + 32, dtype=torch.uint8, device='cuda')
            rc = _ffi.lib().ssdk_photometric(_ffi.context(), C.c_void_p(src.data_ptr() + s_off), C.c_void_p(dst.data_ptr() + d_off),
                                             _ffi.dptr(offs), _ffi.dptr(hw), 3, _ffi.dptr(ops_dev), max_ops, _ffi.stream_ptr())
            assert rc == _ffi.SSDK_OK
            np.testing.assert_array_equal(dst.cpu().numpy()[d_off:d_off + flat.size], want, err_msg=str((s_off, d_off)))


def test_launch_count():
    from ssd_keras_b200 import _ffi
    from ssd_keras_b200.data_generator import batch_assembly as ba
    images, ops, px = _voc_batch(9, B=4)
    ba.assemble_images_device(images, ops, 300, 300)
    n0 = _ffi.launch_count()
    ba.assemble_images_device(images, ops, 300, 300)
    n1 = _ffi.launch_count()
    ba.assemble_images_device(images, ops, 300, 300, pixel_ops=px)
    n2 = _ffi.launch_count()
    assert n1 - n0 == 1 and n2 - n1 == 2


def test_refusals_raise_before_any_launch():
    import torch
    from test_oracle_photometric_cpu import REFUSED
    from ssd_keras_b200 import _ffi
    from ssd_keras_b200.data_generator import batch_assembly as ba
    img = case_image(1, 10, 12)
    src = torch.from_numpy(img.reshape(-1)).cuda()
    offs = torch.zeros(1, dtype=torch.int64, device='cuda')
    hw = torch.tensor([10, 12], dtype=torch.int32, device='cuda')
    for name, ops in REFUSED:
        n0 = _ffi.launch_count()
        with pytest.raises(ValueError):
            ba.assemble_images_device([img], None, 10, 12, pixel_ops=[ops])
        raw, max_ops = ba._pack_pixel_ops([ops], 1)
        ops_dev = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
        rc = _ffi.lib().ssdk_photometric(_ffi.context(), _ffi.dptr(src), _ffi.dptr(src), _ffi.dptr(offs), _ffi.dptr(hw), 1,
                                         _ffi.dptr(ops_dev), max_ops, _ffi.stream_ptr())
        assert rc == _ffi.SSDK_ERR_INVALID, name
        assert _ffi.launch_count() == n0, name
    with pytest.raises(ValueError):
        ba.assemble_images_device([img, img], None, 10, 12, pixel_ops=[[]])                 # one list per image
    hw0 = torch.tensor([0, 12], dtype=torch.int32, device='cuda')
    assert _ffi.lib().ssdk_photometric(_ffi.context(), _ffi.dptr(src), _ffi.dptr(src), _ffi.dptr(offs), _ffi.dptr(hw0), 1, C.c_void_p(0), 0,
                                       _ffi.stream_ptr()) == _ffi.SSDK_ERR_INVALID
