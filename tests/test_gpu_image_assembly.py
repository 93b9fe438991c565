"""Device-side image assembly (ssdk_assemble_images): ragged uint8 images through crop/pad, flips and cv2.resize's five modes
into the model's input batch, against the REAL reference's outputs (tests/golden/make_image_golden.py) and against
oracle/augment.py at sizes the goldens do not store; one op list drives pixels and boxes."""
import io
import json
import lzma
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
with lzma.open(os.path.join(HERE, 'golden', 'ref_image_golden.npz.xz')) as _f:
    G = dict(np.load(io.BytesIO(_f.read())))
META = json.load(open(os.path.join(HERE, 'golden', 'ref_image_golden.json')))
CASES = META['cases']
EXPAND_BG = tuple(META['expand_background'])


@pytest.fixture(scope='module', autouse=True)
def _built():
    import __graft_entry__ as entry
    entry.build()


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


def _groups():
    by = {}
    for i, c in enumerate(CASES):
        by.setdefault(tuple(c['out']), []).append(i)
    return sorted(by.items())


@pytest.mark.parametrize('dtype', ['float32', 'uint8'])
def test_device_equals_reference_goldens(dtype):
    """Every stored case, batched by output size.  INTER_CUBIC is bit-exact to OpenCV's portable implementation and within 1
    of the default optimised cv2.resize; every other mode is bit-exact to cv2.resize."""
    import torch
    from ssd_keras_b200.data_generator.batch_assembly import assemble_images_device
    tdt = getattr(torch, dtype)
    for (h, w), idx in _groups():
        imgs = [case_image(CASES[i]['seed'], *CASES[i]['src']) for i in idx]
        out = assemble_images_device(imgs, [encode_ops(CASES[i]['ops']) for i in idx], h, w, dtype=tdt)
        assert out.dtype == tdt and tuple(out.shape) == (len(idx), h, w, 3)
        got = out.cpu().numpy()
        for k, i in enumerate(idx):
            c = CASES[i]
            g = got[k].astype(np.int32)
            ref = G['img%d' % i].astype(np.int32)
            if c.get('generic'):
                np.testing.assert_array_equal(g, G['generic%d' % i].astype(np.int32), err_msg=c['name'])
                assert np.abs(g - ref).max() <= 1, c['name']
            else:
                np.testing.assert_array_equal(g, ref, err_msg=c['name'])


def _voc_batch(seed, B=32):
    """B VOC-sized ragged sources through the SSD chain (expand -> crop -> flip -> resize to 300x300), random mode per image."""
    from ssd_keras_b200.data_generator import batch_assembly as ba
    rng = np.random.default_rng(seed)
    images, labels, ops = [], [], []
    for b in range(B):
        h, w = (375, 500) if b % 2 == 0 else (500, 375)
        images.append(rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
        n = int(rng.integers(1, 6))
        x0 = rng.integers(0, w - 20, n); y0 = rng.integers(0, h - 20, n)
        labels.append(np.stack([rng.integers(1, 21, n), x0, y0, x0 + rng.integers(5, 20, n), y0 + rng.integers(5, 20, n)], 1).astype(np.float64))
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
        lst.append(ba.box_filter())
        ops.append(lst)
    return images, labels, ops


def test_voc_batch_equals_oracle():
    import torch
    from oracle import augment
    from ssd_keras_b200.data_generator.batch_assembly import assemble_images_device
    images, _, ops = _voc_batch(7)
    got = assemble_images_device(images, ops, 300, 300).cpu().numpy()
    want = augment.assemble_images(images, ops, 300, 300)
    bad = np.argwhere((got != want).any(axis=(1, 2, 3))).ravel().tolist()
    assert not bad, [(b, [o[:2] for o in ops[b]]) for b in bad]
    u8 = assemble_images_device(images, ops, 300, 300, dtype=torch.uint8).cpu().numpy()
    np.testing.assert_array_equal(u8.astype(np.float32), want)


def test_augment_batch_boxes_equal_box_path():
    from ssd_keras_b200.data_generator.batch_assembly import assemble_batch_device, augment_batch_device
    images, labels, ops = _voc_batch(11)
    imgs, (gt, offs, stats, total, max_g) = augment_batch_device(images, labels, ops, 300, 300)
    gt2, offs2, stats2, total2, max_g2 = assemble_batch_device(labels, ops)
    assert tuple(imgs.shape) == (32, 300, 300, 3) and (total, max_g) == (total2, max_g2)
    np.testing.assert_array_equal(offs.cpu().numpy(), offs2.cpu().numpy())
    np.testing.assert_array_equal(stats.cpu().numpy(), stats2.cpu().numpy())
    n = int(offs2[-1])
    np.testing.assert_array_equal(gt.cpu().numpy()[:n], gt2.cpu().numpy()[:n])


def test_golden_boxes_through_augment_batch():
    """The boxes the reference chain produced for the stored cases, from the same op lists that produced the pixels."""
    from ssd_keras_b200.data_generator.batch_assembly import augment_batch_device
    for (h, w), idx in _groups():
        imgs = [case_image(CASES[i]['seed'], *CASES[i]['src']) for i in idx]
        _, (gt, offs, _, _, _) = augment_batch_device(imgs, [G['in%d' % i] for i in idx], [encode_ops(CASES[i]['ops']) for i in idx], h, w)
        gt, offs = gt.cpu().numpy(), offs.cpu().numpy()
        for k, i in enumerate(idx):
            np.testing.assert_array_equal(gt[offs[k]:offs[k + 1]].astype(np.float64), G['out%d' % i].astype(np.float32).astype(np.float64),
                                          err_msg=CASES[i]['name'])


def test_model_input_equals_host_assembled():
    """SSD300's y_pred on the device-assembled batch equals y_pred on the oracle-assembled images uploaded from the host."""
    import torch
    import bench
    from oracle import augment
    from ssd_keras_b200.data_generator.batch_assembly import assemble_images_device
    from ssd_keras_b200.models.keras_ssd300 import ssd_300
    images, _, ops = _voc_batch(5)
    model = ssd_300((300, 300, 3), bench.N_CLASSES, mode='inference', scales=bench.SC300, precision='bf16x3')
    model.set_weights(bench._weights())
    dev = assemble_images_device(images, ops, 300, 300)
    host = torch.from_numpy(augment.assemble_images(images, ops, 300, 300)).cuda()
    y_dev = model.forward_device(dev).cpu().numpy()
    y_host = model.forward_device(host).cpu().numpy()
    assert np.isfinite(y_dev).all()
    np.testing.assert_array_equal(y_dev, y_host)


def test_validation_errors():
    import ctypes as C
    import torch
    from ssd_keras_b200 import _ffi
    from ssd_keras_b200.data_generator import batch_assembly as ba
    from ssd_keras_b200.data_generator.batch_assembly import assemble_images_device
    img = np.zeros((10, 12, 3), np.uint8)
    cases = [
        ([img], [[ba.resize(10, 12, 5, 5), ba.resize(5, 5, 6, 6)]], 6, 6),        # two resizes
        ([img], [[ba.resize(10, 12, 5, 5), ba.flip(5)]], 5, 5),                     # flip after the resize
        ([img], [[ba.resize(10, 12, 5, 5), ba.crop_pad(0, 0, 5, 5)]], 5, 5),        # crop/pad after the resize
        ([img], [[ba.resize(10, 12, 5, 5, interpolation_mode=5)]], 5, 5),           # mode outside 0..4
        ([img], [[ba.resize(10, 12, 5, 6)]], 5, 5),                                 # final size
        ([img], [[ba.crop_pad(0, 13, 5, 5), ba.resize(5, 5, 5, 5)]], 5, 5),         # patch origin past the image
        ([img], [[]], 5, 5),                                                         # no ops, wrong size
        ([np.zeros((0, 12, 3), np.uint8)], [[]], 0, 12),                            # empty source
        ([np.zeros((10, 12, 4), np.uint8)], [[ba.resize(10, 12, 5, 5)]], 5, 5),     # four channels
        ([np.zeros((10, 12, 3), np.float32)], [[ba.resize(10, 12, 5, 5)]], 5, 5),   # not uint8
    ]
    for imgs, ops, h, w in cases:
        with pytest.raises(ValueError):
            assemble_images_device(imgs, ops, h, w)
    # the C entry point refuses the same lists on its own (validation of what is on the device, before the launch)
    for ops, h, w in [([ba.resize(10, 12, 5, 5), ba.resize(5, 5, 6, 6)], 6, 6), ([ba.resize(10, 12, 5, 5, interpolation_mode=9)], 5, 5),
                      ([ba.crop_pad(11, 0, 5, 5)], 5, 5), ([ba.resize(10, 12, 5, 6)], 5, 5), ([ba.resize(10, 12, 5, 5), ba.flip(5)], 5, 5)]:
        raw, max_ops = ba._pack_ops([ops], 1)
        ops_dev = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
        src = torch.from_numpy(img.reshape(-1)).cuda()
        offs = torch.zeros(1, dtype=torch.int64, device='cuda')
        hw = torch.tensor([10, 12], dtype=torch.int32, device='cuda')
        out = torch.empty((1, h, w, 3), device='cuda')
        rc = _ffi.lib().ssdk_assemble_images(_ffi.context(), _ffi.dptr(src), _ffi.dptr(offs), _ffi.dptr(hw), 1, _ffi.dptr(ops_dev), max_ops,
                                             h, w, 0, _ffi.dptr(out), _ffi.stream_ptr())
        assert rc == _ffi.SSDK_ERR_INVALID, ops
    hw0 = torch.tensor([0, 12], dtype=torch.int32, device='cuda')
    rc = _ffi.lib().ssdk_assemble_images(_ffi.context(), _ffi.dptr(src), _ffi.dptr(offs), _ffi.dptr(hw0), 1, C.c_void_p(0), 0, 5, 12, 0,
                                         _ffi.dptr(out), _ffi.stream_ptr())
    assert rc == _ffi.SSDK_ERR_INVALID
