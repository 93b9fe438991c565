#!/usr/bin/env python
"""Golden vectors for the device-side photometric distortions: the REAL reference's ConvertDataType / ConvertColor / Brightness /
Contrast / Saturation / Hue / ChannelSwap (data_generator/object_detection_2d_photometric_ops.py) and SSDPhotometricDistortions
(data_augmentation_chain_original_ssd.py:146-206), as installed with OpenCV 4.13 and NumPy 2.

  * ``domains``: sha256 digests of ``cv2.cvtColor`` over whole domains, for ``setUseOptimized(True)`` and ``(False)``:
    COLOR_RGB2HSV and the round trip RGB2HSV -> HSV2RGB over all 2^24 RGB colours (a 4096 x 4096 image, pixel i =
    (i >> 16, (i >> 8) & 255, i & 255)), and COLOR_HSV2RGB over all 181 x 256 x 256 triples with H <= 180 (2896 x 4096, same
    layout; H = 180 is reachable through Hue + ConvertDataType), and the same triples as rows of 16 pixels (``hsv2rgb_rows16``:
    cv2 converts the last (width mod 32) pixels of a row with its scalar code).  Where the two paths differ on the whole
    domains, the inputs and both outputs are stored (``diff_<name>_in`` / ``_opt`` / ``_port``).
  * ``cases``: the reference classes on seeded images, one op at a time and in combinations, with the edge cases named.
  * ``ssd``: ``SSDPhotometricDistortions()(image, labels)`` under ``np.random.seed(s)``; the draws are logged by wrapping
    ``np.random.uniform`` / ``choice`` / ``randint`` during the call, and a digest of ``np.random.get_state()`` afterwards and of
    the output image are stored (the first few outputs in full).
  * ``chains``: photometric (seeded SSDPhotometricDistortions) -> SSDExpand's CropPad -> crop -> flip -> Resize in each of the
    five modes, with output images and boxes.  For INTER_CUBIC the portable resize of the same distorted image is stored too
    (``generic<i>``), like tests/golden/make_image_golden.py does.

Images are regenerated from their seed at test time (``case_image``) and every input stores its digest.
Writes tests/golden/ref_photometric_golden.npz.xz and ref_photometric_golden.json.  Needs the reference checkout and cv2."""
import hashlib
import io
import json
import lzma
import os
import sys

import numpy as np

np.float = float   # noqa
np.int = int       # noqa
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.environ.get('SSD_REFERENCE_ROOT', '/root/reference'))

import cv2                                                                                          # noqa: E402
from data_generator.data_augmentation_chain_original_ssd import SSDPhotometricDistortions          # noqa: E402
from data_generator.object_detection_2d_photometric_ops import (Brightness, ChannelSwap, Contrast, ConvertColor,  # noqa: E402
                                                                ConvertDataType, Hue, RandomChannelSwap, Saturation)
from make_image_golden import EXPAND_BG, MODES, run_chain                                           # noqa: E402

N_SEEDS = 80
N_SEEDS_STORED = 6


def case_image(seed, h, w):
    """Uniform uint8 noise with a few structured rows: greys (H = 0, S = 0), black, white and saturated primaries, so that
    clipping, hue wrap-around and the S = 0 path are all hit."""
    img = np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
    g = np.arange(w, dtype=np.int64) * 255 // max(w - 1, 1)
    img[0] = np.stack([g, g, g], -1)
    img[1] = 0
    img[2] = 255
    img[3, :, 0], img[3, :, 1], img[3, :, 2] = 255, g, 0
    return img


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def rgb_domain():
    i = np.arange(1 << 24, dtype=np.uint32)
    return np.stack([i >> 16, (i >> 8) & 255, i & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)


def hsv_domain():
    i = np.arange(181 << 16, dtype=np.uint32)
    return np.stack([i >> 16, (i >> 8) & 255, i & 255], -1).astype(np.uint8).reshape(2896, 4096, 3)


def reference_op(spec):
    """A reference class instance for one JSON op spec."""
    kind = spec[0]
    if kind == 'convert_data_type':
        return ConvertDataType(to=spec[1])
    if kind == 'convert_color':
        return ConvertColor(current=spec[1], to=spec[2])
    return {'brightness': Brightness, 'contrast': Contrast, 'saturation': Saturation, 'hue': Hue}.get(kind, ChannelSwap)(
        tuple(spec[1]) if kind == 'channel_swap' else spec[1])


def run_specs(image, specs):
    x = image
    for s in specs:
        x = reference_op(s)(x)
    return x


def domains(arrays):
    out = {}

    def both(name, fn, x, store=True):
        cv2.setUseOptimized(True)
        opt = fn(x)
        cv2.setUseOptimized(False)
        port = fn(x)
        cv2.setUseOptimized(True)
        d = (opt != port).any(-1)
        out[name] = {'optimized': digest(opt), 'portable': digest(port), 'n_diff': int(d.sum())}
        if d.any() and store:
            arrays['diff_%s_in' % name] = x[d]
            arrays['diff_%s_opt' % name] = opt[d]
            arrays['diff_%s_port' % name] = port[d]
        return opt

    rgb = rgb_domain()
    both('rgb2hsv', lambda x: cv2.cvtColor(x, cv2.COLOR_RGB2HSV), rgb)
    both('roundtrip', lambda x: cv2.cvtColor(cv2.cvtColor(x, cv2.COLOR_RGB2HSV), cv2.COLOR_HSV2RGB), rgb)
    both('hsv2rgb', lambda x: cv2.cvtColor(x, cv2.COLOR_HSV2RGB), hsv_domain())
    # the same triples in rows of 16 pixels: every pixel is in the last (width mod 32) of its row, which cv2 converts with its
    # scalar code (rounding instead of truncating)
    both('hsv2rgb_rows16', lambda x: cv2.cvtColor(x, cv2.COLOR_HSV2RGB), hsv_domain().reshape(-1, 16, 3),
         store=False)
    out['rgb_input'] = digest(rgb)
    out['hsv_input'] = digest(hsv_domain())
    return out


def main():
    arrays = {}
    meta = {'opencv': cv2.__version__, 'numpy': np.__version__, 'domains': domains(arrays)}

    F, U = ['convert_data_type', 'float32'], ['convert_data_type', 'uint8']
    TO_HSV, TO_RGB = ['convert_color', 'RGB', 'HSV'], ['convert_color', 'HSV', 'RGB']
    cases = []

    def add(name, specs, h=24, w=40):
        cases.append({'name': name, 'seed': 5000 + len(cases), 'src': [h, w], 'ops': specs})

    add('to_float_to_u8', [F, U])
    add('identity_u8_to_u8', [U, U, F, F, U])
    for d in (0.5, -0.5, 1.5, 2.5, -32.0, 31.99, 17.123456789, -4.7e-7):
        add('brightness_%g' % d, [F, ['brightness', d], U])
    for f in (0.5, 1.5, 0.5000001, 1.3333333333, 0.77):
        add('contrast_%g' % f, [F, ['contrast', f], U])
    add('rgb2hsv', [TO_HSV])
    add('hsv_roundtrip', [TO_HSV, TO_RGB])
    for f in (0.5, 1.5, 1.23456789, 0.9):
        add('saturation_%g' % f, [TO_HSV, F, ['saturation', f], U, TO_RGB])
    for d in (-18.0, 18.0, 7.3, -0.5, 0.5, -1e-7, -4.7e-7, 179.9, -180.0, 180.0, 12.5):
        add('hue_%g' % d, [TO_HSV, F, ['hue', d], U, TO_RGB])
    add('hue_to_180_raw_hsv', [TO_HSV, F, ['hue', -1e-7], U])                    # H = 0 -> exactly 180.0 -> 180
    for perm in RandomChannelSwap().permutations:
        add('channel_swap_%d%d%d' % perm, [['channel_swap', list(perm)]])
    add('channel_swap_float_state', [F, ['channel_swap', [2, 1, 0]], ['brightness', 3.25], U])
    add('channel_swap_hsv_state', [TO_HSV, ['channel_swap', [1, 0, 2]], TO_RGB])
    add('ssd_sequence1_all', [F, ['brightness', -12.75], ['contrast', 1.21], U, TO_HSV, F, ['saturation', 1.37], ['hue', -9.6], U,
                              TO_RGB])
    add('ssd_sequence2_all', [F, ['brightness', 20.5], U, TO_HSV, F, ['saturation', 0.61], ['hue', 15.2], U, TO_RGB, F,
                              ['contrast', 0.73], U, ['channel_swap', [2, 0, 1]]])
    add('ssd_sequence_none', [F, U, TO_HSV, F, U, TO_RGB])
    add('constant_chain_order', [F, ['brightness', 5.5], ['contrast', 1.1], U, TO_HSV, F, ['saturation', 1.2], ['hue', 3.3], U,
                                 TO_RGB], 7, 13)
    add('voc_sized', [F, ['brightness', -7.5], ['contrast', 1.05], U, TO_HSV, F, ['saturation', 1.1], ['hue', 4.4], U, TO_RGB],
        375, 500)
    for i, c in enumerate(cases):
        img = case_image(c['seed'], *c['src'])
        c['digest'] = digest(img)
        out = run_specs(img, c['ops'])
        assert out.dtype == np.uint8 and out.shape == img.shape, c['name']
        if out.size > 64 * 1024:
            c['out_digest'] = digest(out)
        else:
            arrays['case%d' % i] = out
    meta['cases'] = cases

    # SSDPhotometricDistortions under np.random.seed(s): the draws, the RNG state afterwards, the output
    ssd = []
    names = ('uniform', 'choice', 'randint')
    orig = {n: getattr(np.random, n) for n in names}
    for k in range(N_SEEDS):
        h, w = (30, 44) if k % 2 else (41, 29)
        img = case_image(9000 + k, h, w)
        log = []

        def wrap(n):
            def f(*a, **kw):
                r = orig[n](*a, **kw)
                log.append([n, [float(v) for v in a], float(r)])
                return r
            return f

        np.random.seed(k)
        for n in names:
            setattr(np.random, n, wrap(n))
        try:
            out, _ = SSDPhotometricDistortions()(img, np.zeros((0, 5)))
        finally:
            for n in names:
                setattr(np.random, n, orig[n])
        st = np.random.get_state()
        rec = {'seed': k, 'src': [h, w], 'digest': digest(img), 'draws': log, 'state': digest(np.concatenate([st[1].view(np.uint8),
               np.asarray([st[2], st[3]], np.int64).view(np.uint8), np.asarray([st[4]], np.float64).view(np.uint8)])),
               'out_digest': digest(out)}
        if k < N_SEEDS_STORED:
            arrays['ssd%d' % k] = out
        ssd.append(rec)
    meta['ssd'] = ssd

    # full chains: photometric -> expand -> crop -> flip -> resize, each mode
    chains = []
    for m in MODES:
        seed = 7000 + m
        h, w = 45, 60
        img = case_image(seed, h, w)
        lab = np.asarray([[1, 5, 6, 30, 40], [3, 20, 10, 58, 44]], np.float64)
        np.random.seed(seed)
        dist, _ = SSDPhotometricDistortions()(img, lab)
        ops = [['crop_pad', -9, -13, 70, 90, False, False, list(EXPAND_BG)], ['crop_pad', 4, 10, 52, 66, True, True, [0, 0, 0]],
               ['flip', 66, 'horizontal'], ['resize', 52, 66, 30, 40, True, m]]
        out, lab_out = run_chain(dist, lab, ops)
        i = len(chains)
        arrays['chain%d' % i] = out
        arrays['chain_in%d' % i] = lab
        arrays['chain_out%d' % i] = np.asarray(lab_out, np.float64).reshape(-1, 5)
        rec = {'name': 'chain_mode%d' % m, 'seed': seed, 'src': [h, w], 'digest': digest(img), 'np_seed': seed, 'ops': ops,
               'out': [30, 40], 'photometric_digest': digest(dist)}
        cv2.setUseOptimized(False)
        gen, _ = run_chain(dist, lab, ops)
        cv2.setUseOptimized(True)
        if not np.array_equal(gen, out):
            arrays['chain_generic%d' % i] = gen
            rec['generic'] = True
        chains.append(rec)
    meta['chains'] = chains

    buf = io.BytesIO()
    np.savez(buf, **arrays)
    path = os.path.join(HERE, 'ref_photometric_golden.npz.xz')
    with open(path, 'wb') as f:
        f.write(lzma.compress(buf.getvalue(), preset=9))
    with open(os.path.join(HERE, 'ref_photometric_golden.json'), 'w') as f:
        json.dump(meta, f, indent=1)
    print('wrote %d cases, %d seeds, %d chains, %d bytes; domains %s' % (len(cases), len(ssd), len(chains), os.path.getsize(path),
                                                                         json.dumps(meta['domains'])))


if __name__ == '__main__':
    main()
