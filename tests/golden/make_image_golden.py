#!/usr/bin/env python
"""Golden vectors for the device-side image assembly: the REAL reference's CropPad / Flip / Resize / BoxFilter
(data_generator/object_detection_2d_patch_sampling_ops.py, ..._geometric_ops.py, ..._image_boxes_validation_utils.py) and
SSDExpand's background (data_augmentation_chain_original_ssd.py) applied to seeded synthetic uint8 images and label arrays.

Images are regenerated from their seed at test time (``case_image``); every case stores a digest of its input image, so a
change in how inputs are generated is reported as such.  Each case stores the output image of the chain (``cv2.resize`` as
installed, OpenCV 4.13) and the output boxes.  For INTER_CUBIC the default optimised ``cv2.resize`` and OpenCV's own
portable implementation (``cv2.setUseOptimized(False)``) differ by 1 on a few percent of values; the portable output is
stored as well (``generic<i>``) where it differs.

Writes tests/golden/ref_image_golden.npz.xz and ref_image_golden.json.  Needs the reference checkout and cv2."""
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
sys.path.insert(0, os.environ.get('SSD_REFERENCE_ROOT', '/root/reference'))

import cv2                                                                                          # noqa: E402
from data_generator.data_augmentation_chain_original_ssd import SSDExpand                          # noqa: E402
from data_generator.object_detection_2d_geometric_ops import Flip, Resize                          # noqa: E402
from data_generator.object_detection_2d_image_boxes_validation_utils import BoxFilter              # noqa: E402
from data_generator.object_detection_2d_patch_sampling_ops import CropPad                          # noqa: E402

MODES = [cv2.INTER_NEAREST, cv2.INTER_LINEAR, cv2.INTER_CUBIC, cv2.INTER_AREA, cv2.INTER_LANCZOS4]
EXPAND_BG = tuple(int(c) for c in SSDExpand().expand.background)


def case_image(seed, h, w):
    """The synthetic input of a case: uniform uint8 noise (the hardest input for an interpolation rule)."""
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


def case_labels(seed, h, w):
    rng = np.random.default_rng(seed + 100000)
    n = int(rng.integers(1, 8))
    x0 = rng.integers(0, max(w - 1, 1), n); y0 = rng.integers(0, max(h - 1, 1), n)
    x1 = np.minimum(x0 + rng.integers(1, max(w // 2, 2), n), w); y1 = np.minimum(y0 + rng.integers(1, max(h // 2, 2), n), h)
    return np.stack([rng.integers(1, 21, n), x0, y0, x1, y1], axis=1).astype(np.float64)


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def run_chain(image, labels, ops):
    """Apply the reference classes in list order; returns (image, labels)."""
    img, lab = image, labels
    for o in ops:
        if o[0] == 'crop_pad':
            _, py, px, ph, pw, filt, clip, bg = o
            bf = BoxFilter(check_overlap=True, check_min_area=False, check_degenerate=False, overlap_criterion='center_point') if filt else None
            img, lab = CropPad(py, px, ph, pw, clip_boxes=clip, box_filter=bf, background=tuple(bg))(img, lab)
        elif o[0] == 'flip':
            img, lab = Flip(dim=o[2])(img, lab)
        elif o[0] == 'resize':
            _, ih, iw, oh, ow, drop, mode = o
            assert img.shape[:2] == (ih, iw)
            bf = BoxFilter(check_overlap=False, check_min_area=False, check_degenerate=True) if drop else None
            img, lab = Resize(height=oh, width=ow, interpolation_mode=mode, box_filter=bf)(img, lab)
        else:
            raise ValueError(o[0])
    return img, lab


def main():
    cases = []

    def add(name, h, w, ops, out_hw):
        cases.append({'name': name, 'seed': 1000 + len(cases), 'src': [h, w], 'ops': ops, 'out': list(out_hw)})

    OH, OW = 60, 80
    shapes = {'up': (23, 31), 'down': (157, 203), 'int2': (2 * OH, 2 * OW), 'int3': (3 * OH, 3 * OW), 'thin_w': (500, 7),
              'thin_h': (7, 500)}
    for m in MODES:
        for tag, (h, w) in shapes.items():
            add('mode%d_%s' % (m, tag), h, w, [['resize', h, w, OH, OW, True, m]], (OH, OW))
        add('mode%d_1x1' % m, 1, 1, [['resize', 1, 1, OH, OW, True, m]], (OH, OW))
        # the SSD chain: expand -> crop -> flip h -> resize
        add('mode%d_ssd_chain' % m, 75, 100, [['crop_pad', -21, -34, 130, 170, False, False, EXPAND_BG],
                                              ['crop_pad', 12, 40, 97, 118, True, True, [0, 0, 0]],
                                              ['flip', 118, 'horizontal'], ['resize', 97, 118, OH, OW, True, m]], (OH, OW))
    add('expand_only', 40, 50, [['crop_pad', -10, -7, 70, 80, False, False, EXPAND_BG]], (70, 80))
    add('crop_only_past_edge', 50, 60, [['crop_pad', 20, 30, 45, 50, True, True, [9, 200, 77]]], (45, 50))
    add('crop_inside', 50, 60, [['crop_pad', 5, 8, 30, 40, True, True, [0, 0, 0]]], (30, 40))
    add('flip_v', 30, 40, [['flip', 30, 'vertical'], ['resize', 30, 40, OH, OW, True, cv2.INTER_LINEAR]], (OH, OW))
    add('flip_hv', 30, 40, [['flip', 40, 'horizontal'], ['flip', 30, 'vertical']], (30, 40))
    add('no_resize_target', 90, 100, [['crop_pad', 10, 15, OH, OW, True, True, [0, 0, 0]], ['flip', OW, 'horizontal']], (OH, OW))
    add('crop_on_expand_background', 20, 20, [['crop_pad', -30, -30, 100, 100, False, False, EXPAND_BG],
                                              ['crop_pad', 0, 0, 25, 25, True, True, [0, 0, 0]],
                                              ['resize', 25, 25, OH, OW, True, cv2.INTER_CUBIC]], (OH, OW))
    add('two_backgrounds', 20, 30, [['crop_pad', -10, -10, 40, 50, False, False, EXPAND_BG],
                                    ['crop_pad', -4, 30, 50, 30, True, True, [250, 3, 40]],
                                    ['resize', 50, 30, OH, OW, True, cv2.INTER_LANCZOS4]], (OH, OW))
    add('expand_crop_flip_resize_voc', 375, 500, [['crop_pad', -120, -300, 750, 1000, False, False, EXPAND_BG],
                                                  ['crop_pad', 80, 250, 400, 420, True, True, [0, 0, 0]],
                                                  ['flip', 420, 'horizontal'], ['resize', 400, 420, 300, 300, True, cv2.INTER_LINEAR]],
        (300, 300))

    arrays = {}
    n_cubic_diff = n_cubic = 0
    for i, c in enumerate(cases):
        h, w = c['src']
        img = case_image(c['seed'], h, w)
        lab = case_labels(c['seed'], h, w)
        c['digest'] = digest(img)
        out, lab_out = run_chain(img, lab, c['ops'])
        assert out.shape == (c['out'][0], c['out'][1], 3), (c['name'], out.shape)
        arrays['img%d' % i] = out
        arrays['in%d' % i] = lab
        arrays['out%d' % i] = np.asarray(lab_out, np.float64).reshape(-1, 5)
        cv2.setUseOptimized(False)
        gen, _ = run_chain(img, lab, c['ops'])
        cv2.setUseOptimized(True)
        if not np.array_equal(gen, out):
            arrays['generic%d' % i] = gen
            c['generic'] = True
            n_cubic_diff += int((gen != out).sum())
        if any(o[0] == 'resize' and o[6] == cv2.INTER_CUBIC for o in c['ops']):
            n_cubic += out.size
    buf = io.BytesIO()
    np.savez(buf, **arrays)
    with open(os.path.join(HERE, 'ref_image_golden.npz.xz'), 'wb') as f:
        f.write(lzma.compress(buf.getvalue(), preset=9))
    with open(os.path.join(HERE, 'ref_image_golden.json'), 'w') as f:
        json.dump({'opencv': cv2.__version__, 'expand_background': list(EXPAND_BG), 'cases': cases}, f, indent=1)
    print('wrote %d cases, %d bytes; cubic: optimised vs portable differ on %d of %d values'
          % (len(cases), os.path.getsize(os.path.join(HERE, 'ref_image_golden.npz.xz')), n_cubic_diff, n_cubic))


if __name__ == '__main__':
    main()
