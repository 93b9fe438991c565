#!/usr/bin/env python
"""Time the device image assembly (assemble_images_device / ssdk_assemble_images) on the SSD chain at B=32.

VOC-sized sources (500x375 and 375x500 uint8, seeded) go through expand (SSDExpand's background) -> crop -> flip h -> resize to
300x300 float32, the interpolation mode drawn per image like ResizeRandomInterp.  The upload of the sources is done once and
the entry point is timed on its own with CUDA events: warm-up, then the median of --iters calls (each call includes the
validation read-back of the op lists).  Reported: microseconds per batch, the algorithmic bytes (source bytes +
B*300*300*3*4 written) and their rate as a fraction of the B200 data-sheet HBM bandwidth (7.7 TB/s).  If cv2 is importable the
same chain is also timed on the host (NumPy canvas + cv2.resize, one image after another) and the host's core count is stated.
The card's name and power limit are read in the same run.

    python tools/augment_bench.py [--iters 200] [--warmup 20] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))
sys.path.insert(0, ROOT)

B, OUT = 32, 300
HBM_BYTES_PER_S = 7.7e12
EXPAND_BG = (123, 117, 104)


def chain(seed):
    from ssd_keras_b200.data_generator import batch_assembly as ba
    rng = np.random.default_rng(seed)
    images, ops, plain = [], [], []
    for b in range(B):
        h, w = (375, 500) if b % 2 == 0 else (500, 375)
        images.append(rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
        r = rng.uniform(1, 4)
        ph, pw = int(h * r), int(w * r)
        ey, ex = -int(rng.integers(0, ph - h + 1)), -int(rng.integers(0, pw - w + 1))
        ch, cw = int(ph * rng.uniform(0.3, 1)), int(pw * rng.uniform(0.3, 1))
        cy, cx = int(rng.integers(0, ph - ch + 1)), int(rng.integers(0, pw - cw + 1))
        mode = int(rng.integers(0, 5))
        ops.append([ba.crop_pad(ey, ex, ph, pw, background=EXPAND_BG), ba.crop_pad(cy, cx, ch, cw, center_point_filter=True),
                    ba.flip(cw), ba.resize(ch, cw, OUT, OUT, interpolation_mode=mode)])
        plain.append((ey, ex, ph, pw, cy, cx, ch, cw, mode))
    return images, ops, plain


def host_chain(images, plain):
    """The reference's image arithmetic on the host: CropPad canvases, [:, ::-1], cv2.resize, float32 stack."""
    import cv2
    out = np.empty((B, OUT, OUT, 3), np.float32)
    for b, (img, (ey, ex, ph, pw, cy, cx, ch, cw, mode)) in enumerate(zip(images, plain)):
        h, w = img.shape[:2]
        canvas = np.empty((ph, pw, 3), np.uint8)
        canvas[:] = EXPAND_BG
        canvas[-ey:-ey + h, -ex:-ex + w] = img
        crop = canvas[cy:cy + ch, cx:cx + cw].copy()
        crop = crop[:, ::-1]
        out[b] = cv2.resize(crop, (OUT, OUT), interpolation=mode)
    return out


def gpu_info():
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True,
                           text=True, timeout=60)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else 'unknown'
    except (OSError, subprocess.SubprocessError):
        return 'unknown'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit('augment_bench.py needs a CUDA device')
    from ssd_keras_b200 import _ffi
    from ssd_keras_b200.build import build_library
    from ssd_keras_b200.data_generator import batch_assembly as ba
    build_library()
    images, ops, plain = chain(2024)
    out = ba.assemble_images_device(images, ops, OUT, OUT)                      # the public call, once (validation + upload)

    # the timed call: the entry point on device-resident sources and op lists
    raw, max_ops = ba._pack_ops(ops, B)
    ops_dev = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
    src = torch.from_numpy(np.concatenate([a.reshape(-1) for a in images])).cuda()
    offs = torch.from_numpy(np.cumsum([0] + [a.size for a in images[:-1]]).astype(np.int64)).cuda()
    hw = torch.from_numpy(np.asarray([a.shape[:2] for a in images], np.int32).reshape(-1)).cuda()
    out2 = torch.empty_like(out)

    def call():
        _ffi.check(_ffi.lib().ssdk_assemble_images(_ffi.context(), _ffi.dptr(src), _ffi.dptr(offs), _ffi.dptr(hw), B, _ffi.dptr(ops_dev),
                                                   max_ops, OUT, OUT, 0, _ffi.dptr(out2), _ffi.stream_ptr()))

    for _ in range(args.warmup):
        call()
    torch.cuda.synchronize()
    times = []
    for _ in range(args.iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) * 1e3)
    assert torch.equal(out, out2)
    med = float(np.median(times))
    src_bytes = int(sum(a.size for a in images))
    alg_bytes = src_bytes + B * OUT * OUT * 3 * 4
    res = {'metric': 'assemble_images_us_per_batch', 'B': B, 'out': [OUT, OUT], 'dtype': 'float32', 'iters': args.iters,
           'warmup': args.warmup, 'median_us': round(med, 2), 'p10_us': round(float(np.percentile(times, 10)), 2),
           'p90_us': round(float(np.percentile(times, 90)), 2), 'algorithmic_bytes': alg_bytes, 'source_bytes': src_bytes,
           'achieved_GBps': round(alg_bytes / (med * 1e-6) / 1e9, 1), 'hbm_fraction': round(alg_bytes / (med * 1e-6) / HBM_BYTES_PER_S, 4),
           'modes': [p[-1] for p in plain], 'gpu': gpu_info(), 'torch': torch.__version__}
    try:
        import cv2
        host_chain(images, plain)
        t = []
        for _ in range(5):
            t0 = time.perf_counter()
            ref = host_chain(images, plain)
            t.append((time.perf_counter() - t0) * 1e6)
        res['host_cv2_us_per_batch'] = round(float(np.median(t)), 1)
        res['host_cores'] = os.cpu_count()
        res['host_cv2_threads'] = cv2.getNumThreads()
        res['host_cv2_version'] = cv2.__version__
        res['host_max_abs_diff'] = int(np.abs(ref - out.cpu().numpy()).max())
    except ImportError:
        res['host_cv2_us_per_batch'] = None
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
