#!/usr/bin/env python
"""Time the device image assembly (assemble_images_device / ssdk_assemble_images) on the SSD chain at B=32.

VOC-sized sources (500x375 and 375x500 uint8, seeded) go through expand (SSDExpand's background) -> crop -> flip h -> resize to
300x300 float32, the interpolation mode drawn per image like ResizeRandomInterp.  The upload of the sources is done once and
the entry point is timed on its own with CUDA events: warm-up, then the median of --iters calls (each call includes the
validation read-back of the op lists).  Reported: microseconds per batch, the algorithmic bytes (source bytes +
B*300*300*3*4 written) and their rate as a fraction of the B200 data-sheet HBM bandwidth (7.7 TB/s).  If cv2 is importable the
same chain is also timed on the host (NumPy canvas + cv2.resize, one image after another) and the host's core count is stated.
The card's name and power limit are read in the same run.

--photometric adds a ``photometric`` object to the result: the same sources with one seeded ``ssd_photometric_distortions()``
list per image (np.random.seed(2024)), timed as the ssdk_photometric pass alone (sources -> a second buffer) and as the whole
chain (ssdk_photometric in place, then ssdk_assemble_images), with the pass's algorithmic bytes (2 x source bytes: read once,
written once) as a fraction of 7.7 TB/s; and, when cv2 is importable, the host equivalent (NumPy float32 ops + cv2.cvtColor, one
image after another).

    python tools/augment_bench.py [--iters 200] [--warmup 20] [--photometric] [--out FILE.json]
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


def host_photometric(images, pixel_ops):
    """SSDPhotometricDistortions' arithmetic on the host, one image after another: NumPy float32 ops and cv2.cvtColor."""
    import cv2
    from ssd_keras_b200 import _ffi as F
    out = []
    for img, ops in zip(images, pixel_ops):
        x = img
        for kind, arg, a0 in ops:
            if kind == F.PIXOP_TO_FLOAT:
                x = x.astype(np.float32)
            elif kind == F.PIXOP_TO_U8:
                x = np.round(x, decimals=0).astype(np.uint8)
            elif kind == F.PIXOP_RGB2HSV:
                x = cv2.cvtColor(x, cv2.COLOR_RGB2HSV)
            elif kind == F.PIXOP_HSV2RGB:
                x = cv2.cvtColor(x, cv2.COLOR_HSV2RGB)
            elif kind == F.PIXOP_BRIGHTNESS:
                x = np.clip(x + a0, 0, 255)
            elif kind == F.PIXOP_CONTRAST:
                x = np.clip(127.5 + a0 * (x - 127.5), 0, 255)
            elif kind == F.PIXOP_SATURATION:
                x[:, :, 1] = np.clip(x[:, :, 1] * a0, 0, 255)
            elif kind == F.PIXOP_HUE:
                x[:, :, 0] = (x[:, :, 0] + a0) % 180.0
            else:
                x = x[:, :, [arg & 255, (arg >> 8) & 255, (arg >> 16) & 255]]
        out.append(x)
    return out


def time_us(fn, iters, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) * 1e3)
    return times


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
    ap.add_argument('--photometric', action='store_true')
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
    if args.photometric:
        res['photometric'] = photometric_rows(args, images, ops, src, offs, hw, ops_dev, max_ops, out2)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')


def photometric_rows(args, images, ops, src, offs, hw, ops_dev, max_ops, out2):
    import torch
    from oracle import photometric
    from ssd_keras_b200 import _ffi
    from ssd_keras_b200.data_generator import batch_assembly as ba
    np.random.seed(2024)
    px = [ba.ssd_photometric_distortions() for _ in range(B)]
    raw, px_max = ba._pack_pixel_ops(px, B)
    px_dev = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
    dst = torch.empty_like(src)
    work = torch.empty_like(src)
    L, ctx = _ffi.lib(), _ffi.context()

    def alone():
        _ffi.check(L.ssdk_photometric(ctx, _ffi.dptr(src), _ffi.dptr(dst), _ffi.dptr(offs), _ffi.dptr(hw), B, _ffi.dptr(px_dev), px_max,
                                      _ffi.stream_ptr()))

    def whole():
        work.copy_(src)                                                    # the in-place pass needs fresh sources each time
        _ffi.check(L.ssdk_photometric(ctx, _ffi.dptr(work), _ffi.dptr(work), _ffi.dptr(offs), _ffi.dptr(hw), B, _ffi.dptr(px_dev), px_max,
                                      _ffi.stream_ptr()))
        _ffi.check(L.ssdk_assemble_images(ctx, _ffi.dptr(work), _ffi.dptr(offs), _ffi.dptr(hw), B, _ffi.dptr(ops_dev), max_ops, OUT, OUT, 0,
                                          _ffi.dptr(out2), _ffi.stream_ptr()))

    def copy_only():
        work.copy_(src)

    t_alone = time_us(alone, args.iters, args.warmup)
    t_whole = time_us(whole, args.iters, args.warmup)
    t_copy = time_us(copy_only, args.iters, args.warmup)
    want = photometric.apply_images(images, px)
    got = dst.cpu().numpy()
    pos = 0
    for w in want:
        assert np.array_equal(got[pos:pos + w.size], w.reshape(-1))
        pos += w.size
    src_bytes = int(sum(a.size for a in images))
    med = float(np.median(t_alone))
    r = {'pass_median_us': round(med, 2), 'pass_p10_us': round(float(np.percentile(t_alone, 10)), 2),
         'pass_p90_us': round(float(np.percentile(t_alone, 90)), 2), 'pass_algorithmic_bytes': 2 * src_bytes,
         'pass_achieved_GBps': round(2 * src_bytes / (med * 1e-6) / 1e9, 1),
         'pass_hbm_fraction': round(2 * src_bytes / (med * 1e-6) / HBM_BYTES_PER_S, 4),
         'chain_median_us': round(float(np.median(t_whole)) - float(np.median(t_copy)), 2),
         'chain_note': 'photometric in place + assemble_images, minus the median of the source copy each timed call makes',
         'source_copy_median_us': round(float(np.median(t_copy)), 2), 'pixel_ops_per_image': [len(p) for p in px]}
    try:
        import cv2
        host_photometric(images, px)
        t = []
        for _ in range(5):
            t0 = time.perf_counter()
            h = host_photometric(images, px)
            t.append((time.perf_counter() - t0) * 1e6)
        r['host_us_per_batch'] = round(float(np.median(t)), 1)
        r['host_cores'] = os.cpu_count()
        r['host_cv2_threads'] = cv2.getNumThreads()
        r['host_cv2_version'] = cv2.__version__
        r['host_max_abs_diff'] = int(max(np.abs(a.astype(int) - b.astype(int)).max() for a, b in zip(h, want)))
    except ImportError:
        r['host_us_per_batch'] = None
    return r


if __name__ == '__main__':
    main()
