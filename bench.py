#!/usr/bin/env python
"""bench.py -- SSD300 images/sec (forward + DecodeDetections) on N B200s, plus the reference CPU arm.

  python bench.py --gpus 1 --steps 20 --warmup 3                   # this framework (one JSON line on stdout)
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
         bench.py --gpus N --steps K --warmup W                     # N ranks, NCCL, weak scaling (32 images / GPU)
  python bench.py --impl reference --steps 3 --warmup 1             # the reference's CPU path (oracle port) on host cores
  python bench.py --steps 20 --warmup 3 --dump-outputs DIR          # also write the last timed step's detections to DIR

Workload (BASELINE.json configs[1]): SSD300, batch 32 synthetic 300x300x3 float32 images, 21 classes, 8732 priors,
he_normal random weights (conv1_1 scaled by 1/64, see _weights), DecodeDetections(conf 0.01, iou 0.45, top_k 200, nms cap 400).
A step = one forward + decode of one batch.  `value` = images/s with inputs resident in HBM (CUDA events, max over
ranks); `e2e` = the same through SSDModel.predict with pinned host images copied H2D and the (B,200,6) result copied
D2H inside the timed region.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SC300 = [0.1, 0.2, 0.37, 0.54, 0.71, 0.88, 1.05]
BATCH = 32
N_CLASSES = 20
METRIC = 'SSD300 images/sec (fwd+decode)'
WORKLOAD = ('SSD300 inference, batch 32 per GPU, synthetic 300x300x3 float32, 21 classes, 8732 priors, he_normal random '
            'weights (conv1_1 scaled by 1/64), DecodeDetections(0.01/0.45/200/400)')


def _peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, 'measured (MEASURED_PEAKS.json)'
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}, 'fallback (B200_PROFILING.md)'


def _weights():
    """he_normal weights, zero biases, conv1_1 scaled by 1/64.  With zero biases the ReLU network is linear in the scale of its
    input, and the default preprocessing leaves pixels within +-128: unscaled, the box regressions of the heads after conv4_3
    reach ~1000, exp() overflows float32 in the decoder (infinite box coordinates) and every score saturates to 1.0.  The
    scaled first layer keeps activations in the O(1) range that trained weights produce, so the detections are finite and
    ranked by distinct scores."""
    from oracle import synth
    from oracle.model import vgg_weight_shapes
    w = synth.synth_weights(1, vgg_weight_shapes(300, N_CLASSES), bias_scale=0.0)
    w['conv1_1/kernel'] = w['conv1_1/kernel'] / np.float32(64.0)
    w['conv4_3_norm/gamma'] = np.full((512,), 20.0, np.float32)
    return w


class ClockSampler:
    """Samples SM clock / throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {'hw_slowdown': getattr(nv, 'nvmlClocksThrottleReasonHwSlowdown', 0x8),
                 'hw_thermal_slowdown': getattr(nv, 'nvmlClocksThrottleReasonHwThermalSlowdown', 0x40),
                 'sw_thermal_slowdown': getattr(nv, 'nvmlClocksThrottleReasonSwThermalSlowdown', 0x20),
                 'sw_power_cap': getattr(nv, 'nvmlClocksThrottleReasonSwPowerCap', 0x4)}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        if self._t:
            self._stop.set()
            self._t.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {'sm_mhz': med, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons), 'samples': len(self.samples)}


# ------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference CPU path, on the host cores
# ------------------------------------------------------------------------------------------------------
_POOL = None


def _decode_one(y):
    """worker: DecodeDetections restatement for one image.  The greedy NMS it delegates to tf.image.non_max_suppression -- compiled
    C++ in TensorFlow -- runs through the C restatement oracle/tf_nms.c (bit-identical to the NumPy one, which stays the fallback
    where no compiler exists): a Python NMS loop would make the CPU arm slower than the reference really is."""
    from oracle.decoder import decode_layer, tf_nms_c
    with np.errstate(all='ignore'):                 # overflowing boxes, should other weights produce them, are handled as TensorFlow does
        return decode_layer(y, 0.01, 0.45, 200, 400, True, 300, 300, nms=tf_nms_c)


def _close_pool():
    global _POOL
    if _POOL is not None:
        _POOL.close(); _POOL.join(); _POOL = None


def _decode_pool(n):
    global _POOL
    if _POOL is None:
        import multiprocessing as mp
        _POOL = mp.get_context('spawn').Pool(n)
        _POOL.map(_decode_one, [np.zeros((1, 16, N_CLASSES + 12), np.float32)] * n)      # import numpy / oracle in every worker
    return _POOL


def cpu_reference_step(images, weights, pool=None):
    """One bounded sample of the workload on the CPU: torch-CPU restatement of the Keras graph (all host threads)
    followed by the DecodeDetections restatement (NumPy + the C NMS of oracle/tf_nms.c; one image per worker process).  Returns the
    (n,200,6) detections."""
    from oracle.model import ssd_vgg_forward
    y = ssd_vgg_forward(images, weights, 300, N_CLASSES, scales=SC300)
    if pool is None:
        return _decode_one(y)
    return np.concatenate(pool.map(_decode_one, [y[i:i + 1] for i in range(y.shape[0])]), axis=0)


def _pick_threads(x, w):
    """torch's CPU convolutions do not scale to every core of a many-core host at this batch size (128 threads were 7x
    slower than 32 on the GPU boxes): time one forward per candidate thread count and keep the fastest."""
    import torch
    from oracle.model import ssd_vgg_forward
    ncpu = os.cpu_count() or 1
    best, best_t = None, 0
    for t in sorted({min(ncpu, c) for c in (8, 16, 32, 64, ncpu)}):
        torch.set_num_threads(t)
        ssd_vgg_forward(x[:1], w, 300, N_CLASSES, scales=SC300)           # warm the thread pool
        t0 = time.perf_counter()
        ssd_vgg_forward(x, w, 300, N_CLASSES, scales=SC300)
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, best_t = dt, t
    torch.set_num_threads(best_t)
    return best_t


def time_cpu_reference(n_images, reps, warmup):
    import torch
    from oracle import synth
    from oracle.decoder import decode_layer
    from oracle.model import ssd_vgg_forward
    w = _weights()
    x = synth.synth_images(0, n_images, 300, 300)
    threads = _pick_threads(x, w)
    pool = _decode_pool(min(n_images, os.cpu_count() or 1))
    for _ in range(warmup):
        cpu_reference_step(x, w, pool)
    t_fwd = t_dec = 0.0
    for _ in range(reps):
        t0 = time.perf_counter()
        y = ssd_vgg_forward(x, w, 300, N_CLASSES, scales=SC300)
        t1 = time.perf_counter()
        pool.map(_decode_one, [y[i:i + 1] for i in range(y.shape[0])])
        t2 = time.perf_counter()
        t_fwd += t1 - t0; t_dec += t2 - t1
    _close_pool()
    n = max(reps, 1)
    dt = (t_fwd + t_dec) / n
    return n_images / dt, dt, max(threads, min(n_images, os.cpu_count() or 1)), t_fwd / n, t_dec / n


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    n_img = int(os.environ.get('SSDK_REF_SAMPLE', '16'))          # images per step of the bounded CPU sample
    ips, dt, threads, t_fwd, t_dec = time_cpu_reference(n_img, args.steps, args.warmup)
    line = {'impl': 'reference', 'metric': METRIC, 'value': ips, 'unit': 'images/s', 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'sample': '%d of 32 images per step' % n_img},
            'cpu_baseline': {'value': ips, 'unit': 'images/s', 'cores': threads, 'kind': 'port',
                             'sample': '%d images per step: torch-CPU restatement of models/keras_ssd300.py (TF1/Keras2 not '
                                       'installable offline; thread count picked by calibration) %.2f s + restatement of DecodeDetections (NumPy, '
                                       'greedy NMS in compiled C like TensorFlow\'s kernel, one worker process per image) %.2f s' % (n_img, t_fwd, t_dec)},
            'e2e': {'value': ips, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
# micro-benchmarks reported under "extra" (BASELINE metric part 2: IoU-match + NMS boxes/sec)
# ------------------------------------------------------------------------------------------------------
def _time_cuda(fn, iters=10, warm=3, inner=1):
    """Median time of one call in ms: CUDA events around `inner` back-to-back calls (so that launch-bound ops are timed by the
    GPU's rate, not by the latency of a single enqueue), `iters` samples after `warm` untimed calls."""
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(inner):
            fn()
        b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / inner)
    return float(np.median(ts))


def micro_benchmarks(peaks):
    """config 3 (encode + loss at SSD300 B=32) and config 5 (P=1e5 x G=128 encode and NMS at B=256, the stated size)."""
    import torch
    from oracle import synth
    from ssd_keras_b200.keras_loss_function.keras_ssd_loss import SSDLoss
    from ssd_keras_b200.ssd_encoder_decoder.ssd_input_encoder import SSDInputEncoder
    from ssd_keras_b200.ssd_encoder_decoder.ssd_output_decoder import nms_device
    hbm = peaks['hbm_gbs']
    out = {}
    # --- encode, SSD300/VOC B=32 G=8 (config 3): ONE launch per batch, output buffer reused
    ps = [(38, 38), (19, 19), (10, 10), (5, 5), (3, 3), (1, 1)]
    from oracle.model import SSD300_AR
    enc = SSDInputEncoder(300, 300, 20, ps, scales=SC300, aspect_ratios_per_layer=SSD300_AR, steps=[8, 16, 32, 64, 100, 300],
                          offsets=[0.5] * 6, pos_iou_threshold=0.5, neg_iou_limit=0.5)
    gt = synth.synth_gt(2, 32, 8, 300, 300, 20)
    offs = np.cumsum([0] + [g.shape[0] for g in gt]).astype(np.int32)
    gdev = torch.from_numpy(np.concatenate(gt)).cuda()
    ybuf = torch.empty((32, 8732, 33), dtype=torch.float32, device='cuda')
    ms = _time_cuda(lambda: enc.encode_device(gdev, offs, out=ybuf), iters=10, warm=5, inner=50)
    bytes_ = 32 * (8732 * 16 + 8 * 20 + 8732 * 4 * 33)
    out['encode_ssd300_b32'] = {'ms': ms, 'images_per_s': 32e3 / ms, 'algorithmic_GB': bytes_ / 1e9, 'GBps': bytes_ / ms / 1e6,
                                'frac_hbm': bytes_ / ms / 1e6 / hbm, 'launches_per_call': 1,
                                'kernels': 'enc_tiles_kernel (G <= 16: no lower-bound pre-pass)', 'timing': '50 back-to-back calls between two CUDA events, median of 10'}
    del ybuf
    y_true = enc.encode_device(gdev, offs)
    y_pred = torch.from_numpy(synth.synth_y_pred(3, 32, enc.anchors, 21, sharp=2.0)).cuda()
    L = SSDLoss()
    ms = _time_cuda(lambda: L.loss_and_stats(y_true, y_pred), iters=10, warm=5, inner=20)
    bytes_ = 2 * 8732 * 25 * 4 * 32
    out['ssd_loss_fwd_b32'] = {'ms': ms, 'algorithmic_GB': bytes_ / 1e9, 'GBps': bytes_ / ms / 1e6, 'frac_hbm': bytes_ / ms / 1e6 / hbm,
                               'launches_per_call': 2, 'kernels': 'ssd_loss_kernel (cooperative, all phases) + a 16-byte fill of the statistics',
                               'timing': '20 back-to-back calls between two CUDA events, median of 10'}
    # --- config 5 at its stated size: P = 100000, G = 128, B = 256 (3.4 GB of targets per call)
    Bm = int(os.environ.get('SSDK_MICRO_B', '256'))
    encm = SSDInputEncoder(1000, 1600, 20, [(125, 200)], scales=[0.1, 0.2], aspect_ratios_global=[0.5, 1.0, 2.0],
                           pos_iou_threshold=0.5, neg_iou_limit=0.5)
    gtm = synth.synth_gt(4, Bm, 128, 1600, 1000, 20)
    offm = np.cumsum([0] + [g.shape[0] for g in gtm]).astype(np.int32)
    gm = torch.from_numpy(np.concatenate(gtm)).cuda()
    ybuf = torch.empty((Bm, 100000, 33), dtype=torch.float32, device='cuda')
    ms = _time_cuda(lambda: encm.encode_device(gm, offm, out=ybuf), iters=7, warm=2)
    bytes_ = Bm * (100000 * 16 + 128 * 20 + 100000 * 4 * 33)
    out['encode_micro_p1e5_g128'] = {'batch': Bm, 'ms': ms, 'priors_per_s': Bm * 1e5 / ms * 1e3, 'iou_pairs_per_s': Bm * 1.28e7 / ms * 1e3,
                                     'algorithmic_GB': bytes_ / 1e9, 'GBps': bytes_ / ms / 1e6, 'frac_hbm': bytes_ / ms / 1e6 / hbm,
                                     'launches_per_call': 2, 'kernels': 'enc_lb_kernel (row-maximum lower bounds, ~10% of the time) + enc_tiles_kernel'}
    del ybuf
    anc = torch.from_numpy(encm.anchors_f32.copy()).cuda()
    boxes = torch.stack([anc[:, 0] - anc[:, 2] / 2, anc[:, 1] - anc[:, 3] / 2, anc[:, 0] + anc[:, 2] / 2, anc[:, 1] + anc[:, 3] / 2], 1)
    boxes = (boxes * torch.tensor([1600., 1000., 1600., 1000.], device='cuda')).unsqueeze(0).expand(Bm, -1, -1).contiguous()
    scores = torch.from_numpy(np.stack([np.random.default_rng(5 + i).uniform(0, 1, 100000) for i in range(Bm)]).astype(np.float32)).cuda()
    ms = _time_cuda(lambda: nms_device(boxes, scores, 0.01, 0.45, 400, 200), iters=5, warm=2)
    bytes_ = Bm * (100000 * 20 + 200 * 4)
    out['nms_micro_p1e5'] = {'batch': Bm, 'ms': ms, 'boxes_per_s': Bm * 1e5 / ms * 1e3, 'algorithmic_GB': bytes_ / 1e9,
                             'GBps': bytes_ / ms / 1e6, 'frac_hbm': bytes_ / ms / 1e6 / hbm}
    del boxes, scores, gm
    # --- config 3: SSD300 training step, B = 32 per GPU (forward + loss + backward + SGD-momentum update; no all-reduce here,
    #     this leg runs on rank 0 only)
    from ssd_keras_b200.models.keras_ssd300 import ssd_300
    from ssd_keras_b200.training import SSDTrainer
    Bt = 32
    mt = ssd_300((300, 300, 3), 20, mode='training', scales=SC300)
    tr = SSDTrainer(mt, Bt, lr=1e-4, momentum=0.9)
    xt = torch.from_numpy(synth.synth_images(0, Bt, 300, 300)).cuda()

    def train_step():
        tr.forward_backward(xt, y_true)
        tr.apply(1.0)
    ms = _time_cuda(train_step, iters=5, warm=2)
    fl = 3.0 * mt.flops(Bt)[0]
    out['train_step_ssd300_b32'] = {'ms': ms, 'images_per_s': Bt * 1e3 / ms, 'algorithmic_TFLOPs': fl / ms / 1e9,
                                    'frac_tensor_peak': fl / ms / 1e9 / peaks['bf16_tflops_sustained'], 'n_params': tr.n_params}
    return out


def dump_outputs(path, arrays):
    """Writes every array as `path/<name>.npy` in float32, so that two builds can be compared output for output (the inputs
    and weights are seeded: the same arguments give the same inputs)."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), np.ascontiguousarray(a, dtype=np.float32))


def _max_over_ranks(ms, dist):
    import torch
    t = torch.tensor([ms], device='cuda', dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def dist_extras(world, rank, peaks, model_inf_weights):
    """Runs on EVERY rank when world > 1 (all collectives are real NCCL calls): BASELINE config 3's training step with the
    gradient exchange overlapped with the backward pass, the same step with one exchange after the backward pass, a fixed
    global batch of 32 split over the ranks (strong scaling), and a correctness check of both loss modes against the float64
    oracle.  Times are CUDA events, max over ranks."""
    import importlib.util
    import torch
    import torch.distributed as dist
    from oracle import synth
    from ssd_keras_b200.distributed import all_gather_detections, all_reduce_buckets_, shard_bounds, ssd_loss_global
    from ssd_keras_b200.models.keras_ssd300 import ssd_300
    from ssd_keras_b200.ssd_encoder_decoder.ssd_input_encoder import SSDInputEncoder
    from ssd_keras_b200.training import SSDTrainer
    out = {}

    def timed(fn, steps=5, warm=2):
        for _ in range(warm):
            fn()
        dist.barrier(); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        dist.barrier(); torch.cuda.synchronize()
        return _max_over_ranks(a.elapsed_time(b) / steps, dist)

    # --- config 3, weak scaling: 32 images per rank, encode on the device + forward + loss + backward + exchange + update
    Bt = 32
    from oracle.model import SSD300_AR
    mt = ssd_300((300, 300, 3), 20, mode='training', scales=SC300)
    enc = SSDInputEncoder(300, 300, 20, mt.predictor_sizes, scales=SC300, aspect_ratios_per_layer=SSD300_AR, steps=[8, 16, 32, 64, 100, 300],
                          offsets=[0.5] * 6, pos_iou_threshold=0.5, neg_iou_limit=0.5)
    gt = synth.synth_gt(2 + rank, Bt, 8, 300, 300, 20)
    offs = np.cumsum([0] + [g.shape[0] for g in gt]).astype(np.int32)
    gdev = torch.from_numpy(np.concatenate(gt)).cuda()
    xt = torch.from_numpy(synth.synth_images(50 + rank, Bt, 300, 300)).cuda()
    ybuf = torch.empty((Bt, 8732, 33), dtype=torch.float32, device='cuda')
    tr = SSDTrainer(mt, Bt, lr=1e-4, momentum=0.9)

    def step(overlap):
        tr.train_on_batch(xt, enc.encode_device(gdev, offs, out=ybuf), overlap=overlap)
    ms_overlap = timed(lambda: step(True))                      # gradient buckets on a side stream under the backward pass
    ms_serial = timed(lambda: step(False))                      # one all-reduce when the backward pass is over
    ms_default = ms_overlap if world > 2 else ms_serial         # what train_on_batch(overlap=None) runs at this world size

    def step_local():                                           # the same step without any exchange (what a single GPU does)
        loss, _, dy = tr._loss_and_dy(xt, enc.encode_device(gdev, offs, out=ybuf))
        tr._backward_layers(dy, len(mt.specs) - 1, 0)
        tr.apply(1.0)
    ms_local = timed(step_local)
    nbytes = tr.n_params * 4
    out['train_step_ssd300_b32_per_gpu'] = {
        'ms_overlapped_buckets': ms_overlap, 'ms_single_allreduce_after_backward': ms_serial, 'ms_no_exchange': ms_local,
        'ms_default': ms_default, 'default': 'bucketed from 4 ranks on, single exchange below (SSDTrainer.train_on_batch)',
        'images_per_s': world * Bt * 1e3 / ms_default, 'allreduce_MB': nbytes / 1e6, 'buckets': len(tr.buckets()),
        'exposed_exchange_ms': ms_overlap - ms_local, 'unoverlapped_exchange_ms': ms_serial - ms_local,
        'allreduce_busbw_GBps_if_serial': (2.0 * (world - 1) / world * nbytes / 1e9) / max((ms_serial - ms_local) * 1e-3, 1e-9),
        'scaling': 'weak', 'loss_mode': 'replica'}
    del tr, mt, xt, ybuf
    torch.cuda.empty_cache()

    # --- configs 1/2 as the survey partitions them: a FIXED global batch of 32 images, 32 / world per rank (strong scaling)
    if 32 % world == 0:
        bl = 32 // world
        ms_ = ssd_300((300, 300, 3), 20, mode='inference', scales=SC300)
        ms_.set_weights(model_inf_weights)
        lo, hi = shard_bounds(32, rank, world)
        xs = [torch.from_numpy(synth.synth_images(200 + i, 32, 300, 300)[lo:hi]).cuda() for i in range(2)]
        state = {'i': 0}

        def infer():
            state['i'] += 1
            return all_gather_detections(ms_.predict_device(xs[state['i'] & 1]))
        t = timed(infer, steps=10, warm=3)
        out['strong_b32'] = {'global_batch': 32, 'images_per_rank': bl, 'ms_per_step': t, 'images_per_s': 32e3 / t, 'scaling': 'strong',
                             'note': 'SSD300 forward + DecodeDetections + all-gather of the (32,200,6) boxes'}
        del ms_, xs
        torch.cuda.empty_cache()

    # --- correctness of the exchange against the float64 oracle (small graph, 2 images per rank) and of the global-batch-exact loss
    spec = importlib.util.spec_from_file_location('train_check', os.path.join(ROOT, 'tools', 'train_check.py'))
    tc = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(tc)
    case = tc.CASES[2]
    m, w, n_cls = tc.build(case)
    hw, per = case[1], 2
    Bg = per * world
    rng = np.random.default_rng(11)
    x_all = rng.integers(0, 256, size=(Bg, hw, hw, 3)).astype(np.float32)
    from oracle.encoder import OracleEncoder
    oenc = OracleEncoder(hw, hw, n_cls - 1, m.predictor_sizes, scales=m.anchor_cfg['scales'], aspect_ratios_per_layer=m.anchor_cfg['aspect_ratios_per_layer'],
                         variances=[0.1, 0.1, 0.2, 0.2], pos_iou_threshold=0.3, neg_iou_limit=0.2)
    y_all = oenc(tc.small_gt(5, Bg, 3, hw, n_cls - 1)).astype(np.float32)
    lo, hi = rank * per, (rank + 1) * per
    xd, yd = torch.from_numpy(x_all[lo:hi]).cuda(), torch.from_numpy(y_all[lo:hi]).cuda()
    check = {}
    for mode in ('replica', 'global'):
        trc = SSDTrainer(m, per, lr=1e-3, momentum=0.9, l2_regularization=0.0, loss_mode=mode)
        loss, y_pred, dy = trc._loss_and_dy(xd, yd)
        all_reduce_buckets_(trc.grad, trc.buckets(1 << 12), lambda a, b: trc._backward_layers(dy, a, b))
        torch.cuda.synchronize()
        grads = trc.gradients()
        losses = [torch.zeros_like(loss) for _ in range(world)]
        dist.all_gather(losses, loss)
        if rank == 0:
            from oracle import graph as og
            params = og.make_params(m.specs, w, dtype=torch.float64)
            yp, _ = og.forward(m.specs, params, x_all, n_cls, m.anchors, [0.1, 0.1, 0.2, 0.2], dtype=torch.float64)
            if mode == 'replica':                # every rank: the reference loss on its own shard, mean over the shard; gradients summed
                lv = torch.cat([og.ssd_loss_torch(y_all[r * per:(r + 1) * per], yp[r * per:(r + 1) * per]) for r in range(world)])
                torch.stack([lv[r * per:(r + 1) * per].mean() for r in range(world)]).sum().backward()
            else:                                # the single-process reference on the whole batch
                lv = og.ssd_loss_torch(y_all, yp)
                lv.mean().backward()
            ref_l = lv.detach().numpy()
            got_l = torch.cat(losses).cpu().numpy()
            gerr = max(float(np.abs(grads[k] - params[k].grad.numpy()).max() / (np.abs(params[k].grad.numpy()).max() + 1e-30)) for k in grads)
            lerr = float(np.abs(got_l - ref_l).max() / np.abs(ref_l).max())
            check[mode] = {'loss_rel_err': lerr, 'grad_rel_err_max': gerr, 'pass': bool(lerr < 1e-4 and gerr < 2e-3)}
        del trc
    if rank == 0:
        check['pass'] = bool(all(v['pass'] for v in check.values()))
        check['what'] = ('%d ranks x 2 images, small SSD graph (conv / l2norm / pool / two heads): all-reduced gradients and gathered '
                         'losses against float64 autograd of the oracle graph; replica-local loss and global-batch-exact loss' % world)
        out['nccl_check'] = check
    return out


# ------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import __graft_entry__
    __graft_entry__.build()
    from oracle import synth                     # synthetic input generator only (not measured, not shipped)
    from ssd_keras_b200 import _ffi
    from ssd_keras_b200.models.keras_ssd300 import ssd_300

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    peaks, peaks_src = _peaks()

    precision = 'bf16' if args.fast else 'bf16x3'
    model = ssd_300((300, 300, 3), N_CLASSES, mode='inference', scales=SC300, precision=precision)
    model.set_weights(_weights())
    # several distinct input batches so that a step never finds its images in L2 (4 x 34.6 MB > 126 MB L2)
    n_in = 4
    host = [torch.from_numpy(synth.synth_images(100 * rank + i, BATCH, 300, 300)).pin_memory() for i in range(n_in)]
    dev = [h.cuda() for h in host]
    from ssd_keras_b200.distributed import all_gather_detections

    def step_device(i):
        out = model.predict_device(dev[i % n_in])
        if world > 1:
            out = all_gather_detections(out)            # decoded boxes of every rank (SURVEY 8e, C2)
        return out

    pinned_out = torch.empty((world * BATCH, 200, 6), dtype=torch.float32).pin_memory()
    out_np = pinned_out.numpy()

    def run_e2e(steps):
        """`steps` batches from pinned host memory through the public streaming call (SSDModel.predict_stream, what
        predict_generator / predict run on): every batch is uploaded, computed and its result downloaded inside this call; the
        upload of batch i+1 and the host's read of result i-1 overlap the kernels of batch i.  Returns when the LAST result is
        on the host."""
        post = all_gather_detections if world > 1 else None
        n = 0
        for res in model.predict_stream((host[i % n_in] for i in range(steps)), post=post):
            np.copyto(out_np, res.numpy())               # the consumer's read of every result (plain host memcpy, 154 kB per rank;
                                                         # a torch CPU copy_ would wake the OpenMP pool next to the launching thread)
            n += 1
        assert n == steps
        return pinned_out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        """Returns the time of `steps` calls, the clocks, the launch count and what the last call returned."""
        for i in range(warmup):
            fn(i)
        barrier()
        sampler = ClockSampler(local)
        sampler.start()
        l0 = _ffi.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for i in range(steps):
            out = fn(warmup + i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        clocks = sampler.stop()
        launches = _ffi.launch_count() - l0
        if world > 1:
            t = torch.tensor([ms], device='cuda'); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
            c = torch.tensor([launches], device='cuda', dtype=torch.int64); dist.all_reduce(c); launches = int(c.item())
        return ms, clocks, launches, out

    ms_dev, clocks, launches, last = timed(step_device, args.steps, max(args.warmup, 3))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'detections': last.cpu().numpy()})
    # end to end: one untimed pipelined pass, then K batches in ONE timed pipelined pass (K uploads + K downloads inside it)
    run_e2e(max(args.warmup, 3))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run_e2e(args.steps)
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_e2e], device='cuda'); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms_e2e = float(t.item())
    ips = world * BATCH * args.steps / (ms_dev * 1e-3)
    ips_e2e = world * BATCH * args.steps / (ms_e2e * 1e-3)

    # dominant kernel: the tcgen05 convolution.  Time of all conv launches of one step via CUDA events on the launch
    # stream (instrumented passes outside the timed region).
    model.set_timing(BATCH, True)
    conv_ms = []
    for i in range(3):
        step_device(i)
        torch.cuda.synchronize()
        conv_ms.append(model.last_conv_ms(BATCH))
    model.set_timing(BATCH, False)
    conv_ms = float(np.median(conv_ms))
    fl_algo, fl_issued = model.flops(BATCH)
    peak = peaks.get('bf16_tflops_sustained', peaks.get('bf16_tflops'))
    traffic, traffic_src = None, None
    for name in ('r02_conv_traffic.json', 'r01_conv_traffic.json'):       # newest ncu --set full capture of this workload first
        tp = os.path.join(ROOT, 'profiles', name)
        if os.path.exists(tp):
            with open(tp) as f:
                tj = json.load(f)
            traffic = tj.get('dram_bytes_per_step')
            traffic_src = 'profiles/%s (dram read+write bytes of the %d conv launches of one step, ncu --set full; %s)' % (
                name, tj.get('launches_per_step', 0), tj.get('source', ''))
            break
    roofline = {'bound': 'tensor', 'kernel': 'conv_tcgen05_kernel (all conv launches of one step)',
                'achieved': fl_algo / conv_ms / 1e9, 'peak': peak, 'unit': 'TFLOP/s', 'frac': fl_algo / conv_ms / 1e9 / peak,
                'peak_source': peaks_src + ', bf16_tflops_sustained', 'traffic': traffic, 'traffic_unit': 'bytes per step',
                'traffic_source': traffic_src,
                'algorithmic_tflop_per_step': fl_algo / 1e12, 'issued_mma_tflop_per_step': fl_issued / 1e12,
                'issued_tflops': fl_issued / conv_ms / 1e9, 'issued_frac': fl_issued / conv_ms / 1e9 / peak,
                'conv_ms_per_step': conv_ms}

    line = {'metric': METRIC, 'value': ips, 'unit': 'images/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': ms_dev / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'bf16x3 (bf16 hi+lo operands, 3 tcgen05 MMAs per product, fp32 accumulate)' if not args.fast else 'bf16',
            'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'global_batch': world * BATCH, 'parallelism': 'dp%d' % world, 'precision': precision,
                       'l2': 'no explicit flush: %d distinct 34.6 MB input batches are rotated and each step streams >4 GB of '
                             'activations through the 126 MB L2' % n_in},
            'e2e': {'value': ips_e2e, 'unit': 'images/s', 'h2d_bytes_per_step': world * BATCH * 300 * 300 * 3 * 4,
                    'd2h_bytes_per_step': world * BATCH * 200 * 6 * 4, 'ms_per_step': ms_e2e / args.steps,
                    'note': 'SSDModel.predict_stream (the pipeline behind predict / predict_generator) on pinned-host inputs: the H2D '
                            'of batch i+1 runs on a copy stream under the kernels of batch i, every result is copied to pinned host '
                            'memory and read by the host while the next batch runs; K uploads + K downloads + the final wait are '
                            'inside the timed region'},
            'gpu_launches': launches, 'clocks': clocks, 'roofline': roofline}
    if world > 1:
        # every rank takes part in the extras (real NCCL collectives).  They must never cost the headline line: a watchdog
        # prints it without them and leaves if they hang (a rank that failed while the others wait in a collective)
        import threading

        def _bail():
            # runs on its own thread: the main thread may be blocked inside a CUDA / NCCL call that never returns (a signal
            # handler would not get to run there)
            if rank == 0:
                line['extra'] = {'error': 'multi-rank extras timed out'}
                print(json.dumps(line), flush=True)
            os._exit(0)
        if not args.no_micro:
            dog = threading.Timer(float(os.environ.get('SSDK_EXTRAS_TIMEOUT', '420')), _bail)
            dog.daemon = True
            dog.start()
            try:
                extra = dist_extras(world, rank, peaks, _weights())
            except Exception as e:
                import traceback
                extra = {'error': repr(e), 'trace': traceback.format_exc()[-1500:]}
            dog.cancel()
            line['extra'] = extra
        if rank == 0:
            print(json.dumps(line), flush=True)
        if isinstance(line.get('extra'), dict) and 'error' in line['extra']:
            os._exit(0)                                  # peers may be stuck in a collective: do not wait for them in a clean-up
        try:
            dist.destroy_process_group()
        except Exception:
            pass
        return
    if world == 1:
        if not args.no_cpu:
            v, dt, threads, t_fwd, t_dec = time_cpu_reference(16, 2, 1)
            line['cpu_baseline'] = {'value': v, 'unit': 'images/s', 'cores': threads, 'kind': 'port',
                                    'sample': '16 of 32 images, 2 repetitions after 1 warm-up (%.1f s each): torch-CPU restatement of '
                                              'the Keras graph (%.2f s, thread count picked by calibration) + restatement of DecodeDetections '
                                              '(NumPy + compiled C NMS, %.2f s, one worker process per image)' % (dt, t_fwd, t_dec)}
        if not args.no_micro:
            try:
                line['extra'] = micro_benchmarks(peaks)
            except Exception as e:                    # the headline number must not depend on the extras
                line['extra'] = {'error': repr(e)}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--fast', action='store_true', help='single-pass bf16 convolutions instead of bf16x3')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-micro', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the (world*32, 200, 6) detections of the last timed step to DIR/detections.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes what the CUDA path computed: it needs --impl ours')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
