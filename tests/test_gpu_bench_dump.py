"""bench.py --dump-outputs: the file holds the detections of the LAST timed step, as the public call returns them."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', '3', '--warmup', '1', '--no-cpu',
                        '--no-micro', '--dump-outputs', str(tmp_path)], capture_output=True, text=True, timeout=1200, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith('{')][-1])
    assert line['steps'] == 3 and line['warmup'] == 3
    got = np.load(tmp_path / 'detections.npy')
    assert got.dtype == np.float32 and got.shape == (32, 200, 6)
    assert np.isfinite(got).all()

    # steps 0-2 warm up, 3-5 are timed; step i reads input batch i % 4, so the last timed step read batch 1 (seed 1)
    import torch
    import bench
    from oracle import synth
    from ssd_keras_b200.models.keras_ssd300 import ssd_300
    model = ssd_300((300, 300, 3), bench.N_CLASSES, mode='inference', scales=bench.SC300, precision='bf16x3')
    model.set_weights(bench._weights())
    want = model.predict_device(torch.from_numpy(synth.synth_images(1, bench.BATCH, 300, 300)).cuda()).cpu().numpy()
    assert (want[:, :, 1] > 0).any()
    np.testing.assert_array_equal(got[:, :, 0], want[:, :, 0])
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-5)
