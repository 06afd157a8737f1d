"""GPU: `bench.py --dump-outputs` writes what the last timed step of the flagship workload computed, and `--steps` is the
number of timed steps (one launch each at N = 1)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', '3', '--warmup', '1',
                          '--no-extras', '--no-cpu-baseline', '--dump-outputs', str(tmp_path)],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip().startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['steps'] == 3 and d['gpu_launches'] == 3, (d['steps'], d['gpu_launches'])
    from oracle import loco_oracle as O
    from monoloco_b200 import synthetic
    assert sorted(os.listdir(tmp_path)) == ['dec.npy', 'raw.npy']
    raw, dec = np.load(tmp_path / 'raw.npy'), np.load(tmp_path / 'dec.npy')
    assert raw.dtype == dec.dtype == np.float32 and raw.shape == (4096, 9) and dec.shape == (4096, 8)
    sd = synthetic.make_state_dict('loco', 34, 9, 1024, 3, 0)
    ref_raw = O.loco_model_forward(sd, O.preprocess_monoloco(synthetic.make_keypoints(4096, seed=0), synthetic.KITTI_K))
    ok, worst = O.close(raw, ref_raw)
    assert ok, worst
    ok, worst = O.close(dec[:, 0:4], O.extract_outputs(ref_raw)['xyzd'], col_scale=False)
    assert ok, worst
