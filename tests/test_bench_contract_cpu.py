"""CPU: `bench.py --impl reference` prints ONE JSON line with the benchmark's keys (the reference arm) and writes what its
last step computed with --dump-outputs; the row sample that bounds a large dump."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '1',
                          '--batch', '64', '--dump-outputs', str(tmp_path)],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip().startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
              'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert k in d, k
    assert d['impl'] == 'reference' and d['unit'] == 'detections/s' and d['higher_is_better'] is True and d['vs_baseline'] is None
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1 and d['value'] > 0
    assert 'workload' in d['config']
    # the dump: the model outputs of the last step on bench.py's seeded inputs
    from oracle import loco_oracle as O
    from monoloco_b200 import synthetic
    assert sorted(os.listdir(tmp_path)) == ['raw.npy']
    raw = np.load(tmp_path / 'raw.npy')
    assert raw.dtype == np.float32 and raw.shape == (64, 9)
    sd = synthetic.make_state_dict('loco', 34, 9, 1024, 3, 0)
    ok, worst = O.close(raw, O.loco_model_forward(sd, O.preprocess_monoloco(synthetic.make_keypoints(64, seed=0),
                                                                            synthetic.KITTI_K)))
    assert ok, worst


def test_dump_outputs_sample(tmp_path, monkeypatch):
    """Above the size limit every array keeps the same seeded rows, listed in row_index.npy, and the files fit the limit."""
    import bench
    monkeypatch.setattr(bench, 'DUMP_BYTES', 10000)
    raw = np.arange(1000 * 9, dtype=np.float32).reshape(1000, 9)
    dec = -np.arange(1000 * 8, dtype=np.float64).reshape(1000, 8)
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), {'raw': raw, 'dec': dec})
    files = sorted(os.listdir(tmp_path / 'a'))
    assert files == ['dec.npy', 'raw.npy', 'row_index.npy']
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in files) <= 10000
    idx = np.load(tmp_path / 'a' / 'row_index.npy')
    assert idx.dtype == np.float64 and len(idx) > 0 and np.all(np.diff(idx) > 0)
    rows = idx.astype(np.int64)
    got = {f: np.load(tmp_path / 'a' / f) for f in files}
    assert got['raw.npy'].dtype == np.float32 and np.array_equal(got['raw.npy'], raw[rows])
    assert got['dec.npy'].dtype == np.float32 and np.array_equal(got['dec.npy'], dec[rows].astype(np.float32))
    for f in files:
        assert np.array_equal(got[f], np.load(tmp_path / 'b' / f)), f
    bench.dump_outputs(str(tmp_path / 'small'), {'raw': raw[:10]})   # under the limit: whole arrays, no index
    assert sorted(os.listdir(tmp_path / 'small')) == ['raw.npy']
    assert np.array_equal(np.load(tmp_path / 'small' / 'raw.npy'), raw[:10])
