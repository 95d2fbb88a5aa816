"""bench.py contract pieces that run without a GPU: the reference arm (oracle port timed on host
cores) prints one JSON line with the keys the driver reads."""
import json
import os
import subprocess
import sys

import numpy as np

from conftest import ROOT


def test_reference_arm_prints_contract_json():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1',
                          '--warmup', '0', '--ref-sample', '20000'], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith('{')][-1]
    d = json.loads(line)
    for k in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better',
              'scaling', 'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e', 'gpu_launches'):
        assert k in d, k
    assert d['impl'] == 'reference' and d['unit'] == 'triples/s' and d['value'] > 0
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] == 1
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['gpu_launches'] == 0


def test_reference_arm_nonzero_rank_is_silent():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2',
                          '--steps', '1', '--warmup', '0'], capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ''


def test_reference_arm_dumps_outputs_of_the_last_timed_step(tmp_path):
    """--dump-outputs: float .npy files of at most 64 MB in all, identical from run to run, and --steps changes them."""
    def dump(steps, name):
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', str(steps),
                              '--warmup', '1', '--ref-sample', '20000', '--dump-outputs', str(tmp_path / name)],
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        return {f[:-4]: np.load(tmp_path / name / f) for f in os.listdir(tmp_path / name)}
    a, b, c = dump(2, 'a'), dump(2, 'b'), dump(3, 'c')
    assert sorted(a) == ['P', 'Q', 'loss']
    assert all(x.dtype == np.float64 for x in a.values()) and sum(x.nbytes for x in a.values()) <= 64 << 20
    assert a['P'].shape == (1200, 64)                  # 400 users per step, all of them
    assert a['Q'].shape == (57344, 64)                 # 100K float64 rows are above 28 MiB: a seeded sample of them
    assert all(np.array_equal(a[f], b[f]) for f in a)
    assert not np.array_equal(a['P'], c['P']) and a['loss'] != c['loss']
