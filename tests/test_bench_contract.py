"""The bench.py contract, checked without a GPU except where marked.

* `--impl reference` times the oracle port of the reference's path on the host cores and prints ONE JSON line with the
  keys the driver reads (tier framing (4)).
* our arm has no CPU fallback: without a CUDA device it must fail loudly, not print a number.
* `--dump-outputs DIR` writes the placements of the last timed step, identical from run to run.
"""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ['--leaves', '300', '--sites', '300', '--queries-per-gpu', '64', '--steps', '1', '--warmup', '1']


def _run(extra, env_extra=None, base=SMALL):
    env = dict(os.environ)
    env.pop('RANK', None)
    env.pop('WORLD_SIZE', None)
    if env_extra:
        env.update(env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + base + extra, capture_output=True,
                          text=True, cwd=ROOT, env=env, timeout=600)


def test_reference_arm_prints_one_json_line():
    p = _run(['--impl', 'reference', '--cpu-sample', '8'])
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d['impl'] == 'reference'
    assert d['metric'] == 'queries placed/sec' and d['unit'] == 'queries/s' and d['higher_is_better'] is True
    assert d['value'] > 0 and d['steps'] == 1 and d['warmup'] == 1 and d['n_gpus'] == 1
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
    assert d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': 'queries/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert 'workload' in d['config']


def test_reference_arm_other_ranks_exit_quietly():
    p = _run(['--impl', 'reference', '--cpu-sample', '8'], {'RANK': '1', 'WORLD_SIZE': '2', 'LOCAL_RANK': '1'})
    assert p.returncode == 0, p.stderr[-2000:]
    assert p.stdout.strip() == ''


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the behaviour on a box without a CUDA device')
def test_our_arm_fails_loudly_without_cuda():
    p = _run(['--no-cpu-baseline', '--no-e2e'])
    assert p.returncode != 0
    assert p.stdout.strip() == ''
    assert 'CUDA' in p.stderr


def _dumped(path):
    return {n: np.load(os.path.join(path, n + '.npy')) for n in ('edge', 'error', 'distal', 'pendant', 'status')}


def test_reference_arm_dumps_the_last_step(tmp_path):
    """--dump-outputs: the same arguments give the same inputs, so two runs write the same arrays."""
    runs = []
    for k in range(2):
        out = str(tmp_path / str(k))
        p = _run(['--impl', 'reference', '--cpu-sample', '8', '--dump-outputs', out])
        assert p.returncode == 0, p.stderr[-2000:]
        runs.append(_dumped(out))
    for name, a in runs[0].items():
        assert a.dtype == np.float64 and a.shape == (8,), name
        assert a.tobytes() == runs[1][name].tobytes(), name


@pytest.mark.gpu
def test_our_arm_dumps_what_it_timed(tmp_path):
    """--dump-outputs writes the placements of the last timed step: run to run identical, and the records whose hash the
    JSON line carries.  --steps sets the number of timed steps."""
    args = ['--leaves', '300', '--sites', '300', '--queries-per-gpu', '64', '--steps', '2', '--warmup', '1',
            '--no-cpu-baseline', '--no-cli', '--no-e2e']
    runs = []
    for k in range(2):
        out = str(tmp_path / str(k))
        p = _run(['--dump-outputs', out], base=args)
        assert p.returncode == 0, p.stderr[-2000:]
        d = json.loads(p.stdout)
        assert d['steps'] == 2
        runs.append(_dumped(out))
    a = runs[0]
    for name in a:
        assert a[name].dtype == np.float64 and a[name].shape == (64,), name
        assert a[name].tobytes() == runs[1][name].tobytes(), name
    rec = np.empty((64, 4), np.int64)
    rec[:, 0] = (a['edge'].astype(np.int64) & 0xffffffff) | (a['status'].astype(np.int64) << 32)
    rec[:, 1:] = np.stack([a['error'], a['distal'], a['pendant']], axis=1).view(np.int64)
    assert d['result_sha1_per_block'] == [hashlib.sha1(rec.tobytes()).hexdigest()[:16]]
