"""bench.py --impl reference on the CPU: the JSON line carries the keys the contract names; non-zero ranks stay silent.
(The GPU arm is exercised by the driver on a B200; its line is built by the same code path, bench.run_ours.)"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(env_extra, *flags):
    env = dict(os.environ)
    env.update(env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0', '--no-ref-calibrate'] + list(flags),
                          capture_output=True, text=True, env=env, timeout=600)


def test_reference_arm_line():
    r = run({})
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
              'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert k in d, k
    assert d['impl'] == 'reference' and d['unit'] == 'fits/s' and d['higher_is_better'] is True and d['vs_baseline'] is None
    assert d['dtype'] == 'f64' and d['data'] == 'synthetic' and 'workload' in d['config'] and 'model' not in d['config']
    assert d['steps'] == 1 and d['warmup'] == 0 and d['value'] > 0 and abs(d['ms_per_step'] * d['value'] - 1e3) < 1e-6 * 1e3
    cb = d['cpu_baseline']
    assert cb['kind'] == 'port' and cb['cores'] >= 1 and cb['value'] == d['value'] and 'N=' in cb['sample']
    assert d['e2e'] == {'value': d['value'], 'unit': 'fits/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_reference_arm_other_ranks_are_silent():
    r = run({'RANK': '1', 'LOCAL_RANK': '1', 'WORLD_SIZE': '2', 'MASTER_ADDR': '127.0.0.1', 'MASTER_PORT': '29876'}, '--gpus', '2')
    assert r.returncode == 0 and r.stdout.strip() == ''


def test_dump_outputs_is_refused_by_the_reference_arm(tmp_path):
    r = run({}, '--dump-outputs', str(tmp_path / 'out'))
    assert r.returncode == 2 and '--dump-outputs' in r.stderr and not (tmp_path / 'out').exists()


import numpy as np
import pytest


@pytest.mark.gpu
def test_gpu_arm_line(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '2', '--warmup', '3', '--skip-extras', '--no-sweep',
                        '--dump-outputs', str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline',
              'dtype', 'data', 'config', 'roofline', 'cpu_baseline', 'e2e', 'gpu_launches', 'clocks'):
        assert k in d, k
    assert d['n_gpus'] == 1 and d['steps'] == 2 and d['warmup'] == 3 and d['dtype'] == 'f64' and d['scaling'] == 'weak'
    assert 'workload' in d['config'] and d['vs_baseline'] is None
    assert 10.0 < d['value'] < 40.0 and abs(d['ms_per_step'] * d['value'] - 1e3) < 1.0          # fits/s at N=16384 on a B200
    rf = d['roofline']
    assert rf['bound'] == 'tensor' and rf['unit'] == 'TFLOP/s' and 0.5 < rf['frac'] < 1.0
    assert abs(rf['frac'] - rf['achieved'] / rf['peak']) < 1e-9 and rf['traffic'] > 0
    e = d['e2e']
    assert e['h2d_bytes_per_step'] >= 16384 * 9 * 8 and e['d2h_bytes_per_step'] > 0 and 0.8 * d['value'] < e['value'] <= 1.05 * d['value']
    assert d['gpu_launches'] > 100 * d['steps']
    cb = d['cpu_baseline']
    assert cb['kind'] == 'port' and cb['cores'] >= 1 and cb['value'] > 0 and cb['unit'] == 'fits/s'
    assert d['clocks']['sm_mhz'] > 0 and isinstance(d['clocks']['reasons'], list)
    nl, e2e = np.load(tmp_path / 'nlml.npy'), np.load(tmp_path / 'e2e_nlml.npy')
    assert nl.dtype == e2e.dtype == np.float64 and nl.shape == (1,) and e2e.shape == (1, 1)
    assert np.isfinite(nl).all() and np.isfinite(e2e).all() and sorted(os.listdir(tmp_path)) == ['e2e_nlml.npy', 'nlml.npy']
