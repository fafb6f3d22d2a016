"""The bench.py contract, checked on the CPU with the reference arm (no GPU needed): exactly ONE JSON line on stdout
carrying the required keys, whatever libraries print.  The outputs ``--dump-outputs`` writes are checked on the GPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

REQUIRED = ['metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
            'vs_baseline', 'dtype', 'data', 'config', 'e2e', 'gpu_launches', 'cpu_baseline', 'impl']


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, OMP_NUM_THREADS='4')
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0',
           '--cpu-sample', '1', '--nobs', '256']
    out = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    for k in REQUIRED:
        assert k in d, k
    assert d['impl'] == 'reference' and d['unit'] == 'evals/s' and d['higher_is_better'] is True
    assert d['value'] > 0 and d['e2e']['value'] == d['value']
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0
    assert d['cpu_baseline']['kind'] in ('port', 'reference') and d['cpu_baseline']['cores'] >= 1
    assert 'workload' in d['config']


def test_reference_arm_under_torchrun_env_prints_only_on_rank0():
    """N > 1: rank 0 alone runs and prints the line, the other ranks exit 0 without work."""
    env = dict(os.environ, OMP_NUM_THREADS='4', RANK='1', LOCAL_RANK='1', WORLD_SIZE='2')
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2', '--steps', '1',
           '--warmup', '0', '--cpu-sample', '1', '--nobs', '256']
    out = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.strip() == ''


def test_dump_outputs_writes_float64_and_caps_with_one_seeded_sample(tmp_path, monkeypatch):
    import numpy as np
    import bench
    ll, info = np.linspace(-5., 5., 100), np.arange(100, dtype=np.int32) % 3
    bench.dump_outputs(str(tmp_path / 'full'), {'loglik': ll, 'info': info})
    assert sorted(os.listdir(tmp_path / 'full')) == ['info.npy', 'loglik.npy']
    got = np.load(tmp_path / 'full' / 'info.npy')
    assert got.dtype == np.float64 and np.array_equal(got, info)
    monkeypatch.setattr(bench, 'DUMP_LIMIT_BYTES', 8 * 90)
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), {'loglik': ll, 'info': info})
    idx = np.load(tmp_path / 'a' / 'sample_index.npy')
    assert np.array_equal(idx, np.load(tmp_path / 'b' / 'sample_index.npy'))
    assert sum(np.load(tmp_path / 'a' / f).nbytes for f in os.listdir(tmp_path / 'a')) <= 8 * 90
    assert np.array_equal(np.load(tmp_path / 'a' / 'loglik.npy'), ll[idx.astype(int)])


def test_dump_outputs_is_refused_for_the_reference_arm(tmp_path):
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--dump-outputs', str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert out.returncode == 2 and '--dump-outputs' in out.stderr


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(gp, tmp_path):
    """The dumped loglik / info are what the timed path returned for the seeded bench inputs."""
    import numpy as np
    from oracle import sds_oracle as so
    n, B = 256, 8
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '2', '--warmup', '1', '--nobs', str(n),
           '--chains-per-gpu', str(B), '--no-peaks', '--no-e2e', '--no-cpu-baseline', '--no-configs',
           '--dump-outputs', str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    assert json.loads(out.stdout)['steps'] == 2
    ll, info = np.load(tmp_path / 'loglik.npy'), np.load(tmp_path / 'info.npy')
    assert ll.dtype == np.float64 and ll.shape == (B,) and np.all(info == 0)
    G, H = gp.synthetic.loglik_batch(B, n)
    x = np.arange(n, dtype=np.float64).reshape(n, 1)
    ref = np.array([so.loglik_unit(x, G[i], H[i], form='chol') for i in range(B)])
    assert np.max(np.abs(ll - ref) / np.abs(ref)) < 1e-10
