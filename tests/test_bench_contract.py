"""bench.py's reference arm (`--impl reference`: the oracle C port on the host cores) runs without a GPU: check the JSON
line the driver parses.  The own arm needs a GPU; its keys are checked in tests/test_zz_gpu_widening.py."""
import json
import os
import subprocess
import sys

ROOT = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
BASE_KEYS = {'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
             'vs_baseline', 'dtype', 'data', 'config', 'e2e', 'gpu_launches', 'cpu_baseline'}


def _line(args, env=None):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + args, capture_output=True, text=True, timeout=600,
                         env=dict(os.environ, **(env or {})))
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1, out.stdout                      # exactly ONE JSON line
    return json.loads(lines[0])


def test_reference_arm_json_line():
    d = _line(['--impl', 'reference', '--gpus', '1', '--steps', '3', '--warmup', '1'], env={'BENCH_REF_PENV': '0'})
    assert BASE_KEYS <= set(d) and d['impl'] == 'reference'
    assert d['metric'] == json.load(open(os.path.join(ROOT, 'BASELINE.json')))['metric']
    assert d['unit'] == 'env-steps/s' and d['higher_is_better'] is True and d['steps'] == 3 and d['warmup'] == 1
    assert d['value'] > 0 and d['e2e']['value'] == d['value'] and d['e2e']['h2d_bytes_per_step'] == 0
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
    assert d['reference_parallel_env']['available'] is False
    assert 'workload' in d['config'] and 'GoToLocal' in d['config']['workload'] and d['gpu_launches'] == 0


def test_reference_arm_other_ranks_stay_silent():
    """Under torchrun only rank 0 runs and prints the reference arm; the other ranks exit 0 without work."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2', '--steps', '2',
                          '--warmup', '1'], capture_output=True, text=True, timeout=120,
                         env=dict(os.environ, RANK='1', LOCAL_RANK='1', WORLD_SIZE='2'))
    assert out.returncode == 0 and out.stdout.strip() == ''


def test_dump_outputs_keeps_a_fixed_sample_under_the_cap(tmp_path):
    """--dump-outputs writes at most 64 MB: a larger output is cut down to the same seeded sample of environments every time"""
    sys.path.insert(0, ROOT)
    import numpy as np
    from bench import write_outputs
    n = 120000                                                   # 600 bytes per environment: 72 MB in all
    arrays = {'obs': np.arange(n * 147, dtype=np.float32).reshape(n, 7, 7, 3), 'reward': np.arange(n, dtype=np.float32),
              'done': np.zeros(n, np.float32), 'direction': np.ones(n, np.float32)}
    for d in ('a', 'b'):
        write_outputs(str(tmp_path / d), arrays)
    files = sorted(os.listdir(str(tmp_path / 'a')))
    assert files == ['direction.npy', 'done.npy', 'env_index.npy', 'obs.npy', 'reward.npy']
    assert sum(os.path.getsize(str(tmp_path / 'a' / f)) for f in files) <= 64 << 20
    idx = np.load(str(tmp_path / 'a' / 'env_index.npy'))
    assert idx.dtype == np.float64 and np.array_equal(idx, np.load(str(tmp_path / 'b' / 'env_index.npy')))
    assert np.array_equal(np.load(str(tmp_path / 'a' / 'reward.npy')), idx.astype(np.float32))
    assert np.array_equal(np.load(str(tmp_path / 'a' / 'obs.npy')), arrays['obs'][idx.astype(np.int64)])
    write_outputs(str(tmp_path / 'small'), {k: a[:1000] for k, a in arrays.items()})
    assert sorted(os.listdir(str(tmp_path / 'small'))) == ['direction.npy', 'done.npy', 'obs.npy', 'reward.npy']
