"""bench.py contract: the reference arm prints exactly ONE JSON line on stdout with the keys a caller reads, also when a
launcher exports OMP_NUM_THREADS=1 (torchrun does); without a GPU the CUDA arm fails loudly; on the GPU, --dump-outputs
writes what the last timed step computed."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))


def _run(args, env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + args, capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)


def test_reference_arm_prints_one_json_line():
    r = _run(['--impl', 'reference', '--gpus', '1', '--steps', '1', '--warmup', '1', '--photons', '5e4', '--nx', '32', '--nz3', '8'],
             {'OMP_NUM_THREADS': '1'})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'photons/s' and d['unit'] == 'photons/s' and d['higher_is_better'] is True
    assert d['value'] > 0 and d['steps'] == 1 and d['warmup'] == 1 and d['n_gpus'] == 1
    assert d['e2e'] == {'value': d['value'], 'unit': 'photons/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    cb = d['cpu_baseline']
    assert cb['kind'] == 'port' and cb['value'] == d['value'] and cb['cores'] >= 1 and 'photons' in cb['sample']
    # every host thread is used although the launcher exported OMP_NUM_THREADS=1
    assert cb['cores'] == len(os.sched_getaffinity(0))
    assert 'workload' in d['config'] and 'model' not in d['config']


def test_reference_arm_other_ranks_print_nothing():
    r = _run(['--impl', 'reference', '--gpus', '2', '--steps', '1', '--warmup', '1', '--photons', '5e4', '--nx', '32', '--nz3', '8'],
             {'RANK': '1', 'WORLD_SIZE': '2', 'LOCAL_RANK': '1'})
    assert r.returncode == 0 and r.stdout.strip() == ''


@pytest.mark.gpu
def test_cuda_arm_dumps_the_last_timed_step(tmp_path):
    """--dump-outputs writes the tallies of the last timed step.  Every step traces the same seeded job set into zeroed
    tallies, so one timed step and three dump the same arrays, and --steps sets the number of launches timed."""
    small = ['--gpus', '1', '--warmup', '1', '--photons', '1e5', '--nx', '32', '--nz3', '8', '--e2e-steps', '1',
             '--no-cpu-baseline', '--no-accuracy']
    lines, dumps = {}, {}
    for k in (1, 3):
        d = tmp_path / ('steps%d' % k)
        r = _run(small + ['--steps', str(k), '--dump-outputs', str(d)])
        assert r.returncode == 0, r.stderr[-2000:]
        lines[k] = json.loads(r.stdout)
        dumps[k] = {f: np.load(str(d / f)) for f in os.listdir(str(d))}
    assert lines[1]['steps'] == 1 and lines[3]['steps'] == 3
    assert lines[3]['gpu_launches'] == 3 * lines[1]['gpu_launches'] > 0
    a, b = dumps[1], dumps[3]
    assert sorted(a) == sorted(b) == ['rad.npy']
    assert a['rad.npy'].dtype == np.float64 and a['rad.npy'].size == 3 * 32 * 32 and a['rad.npy'].max() > 0.0
    assert np.allclose(a['rad.npy'], b['rad.npy'], rtol=1e-9, atol=1e-15)


def test_cuda_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = _run(['--gpus', '1', '--steps', '1', '--warmup', '1', '--photons', '1e4', '--nx', '32', '--nz3', '8'])
    assert r.returncode != 0
    assert 'no CUDA device' in r.stderr or 'no CPU fallback' in r.stderr
