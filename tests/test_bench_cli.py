"""bench.py contract checks: the reference arm prints one well-formed JSON line (rank 0 only; no GPU needed), and
--dump-outputs writes the same arrays run after run (GPU)."""
import json
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra):
    env = dict(os.environ, **env_extra)
    p = subprocess.run([sys.executable, os.path.join(REPO, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0',
                        '--stage', '1'], capture_output=True, text=True, timeout=600, env=env, cwd=REPO)
    assert p.returncode == 0, p.stderr[-2000:]
    return [l for l in p.stdout.splitlines() if l.startswith('{')]


def test_reference_arm_json_line():
    lines = _run({})
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['unit'] == 'img/s' and d['higher_is_better'] is True
    assert d['value'] > 0 and d['e2e']['value'] == d['value']
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0
    cb = d['cpu_baseline']
    sys.path.insert(0, REPO)
    from oracle import ref_harness as rh
    want = 'reference' if rh.available() else 'port'
    assert cb['kind'] == want and cb['cores'] >= 1 and cb['value'] == d['value'] and 'sample' in cb
    assert d['steps'] == 1 and d['steps_requested'] == 1           # the line reports the steps it actually timed
    assert 'workload' in d['config'] and 'model' not in d['config']


def test_reference_arm_other_ranks_are_silent():
    assert _run({'RANK': '1', 'WORLD_SIZE': '2'}) == []


@pytest.mark.gpu
def test_dump_outputs_repeatable(tmp_path):
    """--dump-outputs: float32 arrays of the last timed step, within 64 MB, and the same arrays from a second run."""
    import numpy as np
    dumps = []
    for run in range(2):
        d = tmp_path / f'run{run}'
        p = subprocess.run([sys.executable, os.path.join(REPO, 'bench.py'), '--workload', 'bcnn_s2', '--batch', '2',
                            '--steps', '2', '--warmup', '1', '--no-e2e', '--no-micro', '--no-eager', '--no-cpu-baseline',
                            '--dump-outputs', str(d)], capture_output=True, text=True, timeout=900, cwd=REPO)
        assert p.returncode == 0, p.stderr[-2000:]
        line = json.loads([l for l in p.stdout.splitlines() if l.startswith('{')][-1])
        assert line['steps'] == 2
        dumps.append({f.name: np.load(f) for f in sorted(d.iterdir())})
    a, b = dumps
    assert set(a) == {'outputs.npy', 'loss.npy', 'state.npy', 'grads.npy'} and set(b) == set(a)
    assert a['outputs.npy'].shape == (2, 200) and a['loss.npy'].shape == ()
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    for k in a:
        assert a[k].dtype == np.float32 and np.isfinite(a[k]).all() and a[k].shape == b[k].shape
        assert np.linalg.norm(a[k] - b[k]) <= 1e-5 * np.linalg.norm(b[k]), k
