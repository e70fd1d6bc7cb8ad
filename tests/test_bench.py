"""bench.py's `--dump-outputs DIR` (what the last timed step returned, for comparing two builds array by array) and
`--steps` (the number of timed steps)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import bench as B  # noqa: E402

BENCH = os.path.join(REPO, 'bench.py')


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_keeps_one_seeded_env_sample_within_the_budget(tmp_path):
    n = 4096
    g = torch.Generator().manual_seed(0)
    arrays = dict(adj=torch.rand(n, 8, 24, 24, generator=g), dones=torch.rand(n, 8, generator=g) > 0.5,
                  agent_id=torch.arange(8, dtype=torch.int32).view(1, 8, 1).expand(n, 8, 1),
                  state=np.random.default_rng(1).random((n, 3)))
    info = B.dump_outputs(str(tmp_path / 'a'), arrays)
    B.dump_outputs(str(tmp_path / 'b'), arrays)
    assert 0 < info['envs'] < n                                   # 75 MB of adjacency alone: sampled
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in os.listdir(tmp_path / 'a')) <= B.DUMP_BYTES
    a, b = _load(tmp_path / 'a'), _load(tmp_path / 'b')
    assert sorted(a) == sorted(arrays)
    idx = np.sort(np.random.default_rng(0).choice(n, info['envs'], replace=False))
    for k, v in arrays.items():
        want = (v.numpy() if torch.is_tensor(v) else v)[idx]
        assert a[k].dtype == (np.float64 if k == 'state' else np.float32), k
        assert np.array_equal(a[k], want.astype(a[k].dtype)), k
        assert np.array_equal(a[k], b[k]), k
    small = torch.rand(5, 2, generator=g)
    assert B.dump_outputs(str(tmp_path / 'c'), dict(obs=small))['envs'] == 5
    assert np.array_equal(np.load(tmp_path / 'c' / 'obs.npy'), small.numpy())


def test_reference_arm_times_the_requested_steps_and_dumps(tmp_path):
    out = subprocess.run([sys.executable, BENCH, '--impl', 'reference', '--steps', '2', '--warmup', '3',
                          '--dump-outputs', str(tmp_path)], capture_output=True, text=True, check=True)
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line['steps'] == line['steps_run'] == 2
    d = _load(tmp_path)
    assert sorted(d) == ['adj', 'dones', 'node_obs', 'obs', 'rewards']
    assert all(v.shape[0] == 1024 and v.dtype == np.float32 for v in d.values())


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, BENCH, '--steps', '0'], capture_output=True, text=True)
    assert out.returncode != 0 and '--steps' in out.stderr


@pytest.mark.gpu
def test_headline_dump_is_the_same_from_run_to_run(tmp_path):
    """Seeded inputs: two runs with the same arguments return identical arrays from their last timed step."""
    cmd = [sys.executable, BENCH, '--steps', '4', '--warmup', '3', '--envs', '256', '--e2e-steps', '3',
           '--no-cpu-baseline', '--no-extra-workloads', '--dump-outputs']
    for d in ('a', 'b'):
        out = subprocess.run(cmd + [str(tmp_path / d)], capture_output=True, text=True)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])['steps'] == 4
    a, b = _load(tmp_path / 'a'), _load(tmp_path / 'b')
    assert sorted(a) == ['adj', 'agent_id', 'dones', 'node_obs', 'obs', 'rewards']
    assert a['adj'].shape == (256, 8, 24, 24) and a['node_obs'].shape[:3] == (256, 8, 24)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
