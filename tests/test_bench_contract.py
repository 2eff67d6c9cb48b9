"""bench.py keeps the driver's contract on the CPU-only reference arm: ONE JSON line on stdout with the required keys."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1',
                        '--warmup', '0', '--cpu-worlds', '2', '--cpu-sim-steps', '1'],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, 'stdout must carry exactly one line'
    d = json.loads(lines[0])
    for k in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better',
              'scaling', 'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert k in d, k
    assert d['impl'] == 'reference' and d['unit'] == 'world-steps/s' and d['value'] > 0
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0
    assert 'workload' in d['config']


class _World:
    """Stand-in for a World3D after a rollout: W worlds of two bodies."""
    W = 6

    def get_p(self):
        return torch.arange(self.W * 14, dtype=torch.float64).reshape(self.W, 14)

    def get_v(self):
        return -torch.arange(self.W * 12, dtype=torch.float64).reshape(self.W, 2, 6)


def test_dump_outputs_writes_float64_arrays_and_samples_worlds_above_the_limit(tmp_path, monkeypatch):
    import bench
    W = _World.W
    grads = {'mass': torch.linspace(0, 1, W, dtype=torch.float64), 'fric_coeff': torch.ones(W, dtype=torch.float64),
             'push': torch.arange(2 * W, dtype=torch.float64).reshape(W, 2)}
    loss = torch.tensor(2.5, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path / 'all'), loss, grads, _World())
    got = {f[:-4]: np.load(str(tmp_path / 'all' / f)) for f in os.listdir(str(tmp_path / 'all'))}
    assert sorted(got) == ['final_p', 'final_v', 'grad_fric_coeff', 'grad_mass', 'grad_push', 'loss', 'world_index']
    assert all(a.dtype == np.float64 for a in got.values())
    assert got['loss'].tolist() == [2.5] and got['world_index'].tolist() == list(range(W))
    np.testing.assert_array_equal(got['grad_push'], grads['push'].numpy())
    np.testing.assert_array_equal(got['final_v'], _World().get_v().reshape(W, -1).numpy())
    # a limit of three worlds' rows: the same seeded three worlds every time
    monkeypatch.setattr(bench, 'DUMP_LIMIT', 8 + 3 * 8 * (1 + 1 + 1 + 2 + 14 + 12))
    picks = []
    for run in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / run), loss, grads, _World())
        idx = np.load(str(tmp_path / run / 'world_index.npy')).astype(int)
        assert len(idx) == 3 and list(idx) == sorted(idx)
        np.testing.assert_array_equal(np.load(str(tmp_path / run / 'final_p.npy')), _World().get_p().numpy()[idx])
        total = sum(os.path.getsize(str(tmp_path / run / f)) - 128 for f in os.listdir(str(tmp_path / run)))
        assert total <= bench.DUMP_LIMIT
        picks.append(idx.tolist())
    assert picks[0] == picks[1]
