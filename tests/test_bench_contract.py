"""bench.py contract checks: the reference arm prints one JSON line with the agreed keys, the B200 arm refuses to run
without a CUDA device (no silent CPU fallback), --dump-outputs writes what the last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0',
                        '--cpu_sample', '16', '--grid_res', '32'], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().split('\n')[-1])
    assert line['impl'] == 'reference' and line['unit'] == 'queries/s' and line['higher_is_better'] is True
    assert line['value'] > 0 and line['n_gpus'] == 1 and line['steps'] == 1
    assert line['metric'].startswith('SDF queries/sec at grid_res=')
    assert 'workload' in line['config']
    cb = line['cpu_baseline']
    assert cb['kind'] == 'port' and cb['cores'] >= 1 and cb['value'] == line['value'] and 'queries' in cb['sample']
    e2e = line['e2e']
    assert e2e['value'] == line['value'] and e2e['h2d_bytes_per_step'] == 0 and e2e['d2h_bytes_per_step'] == 0


def test_b200_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return   # on a GPU box the real arm is exercised by the driver
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '1', '--warmup', '3'], capture_output=True,
                       text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0 and 'no CPU fallback' in (r.stderr + r.stdout)


def test_dump_outputs_writes_float_arrays_and_a_fixed_sample_above_the_limit(tmp_path, monkeypatch):
    idx = np.arange(5000, dtype=np.int32) * 7
    sdf = np.random.RandomState(1).randn(5000).astype(np.float32)
    bench.dump_outputs(str(tmp_path / 'all'), {'voxel_index': idx, 'sdf': sdf})
    a, s = np.load(tmp_path / 'all' / 'voxel_index.npy'), np.load(tmp_path / 'all' / 'sdf.npy')
    assert a.dtype == np.float64 and s.dtype == np.float32
    assert np.array_equal(a, idx) and np.array_equal(s, sdf)
    assert not (tmp_path / 'all' / 'row_index.npy').exists()

    monkeypatch.setattr(bench, 'DUMP_LIMIT_BYTES', 20000)
    for d in ('s1', 's2'):
        bench.dump_outputs(str(tmp_path / d), {'voxel_index': idx, 'sdf': sdf})
    got = {k: np.load(tmp_path / 's1' / (k + '.npy')) for k in ('voxel_index', 'sdf', 'row_index')}
    assert sum(v.nbytes for v in got.values()) <= 20000
    rows = got['row_index'].astype(np.int64)
    assert len(rows) == 20000 // (8 + 4 + 8) and np.all(np.diff(rows) > 0)
    assert np.array_equal(got['voxel_index'], idx[rows]) and np.array_equal(got['sdf'], sdf[rows])
    for k, v in got.items():
        assert np.array_equal(np.load(tmp_path / 's2' / (k + '.npy')), v)


@pytest.mark.gpu
def test_dump_outputs_holds_the_last_timed_step(tmp_path):
    res = 32
    lines = {}
    for steps in (1, 2):
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', str(steps), '--warmup', '0', '--grid_res', str(res),
                            '--cpu_sample', '0', '--skip_mesh_stage', '--skip_sharded', '--dump-outputs', str(tmp_path / str(steps))],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        lines[steps] = json.loads(r.stdout.strip().split('\n')[-1])
        assert lines[steps]['steps'] == steps
    # every timed step runs the same pipeline: the launch count of the timed region scales with --steps
    assert lines[2]['gpu_launches'] == 2 * lines[1]['gpu_launches'] > 0
    Q = lines[2]['config']['queries_per_shape']
    lin = np.load(tmp_path / '2' / 'voxel_index.npy')
    sdf = np.load(tmp_path / '2' / 'sdf.npy')
    assert lin.dtype == np.float64 and sdf.dtype == np.float32 and lin.shape == sdf.shape == (Q,)
    assert np.all(lin == np.round(lin)) and lin.min() >= 0 and lin.max() < res ** 3 and np.all(np.diff(lin) > 0)
    assert np.isfinite(sdf).all() and (sdf != 0).any()
    # same arguments, same inputs: a second run returns the same outputs
    assert np.array_equal(np.load(tmp_path / '1' / 'voxel_index.npy'), lin)
    np.testing.assert_allclose(np.load(tmp_path / '1' / 'sdf.npy'), sdf, rtol=0, atol=1e-6)
