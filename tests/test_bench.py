"""bench.py's command line: --steps sets the number of timed steps, and --dump-outputs writes what the timed path
computed, the same on every run with the same arguments, so that two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from conftest import ROOT, has_cuda


def _bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + list(args), capture_output=True, text=True,
                          timeout=900)


def test_bad_arguments_are_refused():
    for args in (['--steps', '0'], ['--dump-outputs', 'x', '--impl', 'reference'], ['--dump-outputs', 'x', '--workload', 'chain20'],
                 ['--dump-outputs', 'x', '--dense-only']):
        out = _bench(*args)
        assert out.returncode == 2 and 'error' in out.stderr, (args, out.stderr[-500:])


def test_dump_outputs_writes_float64_within_the_limit(tmp_path):
    keys = np.array([0, 3, (1 << 53) - 1], dtype=np.uint64)
    big = np.random.default_rng(5).random(10000)
    bench.dump_outputs(str(tmp_path), {'keys': keys, 'delta': [0.25], 'big': big}, limit=8 * 2 * 3 * 1000)
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(got) == ['big', 'big_index', 'delta', 'keys']
    assert all(a.dtype == np.float64 for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 8 * 2 * 3 * 1000
    assert np.array_equal(got['keys'].astype(np.uint64), keys) and got['delta'].tolist() == [0.25]
    idx = got['big_index'].astype(np.int64)
    assert len(idx) == 1000 and np.all(np.diff(idx) > 0) and np.array_equal(got['big'], big[idx])
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path), {'keys': np.array([1 << 53], dtype=np.uint64)})


@pytest.mark.gpu
@pytest.mark.skipif(not has_cuda(), reason='needs a CUDA device')
def test_dump_outputs_are_reproducible(tmp_path):
    """Two runs with the same arguments dump the same outputs; the line reports the requested steps; the dumped pmf is
    the exact post-selected distribution and the dumped counts hold every shot."""
    lines = []
    for run in ('a', 'b'):
        out = _bench('--workload', 'tree10', '--steps', '2', '--warmup', '3', '--no-cpu-baseline', '--no-dense',
                     '--dump-outputs', str(tmp_path / run))
        assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
        lines.append(json.loads([ln for ln in out.stdout.splitlines() if ln.startswith('{')][-1]))
    assert lines[0]['steps'] == 2 and lines[0]['check']['parity_ok']
    names = sorted(os.listdir(tmp_path / 'a'))
    assert names == sorted(os.listdir(tmp_path / 'b'))
    assert names == sorted(n + '.npy' for n in ('keys', 'pmf', 'delta', 'e2e_pmf', 'e2e_delta', 'e2e_count_keys', 'e2e_counts'))
    a = {n[:-4]: np.load(tmp_path / 'a' / n) for n in names}
    b = {n[:-4]: np.load(tmp_path / 'b' / n) for n in names}
    for n in a:
        assert a[n].dtype == np.float64
        assert np.allclose(a[n], b[n], rtol=1e-12, atol=0), n
    assert np.array_equal(a['keys'], b['keys']) and np.array_equal(a['e2e_count_keys'], b['e2e_count_keys'])
    assert len(a['keys']) == bench.SHOTS and a['e2e_counts'].sum() == bench.SHOTS
    from qcmrf_b200 import workloads
    cliques, _ = workloads.named('tree10')
    pb, db = bench.brute_force_pmf(cliques, workloads.theta_for(cliques, seed=1984))
    assert np.abs(a['pmf'] / a['pmf'].sum() - pb).max() < 1e-5 and abs(a['delta'][0] - db) < 1e-5
