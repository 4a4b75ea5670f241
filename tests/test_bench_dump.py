"""bench.py --dump-outputs and --steps on the host: files, dtypes, the seeded row sample above the size limit, argument checks."""
import os

import numpy as np
import pytest
import torch

import bench


def _arrays(n, k=13):
    g = torch.Generator().manual_seed(1)
    return {'pos': torch.randn(n, 3, generator=g), 'v': torch.randint(0, k, (n,), generator=g),
            'log_v0': torch.randn(n, k, generator=g), 'log_vt': torch.randn(n, k, generator=g)}


def test_dump_outputs_writes_every_array(tmp_path):
    arr = _arrays(50)
    bench.dump_outputs(str(tmp_path), arr)
    assert sorted(os.listdir(tmp_path)) == ['log_v0.npy', 'log_vt.npy', 'pos.npy', 'v.npy']
    for k, v in arr.items():
        got = np.load(tmp_path / (k + '.npy'))
        assert got.dtype in (np.float32, np.float64)
        np.testing.assert_array_equal(got, v.double().numpy() if k == 'v' else v.numpy())


def test_dump_outputs_samples_the_same_rows_above_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, 'DUMP_LIMIT', 4096 + 20 * (124 + 8))
    arr = _arrays(500)
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), arr)
    rows = np.load(tmp_path / 'a' / 'rows.npy')
    assert rows.dtype == np.float64 and len(rows) == 20 and np.all(np.diff(rows) > 0)
    np.testing.assert_array_equal(rows, np.load(tmp_path / 'b' / 'rows.npy'))
    np.testing.assert_array_equal(np.load(tmp_path / 'a' / 'pos.npy'), arr['pos'].numpy()[rows.astype(np.int64)])
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in os.listdir(tmp_path / 'a')) <= bench.DUMP_LIMIT


@pytest.mark.parametrize('argv', [['--steps', '0'], ['--steps', '1001'], ['--impl', 'reference', '--dump-outputs', 'x']])
def test_bench_rejects_bad_arguments(monkeypatch, argv):
    monkeypatch.setattr('sys.argv', ['bench.py'] + argv)
    with pytest.raises(SystemExit):
        bench.parse_args()


def test_bench_steps_is_the_timed_step_count(monkeypatch):
    monkeypatch.setattr('sys.argv', ['bench.py', '--steps', '7', '--warmup', '2'])
    assert bench.parse_args().steps == 7
