"""CPU: bench.py --dump-outputs writes float arrays, caps the total size, and samples large arrays at fixed positions."""
import os

import numpy as np

import bench


def test_dump_outputs_small_arrays_are_written_whole(tmp_path):
    logp = np.random.default_rng(1).normal(size=(4, 25, 49)).astype(np.float32)
    bench.dump_outputs(str(tmp_path / 'd'), {'loss': np.float64(2.5), 'log_probs': logp, 'out_len': np.arange(4.0)})
    assert sorted(os.listdir(tmp_path / 'd')) == ['log_probs.npy', 'loss.npy', 'out_len.npy']
    assert np.array_equal(np.load(tmp_path / 'd' / 'log_probs.npy'), logp)
    assert np.load(tmp_path / 'd' / 'loss.npy') == 2.5


def test_dump_outputs_samples_large_arrays_reproducibly(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, 'DUMP_LIMIT_BYTES', 2 * 4000)
    a = np.arange(10_000, dtype=np.float32)
    for d in ('x', 'y'):
        bench.dump_outputs(str(tmp_path / d), {'a': a, 'b': np.zeros(3)})
    got = np.load(tmp_path / 'x' / 'a.npy')
    assert got.dtype == np.float32 and got.nbytes <= 4000 and got.size == 1000
    assert np.all(np.diff(got) > 0)                                  # positions in order, no repeats
    assert np.array_equal(got, np.load(tmp_path / 'y' / 'a.npy'))
    total = sum(os.path.getsize(tmp_path / 'x' / f) for f in os.listdir(tmp_path / 'x'))
    assert total < 2 * 4000 + 2 * 256                                # + the .npy headers
