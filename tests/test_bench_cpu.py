"""CPU tests of bench.py's --dump-outputs writer: float32 files, the size limit, and the same sample on every run."""
import numpy as np

import bench


def _grads(rng):
  return {'block0/dil0/kernel': rng.standard_normal((2, 8, 16)).astype(np.float32),
          'block0/dil0/bias': rng.standard_normal(16).astype(np.float32),
          'head0/kernel': rng.standard_normal((1, 8, 300)).astype(np.float32)}


def test_dump_writes_loss_and_all_gradients_in_variable_order(tmp_path):
  g = _grads(np.random.default_rng(1))
  bench.dump_outputs(str(tmp_path / 'out'), np.array([2.5, 0.125]), g)
  loss, flat = np.load(tmp_path / 'out' / 'loss.npy'), np.load(tmp_path / 'out' / 'grads.npy')
  assert loss.dtype == np.float32 and loss.tolist() == [2.5, 0.125]
  assert flat.dtype == np.float32 and np.array_equal(flat, np.concatenate([v.ravel() for v in g.values()]))


def test_dump_samples_gradients_over_the_limit_the_same_way_every_run(tmp_path, monkeypatch):
  monkeypatch.setattr(bench, 'DUMP_LIMIT_BYTES', (1 << 12) + 4 * 1000)
  g = _grads(np.random.default_rng(2))
  full = np.concatenate([v.ravel() for v in g.values()])
  for d in ('a', 'b'):
    bench.dump_outputs(str(tmp_path / d), np.zeros(2, np.float32), g)
  a, b = np.load(tmp_path / 'a' / 'grads.npy'), np.load(tmp_path / 'b' / 'grads.npy')
  assert a.size == 1000 - 2 and np.array_equal(a, b)
  assert np.isin(a, full).all()
  assert sum(f.stat().st_size for f in (tmp_path / 'a').iterdir()) <= bench.DUMP_LIMIT_BYTES
