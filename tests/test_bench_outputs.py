"""bench.py --dump-outputs: every output as a float64 .npy file, a fixed sample of trees past the size limit."""
import numpy as np

import bench


def _outputs(B, A, seed):
    gen = np.random.RandomState(seed)
    return {'action': gen.randint(0, A, size=B).astype(np.int32), 'pi': gen.rand(B, A), 'root_value': gen.rand(B),
            'train_loss': np.array([0.5]), 'train_priorities': gen.rand(128).astype(np.float32)}


def test_dump_outputs_writes_every_array_as_float64(tmp_path):
    out = _outputs(64, 82, 0)
    bench.dump_outputs(str(tmp_path), out)
    for k, v in out.items():
        a = np.load(tmp_path / f'{k}.npy')
        assert a.dtype == np.float64 and np.array_equal(a, v.astype(np.float64)), k
    assert not (tmp_path / 'sampled_trees.npy').exists()


def test_dump_outputs_keeps_the_same_sample_of_trees_past_the_limit(tmp_path):
    out = _outputs(5000, 82, 1)
    limit = 1 << 20
    for run in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / run), out, limit=limit)
    assert sum(f.stat().st_size for f in (tmp_path / 'a').iterdir()) <= limit
    rows = np.load(tmp_path / 'a' / 'sampled_trees.npy').astype(np.int64)
    assert np.array_equal(rows, np.load(tmp_path / 'b' / 'sampled_trees.npy'))
    assert 1000 < len(rows) < 5000 and np.all(np.diff(rows) > 0)
    for k in ('action', 'pi', 'root_value'):
        np.testing.assert_array_equal(np.load(tmp_path / 'a' / f'{k}.npy'), out[k][rows].astype(np.float64))
    np.testing.assert_array_equal(np.load(tmp_path / 'a' / 'train_priorities.npy'),
                                  out['train_priorities'].astype(np.float64))
