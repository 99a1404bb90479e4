"""CPU: bench.py --dump-outputs writes float32 / float64 .npy files, keeps their total under the limit with a seeded sample
of chains, and writes the same bytes for the same inputs."""
import os

import numpy as np


def _dump(tmp_path, name, n, d):
    import bench
    rng = np.random.RandomState(1)
    per_chain = {'first_x': rng.normal(size=(n, d)).astype(np.float32), 'last_x': rng.normal(size=(n, d)).astype(np.float32),
                 'last_logl': rng.normal(size=n)}
    out = str(tmp_path / name)
    bench.dump_outputs(out, per_chain, {'scale': 0.25, 'naccept': 12345, 'ncall': 67890})
    return per_chain, {f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out)}


def test_dump_writes_every_output_whole_below_the_limit(tmp_path):
    per_chain, got = _dump(tmp_path, 'small', 1000, 30)
    assert sorted(got) == ['first_x', 'last_logl', 'last_x', 'naccept', 'ncall', 'scale']
    for k, v in per_chain.items():
        assert got[k].dtype == v.dtype and np.array_equal(got[k], v)
    assert got['naccept'].dtype == np.float64 and got['naccept'][0] == 12345 and got['scale'][0] == 0.25


def test_dump_samples_the_same_chains_of_every_output_above_the_limit(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, 'DUMP_LIMIT_BYTES', 1 << 20)
    n, d = 20000, 30                        # 2 x 2.4 MB of float32 states
    per_chain, got = _dump(tmp_path, 'a', n, d)
    assert sum(v.nbytes for v in got.values()) <= bench.DUMP_LIMIT_BYTES
    rows = got['chain_index'].astype(np.int64)
    assert got['chain_index'].dtype == np.float64 and len(rows) < n and np.all(np.diff(rows) > 0)
    for k, v in per_chain.items():
        assert got[k].dtype == v.dtype and np.array_equal(got[k], v[rows])
    _, again = _dump(tmp_path, 'b', n, d)
    assert all(np.array_equal(got[k], again[k]) for k in got)
