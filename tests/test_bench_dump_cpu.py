"""bench.py --dump-outputs without a GPU: which reaches are written, the size bound, and that the files hold exactly
the routed values of those reaches in params-file order, on one rank and assembled from two."""
import os

import numpy as np
import torch

import bench
import river_route_b200 as rr
from river_route_b200 import synth


def test_dump_sample_is_fixed_bounded_and_keeps_outlets():
    down = synth.forest(5000, 30, seed=4)
    outlets = np.flatnonzero(down < 0)
    assert bench.dump_sample(down, 12).shape[0] == down.shape[0]       # a small network is written whole
    for rows in (12, 20000, 300000):
        s = bench.dump_sample(down, rows)
        assert np.array_equal(s, bench.dump_sample(down, rows))
        assert np.all(np.diff(s) > 0) and s[0] >= 0 and s[-1] < down.shape[0]
        assert s.shape[0] * (rows + 1) * 8 <= bench.DUMP_BYTES < 64_000_000
        if s.shape[0] > outlets.shape[0]:
            assert np.isin(outlets, s).all()
        else:
            assert np.isin(s, outlets).all()


class _Gather:
    """torch.distributed.gather for ranks that call it one after the other (``caller``), rank 0 last."""
    def __init__(self, world):
        self.world, self.sent, self.caller = world, {}, None

    def gather(self, t, parts, dst=0):
        self.sent.setdefault(self.caller, []).append(t.clone())
        if parts is not None:
            k = len(self.sent[0]) - 1
            for i in range(self.world):
                parts[i].copy_(self.sent[i][k])


def test_dump_outputs_writes_the_sampled_results(tmp_path, monkeypatch):
    n, rows = 4000, 12
    down = synth.forest(n, 20, seed=2)
    rng = np.random.default_rng(0)
    out, q = rng.random((rows, n)), rng.random(n)
    cpu = torch.device('cpu')
    monkeypatch.setattr(bench, 'DUMP_BYTES', 500 * (rows + 1) * 8)     # a sample, not the whole network
    s = bench.dump_sample(down, rows)
    assert s.shape[0] == 500

    def written(d):
        return np.load(os.path.join(d, 'discharge.npy')), np.load(os.path.join(d, 'channel_state.npy'))

    one = str(tmp_path / 'one')
    bench.dump_outputs(one, torch, None, 0, 1, down, np.arange(n), torch.from_numpy(out), torch.from_numpy(q), rows, cpu)
    d1, q1 = written(one)
    assert d1.dtype == q1.dtype == np.float64
    assert np.array_equal(d1, out[:, s]) and np.array_equal(q1, q[s])

    two = str(tmp_path / 'two')
    part = rr.label_basins(down, 2)[2]
    g = _Gather(2)
    for r in (1, 0):
        idx = np.flatnonzero(part == r)
        assert idx.shape[0] > 0
        g.caller = r
        bench.dump_outputs(two, torch, g, r, 2, down, idx, torch.from_numpy(np.ascontiguousarray(out[:, idx])),
                           torch.from_numpy(q[idx].copy()), rows, cpu)
    d2, q2 = written(two)
    assert np.array_equal(d2, d1) and np.array_equal(q2, q1)
