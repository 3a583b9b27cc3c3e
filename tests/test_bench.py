"""bench.py --dump-outputs: what the timed path hands its caller is written exactly, and within 64 MB through a fixed sample of
the chains when there are more of them than fit."""
import os

import numpy as np

import bench
import timberborn_support_solver_b200 as T


class StandInSearch:
    """The read side of Search (read_chains, best_count, best_layout) over given chain states: no device needed."""

    def __init__(self, n_chains, seed=1):
        rng = np.random.default_rng(seed)
        self.n_chains, self.grid = n_chains, T.WorldGrid(np.ones((16, 16), np.uint8))
        self.state = dict(S=rng.integers(0, 1 << 16, (n_chains, 32), dtype=np.uint32), bestS=rng.integers(0, 1 << 16, (n_chains, 32), dtype=np.uint32),
                          k=rng.integers(15, 40, n_chains, dtype=np.int32), best=rng.integers(15, 40, n_chains, dtype=np.int32),
                          step=rng.integers(0, 1 << 32, n_chains, dtype=np.uint32), scored=rng.integers(0, 1 << 50, n_chains, dtype=np.uint64))

    def read_chains(self):
        return self.state

    def best_count(self):
        return 2

    def best_layout(self):
        return T.PlatformLayout([T.Platform(3, 5, T.PlatformDef(1, 1)), T.Platform(9, 1, T.PlatformDef(1, 1))])


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_outputs_exact_and_bounded(tmp_path):
    for n in (1000, 300_000):                 # all chains / a sample: 300 000 chains x 288 bytes exceed 64 MB
        s = StandInSearch(n)
        out = tmp_path / str(n)
        bench.dump_outputs(str(out), s)
        files = _load(out)
        assert all(a.dtype == np.float64 for a in files.values())
        assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= 64 * 10 ** 6
        idx = files["chain_index"].astype(np.int64)
        assert (len(idx) == n) == (n == 1000) and (np.diff(idx) > 0).all()
        for name, key in (("chain_count", "k"), ("chain_best_count", "best"), ("chain_step", "step"), ("chain_scored", "scored")):
            assert np.array_equal(files[name].astype(s.state[key].dtype), s.state[key][idx]), name
        assert np.array_equal(files["chain_supports"], s.state["S"][idx, :16]) and np.array_equal(files["chain_best_supports"], s.state["bestS"][idx, :16])
        assert files["best_count"].tolist() == [2] and files["best_layout"].tolist() == [[9, 1, 1, 1, 0], [3, 5, 1, 1, 0]]
    again = tmp_path / "again"
    bench.dump_outputs(str(again), StandInSearch(300_000))
    assert np.array_equal(_load(again)["chain_index"], _load(tmp_path / "300000")["chain_index"])     # the sample is fixed
