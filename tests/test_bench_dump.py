"""bench.py --dump-outputs: the paths of the last timed step as float64 arrays, every window when they fit the budget, otherwise a
fixed seeded sample of windows that does."""
import numpy as np

import bench
from augustus_b200.decoder import State, StatePath

NAMES = ("window", "status", "log_prob", "n_states", "type", "begin", "end", "truncated")


def _paths(n):
    rng = np.random.default_rng(3)
    out = []
    for i in range(n):
        k = int(rng.integers(1, 40))
        out.append(StatePath([State(int(rng.integers(0, 47)), 10 * j, 10 * j + 9, j & 1) for j in range(k)], -1000.25 - 0.5 * i))
    return out


def _load(d, prefix=""):
    return {n: np.load(d / (prefix + n + ".npy")) for n in NAMES}


def test_dump_writes_every_window_when_it_fits(tmp_path):
    paths, ids = _paths(50), list(range(7, 107, 2))
    bench.dump_paths(str(tmp_path), ids, paths)
    d = _load(tmp_path)
    assert all(a.dtype == np.float64 for a in d.values())
    assert d["window"].tolist() == ids and d["status"].tolist() == [0] * 50
    assert d["log_prob"].tolist() == [p.log_prob for p in paths]
    assert d["n_states"].tolist() == [len(p.states) for p in paths]
    rows = np.stack([d[n] for n in ("type", "begin", "end", "truncated")], axis=1)
    assert rows.tolist() == [list(s) for p in paths for s in p.as_tuples()]


def test_dump_over_budget_is_a_fixed_sample_of_whole_windows(tmp_path):
    paths, budget = _paths(400), 20000
    bench.dump_paths(str(tmp_path / "a"), range(400), paths, budget)
    bench.dump_paths(str(tmp_path / "b"), range(400), paths, budget, prefix="rank0_")
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b", "rank0_")
    assert all(np.array_equal(a[n], b[n]) for n in NAMES)                   # the same windows on every run
    assert sum(x.nbytes for x in a.values()) <= budget
    w = a["window"].astype(int)
    assert 0 < len(w) < 400 and np.all(np.diff(w) > 0) and w[-1] > 200      # spread over the batch, in index order
    assert a["n_states"].tolist() == [len(paths[k].states) for k in w]
    assert a["begin"].tolist() == [s.begin for k in w for s in paths[k].states]
