"""bench.py --dump-outputs, on the CPU: what is written, in which dtype, and the fixed row sample that keeps a larger output
within the size budget."""
import os

import numpy as np

import bench


def _sol(n, steps=6):
    rng = np.random.default_rng(1)
    S = dict(its=rng.integers(0, 9, size=(4, steps)), its_finalize=2, ts=np.logspace(-1, 8, steps), kappas=np.full(steps, 10.0),
             c_dot_Dz=rng.normal(size=steps), times=rng.random(steps), t_begin=0.5, t_elapsed=1.5, z_unfinalized=rng.normal(size=(n, 2)))
    return dict(z=rng.normal(size=(n, 2)), SOL_main=S, SOL_feasibility=None)


def test_dump_writes_the_whole_solution_in_float64(tmp_path):
    sol = _sol(1000)
    names = bench.dump_outputs(str(tmp_path), sol)
    assert sorted(os.listdir(tmp_path)) == sorted(k + ".npy" for k in names)
    assert set(names) == {"z", "z_unfinalized", "its", "its_finalize", "ts", "kappas", "c_dot_Dz"}
    for k in names:
        a = np.load(tmp_path / (k + ".npy"))
        assert a.dtype == np.float64
        ref = sol[k] if k == "z" else sol["SOL_main"][k]
        assert np.array_equal(a, np.asarray(ref, dtype=np.float64)), k


def test_dump_above_the_budget_is_the_same_row_sample_every_run(tmp_path):
    sol = _sol(100000)                      # 3.2 MB of per-node arrays
    budget = 1 << 20
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), sol, budget=budget)
    a, b = tmp_path / "a", tmp_path / "b"
    assert sum(f.stat().st_size for f in a.iterdir()) <= budget
    rows = np.load(a / "node_rows.npy").astype(np.int64)
    assert rows.size > 10000 and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(a / "z.npy"), sol["z"][rows])
    assert np.array_equal(np.load(a / "z_unfinalized.npy"), sol["SOL_main"]["z_unfinalized"][rows])
    assert np.array_equal(np.load(a / "ts.npy"), sol["SOL_main"]["ts"])
    for f in os.listdir(a):
        assert np.array_equal(np.load(a / f), np.load(b / f)), f
