"""bench.py's synthetic workload: deterministic, and the rank shards tile the global matrix exactly
(INTERLEAVED sharding, xgboost_ray/matrix.py:1100), so the bench trains the SAME dataset at every N.
--dump-outputs writes the trees of the last timed round and the training margin after warm-up + K rounds."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_shards_tile_the_global_matrix():
    n, f = 2500, 12
    X, y = bench.synth_shard(n, f, 0, 1, block_rows=1000)
    X2, y2 = bench.synth_shard(n, f, 0, 1, block_rows=1000)
    assert np.array_equal(X, X2) and np.array_equal(y, y2)           # deterministic
    assert X.shape == (n, f) and X.dtype == np.float32 and 0 <= X.min() and X.max() < 10
    for world in (2, 3, 8):
        parts = [bench.synth_shard(n, f, r, world, block_rows=1000) for r in range(world)]
        for r, (xs, ys) in enumerate(parts):
            assert np.array_equal(xs, X[r::world]) and np.array_equal(ys, y[r::world])
        assert sum(len(p[0]) for p in parts) == n


def test_label_is_learnable_signal():
    X, y = bench.synth_shard(4000, 20, 0, 1)
    a = np.random.default_rng(1234).normal(size=10).astype(np.float32)
    resid = y - (X[:, :10] @ a + np.sin(X[:, 10]))
    assert abs(resid.mean()) < 0.02 and 0.05 < resid.std() < 0.2     # y = sum a_j x_j + sin(x_10) + N(0, 0.1)


def _load_dump(d):
    out = {os.path.basename(f)[:-4]: np.load(f) for f in glob.glob(os.path.join(d, "*.npy"))}
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    return out


def _assert_dump_is_round(dump, or_bst, rounds, leaf_tol):
    """dump = the last of `rounds` oracle rounds: same trees (split exact, leaf values within leaf_tol) and margin."""
    K = or_bst.K
    assert or_bst.num_trees == rounds * K
    trees = [or_bst.tree(i) for i in range(or_bst.num_trees - K, or_bst.num_trees)]
    assert np.array_equal(dump["tree_nodes"], [t.n_nodes for t in trees])
    for k in ("left", "right", "split_feature", "split_bin", "default_left"):
        assert np.array_equal(dump["tree_" + k], np.concatenate([getattr(t, k) for t in trees])), k
    leaf = dump["tree_left"] < 0
    assert np.max(np.abs(dump["tree_value"][leaf] - np.concatenate([t.value for t in trees])[leaf])) <= leaf_tol
    assert dump["margin"].shape == or_bst.margin.shape
    assert np.max(np.abs(dump["margin"] - or_bst.margin)) <= rounds * leaf_tol + 1e-5


def test_dump_outputs_reference_arm(oracle, tmp_path, monkeypatch, capsys):
    n, f, steps = 3000, 12, 2
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--rows", str(n), "--cols", str(f),
                                      "--depth", "4", "--steps", str(steps), "--warmup", "3", "--dump-outputs", str(tmp_path)])
    bench.main()
    assert json.loads(capsys.readouterr().out.strip().splitlines()[-1])["steps"] == steps
    X, y = bench.synth_shard(n, f, 0, 1)
    ob, _ = oracle.train(dict(bench.PARAMS, max_depth=4, hist_qbits=0), X, y, 3 + steps)
    _assert_dump_is_round(_load_dump(str(tmp_path)), ob, 3 + steps, 0.0)


def test_dump_outputs_sample_is_fixed_and_bounded(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MARGIN_VALUES", 3000)
    tree = {k: np.arange(5, dtype=np.int32) for k in bench.TREE_FIELDS}
    tree["cat_bits"] = np.zeros((5, 8), np.uint32)
    margin = np.arange(4000 * 3, dtype=np.float32).reshape(4000, 3)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), [tree, tree], margin)
    a, b = _load_dump(str(tmp_path / "a")), _load_dump(str(tmp_path / "b"))
    assert a["margin"].shape == (1000, 3) and np.array_equal(a["margin"], b["margin"])
    rows = a["margin"][:, 0].astype(np.int64) // 3
    assert np.all(np.diff(rows) > 0) and np.array_equal(a["margin"], margin[rows])
    assert np.array_equal(a["tree_nodes"], [5, 5]) and a["tree_cat_bits"].shape == (10, 8)


@pytest.mark.gpu
def test_dump_outputs_device_arm(oracle, tmp_path):
    n, f, steps = 20000, 12, 2
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--rows", str(n), "--cols", str(f), "--depth", "6",
                        "--steps", str(steps), "--warmup", "3", "--no-cpu-baseline", "--no-e2e", "--no-parity",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
    X, y = bench.synth_shard(n, f, 0, 1)
    ob, _ = oracle.train(dict(bench.PARAMS, max_depth=6), X, y, 3 + steps)
    _assert_dump_is_round(_load_dump(str(tmp_path)), ob, 3 + steps, 1e-5)
