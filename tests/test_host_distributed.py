"""Host-layer tests on CPU: spawned actors (one process each), world_size 2 over `gloo` through the
test-only stand-in engine (tests/cpu_engine.py).  Ports the hot-path subset of
xgboost_ray/tests/test_end_to_end.py, test_xgboost_api.py and test_fault_tolerance.py."""
import os
import pickle

import numpy as np
import pytest


@pytest.fixture(autouse=True)
def use_cpu_engine(monkeypatch):
    """The stand-in engine is a TEST seam: monkeypatched into the driver process here, installed in every actor process
    by a distributed callback that this fixture adds to each RayParams the driver validates."""
    import tests.cpu_engine as ce
    import xgboost_ray_b200.main as M
    import xgboost_ray_b200.xgb as seam
    monkeypatch.setenv("OMP_NUM_THREADS", "1")
    # the stand-in computes on the CPU: the host layer and its actors see no GPU, as on a CPU-only machine, also where
    # CUDA_VISIBLE_DEVICES names one (the host layer would otherwise assign it to the actors, one GPU each)
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    monkeypatch.setattr(seam, "xgboost", ce)
    orig = M._validate_ray_params

    def with_cpu_engine(rp):
        rp = orig(rp)
        cbs = list(rp.distributed_callbacks or [])
        if not any(isinstance(c, ce.UseCpuEngine) for c in cbs):
            rp.distributed_callbacks = [ce.UseCpuEngine()] + cbs
        return rp

    monkeypatch.setattr(M, "_validate_ray_params", with_cpu_engine)
    yield
    M.shutdown_actors()


X_TOY = np.array([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 1], [0, 0, 1, 0]] * 8, np.float32)
Y_TOY = np.array([0, 1, 2, 3] * 8, np.float32)
TOY_PARAMS = {"booster": "gbtree", "nthread": 1, "max_depth": 2, "objective": "multi:softmax", "num_class": 4}


@pytest.mark.timeout(300)
@pytest.mark.parametrize("sharding", ["INTERLEAVED", "BATCH"])
def test_two_actor_training_learns_full_matrix(sharding):
    """test_end_to_end.py:162-211: each half alone over-fits, 2 actors with the exchange step are exact."""
    from xgboost_ray_b200 import RayDMatrix, RayParams, RayShardingMode, predict, train
    mode = getattr(RayShardingMode, sharding)
    evals_result, extra = {}, {}
    dtrain = RayDMatrix(X_TOY, Y_TOY, sharding=mode)
    bst = train(TOY_PARAMS, dtrain, num_boost_round=2, evals=[(dtrain, "train")], evals_result=evals_result,
                additional_results=extra, ray_params=RayParams(num_actors=2, checkpoint_frequency=1))
    assert extra["total_n"] == 32 and extra["training_time_s"] > 0
    assert len(evals_result["train"]["mlogloss"]) == 2
    pred = predict(bst, RayDMatrix(X_TOY, sharding=mode), ray_params=RayParams(num_actors=2))
    assert list(pred) == list(Y_TOY)                  # recombined in original row order
    bst2 = pickle.loads(pickle.dumps(bst))
    assert bst2.get_dump() == bst.get_dump()


@pytest.mark.timeout(300)
def test_callbacks_see_ranks_and_queue_returns():
    from tests.fault_injection import RankRecorder
    from xgboost_ray_b200 import RayDMatrix, RayParams, train
    extra = {}
    train(TOY_PARAMS, RayDMatrix(X_TOY, Y_TOY), num_boost_round=2, additional_results=extra,
          ray_params=RayParams(num_actors=2), callbacks=[RankRecorder()])
    got = sorted(item[1] for per_rank in extra["callback_returns"] for item in per_rank)
    assert got == [0, 1]                               # test_xgboost_api.py:154-178


@pytest.mark.timeout(600)
def test_restart_from_checkpoint_gives_same_model(tmp_path):
    """test_fault_tolerance.py:401-444: failure at round 6, restart from checkpoint 5 == uninterrupted."""
    from tests.fault_injection import DieOnceCallback
    from xgboost_ray_b200 import RayDMatrix, RayParams, train
    rng = np.random.RandomState(0)
    x = rng.uniform(0, 10, size=(400, 4)).astype(np.float32)
    y = (x[:, 0] + x[:, 1] > 10).astype(np.float32)
    params = {"objective": "binary:logistic", "max_depth": 3, "nthread": 1}
    ref = train(params, RayDMatrix(x, y), num_boost_round=10, ray_params=RayParams(num_actors=2, checkpoint_frequency=1))
    extra = {}
    bst = train(params, RayDMatrix(x, y), num_boost_round=10, additional_results=extra,
                ray_params=RayParams(num_actors=2, max_actor_restarts=1, checkpoint_frequency=5),
                callbacks=[DieOnceCallback(str(tmp_path / "lock"), rank=1, at=6)])
    assert os.path.exists(str(tmp_path / "lock"))
    assert bst.num_boosted_rounds() == 10
    assert bst.get_dump() == ref.get_dump()
    with pytest.raises(RuntimeError, match="maximum number of retries"):
        train(params, RayDMatrix(x, y), num_boost_round=10, ray_params=RayParams(num_actors=2, max_actor_restarts=0),
              callbacks=[DieOnceCallback(str(tmp_path / "lock2"), rank=0, at=2)])


@pytest.mark.timeout(300)
def test_validation_errors():
    from xgboost_ray_b200 import RayDMatrix, RayParams, train
    d = RayDMatrix(X_TOY, Y_TOY)
    with pytest.raises(ValueError, match="num_actors"):
        train(TOY_PARAMS, d, ray_params=RayParams())
    with pytest.raises(ValueError, match="RayDMatrix"):
        train(TOY_PARAMS, X_TOY, ray_params=RayParams(num_actors=1))
    with pytest.raises(ValueError, match="exact"):
        train(dict(TOY_PARAMS, tree_method="exact"), d, ray_params=RayParams(num_actors=1))
    with pytest.raises(TypeError, match="invalid keyword"):
        train(TOY_PARAMS, d, ray_params=RayParams(num_actors=1), totally_invalid_kwarg=1)
    with pytest.raises(ValueError, match="no label"):
        train(TOY_PARAMS, RayDMatrix(X_TOY), ray_params=RayParams(num_actors=1))
    # engine error propagates as a training failure (main.py:770-785)
    with pytest.raises(RuntimeError):
        train(dict(TOY_PARAMS, objective="rank:pairwise"), RayDMatrix(X_TOY, Y_TOY), ray_params=RayParams(num_actors=1))


@pytest.mark.timeout(300)
def test_sklearn_estimators():
    """Subset of xgboost_ray/tests/test_sklearn.py: accuracy bars on digits (2-class err < 0.1, :115-141)
    and multiclass, regression fit, RayDMatrix input (test_sklearn_matrix.py)."""
    from sklearn.datasets import load_digits
    from xgboost_ray_b200 import RayDMatrix, RayParams
    from xgboost_ray_b200.sklearn import RayXGBClassifier, RayXGBRegressor
    d = load_digits(n_class=2)
    X, y = d.data.astype(np.float32), d.target
    clf = RayXGBClassifier(n_estimators=10, max_depth=4).fit(X[::2], y[::2], ray_params=RayParams(num_actors=2))
    pred = clf.predict(X[1::2], ray_params=RayParams(num_actors=2))
    assert np.mean(pred != y[1::2]) < 0.1
    proba = clf.predict_proba(X[1::2], ray_params=RayParams(num_actors=1))
    assert proba.shape == (len(X[1::2]), 2) and np.allclose(proba.sum(axis=1), 1.0, atol=1e-5)
    d3 = load_digits(n_class=3)
    clf3 = RayXGBClassifier(n_estimators=5, max_depth=3).fit(d3.data.astype(np.float32), d3.target + 10,
                                                             ray_params=RayParams(num_actors=2))
    p3 = clf3.predict(d3.data.astype(np.float32), ray_params=RayParams(num_actors=2))
    assert set(np.unique(p3)) <= {10, 11, 12} and np.mean(p3 != d3.target + 10) < 0.1
    rng = np.random.RandomState(0)
    Xr = rng.uniform(0, 10, size=(500, 5)).astype(np.float32)
    yr = (Xr[:, 0] * 2 + Xr[:, 1]).astype(np.float32)
    reg = RayXGBRegressor(n_estimators=20, max_depth=4).fit(RayDMatrix(Xr, yr), ray_params=RayParams(num_actors=2))
    assert np.mean((reg.predict(RayDMatrix(Xr), ray_params=RayParams(num_actors=2)) - yr) ** 2) < 1.0


@pytest.mark.timeout(600)
def test_feature_weights_reach_the_engine():
    """test_end_to_end.py:429-467: RayDMatrix(feature_weights=...) is forwarded per actor (set_info, main.py:439-442);
    weights 0..9 with colsample_bynode=0.1 -> feature 0 is never used, feature 9 most."""
    import json
    from xgboost_ray_b200 import RayDMatrix, RayParams, train
    rng = np.random.RandomState(1994)
    X = rng.randn(1000, 10).astype(np.float32)
    y = rng.randn(1000).astype(np.float32)
    fw = np.arange(10, dtype=np.float32)
    bst = train({"objective": "reg:squarederror", "colsample_bynode": 0.1}, RayDMatrix(X, y, feature_weights=fw),
                num_boost_round=40, ray_params=RayParams(num_actors=2, cpus_per_actor=1))
    cnt = np.zeros(10, int)
    for t in bst.get_dump():
        for f in json.loads(t)["split_feature"]:
            if f >= 0:
                cnt[f] += 1
    assert cnt[0] == 0 and cnt.argmax() == 9


@pytest.mark.timeout(600)
def test_custom_objective_and_metric_two_actors():
    """test_xgboost_api.py:77-152: a custom objective (squared log error) and a custom metric through two actors
    give the single-process result; the rounded predictions reproduce the labels."""
    from tests.fault_injection import rmsle, squared_log
    from xgboost_ray_b200 import RayDMatrix, RayParams, predict, train
    x = np.array([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 1], [0, 0, 1, 0]] * 8, np.float32)
    y = np.array([0, 1, 0, 1] * 8, np.float32)
    params = {"booster": "gbtree", "tree_method": "hist", "nthread": 1, "max_depth": 2, "seed": 1000}
    res1, res2 = {}, {}
    d1, d2 = RayDMatrix(x, y), RayDMatrix(x, y)
    b1 = train(params, d1, evals=[(d1, "dtrain")], evals_result=res1, obj=squared_log, feval=rmsle, ray_params=RayParams(num_actors=1))
    b2 = train(params, d2, evals=[(d2, "dtrain")], evals_result=res2, obj=squared_log, feval=rmsle, ray_params=RayParams(num_actors=2))
    p1 = np.round(predict(b1, RayDMatrix(x), ray_params=RayParams(num_actors=1)))
    p2 = np.round(predict(b2, RayDMatrix(x), ray_params=RayParams(num_actors=2)))
    assert list(p1) == list(p2) == list(y)
    assert np.allclose(res1["dtrain"]["PyRMSLE"], res2["dtrain"]["PyRMSLE"], atol=0.1) and len(res2["dtrain"]["PyRMSLE"]) == 10


@pytest.mark.timeout(600)
def test_sklearn_parameters_and_attributes(tmp_path):
    """sklearn.py surface: engine parameters travel from the estimator to xgb.train, None leaves the engine default
    (base_score=None -> estimated like xgboost >= 2.0), importances, unsupported estimators fail loudly."""
    from xgboost_ray_b200 import RayParams
    from xgboost_ray_b200.sklearn import (RayXGBClassifier, RayXGBRanker, RayXGBRegressor, RayXGBRFClassifier,
                                          RayXGBRFRegressor)
    reg = RayXGBRegressor(n_estimators=3, max_depth=3, subsample=0.8, colsample_bynode=0.5, random_state=7,
                          max_delta_step=1.0, eval_metric="rmse")
    p = reg.get_xgb_params()
    assert p["subsample"] == 0.8 and p["colsample_bynode"] == 0.5 and p["seed"] == 7 and p["max_delta_step"] == 1.0
    assert "base_score" not in p and "scale_pos_weight" not in p and p["eval_metric"] == "rmse"
    assert RayXGBClassifier(scale_pos_weight=3.0, base_score=0.4).get_xgb_params()["scale_pos_weight"] == 3.0
    assert set(reg.get_params()) >= {"subsample", "colsample_bytree", "enable_categorical", "early_stopping_rounds"}
    rng = np.random.RandomState(0)
    X = rng.uniform(0, 10, size=(600, 6)).astype(np.float32)
    y = (X[:, 2] * 3 + rng.normal(scale=0.1, size=600)).astype(np.float32)
    reg = RayXGBRegressor(n_estimators=8, max_depth=3, colsample_bynode=0.5, random_state=1).fit(
        X, y, eval_set=[(X, y)], ray_params=RayParams(num_actors=2))
    imp = reg.feature_importances_
    assert imp.shape == (6,) and abs(imp.sum() - 1.0) < 1e-5 and imp.argmax() == 2
    assert "validation_0" in reg.evals_result() and len(reg.evals_result()["validation_0"]["rmse"]) == 8
    with pytest.raises(NotImplementedError):
        RayXGBRanker()
    rf = RayXGBRFRegressor(n_estimators=7, max_depth=3)
    p = rf.get_xgb_params()
    assert p["num_parallel_tree"] == 7 and p["learning_rate"] == 1.0 and p["subsample"] == 0.8 and p["colsample_bynode"] == 0.8
    assert rf.get_num_boosting_rounds() == 1 and rf.get_params()["reg_lambda"] == 1e-5
    from sklearn.base import clone
    assert clone(RayXGBRFClassifier(n_estimators=3, subsample=0.5)).get_params()["subsample"] == 0.5


@pytest.mark.timeout(600)
def test_elastic_training_continues_on_the_remaining_actor(tmp_path):
    """elastic.py / test_fault_tolerance.py:125-167: with elastic_training a dead actor is not waited for -- training
    continues from the last checkpoint on the surviving actors (their shards only) with a new, smaller communicator."""
    from tests.fault_injection import DieOnceCallback
    from xgboost_ray_b200 import RayDMatrix, RayParams, train
    rng = np.random.RandomState(1)
    x = rng.uniform(0, 10, size=(401, 4)).astype(np.float32)
    y = (x[:, 0] + x[:, 1] > 10).astype(np.float32)
    params = {"objective": "binary:logistic", "max_depth": 3, "nthread": 1}
    extra = {}
    bst = train(params, RayDMatrix(x, y), num_boost_round=10, additional_results=extra,
                ray_params=RayParams(num_actors=2, elastic_training=True, max_failed_actors=1, max_actor_restarts=2,
                                     checkpoint_frequency=5),
                callbacks=[DieOnceCallback(str(tmp_path / "lock"), rank=0, at=6)])
    assert bst.num_boosted_rounds() == 10
    assert extra["total_n"] == len(range(1, 401, 2))          # the last attempt trained on the surviving actor's shard only
    with pytest.raises(RuntimeError, match="maximum number of dead actors"):
        train(params, RayDMatrix(x, y), num_boost_round=10,
              ray_params=RayParams(num_actors=2, elastic_training=True, max_failed_actors=1, max_actor_restarts=3),
              callbacks=[DieOnceCallback(str(tmp_path / "l0"), rank=0, at=2), DieOnceCallback(str(tmp_path / "l1"), rank=0, at=1)])
    with pytest.raises(ValueError, match="max_failed_actors"):
        train(params, RayDMatrix(x, y), ray_params=RayParams(num_actors=2, elastic_training=True, max_actor_restarts=1))


@pytest.mark.timeout(600)
def test_actor_pool_shared_memory_and_actor_side_file_loading(tmp_path):
    """Actors are reused between train() and predict() calls (same pids), shards travel as /dev/shm files that disappear
    with the RayDMatrix, and a list of files is read by the actors themselves, one row block per file."""
    import glob
    import pandas as pd
    import xgboost_ray_b200.main as M
    from tests.fault_injection import PidRecorder
    from xgboost_ray_b200 import RayDMatrix, RayParams, predict, train
    rng = np.random.RandomState(2)
    x = rng.uniform(0, 10, size=(600, 5)).astype(np.float32)
    y = (x[:, 0] * 2 + x[:, 1]).astype(np.float32)
    params = {"objective": "reg:squarederror", "max_depth": 3, "nthread": 1}
    e1, e2 = {}, {}
    d = RayDMatrix(x, y)
    b1 = train(params, d, num_boost_round=3, additional_results=e1, ray_params=RayParams(num_actors=2), callbacks=[PidRecorder()])
    shm = [v[1] for sh in d._shared.values() for v in sh.values() if isinstance(v, tuple) and v[0] == "shm"]
    assert shm and all(os.path.exists(p) for p in shm)
    # the feature matrix itself is not copied at all: the actors read their rows out of this process
    assert e1["timing"]["shard_transport"] == "remote" and all(sh["data"][0] == "remote" for sh in d._shared.values())
    assert e1["timing"]["actor0"]["upload_s"] >= 0
    # wall-clock stamps of the driver and of both actors (bench.py reports them with the e2e number)
    stamps = e1["timing"]["actors"]
    assert len(stamps) == 2 and len(e1["timing"]["t_future_done"]) == 2
    for st in stamps:
        assert e1["timing"]["t_dispatch"] <= st["t_enter"] <= st["t_trained"] <= st["t_thread_end"] <= st["t_return"]
    assert max(e1["timing"]["t_future_done"]) >= max(st["t_return"] for st in stamps)
    b2 = train(params, RayDMatrix(x, y), num_boost_round=3, additional_results=e2, ray_params=RayParams(num_actors=2),
               callbacks=[PidRecorder()])
    pids = lambda e: sorted(item[1] for per_rank in e["callback_returns"] for item in per_rank)  # noqa: E731
    assert pids(e1) == pids(e2) and len(set(pids(e1))) == 2          # the same two processes served both calls
    assert b1.get_dump() == b2.get_dump()
    p = predict(b1, RayDMatrix(x), ray_params=RayParams(num_actors=2))
    assert np.mean((p - y) ** 2) < np.var(y)
    d.unload_data()
    assert not any(os.path.exists(p) for p in shm)
    # ---- file list: 4 parquet files, 2 actors -> every actor reads its 2 files itself and keeps them as 2 row blocks
    files = []
    for i in range(4):
        df = pd.DataFrame(x[i * 150:(i + 1) * 150], columns=["a", "b", "c", "d", "e"])
        df["target"] = y[i * 150:(i + 1) * 150]
        f = str(tmp_path / ("part%d.parquet" % i))
        df.to_parquet(f)
        files.append(f)
    df_all = RayDMatrix(files, label="target")
    assert df_all.distributed
    e3 = {}
    b3 = train(params, df_all, num_boost_round=3, additional_results=e3, ray_params=RayParams(num_actors=2))
    assert e3["total_n"] == 600 and not df_all.refs                   # the driver never loaded the rows
    assert b3.get_dump() == b1.get_dump()                             # same rows, same model (row order does not matter)
    M.shutdown_actors()
    # forced file hand-off (what the driver falls back to when the kernel refuses process_vm_readv): same model
    os.environ["B2_SHARD_TRANSPORT"] = "shm"
    try:
        e4 = {}
        d4 = RayDMatrix(x, y)
        b4 = train(params, d4, num_boost_round=3, additional_results=e4, ray_params=RayParams(num_actors=2))
        assert e4["timing"]["shard_transport"] == "shm" and all(sh["data"][0] == "shm" for sh in d4._shared.values())
        assert b4.get_dump() == b1.get_dump()
    finally:
        del os.environ["B2_SHARD_TRANSPORT"]
        M.shutdown_actors()


@pytest.mark.timeout(300)
def test_pandas_category_columns_become_categorical_features():
    """The reference hands the DataFrame to xgb.DMatrix(enable_categorical=True): category dtype -> codes, typed 'c'."""
    import pandas as pd
    from xgboost_ray_b200 import RayDMatrix
    from xgboost_ray_b200.main import _matrix_meta
    df = pd.DataFrame({"num": [0.5, 1.5, 2.5, 3.5], "cat": pd.Categorical(["b", "a", None, "b"], categories=["a", "b"])})
    with pytest.raises(ValueError, match="enable_categorical"):
        RayDMatrix(df, np.zeros(4, np.float32), num_actors=1)
    m = RayDMatrix(df, np.zeros(4, np.float32), enable_categorical=True, num_actors=1)
    shard = m.get_data(0)
    assert np.array_equal(shard["data"][:, 0], np.array([0.5, 1.5, 2.5, 3.5], np.float32))
    assert shard["data"][0, 1] == 1 and shard["data"][1, 1] == 0 and np.isnan(shard["data"][2, 1])
    assert _matrix_meta(m)["feature_types"] == ["q", "c"] and _matrix_meta(m)["enable_categorical"]
