"""
The builder on the GPU: gb_cv_moments against numpy, the fleet's cross-validation scores against sklearn applied to the fold
models' own predictions, and FleetModelBuilder / ModelBuilder end to end (tests/gordo/builder/test_builder.py:160-430).
"""
import json
import os

import numpy as np
import pandas as pd
import pytest
from sklearn import metrics as sk_metrics
from sklearn.preprocessing import MinMaxScaler

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch as t

    if not t.cuda.is_available():
        pytest.skip("needs a B200")
    import __graft_entry__ as ge

    ge.build()
    return t


@pytest.fixture(scope="module")
def engine(torch):
    from gordo_components_b200 import engine as e

    return e


def numpy_moments(yhat, y):
    yhat, y = yhat.astype(np.float64), y.astype(np.float64)
    e, c = yhat - y, y - y[0]
    return np.stack([e.sum(0), (e * e).sum(0), np.abs(e).sum(0), c.sum(0), (c * c).sum(0)])


@pytest.mark.parametrize("T", [1, 5, 64, 100])
def test_cv_moments_match_numpy(engine, torch, T):
    rng = np.random.default_rng(T)
    rows = [700, 1, 33, 2500]
    y = (rng.random((sum(rows) + 50, T)) * 10 + 1000).astype(np.float32)  # a large offset: the shift by the first row matters
    yhat = (rng.random((sum(rows), T)) * 10 + 1000).astype(np.float32)
    y_start = np.array([50, 750, 751, 784])          # jobs read y and yhat at different row offsets
    out_start = np.array([0, 700, 701, 734])
    dev = engine.cuda_device()
    jobs = engine.jobs_to_device(engine.make_jobs(np.arange(4), np.array(rows), y_start, out_start), dev)
    got = engine.cv_moments(jobs, 4, torch.from_numpy(yhat).to(dev), torch.from_numpy(y).to(dev), T).cpu().numpy()
    assert got.shape == (4, 5, T) and got.dtype == np.float64
    for j in range(4):
        want = numpy_moments(yhat[out_start[j] : out_start[j] + rows[j]], y[y_start[j] : y_start[j] + rows[j]])
        np.testing.assert_allclose(got[j], want, rtol=1e-12, atol=1e-9)
    again = engine.cv_moments(jobs, 4, torch.from_numpy(yhat).to(dev), torch.from_numpy(y).to(dev), T).cpu().numpy()
    np.testing.assert_array_equal(got, again)  # fixed summation order
    assert engine.cv_moments(jobs, 0, torch.from_numpy(yhat).to(dev), torch.from_numpy(y).to(dev), T).shape == (0, 5, T)


def _series(rows, tags, seed):
    rng = np.random.default_rng(seed)
    t = np.linspace(0, 25, rows)[:, None]
    values = (0.5 + 0.4 * np.sin(t * rng.uniform(0.5, 2, tags) + rng.uniform(0, 3, tags)) + rng.normal(0, 0.02, (rows, tags))) * rng.uniform(1, 50, tags)
    idx = pd.date_range("2019-01-01", periods=rows, freq="10min", tz="UTC")
    return pd.DataFrame(values.astype(np.float32), index=idx, columns=[f"TAG {i}" for i in range(tags)])


def test_fleet_cv_scores_match_sklearn_on_the_fold_models(engine, torch):
    """The moments route gives what ModelBuilder's scorers give: metric(scaler(y_test), scaler(fold model's prediction))."""
    from gordo_components_b200 import builder, fleet
    from oracle import keras_math as km

    M, N, T, K = 3, 400, 6, 3
    spec = km.ff_hourglass_spec(T)
    eng = engine.FFEngine(spec.dims, spec.acts, spec.l1)
    frames = [_series(N, T, s) for s in range(M)]
    # DataFrame.values of a single-dtype frame is column-major: the kernels take row-major arrays (and _cabi.ptr refuses others)
    x = torch.from_numpy(np.ascontiguousarray(np.concatenate([f.values for f in frames]))).to(eng.device)
    with pytest.raises(ValueError, match="not C-contiguous"):
        engine.cv_moments(engine.jobs_to_device(engine.make_jobs([0], [4], [0]), eng.device), 1, x.t().contiguous().t(), x, T)
    fb = fleet.build_fleet(eng, x, x, rows=N, epochs=2, n_splits=K, seed=3)
    torch.cuda.synchronize()
    assert fb.cv_moments.shape == (M, K, 5, T) and fb.fold_params.shape[:2] == (M, K)
    test = N // (K + 1)
    for m in range(M):
        y = frames[m].values
        scaler = MinMaxScaler().fit(y)
        got = builder.scores_from_moments(fb.cv_moments[m].cpu().numpy(), test, fb.scale[m].cpu().numpy())
        for k in range(K):
            start = N - (K - k) * test
            jobs = engine.jobs_to_device(engine.make_jobs([0], [test], [m * N + start], [0]), eng.device)
            pred = eng.infer_score(fb.fold_params[m, k : k + 1].contiguous(), jobs, 1, test, x, out_rows=test)["model-output"].cpu().numpy()
            yt, yp = scaler.transform(y[start : start + test].astype(np.float64)), scaler.transform(pred.astype(np.float64))
            for name in builder.MOMENT_METRICS:
                func = getattr(sk_metrics, name)
                np.testing.assert_allclose(got[name][1][k], func(yt, yp), rtol=1e-5, atol=1e-7, err_msg=f"{name} fold {k}")
                np.testing.assert_allclose(got[name][0][k], func(yt, yp, multioutput="raw_values"), rtol=1e-5, atol=1e-7, err_msg=f"{name} fold {k}")


AE = {"gordo.machine.model.models.KerasAutoEncoder": {"kind": "feedforward_hourglass", "epochs": 3, "compression_factor": 0.5, "encoding_layers": 2}}
DETECTOR = {"gordo.machine.model.anomaly.diff.DiffBasedAnomalyDetector": {"base_estimator": AE}}
SCALED = {"gordo.machine.model.anomaly.diff.DiffBasedAnomalyDetector": {"base_estimator": {"sklearn.pipeline.Pipeline": {"steps": ["sklearn.preprocessing.MinMaxScaler", AE]}}}}
PIPELINE = {"gordo.machine.model.anomaly.diff.DiffBasedAnomalyDetector": {"base_estimator": {"sklearn.pipeline.Pipeline": {"steps": ["sklearn.preprocessing.StandardScaler", AE]}}}}
LSTM = {"gordo.machine.model.anomaly.diff.DiffBasedAnomalyDetector": {"base_estimator": {"gordo.machine.model.models.KerasLSTMAutoEncoder": {
    "kind": "lstm_hourglass", "lookback_window": 4, "epochs": 1, "encoding_layers": 1}}}}


def test_fleet_model_builder_end_to_end(engine, torch, tmp_path):
    from gordo_components_b200 import builder, serializer
    from gordo_components_b200.machine.model.anomaly.diff import DiffBasedAnomalyDetector

    N, T = 320, 5
    frames = {name: _series(N, T, seed) for seed, name in enumerate(["a-1", "a-2", "a-3", "pipe", "lstm", "s-1", "s-2"])}
    machines = [{"name": n, "model": DETECTOR, "dataset": {"X": frames[n], "y": frames[n]}, "metadata": {"user_defined": {"plant": "X"}}} for n in ("a-1", "a-2", "a-3")]
    machines.insert(1, {"name": "pipe", "model": PIPELINE, "dataset": (frames["pipe"], frames["pipe"])})
    machines.append({"name": "lstm", "model": LSTM, "dataset": {"X": frames["lstm"]}, "evaluation": {"metrics": ["r2_score"], "scoring_scaler": None}})
    machines += [{"name": n, "model": SCALED, "dataset": {"X": frames[n]}} for n in ("s-1", "s-2")]
    results = builder.FleetModelBuilder(machines).build(str(tmp_path))
    assert [m["name"] for _, m in results] == ["a-1", "pipe", "a-2", "a-3", "lstm", "s-1", "s-2"]

    by_name = {m["name"]: (model, m) for model, m in results}
    fleet_scores = by_name["a-2"][1]["metadata"]["build_metadata"]["model"]["cross_validation"]["scores"]
    single_scores = by_name["pipe"][1]["metadata"]["build_metadata"]["model"]["cross_validation"]["scores"]
    assert set(fleet_scores) == set(single_scores) and len(fleet_scores) == 4 * (T + 1)  # batched and per-machine paths write the same keys
    assert set(fleet_scores["r2-score-TAG-3"]) == set(single_scores["r2-score-TAG-3"]) == {"fold-mean", "fold-std", "fold-max", "fold-min", "fold-1", "fold-2", "fold-3"}
    assert set(by_name["lstm"][1]["metadata"]["build_metadata"]["model"]["cross_validation"]["scores"]) == {"r2-score"} | {f"r2-score-TAG-{i}" for i in range(T)}

    for name, (model, machine) in by_name.items():
        block = machine["metadata"]["build_metadata"]
        assert type(model) is DiffBasedAnomalyDetector
        assert set(block["model"]) == {"model_offset", "model_creation_date", "model_builder_version", "model_training_duration_sec", "cross_validation", "model_meta"}
        assert block["model"]["model_offset"] == (3 if name == "lstm" else 0)  # lookback_window - 1 (test_builder.py:99-115)
        splits = block["model"]["cross_validation"]["splits"]
        assert splits["fold-1-n-train"] == 80 and splits["fold-3-test-end"] == frames[name].index[-1]
        meta = block["model"]["model_meta"]
        assert len(meta["history"]["loss"]) == (1 if name == "lstm" else 3) and len(meta["feature-thresholds"]) == T
        assert set(meta["feature-thresholds-per-fold"]) == set(frames[name].columns)  # DataFrame.to_dict(): tag -> fold -> value
        assert set(meta["aggregate-thresholds-per-fold"]) == {"fold-0", "fold-1", "fold-2"}
        assert np.isfinite(meta["aggregate-threshold"])
        for key, val in block["model"]["cross_validation"]["scores"].items():
            assert np.isfinite(list(val.values())).all(), key
            if key.startswith("mean-"):
                assert val["fold-min"] >= 0.0
            else:
                assert val["fold-max"] <= 1.0
        # what was written is what gordo.server reads: model.pkl + metadata.json (serializer.py:149-196)
        loaded = serializer.load(os.path.join(tmp_path, name))
        on_disk = serializer.load_metadata(os.path.join(tmp_path, name))
        assert on_disk["name"] == name and on_disk["metadata"]["build_metadata"]["model"]["model_offset"] == block["model"]["model_offset"]
        json.dumps(on_disk)
        frame = loaded.anomaly(frames[name], frames[name], frequency=pd.Timedelta("10min"))
        np.testing.assert_array_equal(frame["model-output"].values, model.anomaly(frames[name], frames[name], frequency=pd.Timedelta("10min"))["model-output"].values)
        assert len(frame) == N - block["model"]["model_offset"] and "total-anomaly-confidence" in frame

    # a batched machine behind an input scaler: the Pipeline's MinMaxScaler carries sklearn's own statistics of the training
    # data, and the detector answers exactly like the Pipeline run step by step on the host in float64
    model, _ = by_name["s-2"]
    pipe = model.base_estimator
    want = MinMaxScaler().fit(frames["s-2"].values.astype(np.float64))
    np.testing.assert_allclose(pipe.steps[0][1].scale_, want.scale_, rtol=1e-14)
    np.testing.assert_allclose(pipe.steps[0][1].min_, want.min_, rtol=1e-14, atol=1e-14)
    np.testing.assert_allclose(pipe.steps[0][1].data_max_, want.data_max_, rtol=1e-12)
    scaled_x = want.transform(frames["s-2"].values.astype(np.float64)).astype(np.float32)
    direct = pipe.steps[1][1].predict(scaled_x)
    np.testing.assert_allclose(model.predict(frames["s-2"]), direct, rtol=1e-5, atol=1e-5)
    s_loss = by_name["s-1"][1]["metadata"]["build_metadata"]["model"]["model_meta"]["history"]["loss"]
    assert s_loss[-1] < s_loss[0]
    assert set(by_name["s-1"][1]["metadata"]["build_metadata"]["model"]["cross_validation"]["scores"]) == set(fleet_scores)

    # the batched machines keep their own definition and user metadata, and trained (loss falls)
    model, machine = by_name["a-3"]
    assert model.base_estimator.kind == "feedforward_hourglass" and model.base_estimator.kwargs["compression_factor"] == 0.5
    assert serializer.into_definition(model) == serializer.into_definition(serializer.from_definition(serializer.into_definition(model)))
    assert machine["metadata"]["user_defined"] == {"plant": "X"}
    loss = machine["metadata"]["build_metadata"]["model"]["model_meta"]["history"]["loss"]
    assert loss[-1] < loss[0]

    # cross_val_only stops before the final fit (build_model.py:291-306)
    only, m = builder.ModelBuilder({**machines[0], "evaluation": {"cv_mode": "cross_val_only"}}).build()
    assert set(m["metadata"]["build_metadata"]["model"]) == {"cross_validation"} and m["metadata"]["build_metadata"]["model"]["cross_validation"]["scores"]


def test_dropin_definition_on_the_gpu(engine, torch):
    """
    tests/golden/make_golden.py runs the INTEGRATION.md definition through the REFERENCE'S from_definition / ModelBuilder._build /
    serializer.dumps+loads (with the kernels mocked by the oracle) and commits the metadata key tree and the anomaly frame's columns
    it produced (tests/golden/dropin.json).  Here the same definition and data run on the
    real kernels -- per machine (`ModelBuilder`) and through the batched fleet path -- and must produce the same tree and columns.
    """
    import pickle

    from test_reference_dropin import frame, key_tree

    from gordo_components_b200 import builder

    with open(os.path.join(os.path.dirname(__file__), "golden", "dropin.json")) as f:
        want = json.load(f)
    data = frame(**want["frame"])
    machine = {"name": "dropin-machine", "model": want["definition"], "dataset": (data, data), "evaluation": want["evaluation"]}
    single = builder.ModelBuilder(dict(machine)).build()
    fleet = builder.FleetModelBuilder([dict(machine)]).build()[0]
    for model, built in (single, fleet):
        mb = dict(built["metadata"]["build_metadata"]["model"])
        for k in ("model_creation_date", "model_training_duration_sec"):
            mb.pop(k, None)
        tree = json.loads(json.dumps(key_tree(mb)))
        tree["cross_validation"].pop("cv_duration_sec", None)
        assert tree == want["model_build_metadata_keys"]
        model = pickle.loads(pickle.dumps(model))  # gordo/serializer/serializer.py:22-64 is pickle
        X = data.iloc[-40:]
        got = model.anomaly(X, X, frequency=pd.Timedelta("10min"))
        assert [list(c) for c in got.columns] == want["anomaly_columns"]
        assert np.isfinite(got["total-anomaly-confidence"].values).all() and len(got) == 40
