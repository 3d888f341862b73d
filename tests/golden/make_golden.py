"""
Regenerates the golden fixtures in this directory by running the **reference's own code**
(unmodified, from /root/reference, via oracle/reference_loader.py).  Run in the build
container only -- /root/reference does not exist on the GPU box:

    python tests/golden/make_golden.py

Fixtures written:
  hourglass_dims.json        reference hourglass_calc_dims over a grid + the reference test table
  anomaly_<case>.npz         X, y, per-fold predictions/scalers/thresholds, and every column
                             block of DiffBasedAnomalyDetector.anomaly() from the reference
  ffnet_anomaly.npz          the same, with the base estimator being a fixed-weight hourglass
                             net (oracle/keras_math.ff_forward): pins net -> anomaly end to end
  detector_sma_seed<s>.npz   a fitted DiffBasedAnomalyDetector (LinearRegression base, SMA
                             smoothing): its predictions, thresholds and anomaly frame
  dropin.{json,npz}          the INTEGRATION.md definition driven through the reference's
                             from_definition / into_definition / ModelBuilder._build /
                             serializer, with this package's estimators on the CPU oracle
"""
from __future__ import annotations

import json
import os
import sys
import warnings

import numpy as np
import pandas as pd

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))

from oracle import keras_math as km  # noqa: E402
from oracle.reference_loader import load_reference  # noqa: E402

warnings.filterwarnings("ignore")
ref = load_reference()

from sklearn.base import BaseEstimator  # noqa: E402
from sklearn.linear_model import LinearRegression  # noqa: E402
from sklearn.model_selection import TimeSeriesSplit  # noqa: E402
from sklearn.multioutput import MultiOutputRegressor  # noqa: E402
from sklearn.preprocessing import MinMaxScaler  # noqa: E402


class FixedNet(BaseEstimator):
    """sklearn-style estimator around a fixed-weight oracle Dense stack (fit is a no-op)."""

    def __init__(self, n_features=8, seed=0):
        self.n_features = n_features
        self.seed = seed

    def _net(self):
        spec = km.ff_hourglass_spec(self.n_features)
        w = km.init_ff_weights(spec, np.random.default_rng(self.seed))
        # non-zero biases so the bias path is pinned too
        rng = np.random.default_rng(self.seed + 1)
        w = [(W, rng.uniform(-0.1, 0.1, size=b.shape).astype(np.float32)) for W, b in w]
        return spec, w

    def fit(self, X, y=None):
        return self

    def predict(self, X):
        spec, w = self._net()
        return km.ff_predict(spec, w, np.asarray(getattr(X, "values", X)))

    def score(self, X, y, sample_weight=None):
        return 0.0


def dims_fixture():
    table = []
    for cf in (0.0, 0.1, 0.2, 0.3, 0.5, 0.6, 0.75, 1.0):
        for layers in (1, 2, 3, 4, 5):
            for n in (1, 3, 4, 5, 8, 10, 64, 100, 128, 1000):
                table.append([cf, layers, n, list(ref.hourglass_calc_dims(cf, layers, n))])
    ref_test_table = [  # tests/gordo/machine/model/test_factories_utils.py:8-24
        [0.2, 4, 5, [4, 3, 2, 1]],
        [0.5, 3, 10, [8, 7, 5]],
        [0.5, 3, 3, [3, 2, 2]],
        [0.3, 3, 10, [8, 5, 3]],
        [1, 3, 10, [10, 10, 10]],
        [0, 3, 100000, [66667, 33334, 1]],
    ]
    for cf, layers, n, want in ref_test_table:
        assert list(ref.hourglass_calc_dims(cf, layers, n)) == want
    with open(os.path.join(HERE, "hourglass_dims.json"), "w") as f:
        json.dump({"grid": table, "reference_test_table": ref_test_table}, f)


def anomaly_fixture(name, n_rows, n_tags, window, method, datetime_index, base="linear", seed=0):
    rng = np.random.default_rng(seed)
    cols = [f"tag-{i}" for i in range(n_tags)]
    index = pd.date_range("2019-01-01", periods=n_rows, freq="10min", tz="UTC") if datetime_index else pd.RangeIndex(n_rows)
    X = pd.DataFrame(rng.random((n_rows, n_tags)), columns=cols, index=index)
    if base == "linear":
        y = pd.DataFrame(rng.random((n_rows, n_tags)) * np.arange(1, n_tags + 1), columns=cols, index=index)
        est = MultiOutputRegressor(LinearRegression())
    else:
        y = X.copy()
        est = FixedNet(n_features=n_tags, seed=seed)
    det = ref.DiffBasedAnomalyDetector(base_estimator=est, scaler=MinMaxScaler(), window=window, smoothing_method=method)
    cv = TimeSeriesSplit(n_splits=3)
    cvo = det.cross_validate(X=X, y=y, cv=cv)
    save = dict(X=X.values, y=y.values, n_splits=3, window=-1 if window is None else window, method=str(method),
                datetime_index=bool(datetime_index))
    for i, ((tr, te), fold) in enumerate(zip(cv.split(X, y), cvo["estimator"])):
        save[f"fold{i}_pred"] = np.asarray(fold.predict(X.iloc[te]))
        save[f"fold{i}_scale"] = fold.scaler.scale_
        save[f"fold{i}_min"] = fold.scaler.min_
        save[f"fold{i}_test_start"] = te[0]
        save[f"fold{i}_test_len"] = len(te)
    save["feature_thresholds_per_fold"] = det.feature_thresholds_per_fold_.values.astype(np.float64)
    save["aggregate_thresholds_per_fold"] = np.array([det.aggregate_thresholds_per_fold_[f"fold-{i}"] for i in range(3)])
    save["feature_thresholds"] = det.feature_thresholds_.values.astype(np.float64)
    save["aggregate_threshold"] = np.float64(det.aggregate_threshold_)
    if window is not None:
        save["smooth_feature_thresholds"] = det.smooth_feature_thresholds_.values.astype(np.float64)
        save["smooth_aggregate_threshold"] = np.float64(det.smooth_aggregate_threshold_)
    det.fit(X, y)
    save["scale"], save["min"] = det.scaler.scale_, det.scaler.min_
    save["pred"] = np.asarray(det.predict(X))
    frame = det.anomaly(X, y, frequency=pd.Timedelta("10min") if datetime_index else None)
    save["columns_level0"] = np.array(list(dict.fromkeys(frame.columns.get_level_values(0))))
    save["columns"] = np.array(["|".join(map(str, c)) for c in frame.columns])
    for top in dict.fromkeys(frame.columns.get_level_values(0)):
        block = frame[top]
        if top in ("start", "end"):
            save[f"frame_{top}"] = np.array([str(v) for v in np.asarray(block).ravel()])
        else:
            save[f"frame_{top}"] = np.asarray(block, dtype=np.float64)
    if base != "linear":
        spec, w = est._net()
        save["net_dims"] = np.array(spec.dims)
        for l, (W, b) in enumerate(w):
            save[f"W{l}"], save[f"b{l}"] = W, b
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), **save)
    print(name, "ok", frame.shape)


def kfcv_fixture(name, n_rows, n_tags, window, method, q, seed):
    """DiffBasedKFCVAnomalyDetector (diff.py:461-635) from the reference itself, LinearRegression base estimator."""
    rng = np.random.default_rng(seed)
    cols = [f"tag-{i}" for i in range(n_tags)]
    index = pd.date_range("2019-01-01", periods=n_rows, freq="10min", tz="UTC")
    X = pd.DataFrame(rng.random((n_rows, n_tags)), columns=cols, index=index)
    y = pd.DataFrame(rng.random((n_rows, n_tags)) * np.arange(1, n_tags + 1), columns=cols, index=index)
    det = ref.DiffBasedKFCVAnomalyDetector(base_estimator=MultiOutputRegressor(LinearRegression()), scaler=MinMaxScaler(), window=window,
                                           smoothing_method=method, threshold_percentile=q)
    det.cross_validate(X=X, y=y)
    det.fit(X, y)
    frame = det.anomaly(X, y, frequency=pd.Timedelta("10min"))
    save = dict(X=X.values, y=y.values, window=window, method=str(method), q=q, feature_thresholds=np.asarray(det.feature_thresholds_, dtype=np.float64),
                aggregate_threshold=np.float64(det.aggregate_threshold_), columns_level0=np.array(list(dict.fromkeys(frame.columns.get_level_values(0)))))
    for top in ("total-anomaly-confidence", "anomaly-confidence", "smooth-total-anomaly-scaled", "smooth-tag-anomaly-unscaled"):
        save[f"frame_{top}"] = np.asarray(frame[top], dtype=np.float64)
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), **save)
    print(name, "ok", frame.shape)


# ------------------------------------------------------------------------------------------------ the path's callers
# definitions whose class paths exist here (sklearn / numpy only): the reference expands them with its own serializer
CALLER_DEFINITIONS = [
    "sklearn.preprocessing.MinMaxScaler",
    {"sklearn.preprocessing.MinMaxScaler": {"feature_range": [-1, 1]}},
    {"sklearn.pipeline.Pipeline": {"steps": ["sklearn.preprocessing.MinMaxScaler", {"sklearn.decomposition.PCA": {"n_components": 2}}]}},
    {"sklearn.pipeline.Pipeline": ["sklearn.preprocessing.StandardScaler", {"sklearn.linear_model.Ridge": {"alpha": 0.5}}]},
    {"sklearn.pipeline.Pipeline": {"steps": [
        {"sklearn.preprocessing.FunctionTransformer": {"func": "numpy.log1p", "inverse_func": "numpy.expm1"}},
        {"sklearn.pipeline.FeatureUnion": {"transformer_list": [
            {"sklearn.decomposition.PCA": {"n_components": 3}},
            {"sklearn.pipeline.Pipeline": ["sklearn.preprocessing.MinMaxScaler", {"sklearn.decomposition.TruncatedSVD": {"n_components": 2}}]}]}},
        "sklearn.linear_model.LinearRegression"]}},
    {"sklearn.multioutput.MultiOutputRegressor": {"estimator": "sklearn.tree.DecisionTreeRegressor"}},
    {"sklearn.multioutput.MultiOutputRegressor": {"estimator": {"sklearn.tree.DecisionTreeRegressor": {"max_depth": 3}}}},
    {"sklearn.compose.TransformedTargetRegressor": {"transformer": "sklearn.preprocessing.MinMaxScaler", "regressor": {
        "sklearn.pipeline.Pipeline": {"steps": ["sklearn.preprocessing.RobustScaler", {"sklearn.linear_model.Ridge": {"alpha": 2.0}}]}}}},
    {"sklearn.pipeline.Pipeline": {"steps": [{"sklearn.cluster.FeatureAgglomeration": {"n_clusters": 2, "pooling_func": "numpy.median"}},
                                             "sklearn.linear_model.LinearRegression"], "memory": None, "verbose": True}},
]

BUILD_MODEL = {"sklearn.pipeline.Pipeline": {"steps": ["sklearn.preprocessing.MinMaxScaler", {"sklearn.linear_model.Ridge": {"alpha": 0.1}}]}}
BUILD_EVALUATIONS = {
    "default": {"cv_mode": "full_build", "scoring_scaler": "sklearn.preprocessing.MinMaxScaler",
                "metrics": ["explained_variance_score", "r2_score", "mean_squared_error", "mean_absolute_error"]},
    "five_folds_unscaled": {"cv_mode": "full_build", "scoring_scaler": None, "metrics": ["sklearn.metrics.r2_score", "max_error" if False else "mean_absolute_error"],
                            "cv": {"sklearn.model_selection.TimeSeriesSplit": {"n_splits": 5}}, "seed": 3},
    "cv_only": {"cv_mode": "cross_val_only", "scoring_scaler": "sklearn.preprocessing.RobustScaler", "metrics": ["mean_squared_error"]},
}


def _jsonable(obj):
    if isinstance(obj, dict):
        return {str(k): _jsonable(v) for k, v in obj.items()}
    if isinstance(obj, (list, tuple)):
        return [_jsonable(v) for v in obj]
    if isinstance(obj, (np.floating, np.integer)):
        return obj.item()
    if isinstance(obj, (pd.Timestamp,)):
        return str(obj)
    if hasattr(obj, "to_dict") and not isinstance(obj, (pd.DataFrame, pd.Series)):
        return _jsonable(obj.to_dict())
    return obj


def build_frame(rows=240, tags=4, seed=11):
    rng = np.random.default_rng(seed)
    t = np.linspace(0, 20, rows)[:, None]
    values = (0.5 + 0.4 * np.sin(t * rng.uniform(0.5, 2, tags) + rng.uniform(0, 3, tags)) + rng.normal(0, 0.05, (rows, tags))) * rng.uniform(1, 40, tags) + rng.uniform(-5, 100, tags)
    values[:, -1] = 3.25  # a constant tag: the zero-variance conventions of the ratio metrics
    idx = pd.date_range("2020-03-01", periods=rows, freq="10min", tz="UTC")
    return pd.DataFrame(values, index=idx, columns=[f"TAG {i}" for i in range(tags)])


def callers_fixture():
    """Golden outputs of the reference's serializer, builder, server wire formats and InfImputer (tests/golden/callers.json + callers.npz)."""
    from oracle.reference_loader import load_reference_callers

    rc = load_reference_callers()
    out, arrays = {}, {}

    # ---- serializer: into_definition(from_definition(d)), the expansion `gordo build` applies before hashing (cli.py:142-144)
    out["expansions"] = [{"definition": d, "expanded": _jsonable(rc.into_definition(rc.from_definition(d)))} for d in CALLER_DEFINITIONS]

    # ---- builder: ModelBuilder._build (build_model.py:192-339) on stand-in Machine objects
    frame = build_frame()
    out["build"] = {}
    for name, evaluation in BUILD_EVALUATIONS.items():
        class Dataset:
            def get_data(self):
                return frame, frame

            def get_metadata(self):
                return {"rows": len(frame)}

        rc.GordoBaseDataset.registry["fixture"] = Dataset()
        machine = rc.Record(name="fixture-machine", project_name="p", model=BUILD_MODEL, evaluation=dict(evaluation), runtime={},
                            dataset=rc.Record(key="fixture"), metadata=rc.Record(user_defined={"k": 1}))
        builder = rc.ModelBuilder.__new__(rc.ModelBuilder)
        builder.machine, builder.back_compatibles, builder.default_data_provider = machine, None, None
        model, built = builder._build()
        block = _jsonable(built.metadata.build_metadata)
        for k in ("model_creation_date", "model_training_duration_sec"):
            block["model"].pop(k, None)
        block["model"]["cross_validation"].pop("cv_duration_sec", None)
        block["dataset"].pop("query_duration_sec", None)
        out["build"][name] = {"evaluation": evaluation, "build_metadata": block}
        if evaluation["cv_mode"] == "full_build":
            arrays[f"build_{name}_prediction"] = np.asarray(model.predict(frame), dtype=np.float64)
    # the same build with the model wrapped in the reference's DiffBasedAnomalyDetector: thresholds land in model_meta
    detector_model = {"gordo.machine.model.anomaly.diff.DiffBasedAnomalyDetector": {"base_estimator": BUILD_MODEL}}
    machine = rc.Record(name="fixture-detector", project_name="p", model=detector_model, evaluation=dict(BUILD_EVALUATIONS["default"]), runtime={},
                        dataset=rc.Record(key="fixture"), metadata=rc.Record(user_defined={}))
    builder = rc.ModelBuilder.__new__(rc.ModelBuilder)
    builder.machine, builder.back_compatibles, builder.default_data_provider = machine, None, None
    model, built = builder._build()
    block = _jsonable(built.metadata.build_metadata)
    out["build_detector"] = {"model": detector_model, "scores": block["model"]["cross_validation"]["scores"], "model_offset": block["model"]["model_offset"],
                             "model_meta": _jsonable(block["model"]["model_meta"])}
    anomaly = model.anomaly(frame.iloc[-50:], frame.iloc[-50:], frequency=pd.Timedelta("10min"))
    arrays["build_detector_total_confidence"] = np.asarray(anomaly["total-anomaly-confidence"], dtype=np.float64).ravel()
    arrays["build_detector_tag_scaled"] = np.asarray(anomaly["tag-anomaly-scaled"], dtype=np.float64)
    arrays["build_frame"] = frame.values
    out["build_model"] = BUILD_MODEL
    out["default_evaluation"] = rc.default_evaluation
    out["build_frame"] = {"rows": len(frame), "columns": list(frame.columns), "start": str(frame.index[0]), "freq": "10min", "seed": 11}

    # ---- server wire formats (gordo/server/utils.py:47-247)
    idx = pd.date_range("2016-01-01", periods=4, freq="10min", tz="UTC")
    cols = pd.MultiIndex.from_tuples([("start", ""), ("model-output", "tag 0"), ("model-output", "tag 1"), ("total-anomaly-scaled", "")])
    multi = pd.DataFrame(np.arange(16.0).reshape(4, 4) / 7.0, columns=cols, index=idx)
    multi[("start", "")] = [t.isoformat() for t in idx]
    plain = pd.DataFrame(np.arange(8.0).reshape(4, 2) / 3.0, columns=["a", "b"], index=idx)
    numbered = pd.DataFrame({"a": [1.5, 2.5, 3.5]}, index=[2, 0, 1])
    out["wire"] = {"multi": rc.dataframe_to_dict(multi), "plain": rc.dataframe_to_dict(plain), "numbered": _jsonable(rc.dataframe_to_dict(numbered))}
    back = rc.dataframe_from_dict(json.loads(json.dumps(out["wire"]["multi"])))
    out["wire"]["multi_back"] = {"columns": [list(c) for c in back.columns], "index": [str(t) for t in back.index],
                                 "model_output": back["model-output"].values.tolist()}
    nb = rc.dataframe_from_dict(json.loads(json.dumps(out["wire"]["numbered"])))
    out["wire"]["numbered_back"] = {"index": [int(i) for i in nb.index], "a": nb["a"].tolist()}
    expected = ["tag-0", "tag-1", "tag-2"]
    verify = {}
    for case, df in (("unlabelled", pd.DataFrame(np.zeros((2, 3)))), ("shuffled_superset", pd.DataFrame(np.zeros((2, 4)), columns=["tag-2", "x", "tag-0", "tag-1"])),
                     ("too_wide", pd.DataFrame(np.zeros((2, 4)))), ("multi_level", multi)):
        res = rc.verify_dataframe(df, expected)
        verify[case] = {"columns": [str(c) for c in res.columns]} if isinstance(res, pd.DataFrame) else {"status": res[-1], "message": res[0]["message"]}
    out["wire"]["verify"] = verify

    # ---- InfImputer (gordo/machine/model/transformers/imputer.py:12-127)
    rng = np.random.default_rng(5)
    for dtype in ("float32", "float64"):
        base = rng.random((50, 6)).astype(dtype) * 10 - 3
        flat = base.ravel()
        flat[rng.integers(0, flat.size, 30)] = np.inf
        flat[rng.integers(0, flat.size, 30)] = -np.inf
        arrays[f"imputer_{dtype}_input"] = base.copy()
        arrays[f"imputer_{dtype}_minmax"] = rc.InfImputer(strategy="minmax", delta=2.0).fit_transform(base.copy())
        arrays[f"imputer_{dtype}_extremes"] = rc.InfImputer(strategy="extremes").fit_transform(base.copy())
        arrays[f"imputer_{dtype}_filled"] = rc.InfImputer(inf_fill_value=99.0, neg_inf_fill_value=-99.0, strategy=None).fit_transform(base.copy())
        arrays[f"imputer_{dtype}_half"] = rc.InfImputer(inf_fill_value=99.0, delta=0.5).fit_transform(base.copy())

    with open(os.path.join(HERE, "callers.json"), "w") as f:
        json.dump(out, f, indent=1, default=str)
    np.savez_compressed(os.path.join(HERE, "callers.npz"), **arrays)
    print("callers ok:", len(out["expansions"]), "expansions;", {k: len(v["build_metadata"]["model"]["cross_validation"]["scores"]) for k, v in out["build"].items()})


def detector_fixture(seed):
    """The reference's DiffBasedAnomalyDetector cross-validated and fitted on random frames (tests/test_oracle_golden.py)."""
    rng = np.random.default_rng(seed)
    X = pd.DataFrame(rng.random((240, 5)))
    y = pd.DataFrame(rng.random((240, 5)) * 3.0)
    det = ref.DiffBasedAnomalyDetector(base_estimator=MultiOutputRegressor(LinearRegression()), scaler=MinMaxScaler(), window=10, smoothing_method="sma")
    det.cross_validate(X=X, y=y)
    det.fit(X, y)
    frame = det.anomaly(X, y)
    save = dict(X=X.values, y=y.values, window=10, method="sma", pred=np.asarray(det.predict(X), dtype=np.float64),
                feature_thresholds=det.feature_thresholds_.values.astype(np.float64), aggregate_threshold=np.float64(det.aggregate_threshold_),
                hourglass_dims_0p5_3_64=np.array(ref.hourglass_calc_dims(0.5, 3, 64)))
    for top in dict.fromkeys(frame.columns.get_level_values(0)):
        if top not in ("start", "end"):
            save[f"frame_{top}"] = np.asarray(frame[top], dtype=np.float64)
    np.savez_compressed(os.path.join(HERE, f"detector_sma_seed{seed}.npz"), **save)
    print(f"detector_sma_seed{seed} ok", frame.shape)


def dropin_fixture():
    """
    The drop-in definition of tests/test_reference_dropin.py through the reference's own callers: its definition expansion, the
    build metadata of ModelBuilder._build (this package's estimators computing with the CPU oracle of tests/cpu_engine.py) and the
    anomaly frame of the model after the reference serializer's dumps/loads.
    """
    sys.path.insert(0, os.path.dirname(HERE))
    from cpu_engine import patched_engine
    from test_reference_dropin import DEFINITION, EVALUATION, frame, key_tree

    from gordo_components_b200.machine.model import base as b200_base
    from gordo_components_b200.machine.model.anomaly import base as b200_abase
    from oracle.reference_loader import load_reference_callers

    rc = load_reference_callers()
    # gordo only exists once the loader has executed it, so the import-time registration of machine/model/base.py is repeated here
    assert b200_base.register_with_gordo("gordo.machine.model.base", "GordoBase", b200_base.GordoBase)
    assert b200_base.register_with_gordo("gordo.machine.model.anomaly.base", "AnomalyDetectorBase", b200_abase.AnomalyDetectorBase)
    data = frame()
    expanded = rc.into_definition(rc.from_definition(DEFINITION))

    class Dataset:
        def get_data(self):
            return data, data

        def get_metadata(self):
            return {"rows": len(data)}

    rc.GordoBaseDataset.registry["dropin"] = Dataset()
    machine = rc.Record(name="dropin-machine", project_name="p", model=DEFINITION, evaluation=dict(EVALUATION), runtime={},
                        dataset=rc.Record(key="dropin"), metadata=rc.Record(user_defined={}))
    builder = rc.ModelBuilder.__new__(rc.ModelBuilder)
    builder.machine, builder.back_compatibles, builder.default_data_provider = machine, None, None
    with patched_engine():
        model, built = builder._build()
        loaded = rc.serializer.loads(rc.serializer.dumps(model))
        X = data.iloc[-40:]
        anomaly = loaded.anomaly(X, X, frequency=pd.Timedelta("10min"))
    mb = built.metadata.build_metadata.to_dict()["model"]
    tree = key_tree({k: v for k, v in mb.items() if k not in ("model_creation_date", "model_training_duration_sec")})
    tree["cross_validation"].pop("cv_duration_sec", None)
    fixture = {"definition": DEFINITION, "evaluation": EVALUATION, "frame": {"rows": 160, "tags": 4, "seed": 5},
               "model_build_metadata_keys": tree, "anomaly_columns": [list(c) for c in anomaly.columns],
               "expanded": _jsonable(expanded), "model_offset": mb["model_offset"], "model_meta": _jsonable(mb["model_meta"]),
               "scores": _jsonable(mb["cross_validation"]["scores"]), "splits": _jsonable(mb["cross_validation"]["splits"])}
    with open(os.path.join(HERE, "dropin.json"), "w") as f:
        json.dump(fixture, f, indent=1, sort_keys=True)
    arrays = {f"frame_{top}": np.asarray(anomaly[top], dtype=np.float64)
              for top in dict.fromkeys(anomaly.columns.get_level_values(0)) if top not in ("start", "end")}
    np.savez_compressed(os.path.join(HERE, "dropin.npz"), **arrays)
    print("dropin ok", anomaly.shape)


if __name__ == "__main__":
    dims_fixture()
    kfcv_fixture("kfcv_smm", 300, 3, 12, "smm", 0.99, seed=6)
    kfcv_fixture("kfcv_ewma", 400, 4, 24, "ewma", 0.9, seed=7)
    anomaly_fixture("anomaly_plain", 300, 3, None, None, False)
    anomaly_fixture("anomaly_smm", 300, 3, 12, "smm", True, seed=1)
    anomaly_fixture("anomaly_sma", 200, 4, 12, "sma", True, seed=2)
    anomaly_fixture("anomaly_ewma", 200, 4, 12, "ewma", False, seed=3)
    anomaly_fixture("ffnet_anomaly", 400, 8, None, None, True, base="net", seed=4)
    anomaly_fixture("ffnet_anomaly_t64", 200, 64, None, None, True, base="net", seed=5)
    callers_fixture()
    for s in (11, 12):
        detector_fixture(s)
    dropin_fixture()
