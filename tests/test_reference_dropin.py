"""
The drop-in boundary, driven the way gordo's own callers drive it (SURVEY section 8b): the model definition of INTEGRATION.md -- class
paths under ``gordo_components_b200`` -- goes through

    gordo/serializer/from_definition.py:23-66, 176-191   from_definition / into_definition
    gordo/builder/build_model.py:192-339 ``ModelBuilder._build``  (seeds, cross validation with gordo's scorers, final fit, offset,
                                                                   ``_extract_metadata_from_model``)
    gordo/serializer/serializer.py:22-64 ``dumps`` / ``loads``    (pickle)

and the unpickled object answers ``.predict`` / ``.anomaly`` as the server's views call it (gordo/server/blueprints/anomaly.py:50).
tests/golden/make_golden.py ran that chain with the reference's own code and committed what it produced (tests/golden/dropin.json,
dropin.npz): the definition expansion, the build metadata and the anomaly frame.  Here this package's serializer and builder, which
restate those callers, run the same definition on the same data and must reproduce it; gordo's base classes and its builder are
stood in for by minimal modules, so what is under test is the protocol -- every attribute, hook, exception type and metadata key
gordo's callers rely on.  The kernels behind the classes are replaced by the CPU oracle (tests/cpu_engine.py: test infrastructure,
the product has no CPU path), as they were when the fixture was made; the same definition is held to the key tree on a B200 with the
real kernels (tests/test_gpu_builder.py::test_dropin_definition_on_the_gpu).
"""
import abc
import json
import os
import sys
import types

import numpy as np
import pandas as pd
import pytest

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")

# INTEGRATION.md section 1, "after" (epochs shortened; examples/config.yaml:74-81 with the package prefix swapped)
DEFINITION = {
    "gordo_components_b200.machine.model.anomaly.diff.DiffBasedAnomalyDetector": {
        "base_estimator": {
            "sklearn.pipeline.Pipeline": {
                "steps": [
                    "sklearn.preprocessing.MinMaxScaler",
                    {"gordo_components_b200.machine.model.models.KerasAutoEncoder": {"kind": "feedforward_hourglass", "epochs": 3, "batch_size": 16}},
                ]
            }
        }
    }
}
EVALUATION = {"cv_mode": "full_build", "scoring_scaler": "sklearn.preprocessing.MinMaxScaler",
              "metrics": ["explained_variance_score", "r2_score", "mean_squared_error", "mean_absolute_error"]}


def frame(rows=160, tags=4, seed=5):
    rng = np.random.default_rng(seed)
    t = np.linspace(0, 12, rows)[:, None]
    values = (0.5 + 0.4 * np.sin(t * rng.uniform(0.5, 2, tags) + rng.uniform(0, 3, tags)) + rng.normal(0, 0.03, (rows, tags))) * rng.uniform(1, 30, tags)
    return pd.DataFrame(values, index=pd.date_range("2020-03-01", periods=rows, freq="10min", tz="UTC"), columns=[f"TAG {i}" for i in range(tags)])


def key_tree(obj):
    """Nested keys with leaf *types* -- what a consumer of metadata.json can rely on."""
    if isinstance(obj, dict):
        return {str(k): key_tree(v) for k, v in sorted(obj.items(), key=lambda kv: str(kv[0]))}
    if isinstance(obj, (list, tuple)):
        return [f"list[{len(obj)}]", key_tree(obj[0]) if obj else None]
    if isinstance(obj, (bool, np.bool_)):
        return "bool"
    if isinstance(obj, (int, np.integer)):
        return "int"
    if isinstance(obj, (float, np.floating)):
        return "float"
    return type(obj).__name__




@pytest.fixture(scope="module")
def golden():
    with open(os.path.join(GOLDEN, "dropin.json")) as f:
        return json.load(f), np.load(os.path.join(GOLDEN, "dropin.npz"))


def assert_same_values(got, want, rtol, atol, where="model"):
    """`want` is JSON as the reference's run wrote it (keys sorted): same keys, numbers within tolerance, anything else equal."""
    if isinstance(want, dict):
        got = {str(k): v for k, v in got.items()}
        assert sorted(got) == sorted(want), where
        for k, w in want.items():
            assert_same_values(got[k], w, rtol, atol, f"{where}/{k}")
    elif isinstance(want, list):
        assert len(got) == len(want), where
        for i, (v, w) in enumerate(zip(got, want)):
            assert_same_values(v, w, rtol, atol, f"{where}[{i}]")
    elif isinstance(want, (int, float)) and not isinstance(want, bool):
        np.testing.assert_allclose(got, want, rtol=rtol, atol=atol, err_msg=where)
    else:
        assert got == want or str(got) == want, where


def _stand_in(monkeypatch, name, **attrs):
    mod = types.ModuleType(name)
    mod.__dict__.update(attrs)
    monkeypatch.setitem(sys.modules, name, mod)
    return mod


def test_model_builder_class_hook(monkeypatch):
    """MODEL_BUILDER_CLASS (gordo/builder/utils.py:8-17 imports the class path and requires a subclass of gordo's ModelBuilder): the
    class path resolves to a subclass of gordo's builder that inherits its build logic and seeds NumPy."""
    from gordo_components_b200 import builder, gordo_hooks, serializer

    class ModelBuilder:  # gordo.builder.build_model.ModelBuilder: only its identity and inherited methods matter here
        def _build(self):
            return "gordo's _build"

        def set_seed(self, seed):
            raise AssertionError("gordo's set_seed seeds TensorFlow, which the hook replaces")

    _stand_in(monkeypatch, "gordo.builder.build_model", ModelBuilder=ModelBuilder)
    monkeypatch.setattr(gordo_hooks, "_cache", {})
    cls = serializer.locate("gordo_components_b200.gordo_hooks.B200ModelBuilder")
    assert issubclass(cls, ModelBuilder) and cls is not ModelBuilder and cls._build is ModelBuilder._build
    builder_ = cls.__new__(cls)
    builder_.set_seed(3)
    a = np.random.random()
    builder_.set_seed(3)
    assert np.random.random() == a
    assert not issubclass(builder.ModelBuilder, ModelBuilder)  # the stand-alone builder is not a gordo subclass: gordo raises ValueError


def test_reference_callers_drive_these_classes(golden, monkeypatch):
    want, arrays = golden
    # gordo's callers test isinstance(obj, gordo.machine.model.base.GordoBase) (build_model.py:552-553, 566): where gordo is installed
    # this package's protocol classes register with its ABCs
    from gordo_components_b200 import builder, serializer
    from gordo_components_b200.machine.model import base as b200_base
    from gordo_components_b200.machine.model.anomaly import base as b200_abase
    from gordo_components_b200.machine.model.anomaly.diff import DiffBasedAnomalyDetector
    from gordo_components_b200.machine.model.models import KerasAutoEncoder

    class GordoBase(abc.ABC):
        pass

    class AnomalyDetectorBase(GordoBase):
        pass

    _stand_in(monkeypatch, "gordo.machine.model.base", GordoBase=GordoBase)
    _stand_in(monkeypatch, "gordo.machine.model.anomaly.base", AnomalyDetectorBase=AnomalyDetectorBase)
    assert b200_base.register_with_gordo("gordo.machine.model.base", "GordoBase", b200_base.GordoBase)
    assert b200_base.register_with_gordo("gordo.machine.model.anomaly.base", "AnomalyDetectorBase", b200_abase.AnomalyDetectorBase)

    from cpu_engine import patched_engine

    # ---- from_definition builds THIS package's classes through their hooks
    model = serializer.from_definition(DEFINITION)
    assert type(model) is DiffBasedAnomalyDetector and isinstance(model, AnomalyDetectorBase)
    ae = model.base_estimator.steps[-1][1]
    assert type(ae) is KerasAutoEncoder and isinstance(ae, GordoBase)
    assert ae.kind == "feedforward_hourglass" and ae.kwargs == {"epochs": 3, "batch_size": 16}
    # ... and into_definition expands it as the reference's did (what `gordo build` hashes, cli.py:142-144)
    expanded = serializer.into_definition(model)
    assert json.loads(json.dumps(expanded)) == want["expanded"]
    top = "gordo_components_b200.machine.model.anomaly.diff.DiffBasedAnomalyDetector"
    steps = expanded[top]["base_estimator"]["sklearn.pipeline.Pipeline"]["steps"]
    assert steps[1] == {"gordo_components_b200.machine.model.models.KerasAutoEncoder": {"kind": "feedforward_hourglass", "epochs": 3, "batch_size": 16}}
    assert type(serializer.from_definition(expanded)) is DiffBasedAnomalyDetector  # the expansion is itself a definition

    data = frame(**want["frame"])
    with patched_engine():
        # ---- ModelBuilder._build: cross_validate with gordo's scorers, fit, offset, metadata extraction
        machine = {"name": "dropin-machine", "model": DEFINITION, "dataset": (data, data), "evaluation": EVALUATION}
        built_model, built = builder.ModelBuilder(machine).build()
        mb = built["metadata"]["build_metadata"]["model"]
        assert mb["model_offset"] == want["model_offset"] == 0
        meta = mb["model_meta"]
        # the detector's and the network's get_metadata() were both collected
        assert {"feature-thresholds", "aggregate-threshold", "feature-thresholds-per-fold", "aggregate-thresholds-per-fold", "history"} <= set(meta)
        assert set(meta["history"]) == {"loss", "accuracy", "params"} and len(meta["history"]["loss"]) == 3
        assert meta["history"]["params"] == {"verbose": 0, "epochs": 3, "steps": 10}
        assert len(meta["feature-thresholds"]) == 4 and np.isfinite(meta["feature-thresholds"]).all() and meta["aggregate-threshold"] > 0
        assert_same_values(meta, want["model_meta"], rtol=1e-6, atol=0.0)
        scores = mb["cross_validation"]["scores"]
        assert "r2-score-TAG-1" in scores and set(scores["mean-squared-error"]) == {"fold-mean", "fold-std", "fold-max", "fold-min", "fold-1", "fold-2", "fold-3"}
        assert np.isfinite([v for s in scores.values() for v in s.values()]).all()
        assert_same_values(scores, want["scores"], rtol=1e-5, atol=1e-7)
        assert {k: str(v) for k, v in mb["cross_validation"]["splits"].items()} == {k: str(v) for k, v in want["splits"].items()}
        assert mb["cross_validation"]["splits"]["fold-3-n-train"] == 120

        # ---- serializer.dumps / loads (pickle), then the calls the server views make
        blob = serializer.dumps(built_model)
        loaded = serializer.loads(blob)
        assert type(loaded) is DiffBasedAnomalyDetector
        X = data.iloc[-40:]
        np.testing.assert_array_equal(loaded.predict(X), built_model.predict(X))
        got = loaded.anomaly(X, X, frequency=pd.Timedelta("10min"))
        pd.testing.assert_frame_equal(got, built_model.anomaly(X, X, frequency=pd.Timedelta("10min")))
        assert list(dict.fromkeys(got.columns.get_level_values(0))) == [
            "start", "end", "model-input", "model-output", "tag-anomaly-scaled", "total-anomaly-scaled", "tag-anomaly-unscaled",
            "total-anomaly-unscaled", "anomaly-confidence", "total-anomaly-confidence"]
        for name in arrays.files:
            np.testing.assert_allclose(np.asarray(got[name[len("frame_"):]], dtype=np.float64), arrays[name], rtol=1e-5, atol=1e-7, err_msg=name)
        np.testing.assert_allclose(got["anomaly-confidence"].values, got["tag-anomaly-unscaled"].values / np.asarray(meta["feature-thresholds"]), rtol=1e-5)
        # the server maps these exceptions to HTTP codes (blueprints/anomaly.py:49-55 -> 422, base.py:75-81 -> 400)
        fresh = serializer.from_definition(DEFINITION)
        fresh.fit(data, data)
        with pytest.raises(AttributeError):
            fresh.anomaly(X, X)
        with pytest.raises(ValueError):
            loaded.predict(X[list(X.columns[:2])])

    tree = key_tree({k: v for k, v in mb.items() if k not in ("model_creation_date", "model_training_duration_sec")})
    tree["cross_validation"].pop("cv_duration_sec", None)
    assert json.loads(json.dumps(tree)) == want["model_build_metadata_keys"]
    assert [list(c) for c in got.columns] == want["anomaly_columns"]
