"""
Pins the CPU oracle (oracle/) against (1) fixtures produced by the reference's own code
(tests/golden/make_golden.py), (2) the golden tables/batches the reference's tests hold.
"""
import glob
import json
import os

import numpy as np
import pandas as pd
import pytest

from oracle import anomaly_math as am
from oracle import keras_math as km

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
ANOMALY_CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*anomaly*.npz")))


def test_hourglass_dims_table():
    with open(os.path.join(GOLDEN, "hourglass_dims.json")) as f:
        tab = json.load(f)
    for cf, layers, n, want in tab["reference_test_table"] + tab["grid"]:
        assert list(km.hourglass_calc_dims(cf, layers, n)) == want, (cf, layers, n)


def test_hourglass_dims_errors():
    # reference tests/gordo/machine/model/test_feedforward_autoencoder.py:182-196
    with pytest.raises(ValueError):
        km.hourglass_calc_dims(1.5, 3, 10)
    with pytest.raises(ValueError):
        km.hourglass_calc_dims(-0.1, 3, 10)
    with pytest.raises(ValueError):
        km.hourglass_calc_dims(0.5, 0, 10)


def test_factory_docstring_pins():
    # feedforward_autoencoder.py:225-238 / lstm_autoencoder.py:235-248 doctests
    assert km.ff_hourglass_spec(10).dims[1:] == [8, 7, 5, 5, 7, 8, 10]
    assert km.ff_hourglass_spec(5).dims[1:] == [4, 4, 3, 3, 4, 4, 5]
    assert km.ff_hourglass_spec(10, compression_factor=0.2).dims[1:] == [7, 5, 2, 2, 5, 7, 10]
    assert km.ff_hourglass_spec(10, encoding_layers=1).dims[1:] == [5, 5, 10]
    s = km.lstm_hourglass_spec(10)
    assert s.units + [s.n_features_out] == [8, 7, 5, 5, 7, 8, 10]
    # SURVEY A.4 parameter counts
    assert km.ff_hourglass_spec(64).n_params == 15438
    assert km.ff_hourglass_spec(8).n_params == 278
    assert km.ff_hourglass_spec(128).n_params == 61198
    ls = km.lstm_symmetric_spec(128, lookback_window=144)
    assert ls.n_params == 1199744 and ls.flop_per_window == 335085568


def test_l1_placement():
    # encoder layers i>=1 carry the activity regulariser, nothing else does (feedforward_autoencoder.py:76-87)
    s = km.ff_hourglass_spec(64)
    assert s.l1 == [0.0, 10e-5, 10e-5, 0.0, 0.0, 0.0, 0.0]
    assert s.acts == ["tanh"] * 6 + ["linear"]


@pytest.mark.parametrize(
    "L,k,b1x,b1y,b2x,b2y",
    [  # tests/gordo/machine/model/test_model.py:239-311
        (3, 0, [[[0, 1], [2, 3], [4, 5]], [[2, 3], [4, 5], [6, 7]]], [[4, 5], [6, 7]], [[[4, 5], [6, 7], [8, 9]]], [[8, 9]]),
        (2, 1, [[[0, 1], [2, 3]], [[2, 3], [4, 5]]], [[4, 5], [6, 7]], [[[4, 5], [6, 7]]], [[8, 9]]),
        (2, 2, [[[0, 1], [2, 3]], [[2, 3], [4, 5]]], [[6, 7], [8, 9]], None, None),
    ],
)
def test_timeseries_generator_golden(L, k, b1x, b1y, b2x, b2y):
    X = np.array([[0, 1], [2, 3], [4, 5], [6, 7], [8, 9]])
    batches = km.timeseries_batches(X, X.copy(), batch_size=2, lookback_window=L, lookahead=k)
    assert batches[0][0].tolist() == b1x and batches[0][1].tolist() == b1y
    if b2x is None:
        assert len(batches) == 1
    else:
        assert batches[1][0].tolist() == b2x and batches[1][1].tolist() == b2y


def test_timeseries_generator_negative_lookahead():
    with pytest.raises(ValueError):
        km.timeseries_windows(5, 2, -1)


def test_timeseries_doctest_len():
    # models.py:753-768: 100 rows, lookback 20, batch 10 -> 9 batches
    X = np.random.rand(100, 2)
    assert len(km.timeseries_batches(X, X, 10, 20, 0)) == 9


@pytest.mark.parametrize("case", ANOMALY_CASES)
def test_anomaly_oracle_matches_reference_fixture(case):
    g = np.load(os.path.join(GOLDEN, case + ".npz"), allow_pickle=False)
    X, y = g["X"], g["y"]
    n = len(X)
    window = None if int(g["window"]) < 0 else int(g["window"])
    method = None if str(g["method"]) == "None" else str(g["method"])
    # CV geometry
    splits = am.time_series_split(n, 3)
    for i, (tr, te) in enumerate(splits):
        assert te[0] == int(g[f"fold{i}_test_start"]) and len(te) == int(g[f"fold{i}_test_len"])
        assert tr[0] == 0 and tr[-1] == te[0] - 1
        # fold scaler = MinMax fitted on the fold's training targets (diff.py:173 inside sklearn cross_validate)
        sc, mn = am.minmax_fit(y[tr])
        np.testing.assert_allclose(sc, g[f"fold{i}_scale"], rtol=1e-12)
        np.testing.assert_allclose(mn, g[f"fold{i}_min"], rtol=1e-12, atol=1e-15)
        ft, at = am.fold_thresholds(y[te], g[f"fold{i}_pred"], sc, mn, 6)
        # float32 predictions are scaled in float32 by sklearn in the reference -> ~1e-7 relative noise
        np.testing.assert_allclose(ft, g["feature_thresholds_per_fold"][i], rtol=2e-6)
        np.testing.assert_allclose(at, g["aggregate_thresholds_per_fold"][i], rtol=2e-6)
        if window is not None and i == 2:
            fts, ats = am.fold_thresholds(y[te], g[f"fold{i}_pred"], sc, mn, window)
            np.testing.assert_allclose(fts, g["smooth_feature_thresholds"], rtol=2e-6)
            np.testing.assert_allclose(ats, g["smooth_aggregate_threshold"], rtol=2e-6)
    np.testing.assert_allclose(g["feature_thresholds"], g["feature_thresholds_per_fold"][2])
    # final scaler + anomaly frame
    sc, mn = am.minmax_fit(y)
    np.testing.assert_allclose(sc, g["scale"], rtol=1e-12)
    np.testing.assert_allclose(mn, g["min"], rtol=1e-12, atol=1e-15)
    out = am.anomaly_arrays(g["pred"], y, sc, mn, g["feature_thresholds"], float(g["aggregate_threshold"]), window, method)
    level0 = [str(s) for s in g["columns_level0"]]
    for top in level0:
        if top in ("start", "end", "model-input"):
            continue
        want = g[f"frame_{top}"]
        got = out[top]
        if got.ndim == 1:
            want = want.reshape(-1)
        # the reference scales yhat in float32 (sklearn keeps dtype) -> 1e-6 relative noise
        np.testing.assert_allclose(got, want, rtol=2e-6, atol=2e-7, equal_nan=True, err_msg=top)
    np.testing.assert_array_equal(g["frame_model-input"], X)
    # column order (Appendix A.1)
    expect = ["start", "end", "model-input", "model-output", "tag-anomaly-scaled", "total-anomaly-scaled",
              "tag-anomaly-unscaled", "total-anomaly-unscaled"]
    if window is not None:
        expect += ["smooth-tag-anomaly-scaled", "smooth-total-anomaly-scaled", "smooth-tag-anomaly-unscaled", "smooth-total-anomaly-unscaled"]
    expect += ["anomaly-confidence", "total-anomaly-confidence"]
    assert level0 == expect


@pytest.mark.parametrize("case", ["ffnet_anomaly", "ffnet_anomaly_t64"])
def test_ffnet_fixture_prediction_is_oracle_forward(case):
    g = np.load(os.path.join(GOLDEN, case + ".npz"))
    dims = [int(d) for d in g["net_dims"]]
    spec = km.ff_hourglass_spec(dims[0])
    assert spec.dims == dims
    w = [(g[f"W{l}"], g[f"b{l}"]) for l in range(spec.n_layers)]
    pred = km.ff_forward(spec, w, g["X"])
    np.testing.assert_allclose(pred, g["pred"], rtol=1e-5, atol=1e-6)
    # float64 evaluation agrees with float32 to well under the 1e-4 parity budget
    pred64 = km.ff_forward(spec, w, g["X"], dtype=np.float64)
    np.testing.assert_allclose(pred, pred64, rtol=2e-5, atol=2e-6)


def test_base_frame_layout():
    idx = pd.date_range("2019-01-01", periods=5, freq="10min", tz="UTC")
    X = np.arange(15.0).reshape(5, 3)
    out = np.ones((3, 3), np.float32)
    f = am.base_frame(["a", "b", "c"], X, out, index=idx, frequency=pd.Timedelta("10min"))
    assert len(f) == 3 and f.index[0] == idx[2]
    assert f[("start", "")].iloc[0] == idx[2].isoformat()
    assert f[("end", "")].iloc[0] == (idx[2] + pd.Timedelta("10min")).isoformat()
    np.testing.assert_array_equal(f["model-input"].values, X[-3:])


@pytest.mark.parametrize("seed", [11, 12])
def test_live_reference_agrees_with_oracle(seed):
    """The reference's DiffBasedAnomalyDetector, cross-validated and fitted on these frames by tests/golden/make_golden.py: its
    predictions and thresholds through the oracle give its anomaly frame."""
    g = np.load(os.path.join(GOLDEN, f"detector_sma_seed{seed}.npz"), allow_pickle=False)
    rng = np.random.default_rng(seed)
    X, y = rng.random((240, 5)), rng.random((240, 5)) * 3.0
    np.testing.assert_array_equal(g["X"], X)
    np.testing.assert_array_equal(g["y"], y)
    sc, mn = am.minmax_fit(y)
    out = am.anomaly_arrays(g["pred"], y, sc, mn, g["feature_thresholds"], float(g["aggregate_threshold"]), int(g["window"]), str(g["method"]))
    for k, v in out.items():
        want = g[f"frame_{k}"]
        np.testing.assert_allclose(v, want.reshape(v.shape), rtol=1e-9, atol=1e-12, equal_nan=True, err_msg=k)
    assert tuple(g["hourglass_dims_0p5_3_64"]) == km.hourglass_calc_dims(0.5, 3, 64) == (53, 43, 32)


def test_ff_fit_reduces_loss_and_history_contract():
    rng = np.random.default_rng(0)
    spec = km.ff_hourglass_spec(8)
    w0 = km.init_ff_weights(spec, rng)
    t = np.linspace(0, 20, 512)[:, None]
    X = (0.5 + 0.4 * np.sin(t * np.arange(1, 9))).astype(np.float32)
    w1, hist, _ = km.ff_fit(spec, w0, X, X, epochs=5, batch_size=32, rng=np.random.default_rng(1))
    assert hist["loss"][-1] < hist["loss"][0]
    assert set(hist) == {"loss", "accuracy", "params"} and hist["params"]["steps"] == 16 and hist["params"]["epochs"] == 5


def test_ff_grads_match_finite_differences():
    rng = np.random.default_rng(3)
    spec = km.ff_hourglass_spec(6)
    w = km.init_ff_weights(spec, rng)
    w = [(W.astype(np.float64), rng.normal(0, 0.1, b.shape)) for W, b in w]
    xb = rng.random((7, 6))
    loss, _, grads, _ = km.ff_loss_and_grads(spec, w, xb, xb, dtype=np.float64)
    for l in (0, 2, 6):
        W = w[l][0]
        for (i, j) in ((0, 0), (1, 2)):
            h = 1e-6
            Wp = W.copy(); Wp[i, j] += h
            Wm = W.copy(); Wm[i, j] -= h
            lp = km.ff_loss_and_grads(spec, w[:l] + [(Wp, w[l][1])] + w[l + 1:], xb, xb, dtype=np.float64)[0]
            lm = km.ff_loss_and_grads(spec, w[:l] + [(Wm, w[l][1])] + w[l + 1:], xb, xb, dtype=np.float64)[0]
            assert abs((lp - lm) / (2 * h) - grads[l][0][i, j]) < 1e-6


def test_lstm_bptt_gradients_match_finite_differences():
    """The oracle's back-propagation through time (the checker of gb_lstm_fit) against central differences in float64."""
    from oracle import keras_math as km

    spec = km.lstm_model_spec(3, 2, lookback_window=4, encoding_dim=(5,), encoding_func=("tanh",), decoding_dim=(4,), decoding_func=("sigmoid",), out_func="tanh")
    rng = np.random.default_rng(0)
    w = km.init_lstm_weights(spec, rng)
    flat = [a.astype(np.float64) for a in km._lstm_flat(w)]
    win, tg = rng.random((6, 4, 3)), rng.random((6, 2))
    _, grads, _ = km.lstm_loss_and_grads(spec, km._lstm_unflat(flat, 2), win, tg, np.float64)
    gflat = km._lstm_flat(grads)
    for k, a in enumerate(flat):
        for _ in range(5):
            idx = tuple(rng.integers(0, s) for s in a.shape)
            old, h = a[idx], 1e-6
            a[idx] = old + h
            lp = km.lstm_loss_and_grads(spec, km._lstm_unflat(flat, 2), win, tg, np.float64)[0]
            a[idx] = old - h
            lm = km.lstm_loss_and_grads(spec, km._lstm_unflat(flat, 2), win, tg, np.float64)[0]
            a[idx] = old
            fd = (lp - lm) / (2 * h)
            assert abs(fd - gflat[k][idx]) <= 1e-5 * max(1e-3, abs(fd)), (k, idx, fd, gflat[k][idx])


def test_lstm_fit_control_flow():
    """models.py:557-616: primer step + ordered batches; the history has one entry per epoch and the loss falls."""
    from oracle import keras_math as km

    spec = km.lstm_model_spec(3, 3, lookback_window=4, encoding_dim=(5,), encoding_func=("tanh",), decoding_dim=(4,), decoding_func=("tanh",))
    X = np.random.default_rng(2).random((40, 3)).astype(np.float32)
    w, hist = km.lstm_fit(spec, km.init_lstm_weights(spec, np.random.default_rng(1)), X, X, epochs=3, batch_size=8)
    assert len(hist["loss"]) == 3 and hist["loss"][2] < hist["loss"][0] and hist["params"]["steps"] == 5


@pytest.mark.parametrize("case", ["kfcv_smm", "kfcv_ewma"])
def test_oracle_kfcv_thresholds_match_reference_fixture(case):
    """oracle/anomaly_math.kfcv_thresholds against the reference's own DiffBasedKFCVAnomalyDetector (fixture generated by
    tests/golden/make_golden.py from /root/reference): K-fold predictions of a LinearRegression, fold scalers, smoothing, percentile."""
    from sklearn.linear_model import LinearRegression
    from sklearn.model_selection import KFold
    from sklearn.multioutput import MultiOutputRegressor
    from sklearn.utils import shuffle as sk_shuffle

    from oracle import anomaly_math as am

    g = np.load(os.path.join(GOLDEN, f"{case}.npz"), allow_pickle=False)
    X, y = np.ascontiguousarray(g["X"]), np.ascontiguousarray(g["y"])
    abs_err, mse = np.zeros_like(y), np.zeros(len(y))
    for tr, te in KFold(n_splits=5, shuffle=True, random_state=0).split(X, y):
        Xs, ys = sk_shuffle(X[tr], y[tr], random_state=0)  # the KFCV detector shuffles in fit by default (diff.py:469)
        pred = MultiOutputRegressor(LinearRegression()).fit(Xs, ys).predict(X[te])
        scale, mn = am.minmax_fit(y[tr])
        abs_err[te] = np.abs(pred - y[te])
        mse[te] = ((am.minmax_transform(pred, scale, mn) - am.minmax_transform(y[te], scale, mn)) ** 2).mean(axis=1)
    feat, agg = am.kfcv_thresholds(abs_err, mse, int(g["window"]), str(g["method"]), float(g["q"]))
    np.testing.assert_allclose(feat, g["feature_thresholds"], rtol=1e-9)
    np.testing.assert_allclose(agg, float(g["aggregate_threshold"]), rtol=1e-9)
