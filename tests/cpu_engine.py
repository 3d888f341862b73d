"""
TEST INFRASTRUCTURE ONLY.  A CPU stand-in for the compute entry points of ``gordo_components_b200.engine``, built on the
oracle (``oracle/keras_math.py``, ``oracle/anomaly_math.py``), so that the *host-side* protocol of the estimator classes --
what gordo's serializer, ModelBuilder and server call on them -- can be exercised end to end without a GPU
(tests/test_reference_dropin.py, and tests/golden/make_golden.py for its fixture).

The product has no CPU path: this module is never imported by the package, and the numbers it produces are the oracle's, not
a parity claim about the kernels (those are tests/test_gpu_*.py on a B200).  ``patched_engine()`` swaps the entry points in and
restores them on exit.
"""
from __future__ import annotations

import contextlib

import numpy as np
import torch

from gordo_components_b200 import _cabi, engine
from oracle import anomaly_math as am
from oracle import keras_math as km

CPU = torch.device("cpu")


def _jobs(jobs_dev) -> np.ndarray:
    return jobs_dev.cpu().numpy().view(_cabi.JOB_DTYPE)


def _np(t):
    return None if t is None else t.detach().cpu().numpy()


class _FFEngine(engine.FFEngine):
    """The real engine's bookkeeping (parameter layout from the C library, which loads without a GPU) with oracle arithmetic."""

    def _spec(self):
        return km.FFSpec(list(self.dims), list(self.acts), list(self.l1))

    def infer_score(self, params, jobs_dev, n_jobs, max_rows, x, y=None, scale=None, feat_thr=None, agg_thr=None, out_rows=None,
                    want=engine.SCORE_KEYS, variant=0, out=None):
        total = int(out_rows if out_rows is not None else x.shape[0])
        weights = self.unpack_params(params)
        X, Y = _np(x), _np(y)
        res = {"model-output": np.zeros((total, self.n_out), np.float32)}
        sel = set(want) if y is not None else set()
        if scale is None:
            sel -= {"tag-anomaly-scaled", "total-anomaly-scaled", "total-anomaly-confidence"}
        if feat_thr is None:
            sel.discard("anomaly-confidence")
        if agg_thr is None:
            sel.discard("total-anomaly-confidence")
        for name in sel:
            res[name] = np.zeros((total, self.n_out) if name.startswith(("tag-", "anomaly-")) else (total,), np.float32)
        for job in _jobs(jobs_dev)[:n_jobs]:
            s, n, xr, orow = int(job["slot"]), int(job["n_rows"]), int(job["x_row"]), int(job["out_row"])
            pred = km.ff_forward(self._spec(), weights[s], X[xr:xr + n])
            res["model-output"][orow:orow + n] = pred
            if sel:
                sc = _np(scale)[s].astype(np.float64) if scale is not None else np.ones(self.n_out)
                cols = am.anomaly_arrays(pred, Y[xr:xr + n], sc, np.zeros_like(sc), None if feat_thr is None else _np(feat_thr)[s],
                                         None if agg_thr is None else float(_np(agg_thr)[s]))
                for name in sel:
                    res[name][orow:orow + n] = cols[name]
        return {k: torch.from_numpy(v) for k, v in res.items()}

    def fit(self, params, jobs_dev, n_jobs, max_rows, x, y, epochs=1, batch_size=32, shuffle=True, perm=None, adam=None, seed=0,
            l1_div_batch=False, state=None, step0=0):
        adam = adam or {}
        weights = self.unpack_params(params)
        X, Y = _np(x), _np(y)
        loss = np.zeros((n_jobs, epochs), np.float32)
        acc = np.zeros((n_jobs, epochs), np.float32)
        state = state if state is not None else {}
        host = params.numpy()
        for i, job in enumerate(_jobs(jobs_dev)[:n_jobs]):
            s, n, xr = int(job["slot"]), int(job["n_rows"]), int(job["x_row"])
            perms = None if perm is None else [_np(perm)[i, e, :n] for e in range(epochs)]
            w, hist, st = km.ff_fit(self._spec(), weights[s], X[xr:xr + n], Y[xr:xr + n], epochs=epochs, batch_size=batch_size, shuffle=bool(shuffle),
                                    perms=perms, rng=np.random.default_rng(int(seed) + 7919 * s), lr=adam.get("lr", 1e-3), b1=adam.get("beta1", 0.9),
                                    b2=adam.get("beta2", 0.999), eps=adam.get("eps", 1e-7), l1_div_batch=l1_div_batch, state=state.get(s))
            state[s] = st
            loss[i], acc[i] = hist["loss"], hist["accuracy"]
            ofs = 0
            for W, b in w:
                host[s, ofs:ofs + W.size] = W.ravel()
                ofs += W.size
                host[s, ofs:ofs + b.size] = b
                ofs += b.size
        return torch.from_numpy(loss), torch.from_numpy(acc), state


def _ff_engine_for(spec, device=None):
    return _FFEngine(spec.dims, spec.acts, spec.l1, CPU)


def _minmax_f64(jobs_dev, n_jobs, max_rows, y64, n_slots):
    y = _np(y64)
    lo = np.full((n_slots, y.shape[1]), np.inf)
    hi = np.full((n_slots, y.shape[1]), -np.inf)
    for job in _jobs(jobs_dev)[:n_jobs]:
        rows = y[int(job["x_row"]):int(job["x_row"]) + int(job["n_rows"])]
        lo[int(job["slot"])], hi[int(job["slot"])] = np.nanmin(rows, axis=0), np.nanmax(rows, axis=0)
    return torch.from_numpy(lo), torch.from_numpy(hi)


def _thresholds(jobs_dev, n_jobs, max_rows, tag_unscaled, total_scaled, n_out, n_slots, window, device):
    tu, ts = _np(tag_unscaled), _np(total_scaled)
    feat = np.full((n_slots, n_out), np.nan, tu.dtype)
    agg = np.full((n_slots,), np.nan, tu.dtype)
    for job in _jobs(jobs_dev)[:n_jobs]:
        sl = slice(int(job["out_row"]), int(job["out_row"]) + int(job["n_rows"]))
        feat[int(job["slot"])] = am.rolling_min_then_max(tu[sl], window)
        agg[int(job["slot"])] = am.rolling_min_then_max(ts[sl], window)
    return torch.from_numpy(feat), torch.from_numpy(agg)


def _anomaly_score(jobs_dev, n_jobs, max_rows, yhat, y, n_out, scale=None, feat_thr=None, agg_thr=None, want=engine.SCORE_KEYS, device=None):
    P, Y = _np(yhat), _np(y)
    sel = set(want)
    if scale is None:
        sel -= {"tag-anomaly-scaled", "total-anomaly-scaled", "total-anomaly-confidence"}
    if feat_thr is None:
        sel.discard("anomaly-confidence")
    if agg_thr is None:
        sel.discard("total-anomaly-confidence")
    res = {name: np.zeros((len(P), n_out) if name.startswith(("tag-", "anomaly-")) else (len(P),), P.dtype) for name in sel}
    for job in _jobs(jobs_dev)[:n_jobs]:
        s, n, xr, orow = int(job["slot"]), int(job["n_rows"]), int(job["x_row"]), int(job["out_row"])
        sc = _np(scale)[s].astype(np.float64) if scale is not None else np.ones(n_out)
        cols = am.anomaly_arrays(P[orow:orow + n], Y[xr:xr + n], sc, np.zeros_like(sc), None if feat_thr is None else _np(feat_thr)[s],
                                 None if agg_thr is None else float(_np(agg_thr)[s]))
        for name in sel:
            res[name][orow:orow + n] = cols[name]
    return {k: torch.from_numpy(v) for k, v in res.items()}


def _affine_f64(jobs_dev, n_jobs, max_rows, x64, a, b, out_rows=None):
    X, A, B = _np(x64), _np(a), _np(b)
    out = np.zeros((int(out_rows if out_rows is not None else len(X)), X.shape[1]), np.float32)
    for job in _jobs(jobs_dev)[:n_jobs]:
        s, n, xr, orow = int(job["slot"]), int(job["n_rows"]), int(job["x_row"]), int(job["out_row"])
        out[orow:orow + n] = (X[xr:xr + n] * A[s] + B[s]).astype(np.float32)
    return torch.from_numpy(out)


def _smooth(jobs_dev, n_jobs, arr, window, method, max_rows=None):
    a = _np(arr)
    out = np.full_like(a, np.nan)
    for job in _jobs(jobs_dev)[:n_jobs]:
        sl = slice(int(job["out_row"]), int(job["out_row"]) + int(job["n_rows"]))
        out[sl] = am.smoothing(a[sl].astype(np.float64), window, method)
    return torch.from_numpy(out)


@contextlib.contextmanager
def patched_engine():
    """Inside the block ``gordo_components_b200.engine`` computes on the CPU with the oracle (tests only)."""
    saved = {n: getattr(engine, n) for n in ("cuda_device", "ff_engine_for", "minmax_f64", "thresholds", "anomaly_score", "affine_f64", "smooth")}
    engine.cuda_device = lambda device=None: CPU
    engine.ff_engine_for = _ff_engine_for
    engine.minmax_f64, engine.thresholds, engine.anomaly_score = _minmax_f64, _thresholds, _anomaly_score
    engine.affine_f64, engine.smooth = _affine_f64, _smooth
    try:
        yield
    finally:
        for n, f in saved.items():
            setattr(engine, n, f)
