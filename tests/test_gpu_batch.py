"""GPU: batched fits (``fit_batch``, ``tpls_fit_batch``; DESIGN.md §4d) -- one CTA per problem, the whole fit inside
it -- against the goldens, the ordinary fit of the same problem, per-fold fits with row weights and the oracle."""

import pickle

import numpy as np
import pytest

from _util import aligned_errors, golden_cases, load_golden

pytestmark = pytest.mark.gpu

FP64_TOL = 1e-8
FP32_TOL = 1e-4


def _state(est):
    if hasattr(est, "Xs_factors"):
        return dict(T=est.factor_T, W=[f[1:] for f in est.Xs_factors], U=est.Y_factors[0], Q=est.Y_factors[1],
                    coef=est.coef_, R2X=est.R2Xs, R2Y=est.R2Y)
    return dict(T=est.X_factors[0], W=[est.X_factors[1:]], U=est.Y_factors[0], Q=est.Y_factors[1],
                coef=est.coef_, R2X=[est.R2X], R2Y=est.R2Y)


def _ordinary(Xs, Y, R, coupled, **kw):
    from cmtf_pls_b200 import ctPLS, tPLS
    est = ctPLS(R) if coupled else tPLS(R)
    est.fit([x.copy() for x in Xs] if coupled else Xs[0].copy(), Y.copy(), **kw)
    return est


def _assert_same(model, ref, tol):
    assert model.n_iter_.tolist() == ref.n_iter_.tolist()
    assert model.converged_.tolist() == ref.converged_.tolist()
    errs = aligned_errors(_state(model), _state(ref))
    assert max(errs.values()) < tol, errs


def _problems(dims, M, R, B, seed0, extra=(), dtype=np.float64, miss=0.0):
    from oracle import tpls_oracle as orc
    Xs, Ys = [], []
    for s in range(B):
        X, Y, _ = orc.synthetic(dims, M, R, error=0.3, seed=seed0 + s, extra_dims=list(extra))
        X = list(X) if isinstance(X, list) else [X]
        if miss:
            rng = np.random.default_rng(seed0 + s)
            X[0][rng.random(X[0].shape) < miss] = np.nan
        Xs.append([x.astype(dtype) for x in X])
        Ys.append(Y)
    return [np.stack([p[l] for p in Xs]) for l in range(len(Xs[0]))], np.stack(Ys)


@pytest.mark.parametrize("case", golden_cases())
def test_golden_cases_as_a_batch(case):
    from cmtf_pls_b200 import fit_batch
    g = load_golden(case)
    coupled = bool(g["coupled"])
    R = int(g["n_components"])
    kw = {"max_iter": 4} if "maxiter" in case else {}
    Xb = [np.stack([x] * 3) for x in g["Xs"]]
    Yb = np.stack([g["Y"]] * 3)
    models = fit_batch(Xb if coupled else Xb[0], Yb, R, **kw)
    M = 1 if g["Y"].ndim == 1 else g["Y"].shape[1]
    tol = FP32_TOL if "f32" in case else FP64_TOL
    for est in models:
        assert est.stats_["batch"] == ("kernel" if M <= 8 else "loop")
        assert est.n_iter_.tolist() == g["trips"].tolist()
        for k, e in aligned_errors(_state(est), g).items():
            assert e < tol, (case, k, e)
        means = est.Xs_mean if coupled else [est.X_mean]
        for mine, ref in zip(means, g["X_mean"]):
            assert mine.dtype == ref.dtype and mine.shape == ref.shape
            np.testing.assert_allclose(mine, ref, rtol=1e-6 if "f32" in case else 1e-12,
                                       atol=1e-7 if "f32" in case else 1e-14, equal_nan=True)
        np.testing.assert_allclose(est.Y_mean, g["Y_mean"], rtol=1e-12, atol=1e-14)


@pytest.mark.parametrize("name,dims,M,R,extra,dtype", [
    ("configs0_f64", (20, 8, 6), 1, 3, (), np.float64),
    ("configs0_f32", (20, 8, 6), 1, 3, (), np.float32),
    ("configs1_reduced", (300, 32, 16), 4, 5, ((300, 24),), np.float64),
    ("four_way", (40, 8, 6, 4), 3, 3, (), np.float64),
])
def test_against_the_ordinary_fit(name, dims, M, R, extra, dtype):
    from cmtf_pls_b200 import fit_batch
    Xb, Yb = _problems(dims, M, R, 64, 1000, extra=extra, dtype=dtype)
    coupled = len(Xb) > 1
    models = fit_batch(Xb if coupled else Xb[0], Yb, R)
    tol = 1e-6 if dtype == np.float32 else 1e-10
    for b, est in enumerate(models):
        assert est.stats_["batch"] == "kernel"
        _assert_same(est, _ordinary([x[b] for x in Xb], Yb[b], R, coupled), tol)


@pytest.mark.parametrize("dims,smem", [((60, 16, 12), "1"), ((3000, 16, 8), "1"), ((60, 16, 12), "0")])
def test_both_placements(dims, smem, monkeypatch):
    """(60, 16, 12) fp64 fits in shared memory; (3000, 16, 8) fp64 (3 MB of X) takes a slot of the global workspace;
    TPLS_BATCH_SMEM=0 sends the small one there too."""
    from cmtf_pls_b200 import fit_batch
    monkeypatch.setenv("TPLS_BATCH_SMEM", smem)
    Xb, Yb = _problems(dims, 3, 3, 4, 77)
    for b, est in enumerate(fit_batch(Xb[0], Yb, 3)):
        assert est.stats_["batch"] == "kernel"
        _assert_same(est, _ordinary([Xb[0][b]], Yb[b], 3, False), 1e-10)


def _run_fit_state(X, Y, R, w):
    from cmtf_pls_b200 import _core
    return _core.run_fit([X], Y, R, 1e-8, 100, row_weights=w)


def _compare_to_run_fit(est, st, tol):
    assert est.n_iter_.tolist() == st["trips"].tolist()
    ref = dict(T=st["T"], W=[st["W"][0]], U=st["U"], Q=st["Q"], coef=st["coef"], R2X=st["R2X"], R2Y=st["R2Y"])
    errs = aligned_errors(_state(est), ref)
    assert max(errs.values()) < tol, errs


@pytest.mark.parametrize("shape,n_folds,miss", [((30, 8, 6), None, 0.1), ((90, 12, 8), 5, 0.0)])
def test_fold_masks_against_weighted_fits(shape, n_folds, miss):
    from cmtf_pls_b200 import fit_batch
    from cmtf_pls_b200.validate import _folds
    Xb, Yb = _problems(shape, 2, 3, 1, 5, miss=miss)
    X, Y = Xb[0][0], Yb[0]
    folds = _folds(shape[0], n_folds, 1)
    W = np.ones((len(folds), shape[0]))
    for k, f in enumerate(folds):
        W[k, f] = 0.0
    models = fit_batch(X[None], Y[None], 3, row_weights=W)
    for k, est in enumerate(models):
        assert est.stats_["batch"] == "kernel"
        _compare_to_run_fit(est, _run_fit_state(X, Y, 3, W[k]), 1e-10)
        # held-out rows of T are transform() of those rows under the fold's model
        held = folds[k]
        t = est.transform(X[held])
        np.testing.assert_allclose(t, est.X_factors[0][held], rtol=1e-9, atol=1e-9 * np.abs(t).max())


def test_all_nans_in_held_out_rows():
    from cmtf_pls_b200 import fit_batch
    Xb, Yb = _problems((40, 8, 6), 2, 2, 1, 11)
    X, Y = Xb[0][0], Yb[0]
    X[:5, 2, :] = np.nan
    X[3, :, 1] = np.nan
    W = np.ones((2, 40))
    W[0, :5] = 0.0       # every NaN held out
    W[1, 20:25] = 0.0    # NaNs in the training rows
    models = fit_batch(X[None], Y[None], 2, row_weights=W)
    for k, est in enumerate(models):
        assert est.X_hasMiss
        assert np.all(np.isfinite(est.X_factors[0]))
        _compare_to_run_fit(est, _run_fit_state(X, Y, 2, W[k]), 1e-10)
        with pytest.raises(RuntimeError, match="no longer alive"):
            est.X_miss


@pytest.mark.parametrize("shape,coupled,miss", [((90, 12, 8), False, False), ((80, 8, 6, 4), False, False),
                                                ((90, 12, 8), True, False), ((90, 12, 8), False, True)])
def test_q2y_sweep_batch_matches_oracle_refits(shape, coupled, miss):
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import q2y_sweep
    from cmtf_pls_b200.validate import _folds
    X, Y, _ = orc.synthetic(shape, 3, 4, error=0.4, seed=9, extra_dims=[(shape[0], 10)] if coupled else ())
    if miss:
        rng = np.random.default_rng(2)
        X[rng.random(X.shape) < 0.1] = np.nan
    folds = _folds(shape[0], 5, 3)
    q_ref, cv_ref = orc.q2y_kfold(X, Y, 4, folds)
    q, cv = q2y_sweep(X, Y, 4, n_splits=5, seed=3, return_scores=True, algorithm="batch")
    assert np.max(np.abs(q - q_ref)) < 1e-8
    s = np.sign(np.sum(cv * cv_ref, axis=0))
    assert np.max(np.abs(cv * s - cv_ref)) / np.max(np.abs(cv_ref)) < 1e-8


def test_q2y_sweep_batch_leave_one_out():
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import q2y_sweep
    X, Y, _ = orc.synthetic((24, 6, 5), 2, 2, error=0.2, seed=4)
    q_ref, _ = orc.q2y_kfold(X, Y, 2, [np.array([i]) for i in range(24)])
    q = q2y_sweep(X, Y, 2, n_splits=None, algorithm="batch")
    assert np.max(np.abs(q - q_ref)) < 1e-8


def test_more_problems_than_resident_ctas():
    """B = 1000 > co-resident CTAs: every CTA fits several problems in turn (slot / index mix-ups would show)."""
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import fit_batch
    Xb, Yb = _problems((20, 8, 6), 1, 3, 1000, 0)
    models = fit_batch(Xb[0], Yb, 3)
    for b, est in enumerate(models):
        ref = orc.fit([Xb[0][b].copy()], Yb[b].copy(), 3, r2_mode="residual")
        assert est.n_iter_.tolist() == ref["trips"].tolist(), b
        errs = aligned_errors(_state(est), dict(T=ref["T"], W=ref["W"], U=ref["U"], Q=ref["Q"], coef=ref["coef"],
                                                R2X=ref["R2X"], R2Y=ref["R2Y"]))
        assert max(errs.values()) < 1e-8, (b, errs)


def test_broadcast_batch_axes():
    from cmtf_pls_b200 import fit_batch
    Xb, Yb = _problems((30, 6, 5), 2, 2, 4, 21)
    # one X, four Y
    for b, est in enumerate(fit_batch(Xb[0][:1], Yb, 2)):
        _assert_same(est, _ordinary([Xb[0][0]], Yb[b], 2, False), 1e-10)
    # four X, one Y
    for b, est in enumerate(fit_batch(Xb[0], Yb[:1], 2)):
        _assert_same(est, _ordinary([Xb[0][b]], Yb[0], 2, False), 1e-10)


def test_fallback_to_one_by_one(monkeypatch):
    from cmtf_pls_b200 import fit_batch
    Xb, Yb = _problems((30, 6, 5), 10, 2, 3, 31)     # 10 responses: outside the kernel's limits
    for b, est in enumerate(fit_batch(Xb[0], Yb, 2)):
        assert est.stats_["batch"] == "loop"
        _assert_same(est, _ordinary([Xb[0][b]], Yb[b], 2, False), 1e-12)
    Xb, Yb = _problems((30, 6, 5), 2, 2, 3, 41)
    monkeypatch.setenv("TPLS_BATCH", "0")
    for b, est in enumerate(fit_batch(Xb[0], Yb, 2)):
        assert est.stats_["batch"] == "loop"
        _assert_same(est, _ordinary([Xb[0][b]], Yb[b], 2, False), 1e-12)


def test_returned_models_are_usable():
    import torch
    from cmtf_pls_b200 import fit_batch
    Xb, Yb = _problems((50, 8, 6), 3, 3, 3, 51, extra=((50, 7),))
    models = fit_batch([torch.from_numpy(x).cuda() for x in Xb], torch.from_numpy(Yb).cuda(), 3)
    for b, est in enumerate(models):
        assert est.stats_["batch"] == "kernel"
        xs = [x[b] for x in Xb]
        t = est.transform(xs)
        np.testing.assert_allclose(t, est.factor_T, rtol=1e-9, atol=1e-9 * np.abs(t).max())
        pred = est.predict(xs)
        assert pred.shape == (50, 3) and np.all(np.isfinite(pred))
        back = pickle.loads(pickle.dumps(est))
        np.testing.assert_array_equal(back.predict(xs), pred)
        assert back.n_iter_.tolist() == est.n_iter_.tolist()
        rec = back.Xs_reconstructed()
        assert [r.shape for r in rec] == [x.shape for x in xs]
