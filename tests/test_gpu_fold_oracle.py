"""GPU: fold fits (0/1 row weights) against an fp64 oracle refit on the training rows, where the held-out rows hold
NaNs in the patterns cross-validation meets: scattered, a whole row, a whole row of one coupled tensor only, and a
column whose only observation is in a held-out row.

The contract (batch.py, validate.py): the training part of a fold fit is the fit on the training rows alone, and the
held-out rows' scores are exactly ``transform`` of those rows under the fold's model.  So the reference of a fold is
``orc.fit`` on the sliced training rows, with ``orc.transform`` of the held-out rows as their scores; no weighted
fit is involved.  Every fold is checked through the batch kernel (``fit_batch``), the ordinary weighted fit in both
inner loops (``_core.run_fit``) and ``q2y_sweep`` in all three algorithms (against ``orc.q2y_kfold``).

The bar: equal trip counts, equal NaN positions, and 1e-8 (fp64 storage) / 1e-4 (fp32) on the finite values after
per-component sign alignment.  Each oracle refit runs once per module.

The stop quantity ||u_old - u|| of every oracle trip of these folds stays at least 6 % away from tol = 1e-8, so equal
trip counts test the kernels, not rounding.  (Measured by recording that norm at every trip of ``orc.fit``, line
``if np.linalg.norm(old_u - U[:, a]) < tol``; rerun it when a seed, shape or NaN pattern changes.)
"""

import numpy as np
import pytest

from _util import aligned_errors

pytestmark = pytest.mark.gpu

FP64_TOL = 1e-8
FP32_TOL = 1e-4
N = 30
R = 3


def case_data(name, coupled, dtype):
    """(Xs, Y, folds) of a case: orc.synthetic((30, 8, 6), 2 responses, 3 latent) and, coupled, a (30, 10) second
    tensor; NaNs placed as the case says; ``folds`` are the held-out rows of each fold mask."""
    from oracle import tpls_oracle as orc
    X, Y, _ = orc.synthetic((N, 8, 6), 2, R, error=0.3, seed=17, extra_dims=[(N, 10)] if coupled else [])
    Xs = [x.astype(dtype) for x in (X if coupled else [X])]
    rng = np.random.default_rng(5)
    if name == "F1":      # NaNs only in held-out rows; every training row complete
        held = np.array([2, 7, 11, 23])
        for x in Xs:
            sub = x[held]
            sub[rng.random(sub.shape) < 0.3] = np.nan
            x[held] = sub
        folds = [held, np.concatenate([held, [0, 15]])]
    elif name == "F2":    # one held-out row entirely NaN (in every tensor), scattered NaNs elsewhere
        for x in Xs:
            x[rng.random(x.shape) < 0.1] = np.nan
            x[4] = np.nan
        folds = [np.array([4, 9, 15]), np.array([4])]
    elif name == "F3":    # coupled: a held-out row entirely NaN in the first tensor only; the second one dense
        Xs[0][rng.random(Xs[0].shape) < 0.1] = np.nan
        Xs[0][4] = np.nan
        folds = [np.array([4, 9, 15]), np.array([4])]
    elif name == "F4":    # column (3, 2) of the first tensor NaN in every row but held-out row 6
        Xs[0][:, 3, 2] = np.nan
        Xs[0][6, 3, 2] = 1.5
        folds = [np.array([6, 12]), np.array([6])]
    else:
        raise KeyError(name)
    return Xs, Y, folds


CASES = [("F1", False), ("F1", True), ("F2", False), ("F2", True), ("F3", True), ("F4", False), ("F4", True)]
DTYPES = [np.float64, np.float32]
IDS = [f"{n}-{'coupled' if c else 'single'}" for n, c in CASES]

_refs = {}


def oracle_fold(Xs, Y, held):
    """The reference of one fold: the fit on the training rows, the held-out rows' scores by transform."""
    from oracle import tpls_oracle as orc
    train = np.setdiff1d(np.arange(Y.shape[0]), held)
    st = orc.fit([x[train].astype(np.float64) for x in Xs], Y[train], R, r2_mode="residual")
    T = np.empty((Y.shape[0], R))
    T[train] = st["T"]
    T[held] = orc.transform(st, [x[held].astype(np.float64) for x in Xs])
    # coef: the upper triangle (lstsq on the zero-padded scores can leave rounding noise below it)
    return dict(T=T, U=st["U"], train=train, W=st["W"], Q=st["Q"], coef=np.triu(st["coef"]), R2X=st["R2X"], R2Y=st["R2Y"],
                X_mean=st["X_mean"], Y_mean=st["Y_mean"], trips=st["trips"])


@pytest.fixture(scope="module")
def refs():
    """(Xs, Y, folds, [reference per fold]) of a case, computed on first use and kept for the module."""
    def get(name, coupled, dtype):
        key = (name, coupled, np.dtype(dtype).name)
        if key not in _refs:
            Xs, Y, folds = case_data(name, coupled, dtype)
            _refs[key] = (Xs, Y, folds, [oracle_fold(Xs, Y, h) for h in folds])
        return _refs[key]
    yield get
    _refs.clear()


def _masks(folds):
    W = np.ones((len(folds), N))
    for k, h in enumerate(folds):
        W[k, h] = 0.0
    return W


def check_fold(got, ref, tol):
    """``got``: T (all rows), U, W, Q, coef, R2X, R2Y, X_mean, Y_mean, trips of a fold fit."""
    assert np.asarray(got["trips"]).tolist() == ref["trips"].tolist()
    train = ref["train"]
    g = dict(T=np.asarray(got["T"]), U=np.asarray(got["U"])[train], W=got["W"], Q=got["Q"], coef=got["coef"],
             R2X=got["R2X"], R2Y=got["R2Y"])
    r = dict(T=ref["T"], U=ref["U"], W=ref["W"], Q=ref["Q"], coef=ref["coef"], R2X=ref["R2X"], R2Y=ref["R2Y"])
    flat = lambda d: [("T", d["T"]), ("U", d["U"]), ("Q", d["Q"]), ("coef", d["coef"]), ("R2Y", d["R2Y"])] + \
        [(f"R2X{l}", v) for l, v in enumerate(d["R2X"])] + \
        [(f"W{l}.{k}", w) for l, ws in enumerate(d["W"]) for k, w in enumerate(ws)]
    for (k, a), (_, b) in zip(flat(g), flat(r)):
        np.testing.assert_array_equal(np.isnan(np.asarray(a, dtype=np.float64)), np.isnan(b), err_msg=k)
    zero = lambda d: dict(T=np.nan_to_num(d["T"]), U=np.nan_to_num(d["U"]), Q=np.nan_to_num(d["Q"]),
                          coef=np.nan_to_num(d["coef"]), R2Y=np.nan_to_num(d["R2Y"]),
                          R2X=[np.nan_to_num(np.asarray(v, dtype=np.float64)) for v in d["R2X"]],
                          W=[[np.nan_to_num(np.asarray(w, dtype=np.float64)) for w in ws] for ws in d["W"]])
    errs = aligned_errors(zero(g), zero(r))
    assert max(errs.values()) < tol, errs
    for mine, m in zip(got["X_mean"], ref["X_mean"]):
        np.testing.assert_allclose(np.asarray(mine, dtype=np.float64), m, rtol=10 * tol, atol=10 * tol, equal_nan=True)
    np.testing.assert_allclose(got["Y_mean"], ref["Y_mean"], rtol=1e-12, atol=1e-14)


def _tol(dtype):
    return FP32_TOL if dtype == np.float32 else FP64_TOL


@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
@pytest.mark.parametrize("name,coupled", CASES, ids=IDS)
def test_batch_kernel_fold_fits(refs, name, coupled, dtype):
    from cmtf_pls_b200 import fit_batch
    Xs, Y, folds, ref = refs(name, coupled, dtype)
    models = fit_batch([x[None] for x in Xs] if coupled else Xs[0][None], Y[None], R, row_weights=_masks(folds))
    for k, est in enumerate(models):
        assert est.stats_["batch"] == "kernel"
        if coupled:
            got = dict(T=est.factor_T, W=[f[1:] for f in est.Xs_factors], X_mean=est.Xs_mean)
        else:
            got = dict(T=est.X_factors[0], W=[est.X_factors[1:]], X_mean=[est.X_mean])
        got.update(U=est.Y_factors[0], Q=est.Y_factors[1], coef=est.coef_, R2X=est.R2Xs if coupled else [est.R2X],
                   R2Y=est.R2Y, Y_mean=est.Y_mean, trips=est.n_iter_)
        check_fold(got, ref[k], _tol(dtype))


@pytest.mark.parametrize("algorithm", ["stream", "covariance"])
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
@pytest.mark.parametrize("name,coupled", CASES, ids=IDS)
def test_weighted_fit_fold_fits(refs, name, coupled, dtype, algorithm):
    from cmtf_pls_b200 import _core
    Xs, Y, folds, ref = refs(name, coupled, dtype)
    for k, w in enumerate(_masks(folds)):
        st = _core.run_fit([x.copy() for x in Xs], Y.copy(), R, 1e-8, 100, row_weights=w, algorithm=algorithm)
        check_fold(st, ref[k], _tol(dtype))


def _compare_cv(q, cv, q_ref, cv_ref, tol):
    np.testing.assert_array_equal(np.isnan(cv), np.isnan(cv_ref))
    a, b = np.nan_to_num(cv), np.nan_to_num(cv_ref)
    s = np.sign(np.sum(a * b, axis=0))
    s[s == 0] = 1
    assert np.max(np.abs(a * s - b)) <= tol * np.max(np.abs(b))
    fin = np.isfinite(q_ref)
    assert np.max(np.abs(q[fin] - q_ref[fin]), initial=0.0) < tol


@pytest.mark.parametrize("algorithm", ["batch", "covariance", "stream"])
@pytest.mark.parametrize("name,coupled", CASES, ids=IDS)
def test_q2y_sweep_fold_scores(name, coupled, algorithm):
    """One sweep per fold; ``cv`` holds the held-out rows' scores under the fold's model."""
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import q2y_sweep
    Xs, Y, folds = case_data(name, coupled, np.float64)
    X = Xs if coupled else Xs[0]
    for k, held in enumerate(folds):   # the folds of a case overlap: one sweep per fold keeps every score
        key = ("q2y", name, coupled, k)
        if key not in _refs:
            _refs[key] = orc.q2y_kfold([x.copy() for x in Xs], Y.copy(), R, [held])
        q_ref, cv_ref = _refs[key]
        q, cv = q2y_sweep(X, Y, R, folds=[held], return_scores=True, algorithm=algorithm)
        _compare_cv(q, cv[held], q_ref, cv_ref[held], FP64_TOL)


def loo_data(coupled):
    """Leave-one-out data: sample 0 is the only observation of column (2, 1) of the first tensor, so the fold that
    holds it out trains on a column with no observation; scattered NaNs elsewhere."""
    from oracle import tpls_oracle as orc
    X, Y, _ = orc.synthetic((16, 5, 4), 2, 2, error=0.2, seed=8, extra_dims=[(16, 6)] if coupled else [])
    Xs = list(X) if coupled else [X]
    rng = np.random.default_rng(9)
    Xs[0][rng.random(Xs[0].shape) < 0.1] = np.nan
    Xs[0][1:, 2, 1] = np.nan
    Xs[0][0, 2, 1] = 0.7
    return Xs, Y


@pytest.mark.parametrize("algorithm", ["batch", "covariance", "stream"])
@pytest.mark.parametrize("coupled", [False, True], ids=["single", "coupled"])
def test_q2y_sweep_leave_one_out_sparse(coupled, algorithm):
    """F5: leave-one-out where one sample is the only observation of a column.  (A sample with no observation at
    all is held out in the F2 / F3 sweeps above; leave-one-out would also train every other fold on it, a row that
    projects to NaN, where the reference itself fails.)"""
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import q2y_sweep
    Xs, Y = loo_data(coupled)
    key = ("loo", coupled)
    if key not in _refs:
        _refs[key] = orc.q2y_kfold([x.copy() for x in Xs], Y.copy(), 2, [np.array([i]) for i in range(16)])
    q_ref, cv_ref = _refs[key]
    q, cv = q2y_sweep(Xs if coupled else Xs[0], Y, 2, n_splits=None, return_scores=True, algorithm=algorithm)
    _compare_cv(q, cv, q_ref, cv_ref, FP64_TOL)
