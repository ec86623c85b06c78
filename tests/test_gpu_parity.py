"""GPU: the CUDA fit path, called through the estimators -> C ABI, against the
golden vectors of the reference and against the oracle on seeded inputs.

Tolerances (BASELINE.json north_star): 1e-8 relative for fp64 storage, 1e-4
for fp32 storage, on loadings, scores, Q, coef_, R2X, R2Y after per-component
sign alignment; measured per factor column as ||a-b|| / ||b||.
"""

import os

import numpy as np
import pytest

from _util import golden_cases, load_golden, aligned_errors, col_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

FP64_TOL = 1e-8
FP32_TOL = 1e-4


def _state(est, coupled):
    if coupled:
        return dict(T=est.factor_T, W=[f[1:] for f in est.Xs_factors], U=est.Y_factors[0], Q=est.Y_factors[1],
                    coef=est.coef_, R2X=est.R2Xs, R2Y=est.R2Y)
    return dict(T=est.X_factors[0], W=[est.X_factors[1:]], U=est.Y_factors[0], Q=est.Y_factors[1],
                coef=est.coef_, R2X=[est.R2X], R2Y=est.R2Y)


def _fit(g, **kw):
    from cmtf_pls_b200 import tPLS, ctPLS
    R = int(g["n_components"])
    if bool(g["coupled"]):
        est = ctPLS(R)
        est.fit([x.copy() for x in g["Xs"]], g["Y"].copy(), **kw)
    else:
        est = tPLS(R)
        est.fit(g["Xs"][0].copy(), g["Y"].copy(), **kw)
    return est


@pytest.mark.parametrize("loop", ["resident", "streaming"])
@pytest.mark.parametrize("case", golden_cases())
def test_fit_matches_reference_golden(case, loop, monkeypatch):
    """Every golden case through both inner loops: the resident trip loop (the default at these sizes, DESIGN.md §3b) and
    the streaming kernels under the graph WHILE node (what large and sharded fits run)."""
    if loop == "streaming":
        monkeypatch.setenv("TPLS_RESIDENT", "0")
    g = load_golden(case)
    kw = {"max_iter": 4} if "maxiter" in case else {}
    est = _fit(g, **kw)
    M = 1 if g["Y"].ndim == 1 else g["Y"].shape[1]
    assert (est.stats_["resident_loops"] > 0) == (loop == "resident" and M <= 8)
    tol = FP32_TOL if "f32" in case else FP64_TOL
    assert est.n_iter_.tolist() == g["trips"].tolist()
    for k, e in aligned_errors(_state(est, bool(g["coupled"])), g).items():
        assert e < tol, (case, k, e)
    means = est.Xs_mean if bool(g["coupled"]) else [est.X_mean]
    for mine, ref in zip(means, g["X_mean"]):
        assert mine.dtype == ref.dtype and mine.shape == ref.shape
        np.testing.assert_allclose(mine, ref, rtol=1e-6 if "f32" in case else 1e-12, atol=1e-7 if "f32" in case else 1e-14,
                                   equal_nan=True)
    np.testing.assert_allclose(est.Y_mean, g["Y_mean"], rtol=1e-12, atol=1e-14)


@pytest.mark.parametrize("case", [c for c in golden_cases() if c in (
    "t3_60x16x12_m4_r5", "t4_60x8x6x4_m3_r4", "t3_miss_70x12x8_m4_r4", "ct_90x32x16_90x24_m4_r5")])
def test_transform_predict_match_reference_golden(case):
    g = load_golden(case)
    est = _fit(g)
    coupled = bool(g["coupled"])
    new = [x.copy() for x in g["Xsnew"]]
    arg = new if coupled else new[0]
    assert col_err(est.predict(arg), g["predict_new"]) < FP64_TOL
    s, v = est.transform(arg, g["Ynew"].copy())
    assert col_err(s, g["transform_new_X"]) < FP64_TOL
    assert col_err(v, g["transform_new_Y"]) < FP64_TOL
    # the caller's arrays are never modified (tpls.py:128,151)
    for a, b in zip(new, g["Xsnew"]):
        assert np.array_equal(a, b, equal_nan=True)


def test_fit_leaves_inputs_untouched_and_api_surface():
    g = load_golden("t3_60x16x12_m4_r5")
    X, Y = g["Xs"][0].copy(), g["Y"].copy()
    from cmtf_pls_b200 import tPLS
    est = tPLS(3)
    assert est.fit(X, Y) is None
    assert np.array_equal(X, g["Xs"][0]) and np.array_equal(Y, g["Y"])
    assert est.X_dim == 3 and est.X_shape == X.shape and est.Y_shape == Y.shape
    assert [f.shape for f in est.X_factors] == [(60, 3), (16, 3), (12, 3)]
    assert [f.shape for f in est.Y_factors] == [(60, 3), (4, 3)]
    assert est[0] is est.X_factors and est[1] is est.Y_factors and est[2] is est.coef_
    assert est.coef_.shape == (3, 3) and np.allclose(np.tril(est.coef_, -1), 0)
    assert est.X_hasMiss is False and est.X_miss.shape == X.shape and not est.X_miss.any()
    assert est.X_reconstructed().shape == X.shape
    with pytest.raises(ValueError, match="Training X has shape"):
        est.predict(np.zeros((3, 16, 11)))
    with pytest.raises(ValueError, match="Training Y has shape"):
        est.transform(X, np.zeros((60, 5)))
    c = est.copy()
    assert c.X_factors is est.X_factors


@pytest.mark.parametrize("shape,M,R,dtype", [
    ((500, 64, 64), 4, 3, np.float64),      # c4-shaped rows (P = 4096), fp64 -> two column slabs
    ((500, 64, 64), 4, 3, np.float32),      # c4-shaped rows, fp32 -> one slab, 4 groups per lane
    ((400, 32, 16, 8), 4, 3, np.float32),   # c5-shaped rows (4-way)
    ((300, 24), 4, 3, np.float64),          # matrix X
    ((257, 7, 3), 2, 2, np.float32),        # row bytes not a multiple of 16 -> pitched staging
    ((130, 9, 7), 3, 2, np.float64),        # odd P in fp64 -> pitched staging
    ((64, 130, 40), 3, 2, np.float32),      # P = 5200 > one slab
    ((60, 4, 3, 3, 2, 2), 3, 2, np.float64),    # 6-way X: 5-way covariance tensor (rank-1 ALS with 5 modes)
    ((50, 3, 3, 2, 2, 2, 2), 2, 2, np.float64),  # 7-way X: 6-way covariance tensor (wide index records)
])
def test_fit_matches_oracle_seeded(shape, M, R, dtype):
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import tPLS
    X, Y, _ = orc.synthetic(shape, M, 5, error=0.5, seed=215)
    X = X.astype(dtype)
    ref = orc.fit([X.copy()], Y.copy(), R, r2_mode="residual")
    est = tPLS(R)
    est.fit(X, Y)
    tol = FP32_TOL if dtype == np.float32 else FP64_TOL
    assert est.n_iter_.tolist() == ref["trips"].tolist()
    for k, e in aligned_errors(_state(est, False), ref).items():
        assert e < tol, (shape, k, e)


def test_masked_fit_matches_oracle_seeded():
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import tPLS
    rng = np.random.default_rng(3)
    for dtype in (np.float64, np.float32):
        X, Y, _ = orc.synthetic((600, 64, 32), 4, 8, error=0.5, seed=215)
        X[rng.random(X.shape) < 0.2] = np.nan
        X = X.astype(dtype)
        ref = orc.fit([X.copy()], Y.copy(), 3, r2_mode="residual")
        est = tPLS(3)
        est.fit(X, Y)
        assert est.X_hasMiss
        assert est.n_iter_.tolist() == ref["trips"].tolist()
        tol = FP32_TOL if dtype == np.float32 else FP64_TOL
        for k, e in aligned_errors(_state(est, False), ref).items():
            assert e < tol, (dtype, k, e)


def test_torch_cuda_input_is_used_in_place_and_not_modified():
    import torch
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import tPLS
    X, Y, _ = orc.synthetic((300, 16, 8), 3, 4, error=0.3, seed=1)
    ref = orc.fit([X.copy()], Y.copy(), 2, r2_mode="residual")
    Xd = torch.from_numpy(X).cuda()
    Yd = torch.from_numpy(Y).cuda()
    est = tPLS(2)
    est.fit(Xd, Yd)
    assert torch.equal(Xd.cpu(), torch.from_numpy(X))
    assert est.stats_["h2d_bytes"] == 0
    for k, e in aligned_errors(_state(est, False), ref).items():
        assert e < FP64_TOL, (k, e)
    # in-place variant: same numbers, X is consumed
    est2 = tPLS(2)
    est2.fit(Xd, Yd, overwrite_x=True)
    assert not torch.equal(Xd.cpu(), torch.from_numpy(X))
    assert np.array_equal(est2.X_factors[0], est.X_factors[0])


def test_large_shape_properties_fp32():
    """BASELINE-sized rows (P = 4096) at a sample count the oracle cannot follow:
    size-independent properties -- unit-norm loadings, monotone R2, the transform of
    the training data reproduces the scores, nested components."""
    import torch
    from cmtf_pls_b200 import ctPLS
    torch.manual_seed(0)
    n, L = 40000, 6
    T = torch.randn(n, L, dtype=torch.float64, device="cuda")
    A = [torch.randn(64, L, dtype=torch.float64, device="cuda") for _ in range(4)]
    yf = torch.randn(4, L, dtype=torch.float64, device="cuda")
    X0 = (torch.einsum("ir,jr,kr->ijk", T, A[0], A[1]) + torch.randn(n, 64, 64, dtype=torch.float64, device="cuda")).float()
    X1 = (torch.einsum("ir,jr,kr->ijk", T, A[2], A[3]) + torch.randn(n, 64, 64, dtype=torch.float64, device="cuda")).float()
    Y = T @ yf.T + 0.5 * torch.randn(n, 4, dtype=torch.float64, device="cuda")
    est = ctPLS(4)
    est.fit([X0, X1], Y)
    for fs in est.Xs_factors:
        for w in fs[1:]:
            np.testing.assert_allclose(np.linalg.norm(w, axis=0), 1.0, rtol=1e-7)
    np.testing.assert_allclose(np.linalg.norm(est.Y_factors[1], axis=0), 1.0, rtol=1e-7)
    assert np.all(np.diff(est.R2Y) >= 0) and np.all(np.diff(est.R2Xs[0]) >= 0) and np.all(np.diff(est.R2Xs[1]) >= 0)
    assert est.R2Y[-1] > 0.5
    s = est.transform([X0[:5000], X1[:5000]])
    assert col_err(s, est.factor_T[:5000]) < 1e-4
    est2 = ctPLS(2)
    est2.fit([X0, X1], Y)
    assert col_err(est2.factor_T, est.factor_T[:, :2]) < 1e-9
    assert est.stats_["alg_bytes"] > 0 and est.stats_["fit_ms"] > 0


# ---------------------------------------------------------------------------
# covariance mode (SURVEY.md §8f n4): same results, ~2.5 passes over X per component
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("case", [c for c in golden_cases() if "same_xy" not in c])
def test_covariance_mode_matches_reference_golden(case):
    from cmtf_pls_b200 import tPLS, ctPLS
    g = load_golden(case)
    R = int(g["n_components"])
    kw = {"max_iter": 4} if "maxiter" in case else {}
    if bool(g["coupled"]):
        est = ctPLS(R, algorithm="covariance")
        est.fit([x.copy() for x in g["Xs"]], g["Y"].copy(), **kw)
    else:
        est = tPLS(R, algorithm="covariance")
        est.fit(g["Xs"][0].copy(), g["Y"].copy(), **kw)
    M = 1 if g["Y"].ndim == 1 else g["Y"].shape[1]
    expect_cov = M <= 8 and not (M > 4 and any(np.isnan(x).any() for x in g["Xs"]))
    assert bool(est.stats_["covariance_mode"]) == expect_cov
    tol = FP32_TOL if "f32" in case else FP64_TOL
    assert est.n_iter_.tolist() == g["trips"].tolist()
    for k, e in aligned_errors(_state(est, bool(g["coupled"])), g).items():
        assert e < tol, (case, k, e)


def test_covariance_mode_streams_far_fewer_bytes():
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import tPLS
    X, Y, _ = orc.synthetic((2000, 64, 64), 4, 6, error=0.7, seed=3)
    X = X.astype(np.float32)
    a = tPLS(4)
    a.fit(X, Y)
    b = tPLS(4, algorithm="covariance")
    b.fit(X, Y)
    assert b.stats_["covariance_mode"] == 1 and a.stats_["covariance_mode"] == 0
    assert a.n_iter_.tolist() == b.n_iter_.tolist()
    assert b.stats_["streamed_bytes"] < 0.25 * a.stats_["streamed_bytes"]
    for k, e in aligned_errors(_state(b, False), _state(a, False) | {"R2X": [a.R2X]}).items():
        assert e < 1e-7, (k, e)


def test_transform_paths_agree_and_complete_data_is_read_in_place():
    """Complete new data takes the read-only path (R projections + the score recurrence); the same data with a
    single NaN takes the sequential masked path; both must agree with each other and with the oracle."""
    import torch
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import ctPLS, _core
    Xs, Y, _ = orc.synthetic((300, 16, 8), 3, 4, error=0.4, seed=12, extra_dims=[(300, 20)])
    est = ctPLS(4)
    est.fit(Xs, Y)
    ref = orc.fit([x.copy() for x in Xs], Y.copy(), 4, r2_mode="residual")
    Xn, _, _ = orc.synthetic((50, 16, 8), 3, 4, error=0.4, seed=13, extra_dims=[(50, 20)])
    want = orc.transform(ref, [x.copy() for x in Xn])
    Xd = [torch.from_numpy(x).cuda() for x in Xn]
    got = est.transform(Xd)
    eng = _core.get_engine(0)
    assert eng.stats()["last_transform_path"] == 1
    for a, b in zip(Xd, Xn):
        assert torch.equal(a.cpu(), torch.from_numpy(b))          # never written
    assert col_err(got, want) < FP64_TOL
    Xm = [x.copy() for x in Xn]
    Xm[0][3, 2, 1] = np.nan
    got_m = est.transform(Xm)
    assert eng.stats()["last_transform_path"] == 2
    want_m = orc.transform(ref, [x.copy() for x in Xm])
    assert col_err(got_m, want_m) < FP64_TOL
    keep = np.arange(50) != 3
    assert col_err(got_m[keep], got[keep]) < FP64_TOL


def test_pickle_roundtrip_and_convergence_flags():
    import pickle
    g = load_golden("t4_maxiter_20x6x5x4_m5_r2")
    from cmtf_pls_b200 import tPLS
    est = tPLS(2)
    est.fit(g["Xs"][0].copy(), g["Y"].copy(), max_iter=4)
    assert est.n_iter_.tolist() == [4, 4] and not est.converged_.any()      # silent in the reference (tpls.py:79-107)
    est.fit(g["Xs"][0].copy(), g["Y"].copy())
    assert est.converged_.all()
    clone = pickle.loads(pickle.dumps(est))
    assert not hasattr(clone, "_X_ref")
    Xn = g["Xs"][0][:5].copy()
    assert np.array_equal(clone.predict(Xn), est.predict(Xn))


def test_all_missing_row_gives_nan_score_like_the_reference():
    """missingvals.py:37 divides by the number of observed entries of the row: 0/0 -> NaN, unguarded."""
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import tPLS
    X, Y, _ = orc.synthetic((40, 6, 5), 2, 3, error=0.3, seed=2)
    est = tPLS(2)
    est.fit(X, Y)
    Xn = X[:6].copy()
    Xn[2] = np.nan
    Xn[4, 1, 1] = np.nan
    s = est.transform(Xn)
    assert np.isnan(s[2]).all() and np.isfinite(np.delete(s, 2, axis=0)).all()
    ref = orc.fit([X.copy()], Y.copy(), 2, r2_mode="residual")
    want = orc.transform(ref, [Xn.copy()])
    keep = np.arange(6) != 2
    assert col_err(s[keep], want[keep]) < FP64_TOL


# ---------------------------------------------------------------------------
# SURVEY.md §8f n2: single-pass multi-component projection (fp64 tensor-core path) and device reconstruction
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("shape,extra,R,dtype", [((700, 64, 64), [], 10, np.float32), ((333, 33, 17), [(333, 24)], 12, np.float64),
                                                 ((120, 40), [], 3, np.float64), ((90, 8, 6, 4), [(90, 50, 3)], 17, np.float32),
                                                 ((64, 70, 30), [], 30, np.float64)])
def test_single_pass_transform_matches_sequential_and_oracle(shape, extra, R, dtype):
    """One read of X with R accumulators per row (multiproj.cu) == the per-component project/deflate sequence."""
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import ctPLS, _core
    Xs, Y, _ = orc.synthetic(shape, 3, 5, error=0.5, seed=21, extra_dims=extra)
    Xs = [x.astype(dtype) for x in (Xs if extra else [Xs])]
    est = ctPLS(R)
    est.fit(Xs, Y, max_iter=30)
    Xn, _, _ = orc.synthetic((77,) + shape[1:], 3, 5, error=0.5, seed=22, extra_dims=[(77,) + e[1:] for e in extra])
    Xn = [x.astype(dtype) for x in (Xn if extra else [Xn])]
    eng = _core.get_engine(0)
    got = est.transform(Xn)
    st = eng.stats()
    assert st["last_transform_path"] == 1
    assert st["kernel_launches"] == len(Xs) + 1          # one pass per tensor + the finishing kernel
    # the sequential path on the same rows: a NaN in a pad row forces it, the other rows must agree
    Xm = [np.concatenate([x, x[:1]]) for x in Xn]
    Xm[0][-1].reshape(-1)[0] = np.nan
    seq = est.transform(Xm)[:-1]
    assert eng.stats()["last_transform_path"] == 2
    tol = FP32_TOL if dtype == np.float32 else FP64_TOL
    assert col_err(got, seq) < tol
    if R <= 12:   # and the oracle's transform through its own refit (later components of an over-fitted model are noise)
        ref = orc.fit([x.copy() for x in Xs], Y.copy(), R, max_iter=30, r2_mode="residual")
        want = orc.transform(ref, [x.copy() for x in Xn])
        assert col_err(got[:, :3], want[:, :3]) < tol


def test_transform_of_training_rows_reproduces_scores_config4_shape():
    import torch
    from cmtf_pls_b200 import ctPLS
    torch.manual_seed(1)
    n = 20000
    T = torch.randn(n, 5, dtype=torch.float64, device="cuda")
    X0 = (T @ torch.randn(5, 4096, dtype=torch.float64, device="cuda") + torch.randn(n, 4096, dtype=torch.float64, device="cuda")).float().reshape(n, 64, 64)
    X1 = (T @ torch.randn(5, 4096, dtype=torch.float64, device="cuda") + torch.randn(n, 4096, dtype=torch.float64, device="cuda")).float().reshape(n, 64, 64)
    Y = T @ torch.randn(5, 4, dtype=torch.float64, device="cuda")
    est = ctPLS(10)
    est.fit([X0, X1], Y)
    s = est.transform([X0, X1])
    assert col_err(s[:, :5], est.factor_T[:, :5]) < 1e-4


@pytest.mark.parametrize("case", ["t3_60x16x12_m4_r5", "ct_90x32x16_90x24_m4_r5", "t4_miss_f32_50x6x5x4_m3_r3", "t2_50x12_m1_r3"])
def test_device_reconstruction_matches_numpy(case):
    """X_reconstructed (tpls.py:188-189): factors_to_tensor(X_factors) + X_mean, formed by the device writer."""
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import tPLS, ctPLS
    g = load_golden(case)
    R = int(g["n_components"])
    if bool(g["coupled"]):
        est = ctPLS(R)
        est.fit([x.copy() for x in g["Xs"]], g["Y"].copy())
        got, facs, means = est.Xs_reconstructed(), est.Xs_factors, est.Xs_mean
    else:
        est = tPLS(R)
        est.fit(g["Xs"][0].copy(), g["Y"].copy())
        got, facs, means = [est.X_reconstructed()], [est.X_factors], [est.X_mean]
    for xr, f, mu, x in zip(got, facs, means, g["Xs"]):
        want = orc.rank_r_tensor(f) + mu
        assert xr.shape == x.shape and xr.dtype == np.float64
        assert np.max(np.abs(xr - want)) <= 1e-12 * max(1.0, np.max(np.abs(want)))


def test_stop_test_met_on_the_last_allowed_trip_counts_as_converged():
    """ADVICE r1: trips == max_iter does not mean 'not converged'."""
    from cmtf_pls_b200 import tPLS
    g = load_golden("t3_60x16x12_m4_r5")
    est = tPLS(2)
    est.fit(g["Xs"][0].copy(), g["Y"].copy())
    k = int(est.n_iter_[0])
    assert est.converged_.all() and k >= 2
    est2 = tPLS(2)
    est2.fit(g["Xs"][0].copy(), g["Y"].copy(), max_iter=k)      # component 0 meets the test exactly on its last trip
    assert int(est2.n_iter_[0]) == k and bool(est2.converged_[0])
    est3 = tPLS(2)
    est3.fit(g["Xs"][0].copy(), g["Y"].copy(), max_iter=k - 1)
    assert int(est3.n_iter_[0]) == k - 1 and not bool(est3.converged_[0])


def test_fit_runs_as_one_graph_and_reports_its_launches(monkeypatch):
    """The streaming fit is ONE CUDA-graph launch (a WHILE node per component); 3 + 2 L kernels per inner trip."""
    import os
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import ctPLS
    monkeypatch.setenv("TPLS_RESIDENT", "0")         # the streaming kernels, whatever the size (read at every fit)
    Xs, Y, _ = orc.synthetic((400, 16, 8), 3, 4, error=0.4, seed=3, extra_dims=[(400, 20)])
    est = ctPLS(3)
    est.fit(Xs, Y)
    st = est.stats_
    assert st["launches_per_trip"] == 3 + 2 * 2 and st["resident_loops"] == 0
    if os.environ.get("TPLS_NO_GRAPH") is None:
        assert st["graph_launches"] == 1
    first = (est.n_iter_.tolist(), est.factor_T.copy())
    est.fit(Xs, Y)                                   # same key: the instantiated graph is relaunched
    assert est.n_iter_.tolist() == first[0] and np.array_equal(est.factor_T, first[1])
    est.fit(Xs, Y, profile=True)                     # host-enqueued trips, same kernels, same numbers
    assert est.stats_["graph_launches"] == 0
    assert est.n_iter_.tolist() == first[0] and np.array_equal(est.factor_T, first[1])
    ref = orc.fit([x.copy() for x in Xs], Y.copy(), 3, r2_mode="residual")
    assert est.n_iter_.tolist() == ref["trips"].tolist()


@pytest.mark.parametrize("case", ["ct_90x32x16_90x24_m4_r5", "t3_miss_70x12x8_m4_r4", "t4_60x8x6x4_m3_r4", "t3_f32_80x16x8_m4_r4"])
def test_resident_trip_loop_matches_the_streaming_kernels(case, monkeypatch):
    """Working sets that stay in L2 run ALL inner trips of a component in one persistent launch (one CTA per SM, grid
    barriers between the phases of a trip; rank1.cuh `ResidentArgs`).  Same trips, same model as the streaming kernels
    (different summation order: 1e-10), one launch per component; profiled fits keep the streaming kernels."""
    from cmtf_pls_b200 import ctPLS
    g = load_golden(case)
    R = int(g["n_components"])
    fits = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("TPLS_RESIDENT", mode)
        est = ctPLS(R)
        est.fit([x.copy() for x in g["Xs"]], g["Y"].copy())
        fits[mode] = est
        assert est.stats_["resident_loops"] == (R if mode == "1" else 0)
        assert est.n_iter_.tolist() == g["trips"].tolist()
    a, b = fits["1"], fits["0"]
    assert a.stats_["kernel_launches"] < b.stats_["kernel_launches"]
    assert np.max(np.abs(a.factor_T - b.factor_T)) < 1e-10 * max(1.0, np.max(np.abs(b.factor_T)))
    assert np.max(np.abs(a.coef_ - b.coef_)) < 1e-10 and np.max(np.abs(a.R2Y - b.R2Y)) < 1e-12
    for l in range(len(g["Xs"])):
        assert np.max(np.abs(a.R2Xs[l] - b.R2Xs[l])) < 1e-12
    monkeypatch.delenv("TPLS_RESIDENT")
    est = ctPLS(R)
    est.fit([x.copy() for x in g["Xs"]], g["Y"].copy())          # small enough: resident by default
    assert est.stats_["resident_loops"] == R
    est.fit([x.copy() for x in g["Xs"]], g["Y"].copy(), profile=True)
    assert est.stats_["resident_loops"] == 0 and est.n_iter_.tolist() == g["trips"].tolist()


@pytest.mark.parametrize("dtype,nan_frac", [(np.float64, 0.0), (np.float32, 0.15)])
def test_resident_trip_loop_with_a_partly_cached_block(dtype, nan_frac, monkeypatch):
    """Blocks of rows too large for shared memory: the first rows of every CTA's block are read from its shared-memory
    cache, the rest from L2, in both passes of a trip (rank1.cuh).  Same trips and the same model as the streaming
    kernels, complete and masked, coupled with a narrow second tensor."""
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import ctPLS
    Xs, Y, _ = orc.synthetic((6000, 32, 32), 3, 4, error=0.5, seed=11, extra_dims=[(6000, 20)])
    Xs = [x.astype(dtype) for x in Xs]
    if nan_frac:
        rng = np.random.default_rng(5)
        for x in Xs:
            x[rng.random(x.shape) < nan_frac] = np.nan
    fits = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("TPLS_RESIDENT", mode)
        est = ctPLS(3)
        est.fit([x.copy() for x in Xs], Y.copy())
        fits[mode] = est
        assert est.stats_["resident_loops"] == (3 if mode == "1" else 0)
    a, b = fits["1"], fits["0"]
    tol = 1e-10 if dtype == np.float64 else 1e-9     # fp64 arithmetic on the same stored values either way
    assert a.n_iter_.tolist() == b.n_iter_.tolist()
    assert np.max(np.abs(a.factor_T - b.factor_T)) < tol * max(1.0, np.max(np.abs(b.factor_T)))
    assert np.max(np.abs(a.coef_ - b.coef_)) < tol and np.max(np.abs(a.R2Y - b.R2Y)) < 1e-10


def test_tall_narrow_blocks_keep_the_streaming_kernels_and_agree_with_the_forced_resident_loop(monkeypatch):
    """200k rows of 24 columns: a CTA's block is 1352 rows of which ~870 fit in shared memory -- too many rows left in
    L2 for a warp per row, so the fit keeps the streaming kernels by default (driver.cu: resident_ctas).  Forced, the
    resident loop walks its block in two chunks of u = Y q (rank1.cu: kResidentUChunk) and must give the same fit."""
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import tPLS
    X, Y, _ = orc.synthetic((200_000, 6, 4), 3, 4, error=0.5, seed=5)
    fits = {}
    for mode in (None, "1"):
        if mode is None:
            monkeypatch.delenv("TPLS_RESIDENT", raising=False)
        else:
            monkeypatch.setenv("TPLS_RESIDENT", mode)
        est = tPLS(3)
        est.fit(X.copy(), Y.copy())
        fits[mode] = est
        assert est.stats_["resident_loops"] == (0 if mode is None else 3)
    a, b = fits["1"], fits[None]
    assert a.n_iter_.tolist() == b.n_iter_.tolist()
    assert np.max(np.abs(a.X_factors[0] - b.X_factors[0])) < 1e-10 * max(1.0, np.max(np.abs(b.X_factors[0])))
    assert np.max(np.abs(a.coef_ - b.coef_)) < 1e-10 and np.max(np.abs(a.R2Y - b.R2Y)) < 1e-10


@pytest.mark.parametrize("env", [{"TPLS_NO_GRAPH": "1"}, {"TPLS_PDL": "0"}, {"TPLS_NO_GRAPH": "1", "TPLS_PDL": "0"},
                                 {"TPLS_NO_GRAPH": "1", "TPLS_RESIDENT": "0"}, {"TPLS_PDL": "0", "TPLS_RESIDENT": "0"},
                                 {"TPLS_NO_GRAPH": "1", "TPLS_PDL": "0", "TPLS_RESIDENT": "0"}])
def test_host_enqueued_and_plain_launch_paths_give_the_same_fit(env, tmp_path, monkeypatch):
    """The graph-launched fit (default), the host-enqueued trips (profiling / NCCL fallback) and launches without the
    PDL attribute run the same kernels: bit-identical results.  The switches are read once per process, so the
    variants run in a subprocess."""
    import os
    import subprocess
    import sys
    from cmtf_pls_b200 import ctPLS
    g = load_golden("ct_90x32x16_90x24_m4_r5")
    if "TPLS_RESIDENT" in env:      # (read at every fit) the streaming trip body in both processes
        monkeypatch.setenv("TPLS_RESIDENT", env["TPLS_RESIDENT"])
    est = ctPLS(5)
    est.fit([x.copy() for x in g["Xs"]], g["Y"].copy())
    assert (est.stats_["resident_loops"] == 0) == ("TPLS_RESIDENT" in env)
    out = str(tmp_path / "variant.npz")
    code = (
        "import sys, numpy as np\n"
        f"sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {os.path.join(ROOT, 'tests')!r})\n"
        "from _util import load_golden\n"
        "from cmtf_pls_b200 import ctPLS\n"
        "g = load_golden('ct_90x32x16_90x24_m4_r5')\n"
        "est = ctPLS(5)\n"
        "est.fit([x.copy() for x in g['Xs']], g['Y'].copy())\n"
        f"np.savez({out!r}, T=est.factor_T, coef=est.coef_, trips=est.n_iter_, graph=np.array(est.stats_['graph_launches']))\n"
    )
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    v = np.load(out)
    assert v["trips"].tolist() == est.n_iter_.tolist() == g["trips"].tolist()
    assert int(v["graph"]) == (0 if "TPLS_NO_GRAPH" in env else 1)
    assert np.array_equal(v["T"], est.factor_T) and np.array_equal(v["coef"], est.coef_)


# ---------------------------------------------------------------------------
# transform and reconstruction at sizes where the rings of multiproj_kernel and the reconstruction's bounce buffers
# cycle, against the oracle / numpy on a random model (unit-norm loadings, a mean of order 1, data = mean + noise)
# ---------------------------------------------------------------------------
def _random_model(shapes, R, dtypes, seed):
    rng = np.random.default_rng(seed)
    Xs, means, loadings = [], [], []
    for shape, dt in zip(shapes, dtypes):
        ws = [rng.normal(size=(d, R)) for d in shape[1:]]
        loadings.append([w / np.linalg.norm(w, axis=0) for w in ws])
        mu = rng.normal(size=shape[1:]).astype(dt)
        means.append(mu)
        Xs.append((mu + rng.normal(size=shape)).astype(dt))
    return Xs, means, loadings


# multiproj_kernel (multiproj.cu): 16-row tiles through a 3-stage ring, one CTA per (row block, column slab) with
# 148 / n_slabs CTAs per slab.  40001 rows = 2501 tiles, the last one 1 row, so CTAs run different numbers of laps.
_TRANSFORM_CASES = [
    # (64, 64) fp32: NB = 1, 2 -> 8 slabs of 512, 18 CTAs per slab x 138-139 tiles = 46-47 laps
    ([(40001, 64, 64)], 3, [np.float32]),
    ([(40001, 64, 64)], 10, [np.float32]),
    # NB = 3, 4 -> half-width slabs: 16 slabs of 256, 9 CTAs per slab x 277-278 tiles
    ([(40001, 64, 64)], 17, [np.float32]),
    ([(40001, 64, 64)], 32, [np.float32]),
    # fp64, NB = 2: 16 slabs of 256 columns, 9 CTAs per slab
    ([(40001, 64, 64)], 10, [np.float64]),
    # P = 5200: 11 slabs, the last one 80 columns wide, 13 CTAs per slab x 192-193 tiles
    ([(40001, 130, 40)], 10, [np.float32]),
    # odd P = 561 in fp64: pitched staging copy (pitch 562), 3 slabs (256, 256, 50), 49 CTAs per slab x 51-52 tiles
    ([(40001, 33, 17)], 5, [np.float64]),
    # a coupled pair with different P: 8 slabs + 1 slab (148 CTAs x 16-17 tiles), both summed by multiproj_finish
    ([(40001, 64, 64), (40001, 24, 20)], 10, [np.float32, np.float32]),
]


@pytest.mark.parametrize("shapes,R,dtypes", _TRANSFORM_CASES)
def test_transform_at_size_matches_oracle(shapes, R, dtypes):
    """Complete data: the single-pass path (all R projections in one read of X, then the score recurrence) computes
    in fp64 on the stored values and never rounds a deflated value -> 1e-10 per column against the oracle's sequential
    project/deflate in fp64, for host input and for torch CUDA input read in place.  With one NaN in the last tile
    and one all-NaN row the sequential masked path runs instead (deflated values rounded to the stored dtype)."""
    import torch
    from oracle import tpls_oracle as orc
    from cmtf_pls_b200 import _core
    Xs, means, loadings = _random_model(shapes, R, dtypes, seed=sum(s[1] for s in shapes) + R)
    state = {"T": np.empty((0, R)), "X_mean": [m.astype(np.float64) for m in means], "W": loadings}
    want = orc.transform(state, [x.astype(np.float64) for x in Xs])
    eng = _core.get_engine(0)
    for kind in ("host", "cuda"):
        arg = Xs if kind == "host" else [torch.from_numpy(x).cuda() for x in Xs]
        got = _core.run_transform(arg, means, loadings, R)
        assert eng.stats()["last_transform_path"] == 1, kind
        assert col_err(got, want) < 1e-10, (kind, col_err(got, want))
        del arg
    del want
    n = shapes[0][0]
    Xm = [x.copy() for x in Xs]
    del Xs
    Xm[-1][n - 1].reshape(-1)[-1] = np.nan        # one NaN in the last row (the 1-row last tile)
    Xm[0][n // 2] = np.nan                        # one row entirely NaN: NaN scores, like the reference
    got = _core.run_transform(Xm, means, loadings, R)
    assert eng.stats()["last_transform_path"] == 2
    want = orc.transform(dict(state, X_mean=means), Xm)         # on the stored dtype, as the masked path computes
    assert np.array_equal(np.isnan(got), np.isnan(want))
    assert np.isnan(got[n // 2]).all() and np.isnan(got).sum() == R
    keep = ~np.isnan(want[:, 0])
    tol = FP32_TOL if np.float32 in dtypes else FP64_TOL
    assert col_err(got[keep], want[keep]) < tol


# tpls_reconstruct with a host result: blocks of 32 MiB / (8 p) rows through two device blocks and two pinned bounce
# buffers.  n = 5000, p = 4096: 1024-row blocks, 5 of them, the last 904 rows, so both buffers cycle; p = 5200: 806-row
# blocks, 7 of them, the last 164 rows.
@pytest.mark.parametrize("p", [4096, 5200])
@pytest.mark.parametrize("R", [1, 32])
@pytest.mark.parametrize("mean_dtype", [np.float32, np.float64])
def test_reconstruct_host_blocks_match_numpy(p, R, mean_dtype):
    import torch
    from cmtf_pls_b200 import _core
    from cmtf_pls_b200._engine import dtype_code
    rng = np.random.default_rng(p + R)
    n = 5000
    scores = rng.normal(size=(n, R))
    wkron = rng.normal(size=(R, p)) / np.sqrt(p)
    mean = rng.normal(size=p).astype(mean_dtype)
    eng = _core.get_engine(0)
    got = eng.reconstruct(scores, wkron, mean)
    want = scores @ wkron + mean.astype(np.float64)
    assert got.shape == (n, p) and np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want))
    # the device-result branch (one launch over all rows) computes every element the same way: bit for bit
    out = torch.empty((n, p), dtype=torch.float64, device="cuda")
    eng._ck(eng.lib.tpls_reconstruct(eng.h, R, scores.ctypes.data, n, p, wkron.ctypes.data, mean.ctypes.data,
                                     dtype_code(mean), out.data_ptr()))
    assert np.array_equal(out.cpu().numpy(), got)

