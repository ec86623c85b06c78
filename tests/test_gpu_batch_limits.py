"""GPU: the batch kernel (``fit_batch``, csrc/batch.cu) at the edges of its limits, against the oracle.

Each case fits 3 or 4 seeded problems in one launch and compares every problem with ``orc.fit(...,
r2_mode="residual")``: equal trip counts, and 1e-8 (fp64 storage) / 1e-4 (fp32) on T, W, U, Q, coef, R2X and R2Y after
sign alignment.  Just past a limit the problems must be fitted one by one ("loop") with the same results.  Every
case that runs the kernel runs again with its working set in global memory (``TPLS_BATCH_SMEM=0``): placement changes
only where the working set lives, not one operation on it, so the outputs of the two runs must be bit-identical.

What each case reaches:
  * M = 6, 7, 8: Y'Y fills ``gy_s[64]`` and its column reduce is up to 64 wide; M = 9 is past ``kBatchMaxResp``.
  * R = 32 (``kBatchMaxComp``): the Gram / Cholesky of solve_coef at full size.  R = 33 is past the ordinary fit's
    limit too, so there is no loop to fall back on: ``fit_batch`` raises that fit's error.
  * p = 513 and p = 1056: a second (and third) column chunk of ``col_reduce`` with a partial last chunk, and the lane
    loop of the projection with lanes that run one element more than others.
  * n = 5 rows: fewer rows than ``col_reduce``'s row groups, most of which get none.
  * L = 3, 5, 8 coupled tensors (8 = ``kMaxTensors``): averages over a non-power-of-2 L, fp32 and fp64 mixed, one
    masked tensor among dense ones (the masked / dense split of the projection), one tensor broadcast with batch
    stride 0.
  * an 8-way X: a 7-mode covariance tensor (``kMaxZModes``).
  * ``TPLS_BATCH_MB=1``: working sets of about 0.8 MB (kernel) and 1.2 MB (loop), from batch_driver.cu's layout.

The stop quantity ||u_old - u|| of every oracle trip of these inputs stays at least 5 % away from tol = 1e-8, and
3.6 % for R = 32, whose components take 4 to 59 trips, so equal trip counts test the kernel, not rounding.  (Measured
by recording that norm at every trip of ``orc.fit``, line ``if np.linalg.norm(old_u - U[:, a]) < tol``; rerun it when
a seed or shape changes.)  Each oracle fit runs once per module.

The oracle's coef comes from ``lstsq`` on the zero-padded (N, R) score matrix, which can put rounding noise (up to
1e15 for R = 32) into the rows of the components not yet computed, below the diagonal.  Those entries are 0 by
definition (the fit's coef is upper triangular, as the kernel writes it), so the comparison takes the oracle's upper
triangle.
"""

import numpy as np
import pytest

from _util import aligned_errors

pytestmark = pytest.mark.gpu

FP64_TOL = 1e-8
FP32_TOL = 1e-4
F32, F64 = np.float32, np.float64

# name: (tensors [(dims, dtype, masked, broadcast)], responses M, components R, latent factors, problems B,
#        environment, expected path)
_COUPLED_DIMS = [(40, 6, 5), (40, 7), (40, 4, 3, 2), (40, 9), (40, 5, 4), (40, 8), (40, 3, 3, 3), (40, 6)]


def _coupled(L):
    # tensor 1 masked, tensor 2 broadcast over the batch, fp64 and fp32 alternating
    return [(_COUPLED_DIMS[l], F64 if l % 2 == 0 else F32, l == 1, l == 2) for l in range(L)]


CASES = {
    "m6": ([((40, 8, 6), F64, False, False)], 6, 3, 4, 3, {}, "kernel"),
    "m7": ([((40, 8, 6), F64, False, False)], 7, 3, 4, 3, {}, "kernel"),
    "m8": ([((40, 8, 6), F64, False, False)], 8, 3, 4, 3, {}, "kernel"),
    "m6_masked": ([((40, 8, 6), F64, True, False)], 6, 3, 4, 3, {}, "kernel"),
    "m7_masked": ([((40, 8, 6), F64, True, False)], 7, 3, 4, 3, {}, "kernel"),
    "m8_masked": ([((40, 8, 6), F64, True, False)], 8, 3, 4, 3, {}, "kernel"),
    "m9": ([((40, 8, 6), F64, False, False)], 9, 3, 4, 3, {}, "loop"),
    "r32": ([((200, 10, 8), F64, False, False)], 2, 32, 32, 3, {}, "kernel"),
    "r33": ([((200, 10, 8), F64, False, False)], 2, 33, 32, 3, {}, "error"),
    "p513_f64": ([((60, 9, 57), F64, False, False)], 2, 3, 3, 3, {}, "kernel"),
    "p513_f32": ([((60, 9, 57), F32, False, False)], 2, 3, 3, 3, {}, "kernel"),
    "p513_f64_masked": ([((60, 9, 57), F64, True, False)], 2, 3, 3, 3, {}, "kernel"),
    "p513_f32_masked": ([((60, 9, 57), F32, True, False)], 2, 3, 3, 3, {}, "kernel"),
    "p1056_f64": ([((40, 33, 32), F64, False, False)], 2, 3, 3, 3, {}, "kernel"),
    "p1056_f32": ([((40, 33, 32), F32, False, False)], 2, 3, 3, 3, {}, "kernel"),
    "p1056_f64_masked": ([((40, 33, 32), F64, True, False)], 2, 3, 3, 3, {}, "kernel"),
    "p1056_f32_masked": ([((40, 33, 32), F32, True, False)], 2, 3, 3, 3, {}, "kernel"),
    "n5": ([((5, 2, 3), F64, False, False)], 1, 2, 2, 4, {}, "kernel"),
    "n5_masked": ([((5, 2, 3), F64, True, False)], 1, 2, 2, 4, {}, "kernel"),
    "coupled3": (_coupled(3), 2, 3, 3, 3, {}, "kernel"),
    "coupled5": (_coupled(5), 2, 3, 3, 3, {}, "kernel"),
    "coupled8": (_coupled(8), 2, 3, 3, 3, {}, "kernel"),
    "way8": ([((20, 2, 2, 2, 2, 2, 2, 2), F64, False, False)], 1, 2, 2, 3, {}, "kernel"),
    # TPLS_BATCH_MB=1 (1 048 576 bytes): X alone is 800 000 bytes of (400, 25, 10) and 1 200 000 of (400, 25, 15) fp64;
    # see _ws_bytes for the whole working set
    "mb1_small": ([((400, 25, 10), F64, False, False)], 2, 3, 3, 3, {"TPLS_BATCH_MB": "1"}, "kernel"),
    "mb1_large": ([((400, 25, 15), F64, False, False)], 2, 3, 3, 3, {"TPLS_BATCH_MB": "1"}, "loop"),
}

# first seed of each case (problem b takes seed + b) or the seed of each problem, chosen for the stop-quantity margin
# above; 100 where not listed
SEED = {"r32": (10, 44, 51), "r33": (10, 44, 51), "m8": 114, "m6_masked": 121, "m7_masked": 107, "m8_masked": 107,
        "m9": 121, "p1056_f64_masked": 107, "p1056_f32_masked": 107, "coupled3": 107, "coupled5": 114}


def case_data(name):
    """(Xs per problem, Y per problem) of a case: orc.synthetic(..., error=0.3; 0.05 for the 32 latent factors of
    R = 32 / 33) with one seed per problem; masked tensors get 10 % NaNs; a broadcast tensor is problem 0's for every
    problem."""
    from oracle import tpls_oracle as orc
    tensors, M, R, latent, B, _, _ = CASES[name]
    seed = SEED.get(name, 100)
    seeds = list(seed) if isinstance(seed, tuple) else [seed + b for b in range(B)]
    probs, Ys = [], []
    for b in range(B):
        X, Y, _ = orc.synthetic(tensors[0][0], M, latent, error=0.05 if latent == 32 else 0.3, seed=seeds[b],
                                extra_dims=[t[0] for t in tensors[1:]])
        Xs = list(X) if len(tensors) > 1 else [X]
        rng = np.random.default_rng(seeds[b])
        for l, (_, dtype, masked, _) in enumerate(tensors):
            if masked:
                Xs[l][rng.random(Xs[l].shape) < 0.1] = np.nan
            Xs[l] = Xs[l].astype(dtype)
        probs.append(Xs)
        Ys.append(Y)
    for l, (_, _, _, bc) in enumerate(tensors):
        if bc:
            for Xs in probs:
                Xs[l] = probs[0][l]
    return probs, Ys


_refs = {}


@pytest.fixture(scope="module")
def oracle_fits():
    """Oracle fits of a case's problems, computed on first use and kept for the module."""
    from oracle import tpls_oracle as orc

    def get(name):
        if name not in _refs:
            probs, Ys = case_data(name)
            R = CASES[name][2]
            _refs[name] = [orc.fit([x.astype(np.float64) for x in Xs], Y.copy(), R, r2_mode="residual")
                           for Xs, Y in zip(probs, Ys)]
        return _refs[name]
    yield get
    _refs.clear()


def _fit(name, env, monkeypatch):
    from cmtf_pls_b200 import fit_batch
    tensors, M, R, _, _, case_env, _ = CASES[name]
    probs, Ys = case_data(name)
    for k in ("TPLS_BATCH_MB", "TPLS_BATCH_SMEM", "TPLS_BATCH"):
        monkeypatch.delenv(k, raising=False)
    for k, v in {**case_env, **env}.items():
        monkeypatch.setenv(k, v)                       # read at every call
    Xb = [np.stack([p[l] for p in (probs[:1] if bc else probs)]) for l, (_, _, _, bc) in enumerate(tensors)]
    assert all(x.shape[0] == (1 if t[3] else len(probs)) for x, t in zip(Xb, tensors))
    return fit_batch(Xb if len(tensors) > 1 else Xb[0], np.stack(Ys), R)


def _state(est):
    if hasattr(est, "Xs_factors"):
        return dict(T=est.factor_T, W=[f[1:] for f in est.Xs_factors], U=est.Y_factors[0], Q=est.Y_factors[1],
                    coef=est.coef_, R2X=est.R2Xs, R2Y=est.R2Y, trips=est.n_iter_)
    return dict(T=est.X_factors[0], W=[est.X_factors[1:]], U=est.Y_factors[0], Q=est.Y_factors[1],
                coef=est.coef_, R2X=[est.R2X], R2Y=est.R2Y, trips=est.n_iter_)


def _flat(st):
    return [st["T"], st["U"], st["Q"], st["coef"], st["R2Y"], st["trips"]] + list(st["R2X"]) + \
        [w for ws in st["W"] for w in ws]


@pytest.mark.parametrize("name", list(CASES))
def test_batch_kernel_limits_match_oracle(oracle_fits, name, monkeypatch):
    from cmtf_pls_b200._engine import TplsError
    tensors, _, _, _, B, _, path = CASES[name]
    if path == "error":
        with pytest.raises(TplsError, match="n_components must be 1..32"):
            _fit(name, {}, monkeypatch)
        return
    refs = oracle_fits(name)
    tol = FP32_TOL if any(t[1] == F32 for t in tensors) else FP64_TOL
    models = _fit(name, {}, monkeypatch)
    assert len(models) == B
    for b, (est, ref) in enumerate(zip(models, refs)):
        assert est.stats_["batch"] == path
        assert est.n_iter_.tolist() == ref["trips"].tolist(), b
        errs = aligned_errors(_state(est), dict(ref, coef=np.triu(ref["coef"])))
        assert max(errs.values()) < tol, f"problem {b}: {errs}"
    if path == "kernel":
        # the same problems with the working sets in global memory: bit-identical
        again = _fit(name, {"TPLS_BATCH_SMEM": "0"}, monkeypatch)
        for est, other in zip(models, again):
            assert other.stats_["batch"] == "kernel"
            for x, y in zip(_flat(_state(est)), _flat(_state(other))):
                np.testing.assert_array_equal(np.asarray(x), np.asarray(y))


def _ws_bytes(name):
    """Per-problem working set of a one-tensor case as batch_driver.cu lays it out, without the rank-1 workspace
    (a few KB for these covariance matrices)."""
    (dims, dtype, _, _), = CASES[name][0]
    up16 = lambda b: (b + 15) // 16 * 16
    n, p, M, R = dims[0], int(np.prod(dims[1:])), CASES[name][1], CASES[name][2]
    elem = np.dtype(dtype).itemsize
    tensor = up16(n * p * elem) + 4 * up16(p * 8) + up16(sum(dims[1:]) * 8) + up16(n * 8)
    return tensor + up16(n * M * 8) + up16(n * R * 8) + up16(n * 8)


def test_batch_mb_cases_straddle_the_limit():
    assert 0.75 * 2 ** 20 < _ws_bytes("mb1_small") < 0.85 * 2 ** 20
    assert 1.1 * 2 ** 20 < _ws_bytes("mb1_large") < 1.2 * 2 ** 20
