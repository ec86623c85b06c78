"""GPU: whole fits at N = 20 000 against the oracle (oracle/tpls_oracle.py) -- sizes at which the rings of the
streaming kernels wrap many times per pass and the resident loop leaves most rows of its block outside shared memory,
through every inner loop a fit can take: the streaming kernels (Y side fused into the X passes or in passes of its
own), the resident trip loop and the covariance mode.

Each oracle fit runs once per module (it takes 20-60 s on a CPU); every GPU variant of the case is compared with it:
equal trip counts, and 1e-8 (fp64 storage) / 1e-4 (fp32 storage) on T, W, U, Q, coef, R2X and R2Y after sign
alignment.  Every variant also asserts the path it took.

The stop quantity ||u_old - u|| of every oracle trip of these inputs stays more than 1 % away from tol = 1e-8 (closest:
0.954 tol on trip 13 of c5's second component, 0.942 tol on the 83rd and last trip of c3's third), so equal trip counts
test the kernels, not rounding.  Oracle trips: c4 [17, 8, 15], c3 [10, 18, 83], c5 [7, 13, 14], y10 [9, 29, 13],
y6_masked [11, 29, 18].
"""

import numpy as np
import pytest

from _util import aligned_errors

pytestmark = pytest.mark.gpu

FP64_TOL = 1e-8
FP32_TOL = 1e-4
N = 20000
R = 3


def case_data(name):
    """(Xs, Y) of a case: orc.synthetic(..., error=0.5, seed=215), NaNs from default_rng(3) where the case has them."""
    from oracle import tpls_oracle as orc
    dims, M, latent, extra, dtype, nan = {
        # coupled pair, fp32: 2 x 328 MB -- too large for the resident loop by default
        "c4": ((N, 64, 64), 4, 12, [(N, 64, 64)], np.float32, 0.0),
        # 20 % NaN: fp32 164 MB (resident loop, ~23 of ~136 rows per CTA in shared memory), fp64 328 MB (streaming)
        "c3_f32": ((N, 64, 32), 4, 8, [], np.float32, 0.2),
        "c3_f64": ((N, 64, 32), 4, 8, [], np.float64, 0.2),
        # 4-way X: a 3-way covariance tensor per trip
        "c5": ((N, 32, 16, 8), 4, 12, [], np.float32, 0.0),
        # 10 responses (more than the 8 the X passes carry): the Y side runs as passes of its own; fp64 -> two slabs
        "y10": ((N, 64, 64), 10, 12, [], np.float64, 0.0),
        # 6 responses and NaNs: fused Y side, but no covariance mode (masked with more than 4 responses)
        "y6_masked": ((N, 64, 32), 6, 8, [], np.float32, 0.2),
    }[name]
    Xs, Y, _ = orc.synthetic(dims, M, latent, error=0.5, seed=215, extra_dims=extra)
    Xs = [x.astype(dtype) for x in (Xs if extra else [Xs])]
    if nan:
        rng = np.random.default_rng(3)
        for x in Xs:
            x[rng.random(x.shape) < nan] = np.nan
    return Xs, Y


_refs = {}


@pytest.fixture(scope="module")
def oracle_fit():
    """Oracle fit of a case, computed on first use and kept for the module."""
    from oracle import tpls_oracle as orc

    def get(name):
        if name not in _refs:
            _refs.clear()                             # the variants of a case are adjacent: keep one case in memory
            Xs, Y = case_data(name)
            _refs[name] = (Xs, Y, orc.fit([x.copy() for x in Xs], Y.copy(), R, r2_mode="residual"))
        return _refs[name]
    yield get
    _refs.clear()


def _fit(Xs, Y, env, algorithm, monkeypatch):
    from cmtf_pls_b200 import ctPLS
    monkeypatch.delenv("TPLS_RESIDENT", raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)                      # read at every fit
    est = ctPLS(R, algorithm=algorithm)
    est.fit([x.copy() for x in Xs], Y.copy())
    return est


def _check(est, ref, tol):
    assert est.n_iter_.tolist() == ref["trips"].tolist()
    got = dict(T=est.factor_T, W=[f[1:] for f in est.Xs_factors], U=est.Y_factors[0], Q=est.Y_factors[1],
               coef=est.coef_, R2X=est.R2Xs, R2Y=est.R2Y)
    for k, e in aligned_errors(got, ref).items():
        assert e < tol, (k, e)


# (case, variant name, environment, algorithm, expected path)
#   path "resident":  the resident trip loop ran every component
#   path "fused":     streaming kernels, Y side inside the X passes: 3 + 2 L launches per trip
#   path "unfused":   streaming kernels, Y side in passes of its own: more than 3 + 2 L launches per trip
#   path "cov":       covariance mode
_VARIANTS = [
    ("c4", "default", {}, "stream", "fused"),
    # forced: ~136 rows per CTA, 2 x 16 KB each, almost all of them outside shared memory
    ("c4", "resident", {"TPLS_RESIDENT": "1"}, "stream", "resident"),
    ("c4", "covariance", {}, "covariance", "cov"),
    ("c3_f32", "default", {}, "stream", "resident"),
    ("c3_f32", "streaming", {"TPLS_RESIDENT": "0"}, "stream", "fused"),
    ("c3_f32", "covariance", {}, "covariance", "cov"),
    ("c3_f64", "default", {}, "stream", "fused"),
    ("c3_f64", "covariance", {}, "covariance", "cov"),
    ("c5", "default", {}, "stream", "fused"),
    ("c5", "covariance", {}, "covariance", "cov"),
    ("y10", "default", {}, "stream", "unfused"),
    ("y6_masked", "default", {}, "stream", "resident"),
    ("y6_masked", "streaming", {"TPLS_RESIDENT": "0"}, "stream", "fused"),
    ("y6_masked", "covariance", {}, "covariance", "resident"),   # asked for, not supported: the default inner loop
]


@pytest.mark.parametrize("case,variant,env,algorithm,path", _VARIANTS, ids=[f"{v[0]}-{v[1]}" for v in _VARIANTS])
def test_fit_20k_matches_oracle(oracle_fit, case, variant, env, algorithm, path, monkeypatch):
    Xs, Y, ref = oracle_fit(case)
    est = _fit(Xs, Y, env, algorithm, monkeypatch)
    st = est.stats_
    L = len(Xs)
    assert st["covariance_mode"] == (1 if path == "cov" else 0)
    assert st["resident_loops"] == (R if path == "resident" else 0)
    if path == "fused":
        assert st["launches_per_trip"] == 3 + 2 * L
    elif path == "unfused":
        assert st["launches_per_trip"] > 3 + 2 * L
    tol = FP32_TOL if Xs[0].dtype == np.float32 else FP64_TOL
    _check(est, ref, tol)
