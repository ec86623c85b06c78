"""GPU: the single operators of include/tpls_b200.h against numpy on the same
seeded inputs (fp64 accumulate: tolerance 1e-12 relative, Frobenius)."""

import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _rel(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(b), 1e-300)


@pytest.fixture(scope="module")
def eng():
    from cmtf_pls_b200._core import get_engine
    return get_engine(0)


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# Steady state of the streaming rings (148 SMs; passes.cu make_geom, rowpass.cu make_row_geom): 40001 rows of 16 KB
# are 20001 two-row tiles with a 1-row last tile, and a tile count that no grid divides, so CTAs run different lap counts.
_STEADY = [
    # colpass FULL fp32: 296 CTAs x 67-68 tiles = 22-23 laps of a 3-stage ring; rowpass FULL fp32: 2-row tiles, 3 stages and
    # the 3-slot reducer ring (masked counting pass: 1-row tiles, 6 stages, 135-136 tiles per CTA)
    (40001, 4096, np.float32),
    # two 2048-column slabs (colpass and rowpass + row_finish_kernel): 148 CTAs per slab x 135-136 tiles = 45-46 laps
    (40001, 4096, np.float64),
    # colpass / rowpass FULL fp64, one slab: 296 CTAs x 67-68 two-row tiles
    (40001, 2048, np.float64),
]


def _masked_input(rng, n, p, dtype, masked):
    X = rng.normal(size=(n, p)).astype(dtype, copy=False)
    if masked:
        X[rng.random(X.shape) < 0.2] = np.nan
        X[:, p // 2] = np.nan
        if (n, p, dtype) in _STEADY:
            X[-1] = np.nan          # an all-NaN row alone in the short last tile: its score is NaN
    return X


@pytest.mark.parametrize("n,p,dtype", [(1000, 4096, np.float32), (1000, 4096, np.float64), (37, 48, np.float64),
                                       (5000, 24, np.float32), (333, 520, np.float32), (200, 6000, np.float32),
                                       (1, 8, np.float64), (70000, 512, np.float32)] + _STEADY)
@pytest.mark.parametrize("masked", [0, 1])
def test_contract_project(eng, n, p, dtype, masked):
    import torch
    rng = np.random.default_rng(n + p)
    X = _masked_input(rng, n, p, dtype, masked)
    u = rng.normal(size=n)
    w = rng.normal(size=p)
    Xd, ud, wd = _dev(X), _dev(u), _dev(w)
    z = torch.empty(p, dtype=torch.float64, device="cuda")
    t = torch.empty(n, dtype=torch.float64, device="cuda")
    code = 0 if dtype == np.float32 else 1
    lib = eng.lib
    eng._ck(lib.tpls_op_contract(eng.h, Xd.data_ptr(), code, n, p, ud.data_ptr(), masked, z.data_ptr(), None, 1))
    eng._ck(lib.tpls_op_project(eng.h, Xd.data_ptr(), code, n, p, wd.data_ptr(), masked, t.data_ptr(), None, 1))
    ts = [t.cpu().numpy()]
    if masked:   # a second launch in the same call uses the row counts of the first (row pass mode 1, not counting)
        t.fill_(0.0)
        eng._ck(lib.tpls_op_project(eng.h, Xd.data_ptr(), code, n, p, wd.data_ptr(), masked, t.data_ptr(), None, 2))
        ts.append(t.cpu().numpy())
    del Xd
    X64 = X.astype(np.float64, copy=False)        # the only full-size fp64 array (X itself when it is fp64)
    if masked:
        obs = ~np.isnan(X64)
        X64[~obs] = 0.0
        cnt = obs.sum(0)
        with np.errstate(all="ignore"):
            z_ref = np.where(cnt > 0, (X64.T @ u) / cnt * n, 0.0)
            t_ref = (X64 @ w) / obs.sum(1) * p
    else:
        z_ref, t_ref = X64.T @ u, X64 @ w
    assert _rel(z.cpu().numpy(), z_ref) < 1e-12
    good = ~np.isnan(t_ref)
    for tt in ts:
        assert np.array_equal(np.isnan(tt), np.isnan(t_ref))
        assert _rel(tt[good], t_ref[good]) < 1e-12


@pytest.mark.parametrize("n,p,dtype", [(800, 4096, np.float32), (800, 2048, np.float64), (50, 48, np.float64)] + _STEADY)
@pytest.mark.parametrize("masked", [0, 1])
def test_deflate_contract(eng, n, p, dtype, masked):
    import torch
    rng = np.random.default_rng(7)
    X = rng.normal(size=(n, p)).astype(dtype, copy=False)
    if masked:
        X[rng.random(X.shape) < 0.2] = np.nan
        if (n, p, dtype) in _STEADY:
            X[-1] = np.nan          # an all-NaN row alone in the short last tile
    t, u, w = rng.normal(size=n), rng.normal(size=n), rng.normal(size=p) / np.sqrt(p)
    Xd = _dev(X)
    z = torch.empty(p, dtype=torch.float64, device="cuda")
    ss = torch.empty(1, dtype=torch.float64, device="cuda")
    code = 0 if dtype == np.float32 else 1
    td, wd, ud = _dev(t), _dev(w), _dev(u)   # keep the device copies alive across the call
    eng._ck(eng.lib.tpls_op_deflate_contract(eng.h, Xd.data_ptr(), code, n, p, td.data_ptr(), wd.data_ptr(),
                                             ud.data_ptr(), masked, z.data_ptr(), ss.data_ptr(), None, 1))
    got = Xd.cpu().numpy()
    del Xd
    # block by block over the rows, so that the large cases hold one fp64 block at a time besides X and the result
    worst, z_ref, ss_ref = 0.0, np.zeros(p), 0.0
    for r0 in range(0, n, 4096):
        r1 = min(n, r0 + 4096)
        X64, g = X[r0:r1].astype(np.float64), got[r0:r1]
        tw = np.outer(t[r0:r1], w)
        Xn = (X64 - tw).astype(dtype)            # numpy's in-place `X -= outer` rounding
        assert np.array_equal(np.isnan(g), np.isnan(Xn))
        # fused multiply-add vs numpy's multiply-then-subtract: within 2 ulp of the operands' magnitude
        scale = np.abs(X64) + np.abs(tw)
        with np.errstate(all="ignore"):
            worst = max(worst, float(np.nanmax(np.abs(g.astype(np.float64) - Xn.astype(np.float64)) / scale)))
        g64 = np.nan_to_num(g.astype(np.float64))
        z_ref += g64.T @ u[r0:r1]
        ss_ref += np.sum(g64 ** 2)
    assert worst <= 2 * float(np.finfo(dtype).eps), worst
    assert _rel(z.cpu().numpy(), z_ref) < 1e-12
    assert abs(ss.item() - ss_ref) / ss_ref < 1e-12


@pytest.mark.parametrize("dims", [(24,), (64, 64), (38, 65), (65, 38), (32, 16), (8, 6, 4), (32, 16, 8), (5, 4, 3, 3),
                                  (100, 4, 3), (2, 2), (1, 7), (120, 90), (4, 3, 3, 2, 2), (3, 3, 2, 2, 2, 2), (3, 2, 2, 2, 2, 2, 2),
                                  (16, 8, 6, 4), (40, 33, 5)])
def test_rank1_matches_restated_parafac(eng, dims):
    import torch
    from oracle import tpls_oracle as orc
    rng = np.random.default_rng(sum(dims))
    # a covariance-like tensor: dominant rank-1 part + structured noise
    vs = [rng.normal(size=d) for d in dims]
    Z = 3.0 * orc.rank_r_tensor([v[:, None] for v in vs]) if len(dims) > 1 else 3.0 * vs[0]
    Z = Z + rng.normal(size=dims)
    ref = orc.rank1_vectors(Z, 1e-8)
    p = int(np.prod(dims))
    zd = _dev(Z.reshape(-1))
    w = torch.zeros(sum(dims), dtype=torch.float64, device="cuda")
    wk = torch.zeros(p, dtype=torch.float64, device="cuda")
    sweeps = C.c_int(0)
    darr = (C.c_int * len(dims))(*dims)
    eng._ck(eng.lib.tpls_op_rank1(eng.h, zd.data_ptr(), len(dims), darr, 1e-8, 0, w.data_ptr(), wk.data_ptr(),
                                  C.byref(sweeps), None, 1))
    got = np.split(w.cpu().numpy(), np.cumsum(dims)[:-1])
    for g, r in zip(got, ref):
        assert _rel(g, r) < 1e-10, dims           # same signs too (largest-|entry| convention)
    assert _rel(wk.cpu().numpy(), orc.kron_weights(ref)) < 1e-10
    if len(dims) >= 2:
        import tensorly.decomposition._cp as cp
        assert sweeps.value == cp.last_sweeps[-1]


def _rank1_gpu(eng, Z):
    import torch
    dims = Z.shape
    zd = _dev(Z.reshape(-1))
    w = torch.zeros(sum(dims), dtype=torch.float64, device="cuda")
    wk = torch.zeros(Z.size, dtype=torch.float64, device="cuda")
    sweeps = C.c_int(0)
    darr = (C.c_int * len(dims))(*dims)
    eng._ck(eng.lib.tpls_op_rank1(eng.h, zd.data_ptr(), len(dims), darr, 1e-8, 0, w.data_ptr(), wk.data_ptr(),
                                  C.byref(sweeps), None, 1))
    return np.split(w.cpu().numpy(), np.cumsum(dims)[:-1]), wk.cpu().numpy(), sweeps.value


def _orth(rng, d, k):
    return np.linalg.qr(rng.normal(size=(d, k)))[0]


def _spectrum_case(kind, dims, eps):
    from oracle import tpls_oracle as orc
    rng = np.random.default_rng(sum(dims) + len(kind))
    if kind == "near" and len(dims) == 2:
        # U diag(1, 1 - eps, 0.5 * 0.9^k ...) V': the top pair of singular values eps apart
        k = min(dims)
        s = np.concatenate([[1.0, 1.0 - eps], 0.5 * 0.9 ** np.arange(k - 2)])
        return (_orth(rng, dims[0], k) * s) @ _orth(rng, dims[1], k).T
    if kind == "near":
        # two orthogonal rank-1 terms of weight 1 and 1 - eps, plus noise of norm ~1e-3
        fs = [_orth(rng, d, 2) for d in dims]
        Z = orc.rank_r_tensor([f[:, :1] for f in fs]) + (1.0 - eps) * orc.rank_r_tensor([f[:, 1:] for f in fs])
        return Z + 1e-3 * rng.normal(size=dims) / np.sqrt(np.prod(dims))
    if kind == "noise":
        return rng.normal(size=dims)
    assert kind == "rank1"   # exactly rank one: tau = 1 at the first squaring of the Gram matrix
    return orc.rank_r_tensor([rng.normal(size=(d, 1)) for d in dims])


@pytest.mark.parametrize("kind,dims,eps", [("near", d, e) for d in [(64, 64), (38, 65), (8, 6)] for e in (1e-3, 1e-6)]
                         + [("near", d, e) for d in [(32, 16, 8), (16, 8, 6, 4)] for e in (1e-3, 1e-6)]
                         + [("noise", d, 0.0) for d in [(64, 64), (32, 16, 8), (16, 8, 6, 4)]]
                         + [("rank1", d, 0.0) for d in [(64, 64), (32, 16, 8)]])
def test_rank1_hard_spectra_match_restated_parafac(eng, kind, dims, eps):
    """Spectra where the Gram squaring of lead_eig (rank1.cu) and the ALS sweeps work hardest: a top gap of 1e-3 and
    1e-6, pure noise (the oracle's ALS runs 23 and 89 sweeps on the 3- and 4-way cases here) and an exact rank one."""
    from oracle import tpls_oracle as orc
    Z = _spectrum_case(kind, dims, eps)
    ref = orc.rank1_vectors(Z, 1e-8)
    import tensorly.decomposition._cp as cp
    got, wk, sweeps = _rank1_gpu(eng, Z)
    # Perturbing these Z by 1e-15 relative moves the oracle's vectors by at most ~1e-12 -- except for a matrix whose top
    # two singular values are 1e-6 apart: its singular vectors are determined only to ~eps_mach / 1e-6 ~ 1e-10 by the
    # data (the same perturbation moves them by up to 5.7e-10), so there they are held to 5e-9, and sigma_1 = w0' Z w1
    # (quadratic in the vectors' error) to 1e-12 as in every 2-way case.
    tol = 5e-9 if (kind == "near" and len(dims) == 2 and eps < 1e-4) else 1e-10
    for g, r in zip(got, ref):
        assert _rel(g, r) < tol, (kind, dims, eps)         # same signs too (largest-|entry| convention)
    assert _rel(wk, orc.kron_weights(ref)) < tol
    if len(dims) == 2:
        assert abs(got[0] @ Z @ got[1] - np.linalg.svd(Z, compute_uv=False)[0]) < 1e-12
    if kind != "rank1":
        assert sweeps == cp.last_sweeps[-1]
    else:
        # exactly rank one: the oracle's stop quantity |err_k-1 - err_k| is rounding noise (err = sqrt of a cancelling
        # difference, ~1e-8), and a 1e-15 relative perturbation of Z moves its sweep count between 2 and 7
        assert 1 <= sweeps <= 100


@pytest.mark.parametrize("spectrum", ["orthogonal", "top_pair"])
def test_rank1_exactly_degenerate_top_returns_a_valid_pair(eng, spectrum):
    """A tie at the top: the vectors are not unique and the squarings of lead_eig never reach tau = 1 (tau stays at
    1/k), so its 64-squaring loop has to end on its own.  What any answer must satisfy is checked instead."""
    rng = np.random.default_rng(16)
    if spectrum == "orthogonal":                 # every singular value 1
        Z = _orth(rng, 16, 16)
    else:                                        # diag(1, 1, 0.5, 0.45, ...)
        s = np.concatenate([[1.0, 1.0], 0.5 * 0.9 ** np.arange(14)])
        Z = (_orth(rng, 16, 16) * s) @ _orth(rng, 16, 16).T
    (w0, w1), wk, sweeps = _rank1_gpu(eng, Z)
    assert np.all(np.isfinite(w0)) and np.all(np.isfinite(w1)) and sweeps >= 1
    assert abs(np.linalg.norm(w0) - 1.0) < 1e-12 and abs(np.linalg.norm(w1) - 1.0) < 1e-12
    assert abs(w0 @ Z @ w1 - 1.0) < 1e-12                      # sigma_1 = 1 in both cases
    assert np.max(np.abs(wk - np.kron(w0, w1))) < 1e-15
    assert w1[np.argmax(np.abs(w1))] > 0                       # sign convention on the last mode
