"""Batched fits: many small tPLS / ctPLS problems -- or the cross-validation
folds of one -- in ONE launch of the CUDA library, one CTA per problem
(``tpls_fit_batch``, DESIGN.md section 4d).

    models = fit_batch(X, Y, n_components, row_weights=None, tol=1e-8, max_iter=100, device=None)

Every returned model is what ``tPLS.fit`` / ``ctPLS.fit`` (with the same 0/1
row weights) gives for its problem: same attributes, ``transform`` /
``predict`` / ``X_reconstructed`` / pickle work on it.  Unlike ``fit``, the
models do not reference the training arrays, so ``X_miss`` / ``Xs_miss`` of a
model whose data had NaNs raises (``np.isnan`` of the problem's data gives the
same mask).
"""

from __future__ import annotations

import numpy as np

from . import _core, _engine
from .cmtf import ctPLS
from .tpls import tPLS


def _host(a):
    return a.detach().cpu().numpy() if _core._is_torch(a) else np.asarray(a)


def _batched(a, what):
    """numpy array or torch tensor with its leading (batch) axis, C-contiguous, float32 / float64."""
    if _core._is_torch(a):
        import torch
        if a.dtype not in (torch.float32, torch.float64):
            a = a.to(torch.float64)
        return a.contiguous()
    return _core.as_input(a, what)


def _check_shapes(Xs, Y, n_components, row_weights):
    """Batch size B, per-problem shapes and the batch axis of every input; raises before any device call."""
    if not isinstance(n_components, (int, np.integer)) or n_components < 1:
        raise ValueError(f"n_components must be a positive integer, got {n_components!r}")
    if len(Xs) < 1:
        raise ValueError("X must hold at least one tensor")
    for X in Xs:
        if X.ndim < 3:
            raise ValueError(f"every X needs a leading batch axis and at least two modes (B, N, d1, ...); got shape {tuple(X.shape)}")
    if Y.ndim not in (2, 3):
        # Y of one problem is a vector or a matrix (tpls.py:48-49)
        assert Y.ndim <= 3, "Only a matrix (2-mode tensor) Y is acceptable."
        raise ValueError(f"Y needs a leading batch axis: (B, N) or (B, N, M); got shape {tuple(Y.shape)}")
    for X in Xs:
        assert X.shape[1] == Y.shape[1]
    sizes = [int(X.shape[0]) for X in Xs] + [int(Y.shape[0])]
    if row_weights is not None:
        if row_weights.ndim != 2 or int(row_weights.shape[1]) != int(Y.shape[1]):
            raise ValueError(f"row_weights must be (B, N) = (B, {int(Y.shape[1])}); got shape {tuple(row_weights.shape)}")
        sizes.append(int(row_weights.shape[0]))
    B = max(sizes)
    if any(s not in (1, B) for s in sizes):
        raise ValueError(f"batch axes {sizes} do not broadcast: each must be 1 or {B}")
    if row_weights is not None:
        w = _host(row_weights)
        if not np.all((w == 0) | (w == 1)):
            raise ValueError("row_weights must be 0 or 1 (held-out rows have weight 0)")
    return B


def _models(kind, st_list, Xs_shape, Y_shape):
    models = []
    for st in st_list:
        m = kind(st["R"], device=st["device"])
        if kind is tPLS:
            m._set_fitted(st, Xs_shape[0], Y_shape, None, None)
        else:
            m._set_fitted(st, list(Xs_shape), Y_shape, [None] * len(Xs_shape), None)
        models.append(m)
    return models


def fit_batch(X, Y, n_components, row_weights=None, tol=1e-8, max_iter=100, device=None):
    """Fit B independent problems at once; returns a list of B fitted ``tPLS`` (X an array) or ``ctPLS`` (X a list
    of coupled arrays) models.

    ``X``: (B, N, d1, ...) array or torch tensor, or a list of such for coupled tensors.  ``Y``: (B, N) or
    (B, N, M).  ``row_weights``: optional (B, N) 0/1 weights; rows of weight 0 are held out (they are centred,
    projected and deflated, so their scores are ``transform`` of those rows).  A batch axis of size 1 is
    broadcast, so ``fit_batch(X[None], Y[None], R, row_weights=masks)`` fits one data set under B fold masks
    without copying X.  ``stats_["batch"]`` of each model is ``"kernel"`` when the one-launch batch kernel ran, or
    ``"loop"`` when the problems were outside its limits (more than 8 responses, more than 32 components, a working
    set per problem above ``TPLS_BATCH_MB``) and were fitted one by one with the same results.
    """
    coupled = isinstance(X, (list, tuple))
    Xs = [_batched(x, "X") for x in (X if coupled else [X])]
    Yb = Y if _core._is_torch(Y) else np.asarray(Y)
    wb = None if row_weights is None else (row_weights if _core._is_torch(row_weights) else np.asarray(row_weights))
    B = _check_shapes(Xs, Yb, n_components, wb)
    R = int(n_components)
    if _core._is_torch(Yb):
        import torch
        Yb = Yb.to(torch.float64)
        Yb = (Yb.reshape(Yb.shape[0], Yb.shape[1], 1) if Yb.ndim == 2 else Yb).contiguous()
    else:
        Yb = np.ascontiguousarray(np.asarray(Yb, dtype=np.float64))
        Yb = Yb.reshape(Yb.shape[0], Yb.shape[1], 1) if Yb.ndim == 2 else Yb
    if wb is not None:
        w = np.ascontiguousarray(np.broadcast_to(np.asarray(_host(wb), dtype=np.float64), (B, int(Yb.shape[1]))))
    else:
        w = None
    n, M = int(Yb.shape[1]), int(Yb.shape[2])
    Xs_shape = [tuple(int(s) for s in x.shape[1:]) for x in Xs]
    Y_shape = (n, 1) if Y.ndim == 2 else (n, M)
    kind = ctPLS if coupled else tPLS
    dev = _core._device_of(Xs + [Yb], device)

    eng = _core.get_engine(dev)
    L = len(Xs)
    dtypes = [_core.np_dtype_of(x) for x in Xs]
    out = _engine.BatchOut()
    T = np.empty((B, n, R))
    U = np.empty((B, n, R))
    Q = np.empty((B, M, R))
    W = [np.empty((B, sum(s[1:]), R)) for s in Xs_shape]
    coef = np.empty((B, R, R))
    r2x = np.empty((B, L, R))
    r2y = np.empty((B, R))
    x_mean = [np.empty((B,) + s[1:], dtype=dt) for s, dt in zip(Xs_shape, dtypes)]
    y_mean = np.empty((B, M))
    trips = np.empty((B, R), dtype=np.int32)
    conv = np.empty((B, R), dtype=np.int32)
    has_miss = np.empty((B, L), dtype=np.int32)
    out.T, out.U, out.Q, out.coef = T.ctypes.data, U.ctypes.data, Q.ctypes.data, coef.ctypes.data
    out.r2x, out.r2y, out.y_mean = r2x.ctypes.data, r2y.ctypes.data, y_mean.ctypes.data
    out.trips, out.converged, out.has_missing = trips.ctypes.data, conv.ctypes.data, has_miss.ctypes.data
    for l in range(L):
        out.W[l] = W[l].ctypes.data
        out.x_mean[l] = x_mean[l].ctypes.data
    strides = [0 if int(x.shape[0]) == 1 else int(np.prod(x.shape[1:])) for x in Xs]
    y_stride = 0 if int(Yb.shape[0]) == 1 else n * M
    ran = eng.fit_batch(B, Xs, strides, Xs_shape, Yb, y_stride, M, w, R, tol, max_iter, out)

    if ran:
        stats = dict(batch="kernel", batch_size=B, batch_fit_ms=out.fit_ms)
        sts = []
        for b in range(B):
            Ws = []
            for l, s in enumerate(Xs_shape):
                offs = np.cumsum((0,) + s[1:])
                Ws.append([W[l][b, offs[k]:offs[k + 1]] for k in range(len(s) - 1)])
            sts.append(dict(T=T[b], U=U[b], Q=Q[b], W=Ws, coef=coef[b], R2X=[r2x[b, l] for l in range(L)], R2Y=r2y[b],
                            X_mean=[x_mean[l][b] for l in range(L)], Y_mean=y_mean[b],
                            has_miss=[bool(v) for v in has_miss[b]], trips=trips[b], converged=conv[b].astype(bool),
                            stats=dict(stats), profile=None, device=dev, R=R))
        return _models(kind, sts, Xs_shape, Y_shape)

    # outside the kernel's limits: the problems one by one through the ordinary device fit, same results
    sts = []
    for b in range(B):
        xb = [x[b if int(x.shape[0]) > 1 else 0] for x in Xs]
        yb = Yb[b if int(Yb.shape[0]) > 1 else 0]
        st = _core.run_fit(xb, yb, R, tol, max_iter, device=dev, row_weights=None if w is None else w[b])
        st["stats"]["batch"] = "loop"
        st["R"] = R
        sts.append(st)
    return _models(kind, sts, Xs_shape, Y_shape)
