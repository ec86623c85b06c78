"""Cross-validated Q2Y (the reference's cmtf_pls/validate.py:7-37, which is dead
code as shipped: it reads ``pls_tensor.original_X`` that ``fit`` never sets).

Formula kept from the reference (validate.py:35-37):

    Q2Y = 1 - sum (Y_pred - Y)^2 / sum Y^2        (uncentred denominator)

What differs is how the refits are done:
  * folds are 0/1 sample weights handed to the device fit
    (``tpls_set_row_weights``): X is uploaded once and never sliced or copied,
    and the held-out rows' scores come out of the same passes as the training
    rows' (they are exactly ``transform`` of the held-out data);
  * PLS components are nested -- the first k components of an R-component fit
    are the k-component fit, and a truncated model predicts identically
    (SURVEY.md §0.5) -- so a sweep over 1..R components needs ONE R-component
    fit per fold, not R of them.
"""

from __future__ import annotations

import numpy as np

from . import _core


def _folds(n, n_splits, seed):
    if n_splits is None or n_splits >= n:
        return [np.array([i]) for i in range(n)]          # leave-one-out, in order (validate.py:24)
    perm = np.random.default_rng(seed).permutation(n)
    return [np.sort(f) for f in np.array_split(perm, n_splits)]


def _to_device(X, device):
    """One resident copy of the data for all folds."""
    if _core._is_torch(X):
        return X
    import torch
    dev = torch.device("cuda", device if device is not None else torch.cuda.current_device())
    return torch.from_numpy(np.ascontiguousarray(X)).to(dev)


def _device_fold_fit(Xd, Yd, R, tol, max_iter, device, algorithm):
    """The product's fold fit: one R-component device fit with the fold as 0/1 row weights."""
    def fit_fold(w):
        return _core.run_fit(Xd, Yd, R, tol, max_iter, device=device, row_weights=w, algorithm=algorithm)
    return fit_fold


def _sum_over_ranks(arrays, group, device):
    """In-place sum of small host arrays over the ranks of ``group`` (True = default group)."""
    import torch
    import torch.distributed as dist
    pg = None if group is True else group
    on_gpu = dist.get_backend(pg) == "nccl"
    for a in arrays:
        t = torch.from_numpy(a)
        if on_gpu:
            d = t.to(torch.device("cuda", device if device is not None else torch.cuda.current_device()))
            dist.all_reduce(d, group=pg)
            t.copy_(d)
        else:
            dist.all_reduce(t, group=pg)


def q2y_sweep(X, Y, n_components, n_splits=5, seed=0, device=None, tol=1e-8, max_iter=100, folds=None,
              return_scores=False, algorithm="covariance", fold_group=None, _fit_fold=None):
    """Q2Y for 1, 2, ..., ``n_components`` components by K-fold cross-validation.

    ``X`` is one tensor (tPLS) or a list of coupled tensors (ctPLS); ``folds``
    optionally gives the held-out row indices of every fold explicitly.
    Returns an array of ``n_components`` values (and, with ``return_scores``,
    the cross-validated scores of every sample, shape (N, n_components)).

    ``algorithm``: inner loop of the fold fits.  The default is the covariance
    loop (one cross-covariance pass per component; same results as the
    streaming loop to rounding, several times faster), which the library
    replaces by the streaming loop on its own when there are more than 8
    responses (4 with missing values); ``"stream"`` forces the latter.
    ``"batch"`` fits all folds of the sweep in ONE launch of the batch kernel
    (:func:`cmtf_pls_b200.fit_batch`, one CTA per fold; same results): the
    fastest choice for small data sets, e.g. leave-one-out.

    ``fold_group`` (a torch.distributed process group, or True for the default
    one) runs the sweep FOLD-PARALLEL (SURVEY.md §8e: folds are independent
    units): every rank holds the complete X and Y, fits folds rank, rank +
    world, ... on its own GPU with no data-path collective, and only the R
    PRESS sums (and the cross-validated scores when asked for) are summed over
    the ranks at the end.  Every rank returns the same result.
    """
    Xs = list(X) if isinstance(X, (list, tuple)) else [X]
    Yn = Y.detach().cpu().numpy() if _core._is_torch(Y) else np.asarray(Y)
    Y2 = np.asarray(Yn, dtype=np.float64).reshape(Yn.shape[0], -1)
    n, R = Y2.shape[0], int(n_components)
    folds = _folds(n, n_splits, seed) if folds is None else [np.asarray(f) for f in folds]
    rank, world = 0, 1
    if fold_group is not None and fold_group is not False:
        import torch.distributed as dist
        pg = None if fold_group is True else fold_group
        rank, world = dist.get_rank(pg), dist.get_world_size(pg)
    mine = folds[rank::world]
    if algorithm == "batch" and _fit_fold is None:
        # all folds of this rank in ONE launch of the batch kernel: X and Y shared, one 0/1 weight row per fold
        from .batch import fit_batch
        masks = np.ones((len(mine), n))
        for k, held in enumerate(mine):
            masks[k, held] = 0.0
        models = fit_batch([x[None] for x in Xs] if isinstance(X, (list, tuple)) else Xs[0][None], Y2[None], R,
                           row_weights=masks, tol=tol, max_iter=max_iter, device=device) if mine else []
        fits = iter([dict(T=mdl.factor_T if isinstance(X, (list, tuple)) else mdl.X_factors[0], coef=mdl.coef_,
                          Q=mdl.Y_factors[1], Y_mean=mdl.Y_mean) for mdl in models])
        _fit_fold = lambda w: next(fits)  # noqa: E731 -- the folds come back in the order of `mine`
    elif _fit_fold is None:                    # tests inject a CPU fit to exercise the fold plumbing without a GPU
        Xd = [_to_device(x, device) for x in Xs]
        Yd = _to_device(Y2, device)
        _fit_fold = _device_fold_fit(Xd, Yd, R, tol, max_iter, device, algorithm)
    press = np.zeros(R)
    cv_scores = np.zeros((n, R))
    for held in mine:
        w = np.ones(n)
        w[held] = 0.0
        st = _fit_fold(w)
        T = st["T"][held]
        cv_scores[held] = T
        for k in range(1, R + 1):
            pred = T[:, :k] @ st["coef"][:k, :k] @ st["Q"][:, :k].T + st["Y_mean"]
            press[k - 1] += float(np.sum((pred - Y2[held]) ** 2))
    if world > 1:
        _sum_over_ranks([press, cv_scores] if return_scores else [press], fold_group, device)
    q2 = 1.0 - press / float(np.sum(Y2 ** 2))
    return (q2, cv_scores) if return_scores else q2


def get_q2y(pls_tensor, X=None, Y=None, n_splits=None, seed=0):
    """Q2Y of a fitted estimator's configuration (validate.py:7): leave-one-out by
    default like the reference, K-fold when ``n_splits`` is given.  ``X`` / ``Y``
    default to the arrays the estimator was fitted on."""
    def alive(ref):   # the estimators reference their training arrays weakly
        return ref() if ref is not None else None
    if X is None:
        if hasattr(pls_tensor, "_X_ref"):
            X = alive(pls_tensor._X_ref)
        elif hasattr(pls_tensor, "_Xs_ref"):
            X = [alive(r) for r in pls_tensor._Xs_ref]
            X = None if any(x is None for x in X) else X
    if Y is None:
        Y = alive(getattr(pls_tensor, "_Y_ref", None))
    assert X is not None and Y is not None, \
        "PLS Tensor must be fit prior to calculating Q2Y (and its training arrays still alive, or passed as X / Y)"
    q2 = q2y_sweep(X, Y, pls_tensor.n_components, n_splits=n_splits, seed=seed,
                   device=getattr(pls_tensor, "_device", None))
    return float(q2[-1])
