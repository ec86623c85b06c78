"""``tPLS`` -- single-tensor N-PLS estimator with the reference's API
(meyer-lab/cmtf-pls, cmtf_pls/tpls.py:15-189), fitted by the sm_100a CUDA
library.  Same constructor, methods, attribute names, Mapping protocol and
error behaviour; inputs may be numpy arrays (staged to the GPU) or torch CUDA
tensors (used where they are).

Extra, not in the reference: ``device`` / ``process_group`` keyword arguments,
``n_iter_`` (inner trips per component) and ``stats_`` (timings and bytes of
the last fit).  With a process group every rank passes its own block of rows of
X and Y; loadings, Q, coef_, R2X/R2Y and the means are replicated, the scores
``X_factors[0]`` / ``Y_factors[0]`` are this rank's rows.
"""

from collections.abc import Mapping
from copy import copy

import numpy as np

from . import _core


class tPLS(Mapping):
    """Tensor PLS (cmtf_pls/tpls.py:15)."""

    def __init__(self, n_components: int, device=None, process_group=None, algorithm="stream"):
        super().__init__()
        self.n_components = n_components
        self.device = device
        self.process_group = process_group
        # "stream": two passes over X per inner trip (the reference's loop, the benchmark contract);
        # "covariance": one cross-covariance pass per component, inner loop on (P x M) data -- same results
        self.algorithm = algorithm

    # ---- Mapping protocol (tpls.py:23-42) ----
    def __getitem__(self, index):
        if index == 0:
            return self.X_factors
        elif index == 1:
            return self.Y_factors
        elif index == 2:
            return self.coef_
        else:
            raise IndexError

    def __iter__(self):
        yield self.X_factors
        yield self.Y_factors
        yield self.coef_

    def __len__(self):
        return 3

    def copy(self):
        return copy(self)

    def __getstate__(self):
        """Pickle the fitted model, not the references to the training arrays or to a process group."""
        state = dict(self.__dict__)
        for k in ("_X_ref", "_Y_ref", "process_group", "_profile"):
            state.pop(k, None)
        return state

    def __setstate__(self, state):
        self.__dict__.update(state)
        self.__dict__.setdefault("process_group", None)

    # ---- fit (tpls.py:44-120) ----
    def fit(self, X, Y, tol=1e-8, max_iter=100, verbose=0, overwrite_x=False, profile=False):
        assert X.shape[0] == Y.shape[0]
        assert Y.ndim <= 2, "Only a matrix (2-mode tensor) Y is acceptable."
        st = _core.run_fit([X], Y, self.n_components, tol, max_iter, device=self.device,
                           group=self.process_group, overwrite=overwrite_x, profile=profile,
                           algorithm=self.algorithm)
        self._set_fitted(st, tuple(X.shape), (int(Y.shape[0]), 1) if Y.ndim == 1 else tuple(Y.shape),
                         _core.weak_ref(X), _core.weak_ref(Y))
        if self.X_hasMiss:
            print("X has missing values")
        if verbose:
            for a, k in enumerate(self.n_iter_):
                if self.converged_[a]:
                    print("Comp {}: converged after {} iterations".format(a, k - 1))

    def _set_fitted(self, st, X_shape, Y_shape, X_ref, Y_ref):
        """The fitted attributes from the state of a device fit (``fit`` and ``fit_batch``)."""
        self.X_dim = len(X_shape)
        self.X_shape = X_shape
        self.Y_shape = Y_shape
        self.X_factors = [st["T"]] + st["W"][0]
        self.Y_factors = [st["U"], st["Q"]]
        self.R2X = st["R2X"][0]
        self.R2Y = st["R2Y"]
        self.X_hasMiss = st["has_miss"][0]
        self._X_ref = X_ref   # for X_miss / get_q2y only; the caller's arrays are not kept alive
        self._Y_ref = Y_ref
        self.X_mean = st["X_mean"][0]
        self.Y_mean = st["Y_mean"]
        self.coef_ = st["coef"]
        self.n_iter_ = st["trips"]
        # the reference is silent when max_iter is exhausted (tpls.py:79-107); here it can be asked
        self.converged_ = st["converged"]
        self.stats_ = st["stats"]
        self._profile = st["profile"]
        self._device = st["device"]

    @property
    def X_miss(self):
        """Positions of missing values of the training X (tpls.py:64).  The reference materialises this N x P
        boolean tensor in every fit; here it is computed on demand: all False when the fit saw no NaN, else
        from the training array, which is referenced WEAKLY (it is neither kept alive nor pickled)."""
        if not self.X_hasMiss:
            return np.zeros(self.X_shape, dtype=bool)
        return _core.isnan_of(getattr(self, "_X_ref", None), "X_miss")

    @property
    def profile_(self):
        """Per-kernel-class timings of the profiled fits (``fit(..., profile=True)``) since the last read; None
        when the last fit was not profiled."""
        p = getattr(self, "_profile", None)
        return None if p is None else p.get()

    # ---- new data (tpls.py:122-186) ----
    def _scores(self, X):
        if tuple(self.X_shape[1:]) != tuple(X.shape[1:]):
            raise ValueError(f"Training X has shape {self.X_shape}, while the new X has shape {tuple(X.shape)}")
        return _core.run_transform([X], [self.X_mean], [self.X_factors[1:]], self.n_components,
                                   device=getattr(self, "_device", self.device))

    def predict(self, X):
        return self._scores(X) @ self.coef_ @ self.Y_factors[1].T + self.Y_mean

    def transform(self, X, Y=None):
        X_scores = self._scores(X)
        if Y is not None:
            Y_scores = _core.y_scores(Y, self.Y_mean, self.Y_shape, X_scores, self.coef_, self.Y_factors[1])
            return X_scores, Y_scores
        return X_scores

    def X_reconstructed(self):
        return _core.run_reconstruct(self.X_factors, self.X_mean, device=getattr(self, "_device", self.device))
