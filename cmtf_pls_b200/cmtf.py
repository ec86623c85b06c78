"""``ctPLS`` -- coupled tensor PLS over a list of X tensors sharing the sample
mode, with the reference's API (meyer-lab/cmtf-pls, cmtf_pls/cmtf.py:15-237),
fitted by the sm_100a CUDA library.  See :mod:`cmtf_pls_b200.tpls` for the
conventions shared with ``tPLS``.
"""

from collections.abc import Mapping
from copy import copy

import numpy as np

from . import _core


class ctPLS(Mapping):
    """Coupled tensor PLS (cmtf_pls/cmtf.py:15)."""

    def __init__(self, n_components: int, device=None, process_group=None, algorithm="stream"):
        super().__init__()
        self.n_components = n_components
        self.device = device
        self.process_group = process_group
        # "stream": two passes over X per inner trip (the reference's loop, the benchmark contract);
        # "covariance": one cross-covariance pass per component, inner loop on (P x M) data -- same results
        self.algorithm = algorithm

    # ---- Mapping protocol (cmtf.py:23-42) ----
    def __getitem__(self, index):
        if index == 0:
            return self.Xs_factors
        elif index == 1:
            return self.Y_factors
        elif index == 2:
            return self.coef_
        else:
            raise IndexError

    def __iter__(self):
        yield self.Xs_factors
        yield self.Y_factors
        yield self.coef_

    def __len__(self):
        return 3

    def copy(self):
        return copy(self)

    def __getstate__(self):
        """Pickle the fitted model, not the references to the training arrays or to a process group."""
        state = dict(self.__dict__)
        for k in ("_Xs_ref", "_Y_ref", "process_group", "_profile"):
            state.pop(k, None)
        return state

    def __setstate__(self, state):
        self.__dict__.update(state)
        self.__dict__.setdefault("process_group", None)

    # ---- fit (cmtf.py:44-140) ----
    def fit(self, Xs, Y, tol=1e-8, max_iter=100, verbose=0, overwrite_x=False, profile=False):
        assert isinstance(Xs, list)
        for X in Xs:
            assert X.shape[0] == Y.shape[0]
            assert X.ndim >= 2
        assert Y.ndim <= 2, "Only a matrix (2-mode tensor) Y is acceptable."
        st = _core.run_fit(Xs, Y, self.n_components, tol, max_iter, device=self.device,
                           group=self.process_group, overwrite=overwrite_x, profile=profile,
                           algorithm=self.algorithm)
        self._set_fitted(st, [tuple(X.shape) for X in Xs], (int(Y.shape[0]), 1) if Y.ndim == 1 else tuple(Y.shape),
                         [_core.weak_ref(X) for X in Xs], _core.weak_ref(Y))
        if any(self.Xs_hasMiss):
            print("At least one X has missing values")
        if verbose:
            for a, k in enumerate(self.n_iter_):
                if self.converged_[a]:
                    print("Comp {}: converged after {} iterations".format(a, k - 1))

    def _set_fitted(self, st, Xs_shape, Y_shape, Xs_ref, Y_ref):
        """The fitted attributes from the state of a device fit (``fit`` and ``fit_batch``)."""
        self.Xs_len = len(Xs_shape)
        self.Xs_dim = [len(s) for s in Xs_shape]
        self.Xs_shape = Xs_shape
        self.Y_shape = Y_shape
        self.factor_T = st["T"]
        # the shared score matrix is the SAME object in every tensor's factor list (cmtf.py:61-65)
        self.Xs_factors = [[self.factor_T] + ws for ws in st["W"]]
        self.Y_factors = [st["U"], st["Q"]]
        self.coef_ = st["coef"]
        self.R2Xs = st["R2X"]
        self.R2Y = st["R2Y"]
        self.Xs_mean = st["X_mean"]
        self.Y_mean = st["Y_mean"]
        self.Xs_hasMiss = st["has_miss"]
        self._Xs_ref = Xs_ref   # for Xs_miss / get_q2y only; not kept alive
        self._Y_ref = Y_ref
        self.n_iter_ = st["trips"]
        # the reference is silent when max_iter is exhausted (tpls.py:79-107); here it can be asked
        self.converged_ = st["converged"]
        self.stats_ = st["stats"]
        self._profile = st["profile"]
        self._device = st["device"]

    @property
    def Xs_miss(self):
        """Positions of missing values of the training tensors (cmtf.py:80-82), computed on demand."""
        refs = getattr(self, "_Xs_ref", None) or [None] * self.Xs_len
        return [np.zeros(self.Xs_shape[ti], dtype=bool) if not self.Xs_hasMiss[ti]
                else _core.isnan_of(refs[ti], f"Xs_miss[{ti}]") for ti in range(self.Xs_len)]

    @property
    def profile_(self):
        """Per-kernel-class timings of the profiled fits (``fit(..., profile=True)``) since the last read; None
        when the last fit was not profiled."""
        p = getattr(self, "_profile", None)
        return None if p is None else p.get()

    # ---- new data (cmtf.py:142-231) ----
    def _scores(self, Xs):
        assert len(Xs) == self.Xs_len
        for ti, X in enumerate(Xs):
            if tuple(self.Xs_shape[ti][1:]) != tuple(X.shape[1:]):
                raise ValueError(
                    f"Training X[{ti}] has shape {self.Xs_shape[ti]}, while the new X has shape {tuple(X.shape)}")
        return _core.run_transform(Xs, self.Xs_mean, [f[1:] for f in self.Xs_factors], self.n_components,
                                   device=getattr(self, "_device", self.device))

    def predict(self, Xs):
        return self._scores(Xs) @ self.coef_ @ self.Y_factors[1].T + self.Y_mean

    def transform(self, Xs, Y=None):
        X_scores = self._scores(Xs)
        if Y is not None:
            Y_scores = _core.y_scores(Y, self.Y_mean, self.Y_shape, X_scores, self.coef_, self.Y_factors[1])
            return X_scores, Y_scores
        return X_scores

    def Xs_reconstructed(self):
        return [_core.run_reconstruct(self.Xs_factors[ti], self.Xs_mean[ti], device=getattr(self, "_device", self.device))
                for ti in range(self.Xs_len)]
