"""cmtf_pls_b200 -- the tensor-PLS (tPLS / coupled ctPLS) fit path of
meyer-lab/cmtf-pls, rebuilt for NVIDIA B200 (sm_100a).

    from cmtf_pls_b200 import tPLS, ctPLS

The estimators keep the reference's API (cmtf_pls/tpls.py, cmtf_pls/cmtf.py);
the work is done by hand-written CUDA kernels behind the C ABI declared in
include/tpls_b200.h.  There is no CPU fallback.
"""

from .tpls import tPLS
from .cmtf import ctPLS
from .validate import get_q2y, q2y_sweep
from .batch import fit_batch



def trim_memory():
    """Return the device buffers cached between fits (one working copy of X per
    engine) to the CUDA driver."""
    from . import _core
    for eng in _core._engines.values():
        if eng.h is not None:
            eng.trim()


__version__ = "0.1.0"
__all__ = ["tPLS", "ctPLS", "fit_batch", "get_q2y", "q2y_sweep", "trim_memory"]
