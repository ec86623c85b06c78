"""CPU: the host side of batched fits -- the ctypes mirror of ``tpls_batch_out`` against the header, and the shape,
broadcast and weight errors ``fit_batch`` raises before it touches a device."""

import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header():
    with open(os.path.join(ROOT, "include", "tpls_b200.h")) as f:
        return f.read()


def test_batch_out_mirror_matches_header():
    from cmtf_pls_b200 import _engine
    body = re.search(r"typedef struct tpls_batch_out \{(.*?)\} tpls_batch_out;", _header(), re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        ctype, names = decl.split(None, 1) if not decl.startswith("void*") else ("void*", decl[5:])
        if names.startswith("*"):
            ctype, names = ctype + "*", names[1:]
        for name in names.split(","):
            name = name.strip().lstrip("*")
            m = re.match(r"(\w+)\[TPLS_MAX_TENSORS\]", name)
            fields.append((m.group(1) if m else name, ctype, bool(m)))
    mirror = _engine.BatchOut._fields_
    assert [f[0] for f in fields] == [m[0] for m in mirror]
    for (name, ctype, is_array), (mname, mtype) in zip(fields, mirror):
        if is_array:
            assert mtype._length_ == _engine.MAX_TENSORS and mtype._type_ is C.c_void_p, name
        elif ctype.endswith("*"):
            assert mtype is C.c_void_p, name
        else:
            assert ctype == "double" and mtype is C.c_double, name
    # x86-64 layout: 3 + 8 + 3 + 8 + 4 pointers, then the double
    assert C.sizeof(_engine.BatchOut) == 27 * 8
    assert "TPLS_E_BATCH_UNSUPPORTED 2" in _header()
    assert _engine.E_BATCH_UNSUPPORTED == 2


def test_fit_batch_is_exported_and_bound():
    import cmtf_pls_b200
    from cmtf_pls_b200 import _engine
    assert "fit_batch" in cmtf_pls_b200.__all__
    assert callable(cmtf_pls_b200.fit_batch)
    assert "tpls_fit_batch" in _engine.SIGNATURES
    assert "int tpls_fit_batch(" in _header()


def _no_device(monkeypatch):
    """Any device call from here on fails the test: the errors must come first."""
    from cmtf_pls_b200 import _core

    def boom(*a, **k):
        raise AssertionError("a device call was made")
    monkeypatch.setattr(_core, "get_engine", boom)
    monkeypatch.setattr(_core, "run_fit", boom)


@pytest.mark.parametrize("X,Y,w,exc,match", [
    (np.zeros((4, 10, 3, 2)), np.zeros((4, 9)), None, AssertionError, None),                 # sample counts differ
    (np.zeros((4, 10, 3, 2)), np.zeros((4, 10, 2, 2, 2)), None, AssertionError, "Only a matrix"),
    (np.zeros((4, 10, 3, 2)), np.zeros(10), None, ValueError, "batch axis"),
    (np.zeros((10, 3)), np.zeros((4, 10)), None, ValueError, "leading batch axis"),
    (np.zeros((4, 10, 3, 2)), np.zeros((3, 10)), None, ValueError, "broadcast"),
    (np.zeros((4, 10, 3, 2)), np.zeros((1, 10)), np.ones((2, 10)), ValueError, "broadcast"),
    (np.zeros((4, 10, 3, 2)), np.zeros((4, 10)), np.ones((4, 9)), ValueError, "row_weights must be"),
    (np.zeros((4, 10, 3, 2)), np.zeros((4, 10)), np.full((4, 10), 0.5), ValueError, "0 or 1"),
    ([np.zeros((4, 10, 3)), np.zeros((2, 10, 5))], np.zeros((4, 10)), None, ValueError, "broadcast"),
    ([np.zeros((4, 10, 3)), np.zeros((4, 11, 5))], np.zeros((4, 10)), None, AssertionError, None),
])
def test_shape_broadcast_and_weight_errors_before_any_device_call(X, Y, w, exc, match, monkeypatch):
    from cmtf_pls_b200 import fit_batch
    _no_device(monkeypatch)
    with pytest.raises(exc, match=match):
        fit_batch(X, Y, 2, row_weights=w)


@pytest.mark.parametrize("R", [0, -1, 2.5])
def test_bad_component_count(R, monkeypatch):
    from cmtf_pls_b200 import fit_batch
    _no_device(monkeypatch)
    with pytest.raises(ValueError, match="n_components"):
        fit_batch(np.zeros((2, 10, 3, 2)), np.zeros((2, 10)), R)
