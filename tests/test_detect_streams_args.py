"""Argument errors of bgsb_pipeline_detect / bgsb_pool_detect that are found before any device work."""
import ctypes as C
import types

import pytest

from tracking_b200 import blobs, capi


def _call(name, *head, S=2, bds=None):
    bds = (C.c_void_p * S)(*(bds or [None] * S))
    new, res, st = (capi.Blob * S)(), (C.c_int * S)(), (C.c_int * S)()
    return getattr(capi.lib(), name)(*head, bds, None, None, new, res, None, None, st)


def test_null_pipeline_or_pool_and_bad_slot():
    L = capi.lib()
    assert _call("bgsb_pipeline_detect", None) == capi.ERR_ARG
    assert b"null" in L.bgsb_last_error()
    for slot in (0, -1, 8):
        assert _call("bgsb_pool_detect", None, slot) == capi.ERR_ARG
        assert b"slot" in L.bgsb_last_error()
    assert L.bgsb_pool_submit(None, 0, capi.POOL_DETECT) == capi.ERR_ARG
    assert L.bgsb_pool_set_param(None, b"tableRows", 512) == capi.ERR_ARG
    assert L.bgsb_kernel_launch_count() == 0


def test_python_wrapper_raises_the_library_error():
    fake = [types.SimpleNamespace(_h=C.c_void_p()) for _ in range(2)]
    with pytest.raises(capi.BgsbError) as e:
        blobs.detect_streams(capi.lib().bgsb_pipeline_detect, (None,), fake, [[(1, 2, 3, 4)], []])
    assert e.value.code == capi.ERR_ARG
