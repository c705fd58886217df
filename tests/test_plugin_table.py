"""bgsb_create accepts exactly the algorithm ids of the bgsb200.h enum, which are the ids of tracking_b200.ALGOS."""
import ctypes as C
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_ids():
    src = open(os.path.join(ROOT, "include", "bgsb200.h")).read()
    return {int(v) for v in re.findall(r"\bBGSB_ALGO_\w+\s*=\s*(\d+)", src)}


def test_create_accepts_exactly_the_header_ids():
    import tracking_b200 as tb
    from tracking_b200 import _build, capi
    _build.build()
    ids = _header_ids()
    assert len(ids) == 13 and ids == set(tb.ALGOS)
    L = capi.lib()
    for algo in range(-1, 64):
        h = C.c_void_p()
        rc = L.bgsb_create(C.byref(h), algo, 0)
        if h:
            L.bgsb_destroy(h)
        if algo in ids:
            assert rc in (capi.OK, capi.ERR_CUDA), (algo, rc, L.bgsb_last_error())
        else:
            assert rc == capi.ERR_ARG, (algo, rc)
            assert b"unknown algorithm id" in L.bgsb_last_error(), algo
            assert not h
