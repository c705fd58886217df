"""YUV 4:2:0 input ("inputFormat" NV12 / I420), the parts that need no GPU: the restatement of cv::cvtColor's
conversion against cv2 itself, and the argument checks that run before any device work."""

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

from tracking_b200 import bgs, capi
from yuv_restate import yuv420_to_bgr

NV12, I420 = capi.INPUT_NV12, capi.INPUT_I420


def cv2_cvt(img, fmt):
    """cv::cvtColor itself"""
    return cv2.cvtColor(np.ascontiguousarray(img), {NV12: cv2.COLOR_YUV2BGR_NV12, I420: cv2.COLOR_YUV2BGR_I420}[fmt])


def every_triple():
    """One 4096 x 4096 frame holding every (Y, U, V) triple: each 2x2 block carries one of the 65536 (U, V) pairs and
    4 of the 256 Y values; the 64 copies of each pair cover all Y values.  -> (Y, U, V) planes."""
    H = W = 4096
    by, bx = np.mgrid[0:H // 2, 0:W // 2]
    blk = by * (W // 2) + bx
    uv, yg = blk % 65536, blk // 65536
    U, V = (uv & 255).astype(np.uint8), (uv >> 8).astype(np.uint8)
    Y = np.empty((H, W), np.uint8)
    for dy in range(2):
        for dx in range(2):
            Y[dy::2, dx::2] = (yg * 4 + dy * 2 + dx).astype(np.uint8)
    return Y, U, V


def pack(Y, U, V, fmt, pad=0):
    """The (3h/2, w) image of `fmt`; NV12 rows `pad` bytes wider than w (a view into the wider array)."""
    h, w = Y.shape
    if fmt == I420:
        return np.concatenate([Y.reshape(-1), U.reshape(-1), V.reshape(-1)]).reshape(h * 3 // 2, w)
    img = np.concatenate([Y, np.stack([U, V], -1).reshape(h // 2, w)], 0)
    if not pad:
        return img
    wide = np.full((h * 3 // 2, w + pad), 0x5A, np.uint8)
    wide[:, :w] = img
    return wide[:, :w]


def random_planes(h, w, seed):
    rng = np.random.default_rng(seed)
    return (rng.integers(0, 256, (h, w), dtype=np.uint8), rng.integers(0, 256, (h // 2, w // 2), dtype=np.uint8),
            rng.integers(0, 256, (h // 2, w // 2), dtype=np.uint8))


@pytest.mark.parametrize("fmt", [NV12, I420])
def test_restatement_equals_cv2_on_every_triple(fmt):
    Y, U, V = every_triple()
    img = pack(Y, U, V, fmt)
    got = yuv420_to_bgr(img, fmt)
    for threads in (1, 8):
        cv2.setNumThreads(threads)
        assert np.array_equal(got, cv2_cvt(img, fmt)), threads
    # the triples really are all there: 2^24 distinct (Y, U, V)
    Uf = np.repeat(np.repeat(U, 2, 0), 2, 1).astype(np.uint32)
    Vf = np.repeat(np.repeat(V, 2, 0), 2, 1).astype(np.uint32)
    assert np.unique(Y.astype(np.uint32) | Uf << 8 | Vf << 16).size == 1 << 24


@pytest.mark.parametrize("fmt,h,w,pad", [(NV12, 98, 130, 13), (NV12, 6, 10, 3), (NV12, 1080, 1920, 64),
                                         (I420, 98, 130, 0), (I420, 6, 10, 0), (I420, 2, 2, 0), (NV12, 2, 2, 5),
                                         (I420, 1082, 1918, 0), (NV12, 1082, 1918, 2)])
def test_restatement_equals_cv2_on_ragged_and_strided_frames(fmt, h, w, pad):
    """h % 4 == 2 (98, 6, 1082, 2), odd w/2 (130, 10, 1918: I420 chroma rows of odd length), padded NV12 rows"""
    img = pack(*random_planes(h, w, h * w), fmt, pad=pad)
    if pad:
        assert img.strides[0] == w + pad
    assert np.array_equal(yuv420_to_bgr(img, fmt), cv2_cvt(img, fmt))


def test_python_shape_and_format_refusals():
    ok = np.zeros((6, 8), np.uint8)
    img, h, w, grouped = bgs.yuv_frame(ok, NV12)
    assert (h, w, grouped) == (4, 8, False)
    img, h, w, grouped = bgs.yuv_frame(np.zeros((3, 6, 8), np.uint8), I420, nstreams=3)
    assert (h, w, grouped) == (4, 8, True)
    wide = np.zeros((6, 12), np.uint8)[:, :8]
    assert bgs.yuv_frame(wide, NV12)[0].strides[0] == 12            # NV12 keeps the row stride
    assert bgs.yuv_frame(wide, I420)[0].strides[0] == 8             # I420 planes are made dense
    bad = [(np.zeros((6, 8, 3), np.uint8), NV12, 1),                # a BGR frame
           (np.zeros((6, 8), np.uint16), NV12, 1),                  # not 8-bit
           (np.zeros((7, 8), np.uint8), NV12, 1),                   # 7 rows are not 3h/2 of any h
           (np.zeros((6, 7), np.uint8), I420, 1),                   # odd w
           (np.zeros((0, 8), np.uint8), NV12, 1),                   # empty
           (np.zeros((2, 6, 8), np.uint8), NV12, 3),                # wrong group size
           (np.zeros((6, 8), np.uint8), NV12, 2),                   # a group needs the stream axis
           (np.zeros((6, 8), np.uint8), capi.INPUT_BGR, 1),         # not a YUV format
           (np.zeros((6, 8), np.uint8), 3, 1)]                      # unknown format
    for img, fmt, S in bad:
        with pytest.raises(ValueError):
            bgs.yuv_frame(img, fmt, S)
    assert capi.INPUT_BGR == 0 and NV12 == 1 and I420 == 2


def test_header_enum_matches_capi():
    import os
    import re
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "bgsb200.h")).read()
    m = re.search(r"enum\s*\{\s*BGSB_INPUT_BGR\s*=\s*(\d+),\s*BGSB_INPUT_NV12\s*=\s*(\d+),\s*BGSB_INPUT_I420\s*=\s*(\d+)\s*\}", hdr)
    assert m and tuple(int(v) for v in m.groups()) == (capi.INPUT_BGR, NV12, I420)


def test_null_handles_are_refused_before_device_work():
    L = capi.lib()
    assert L.bgsb_set_param(None, b"inputFormat", 1) == capi.ERR_ARG
    assert L.bgsb_pool_set_param(None, b"inputFormat", 1) == capi.ERR_ARG
    assert L.bgsb_kernel_launch_count() == 0
