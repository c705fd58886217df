"""TEST INFRASTRUCTURE ONLY - restatement of cv::cvtColor(COLOR_YUV2BGR_NV12 / COLOR_YUV2BGR_I420) on 8-bit data.

OpenCV's BT.601 limited-range 20-bit fixed point (modules/imgproc/src/color_yuv.simd.hpp), each U,V pair shared by a
2x2 block of Y samples:

    y = max(Y - 16, 0) * CY;  u = U - 128;  v = V - 128
    B = sat_u8((y + 2^19 + CUB * u) >> 20)
    G = sat_u8((y + 2^19 + CVG * v + CUG * u) >> 20)
    R = sat_u8((y + 2^19 + CVR * v) >> 20)

Integer numpy, so it is exact.  Pinned against cv2 on all 2^24 (Y, U, V) triples, on strided NV12, on h % 4 == 2 and on
odd w/2 by tests/test_yuv_input.py; the GPU tests feed its output to the BGR path and to the oracle's plugins.
"""
from __future__ import annotations

import numpy as np

NV12, I420 = 1, 2      # "inputFormat" values (BGSB_INPUT_NV12 / BGSB_INPUT_I420)
CY, CUB, CUG, CVG, CVR, SHIFT = 1220542, 2116026, -409993, -852492, 1673527, 20


def planes(img, fmt):
    """(3h/2, w) image -> (Y [h, w], U [h/2, w/2], V [h/2, w/2]); NV12 rows may be strided (a view into a wider array)"""
    img = np.asarray(img, np.uint8)
    rows, w = img.shape
    h = 2 * rows // 3
    assert img.ndim == 2 and rows == 3 * h // 2 and w % 2 == 0 and h % 2 == 0 and fmt in (NV12, I420)
    Y = img[:h]
    if fmt == NV12:
        uv = img[h:]
        return Y, uv[:, 0::2], uv[:, 1::2]
    flat = np.ascontiguousarray(img).reshape(-1)
    q = (h // 2) * (w // 2)
    return Y, flat[h * w:h * w + q].reshape(h // 2, w // 2), flat[h * w + q:].reshape(h // 2, w // 2)


def yuv420_to_bgr(img, fmt):
    """cv::cvtColor of a (3h/2, w) uint8 image: fmt 1 COLOR_YUV2BGR_NV12, fmt 2 COLOR_YUV2BGR_I420 -> (h, w, 3) BGR"""
    Y, U, V = planes(img, fmt)
    u = np.repeat(np.repeat(U.astype(np.int32) - 128, 2, 0), 2, 1)
    v = np.repeat(np.repeat(V.astype(np.int32) - 128, 2, 0), 2, 1)
    y = np.maximum(Y.astype(np.int32) - 16, 0) * CY + (1 << (SHIFT - 1))
    bgr = np.stack([(y + CUB * u) >> SHIFT, (y + CVG * v + CUG * u) >> SHIFT, (y + CVR * v) >> SHIFT], -1)
    return np.clip(bgr, 0, 255).astype(np.uint8)
