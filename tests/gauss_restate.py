"""Integer restatement of cv::GaussianBlur(img, Size(7, 7), 1.5) on 8-bit images (OpenCV 4.x), the blur the reference's
PreProcessor applies with its gaussianBlur switch.  OpenCV filters CV_8U with the 8-fraction-bit kernel
k = (9, 29, 55, 70, 55, 29, 9) (sum 256) in fixed point, rows then columns, and rounds once at the end:

    H(y, x, c) = sum_j k[j] * I(y, R_w(x + j - 3), c)          <= 65 280
    V(y, x, c) = sum_i k[i] * H(R_h(y + i - 3), x, c)          <  2^24
    out        = (V + 32768) >> 16

R_n is BORDER_REFLECT_101 (... 2 1 | 0 1 ... n-1 | n-2 ...), reflected again as cv::borderInterpolate does when n < 4.
Every channel is filtered on its own.  The reflection indices are computed here, without cv2."""
import numpy as np

K7 = np.array([9, 29, 55, 70, 55, 29, 9], dtype=np.int64)


def reflect101(p, n):
    """cv::borderInterpolate(p, n, BORDER_REFLECT_101)"""
    if n == 1:
        return 0
    while p < 0 or p >= n:
        p = -p if p < 0 else 2 * n - 2 - p
    return p


def gauss7(img):
    """(h, w, c) or (h, w) uint8 -> the same shape, as cv2.GaussianBlur(img, (7, 7), 1.5)"""
    a = np.asarray(img)
    assert a.dtype == np.uint8 and a.ndim in (2, 3)
    h, w = a.shape[:2]
    # the frame padded by 3 reflected pixels on each side, then the taps as shifted views (sums stay below 2^24)
    cols = np.array([reflect101(x, w) for x in range(-3, w + 3)])
    rows = np.array([reflect101(y, h) for y in range(-3, h + 3)])
    x = a.astype(np.int32)[:, cols]
    H = sum(int(K7[j]) * x[:, j:j + w] for j in range(7))[rows]
    V = sum(int(K7[i]) * H[i:i + h] for i in range(7))
    return ((V + 32768) >> 16).astype(np.uint8)


def gauss7_frames(frames):
    """a stack (..., h, w, 3) of frames, each blurred on its own"""
    a = np.asarray(frames)
    flat = a.reshape((-1,) + a.shape[-3:])
    return np.stack([gauss7(f) for f in flat]).reshape(a.shape)
