"""The "gaussianBlur" pre-processing stage on the CPU: the integer restatement (tests/gauss_restate.py) against
cv2.GaussianBlur(img, (7, 7), 1.5) with 1 and 8 threads, and the argument checks that need no GPU."""
import numpy as np
import pytest

from gauss_restate import K7, gauss7, reflect101

cv2 = pytest.importorskip("cv2")


def blur_cv2(img, threads):
    old = cv2.getNumThreads()
    cv2.setNumThreads(threads)
    try:
        return cv2.GaussianBlur(img, (7, 7), 1.5)
    finally:
        cv2.setNumThreads(old)


def same(a, img, what):
    for threads in (1, 8):
        want = blur_cv2(img, threads)
        d = np.flatnonzero(a.reshape(-1) != want.reshape(-1))
        assert d.size == 0, "%s (%d threads): %d bytes differ, first at %s" % (what, threads, d.size, d[:5].tolist())


def contents(h, w, seed):
    """noise, all-255, 0/255 checkerboards of pixels and of channels, and impulses at the corners and edge midpoints"""
    rng = np.random.default_rng(seed)
    yield "noise", rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    yield "all-255", np.full((h, w, 3), 255, np.uint8)
    yy, xx = np.mgrid[0:h, 0:w]
    yield "checker", np.repeat((((yy + xx) & 1) * 255).astype(np.uint8)[..., None], 3, -1)
    cc = (((yy[..., None] + xx[..., None] + np.arange(3)) & 1) * 255).astype(np.uint8)
    yield "channel checker", cc
    imp = np.zeros((h, w, 3), np.uint8)
    for y, x in ((0, 0), (0, w - 1), (h - 1, 0), (h - 1, w - 1), (h // 2, 0), (0, w // 2), (h - 1, w // 2), (h // 2, w - 1)):
        imp[y, x] = (255, 128, 1)
    yield "impulses", imp


def test_kernel_is_opencvs_fixed_point_gaussian():
    """k is the 8-fraction-bit kernel cv::getGaussianKernel(7, 1.5, CV_8U-fixed) rounds to: sum 256, symmetric"""
    assert K7.sum() == 256 and (K7 == K7[::-1]).all()
    g = cv2.getGaussianKernel(7, 1.5).ravel()
    assert np.abs(K7 / 256.0 - g).max() < 1.0 / 256


def test_reflect101_is_cv_border_interpolate():
    for n in range(1, 10):
        for p in range(-9, n + 9):
            assert reflect101(p, n) == cv2.borderInterpolate(p, n, cv2.BORDER_REFLECT_101), (p, n)


@pytest.mark.parametrize("h", range(1, 10))
def test_every_small_shape(h):
    for w in range(1, 10):
        for what, img in contents(h, w, seed=h * 16 + w):
            same(gauss7(img), img, "%d x %d %s" % (h, w, what))


@pytest.mark.parametrize("h,w", [(1080, 1920), (37, 53), (270, 481), (33, 127), (1, 1921), (1081, 1), (1, 64), (64, 1)])
def test_larger_odd_and_one_line_shapes(h, w):
    for what, img in contents(h, w, seed=h + 7 * w):
        same(gauss7(img), img, "%d x %d %s" % (h, w, what))


def test_channels_are_independent():
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, (23, 31, 3), dtype=np.uint8)
    got = gauss7(img)
    for c in range(3):
        assert np.array_equal(got[..., c], gauss7(np.ascontiguousarray(img[..., c])))


def test_plugin_refusals_without_gpu():
    """values other than 0 / 1 and retainInput in either order are refused by the library before any device work"""
    from tracking_b200 import capi
    import tracking_b200 as tb
    try:
        capi.lib()
    except Exception as e:                      # library not built
        pytest.skip("library unavailable: %s" % e)
    try:
        p = tb.ALGOS[0]()
    except capi.BgsbError as e:                 # no CUDA device: a context cannot be created here
        pytest.skip("no device: %s" % e)
    try:
        for bad in (2, -1, 0.5):
            with pytest.raises(capi.BgsbError) as e:
                p.set("gaussianBlur", bad)
            assert e.value.code == capi.ERR_ARG and "gaussianBlur is 0 or 1" in str(e.value)
        p.set("gaussianBlur", 1)
        assert p.get("gaussianBlur") == 1
        with pytest.raises(capi.BgsbError) as e:
            p.set("retainInput", 1)
        assert e.value.code == capi.ERR_ARG and "cannot be combined with gaussianBlur" in str(e.value)
        p.set("gaussianBlur", 0)
        p.set("retainInput", 1)
        with pytest.raises(capi.BgsbError) as e:
            p.set("gaussianBlur", 1)
        assert e.value.code == capi.ERR_ARG and "cannot be combined with retainInput" in str(e.value)
        assert p.get("gaussianBlur") == 0
    finally:
        p.close()
