"""Randomised parameter sweeps (seeded) of every hot-path plugin against the oracle, through the three ways a frame can
reach a kernel (host call, device call, stream group), plus robustness of the C ABI around them: two host threads on
their own contexts, error returns that leave a context usable."""
import threading

import numpy as np
import pytest

from conftest import stress_sequence
from param_draws import scene

pytestmark = pytest.mark.gpu


MOG2_KEYS = {"varThreshold": "Tb", "varThresholdGen": "Tg", "backgroundRatio": "TB", "varInit": "varInit", "varMin": "varMin",
             "varMax": "varMax", "complexityReductionThreshold": "CT", "shadowThreshold": "tau", "detectShadows": "detect_shadows",
             "shadowValue": "shadow_value", "history": "history"}


def random_mog2_params(rng):
    return {"alpha": float(rng.choice([-1.0, 0.001, 0.01, 0.05, 0.2, 0.5, 1.0])),
            "enableThreshold": int(rng.integers(0, 2)), "threshold": int(rng.choice([0, 15, 126, 127, 200, 254, 255])),
            "varThreshold": float(rng.choice([4, 9, 16, 30])), "varThresholdGen": float(rng.choice([3, 9, 16])),
            "backgroundRatio": float(rng.choice([0.5, 0.7, 0.9, 0.99])), "varInit": float(rng.choice([5, 15, 40])),
            "varMin": float(rng.choice([1, 4])), "varMax": float(rng.choice([40, 75, 200])),
            "complexityReductionThreshold": float(rng.choice([0.0, 0.05, 0.2])), "shadowThreshold": float(rng.choice([0.3, 0.5, 0.8])),
            "detectShadows": int(rng.integers(0, 2)), "shadowValue": int(rng.choice([127, 50, 200])), "history": int(rng.choice([10, 50, 500]))}


@pytest.mark.parametrize("trial", range(10))
def test_mog2_random_parameters_all_paths(oracle, trial):
    import torch
    import tracking_b200 as tb
    rng = np.random.default_rng(1000 + trial)
    h, w = int(rng.integers(20, 70)), int(rng.integers(20, 90))
    frames = scene(rng, 24, h, w) if trial % 2 else stress_sequence(24, h, w, seed=trial)
    kw = random_mog2_params(rng)

    def make_oracle():
        o = oracle.MixtureOfGaussianV2BGS(alpha=kw["alpha"], enableThreshold=bool(kw["enableThreshold"]), threshold=kw["threshold"])
        for k, field in MOG2_KEYS.items():
            setattr(o.params, field, type(getattr(o.params, field))(kw[k]))
        return o

    exp = [make_oracle().process(f) for f in [frames[0]]]          # smoke: construction works
    o = make_oracle()
    exp = [o.process(f) for f in frames]
    # host path
    p = tb.MixtureOfGaussianV2BGS(**kw)
    for t, f in enumerate(frames):
        fg, bg = p.process(f)
        assert np.array_equal(fg, exp[t][0]) and np.array_equal(bg, exp[t][1]), (kw, t)
    planes, nm = p.export_state()
    assert np.array_equal(nm, o.nmodes)
    p.close()
    # device path: T = 1 frames, then temporal batches of 7 (fused kernel), as a group of 2 identical streams
    q = tb.MixtureOfGaussianV2BGS(nstreams=2, **kw)
    T = 7
    for t0 in range(0, 21, T):
        host = np.stack([np.stack(frames[t0:t0 + T])] * 2)
        d_in = torch.from_numpy(host).cuda()
        d_fg = torch.zeros((2, T, h, w), dtype=torch.uint8, device="cuda")
        d_bg = torch.zeros((2, T, h, w, 3), dtype=torch.uint8, device="cuda")
        q.process_batch_dev(d_in.data_ptr(), T, w, h, d_fg.data_ptr(), d_bg.data_ptr())
        fg, bg = d_fg.cpu().numpy(), d_bg.cpu().numpy()
        for s in range(2):
            for t in range(T):
                assert np.array_equal(fg[s, t], exp[t0 + t][0]) and np.array_equal(bg[s, t], exp[t0 + t][1]), (kw, s, t0 + t)
    q.close()


@pytest.mark.parametrize("trial", range(6))
def test_simple_plugins_random_parameters(oracle, trial):
    import tracking_b200 as tb
    rng = np.random.default_rng(2000 + trial)
    h, w = int(rng.integers(8, 60)), int(rng.integers(8, 100))
    frames = scene(rng, 14, h, w)
    thr, en = int(rng.choice([0, 5, 15, 40, 254])), int(rng.integers(0, 2))
    gv = int(rng.integers(0, 2))
    cases = [(0, dict(enableThreshold=en, threshold=thr)), (1, dict(enableThreshold=en, threshold=thr)),
             (2, dict(enableThreshold=en, threshold=thr, enableWeight=int(rng.integers(0, 2)))),
             (3, dict(enableThreshold=en, threshold=thr, enableWeight=int(rng.integers(0, 2)))),
             (6, dict(enableThreshold=en, threshold=thr, alpha=float(rng.choice([0.01, 0.05, 0.3, 0.9]))))]
    for aid, kw in cases:
        p = tb.ALGOS[aid](grayVariant=gv, **kw)
        okw = {k: (bool(v) if k.startswith("enable") else v) for k, v in kw.items()}
        o = oracle.ALGOS[aid](gray_variant=gv, **okw)
        for t, f in enumerate(frames):
            fg, bg = p.process(f)
            ofg, obg = o.process(f)
            assert (fg is None) == (ofg is None) and (bg is None) == (obg is None), (aid, t)
            if fg is not None:
                assert np.array_equal(fg, ofg), (aid, kw, gv, t)
            if bg is not None:
                assert np.array_equal(bg, obg), (aid, kw, gv, t)
        p.close()


def test_two_host_threads_on_their_own_contexts(oracle):
    """Distinct contexts are independent: two threads drive a MOG2 and an ABL context at once (the header's contract)."""
    import tracking_b200 as tb
    rng = np.random.default_rng(5)
    frames = scene(rng, 30, 120, 160)
    results, errors = {}, []

    def work(aid):
        try:
            p = tb.ALGOS[aid]()
            out = [p.process(f) for f in frames]
            p.close()
            results[aid] = out
        except Exception as e:          # pragma: no cover
            errors.append(e)

    th = [threading.Thread(target=work, args=(aid,)) for aid in (5, 6, 5 + 0)]
    th[2] = threading.Thread(target=work, args=(3,))
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors, errors
    for aid in (5, 6, 3):
        o = oracle.ALGOS[aid]()
        for t, f in enumerate(frames):
            ofg, obg = o.process(f)
            fg, bg = results[aid][t]
            assert (fg is None) == (ofg is None)
            if fg is not None:
                assert np.array_equal(fg, ofg), (aid, t)
            if bg is not None:
                assert np.array_equal(bg, obg), (aid, t)


def test_errors_leave_the_context_usable(oracle):
    import ctypes as C
    import tracking_b200 as tb
    from tracking_b200 import capi
    p, o = tb.MixtureOfGaussianV2BGS(), oracle.MixtureOfGaussianV2BGS()
    f = stress_sequence(6, 30, 40, seed=3)
    p.process(f[0]); o.process(f[0])
    L = capi.lib()
    fv, bv = C.c_int(0), C.c_int(0)
    buf = np.zeros((30, 40, 3), np.uint8)
    fg = np.zeros((30, 40), np.uint8)
    # stride smaller than a row, null pointers, unknown keys: ERR_ARG, model untouched
    assert L.bgsb_process(p._h, buf.ctypes.data, 40, 30, 10, fg.ctypes.data, 40, None, 0, C.byref(fv), C.byref(bv)) == capi.ERR_ARG
    assert L.bgsb_process(p._h, None, 40, 30, 120, fg.ctypes.data, 40, None, 0, C.byref(fv), C.byref(bv)) == capi.ERR_ARG
    with pytest.raises(tb.BgsbError):
        p.set("noSuchKey", 1)
    with pytest.raises(tb.BgsbError):
        p.set("kernelVariant", 9)                # kernelVariant is 0 or 1
    assert b"kernelVariant" in L.bgsb_last_error()
    assert p.frame_count == 1
    for x in f[1:]:
        fg2, bg2 = p.process(x)
        ofg, obg = o.process(x)
        assert np.array_equal(fg2, ofg) and np.array_equal(bg2, obg)
    # geometry change = re-initialisation, like cv::BackgroundSubtractorMOG2::operator()
    big = stress_sequence(3, 50, 64, seed=4)
    for x in big:
        fg2, bg2 = p.process(x)
        ofg, obg = o.process(x)
        assert np.array_equal(fg2, ofg) and np.array_equal(bg2, obg)
    p.close()
