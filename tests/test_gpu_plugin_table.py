"""Per-plugin facts of the C ABI on a device: every parameter's default right after create, the model size
bgsb_state_bytes reports, and bgsb_process_fanout over all 13 plugins against the oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

F32 = lambda x: float(np.float32(x))       # noqa: E731  (loadConfig float literals read into doubles)

COMMON = {
    "alpha": 0.05, "limit": -1, "learningFrames": 90, "alphaLearn": 0.05, "alphaDetection": 0.05, "enableThreshold": 1,
    "threshold": 15, "samplingRate": 7, "historySize": 16, "ampFactor": 1, "minVar": 15, "maxVar": 255, "weight": 5,
    "gaussians": 3, "enableWeight": 1, "grayVariant": 0, "history": 500, "nmixtures": 5, "varThreshold": 16.0,
    "varThresholdGen": 9.0, "backgroundRatio": F32(0.9), "varInit": 15.0, "varMin": 4.0, "varMax": 75.0,
    "complexityReductionThreshold": F32(0.05), "detectShadows": 1, "shadowValue": 127, "shadowThreshold": 0.5,
    "kernelVariant": 0, "hostBands": 2, "retainInput": 0, "quietGroups": 1, "trace": 0, "ablTable": 1, "ablBlend": 0,
}
DEFAULTS = {
    0: {}, 1: {}, 2: {}, 3: {}, 5: {}, 6: {},
    7: {"threshold": 25},
    9: {"threshold": 40, "samplingRate": 7, "learningFrames": 30},
    11: {"threshold": 25.0, "alpha": 0.001},
    12: {"threshold": 2700, "alpha": F32(1e-6), "learningFrames": 30},
    13: {"threshold": F32(12.25), "alpha": F32(0.005), "learningFrames": 30},
    14: {"threshold": 30, "samplingRate": 5},
    35: {},
}
# bytes per pixel of bgsb_state_bytes at the default parameters
STATE_BPP = {0: 3, 1: 3, 2: 6, 3: 6, 5: 101, 6: 3, 7: 1, 9: 3, 11: 3 * 20 + 1, 12: 12, 13: 16, 14: 16 * 5 + 3, 35: 6}


def frames_of(h, w, n, seed):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    out = [np.clip(base.astype(np.int16) + rng.integers(-12, 13, (h, w, 3)), 0, 255).astype(np.uint8) for _ in range(n)]
    out[4][h // 4:h // 2, w // 4:w // 2] = 255 - out[4][h // 4:h // 2, w // 4:w // 2]
    return out


@pytest.mark.parametrize("aid", sorted(DEFAULTS))
def test_parameter_defaults_after_create(aid):
    import tracking_b200 as tb
    assert set(DEFAULTS) == set(tb.ALGOS)
    p = tb.ALGOS[aid]()
    want = dict(COMMON, **DEFAULTS[aid])
    got = {k: p.get(k) for k in want}
    p.close()
    assert got == want


@pytest.mark.parametrize("aid", sorted(STATE_BPP))
def test_state_bytes(aid):
    """0 before the first frame; the model of the latched parameters afterwards (DPZivkovic's gaussians and
    DPPratiMediod's historySize reach the model on the first frame only); the current parameters after reset()."""
    import tracking_b200 as tb
    h, w = 37, 53
    frames = frames_of(h, w, 5, aid)
    p = tb.ALGOS[aid]()
    assert p.state_bytes() == 0
    p.process(frames[0])
    p.set("gaussians", 5)
    p.set("historySize", 4)
    for f in frames[1:3]:
        p.process(f)
    assert p.frame_count == 3
    assert p.state_bytes() == h * w * STATE_BPP[aid]
    p.reset()
    after_reset = {11: 5 * 20 + 1, 14: 4 * 5 + 3}.get(aid, STATE_BPP[aid])
    assert p.state_bytes() == h * w * after_reset
    p.close()


@pytest.mark.parametrize("shape", [(97, 131), (600, 700)])
def test_fanout_all_plugins_match_oracle(oracle, shape):
    """Every plugin on one uploaded frame == the oracle's plugins run one by one, warm-up frames included;
    (600, 700) takes the row-band pipeline.  Each context then continues through its own process()."""
    import tracking_b200 as tb
    h, w = shape
    frames = frames_of(h, w, 7, 9)
    kw = {14: dict(historySize=2, samplingRate=1)}          # DPPratiMediod: masks from the third frame on
    aids = sorted(tb.ALGOS)
    ps = [tb.ALGOS[a](**kw.get(a, {})) for a in aids]
    os_ = [oracle.ALGOS[a](**kw.get(a, {})) for a in aids]
    for i, f in enumerate(frames[:6]):
        outs = tb.process_fanout(ps, f)
        for a, (fa, ba), o in zip(aids, outs, os_):
            fb, bb = o.process(f)
            assert (fa is None) == (fb is None), (a, i)
            assert (ba is None) == (bb is None), (a, i)
            if fa is not None:
                assert np.array_equal(fa, fb), (a, i)
            if ba is not None:
                assert np.array_equal(ba, bb), (a, i)
    for a, p, o in zip(aids, ps, os_):
        fa, ba = p.process(frames[6])
        fb, bb = o.process(frames[6])
        assert (fa is None) == (fb is None) and (ba is None) == (bb is None), a
        assert np.array_equal(fa, fb), a
        if bb is not None:
            assert np.array_equal(ba, bb), a
        p.close()
