"""The kernels against the C restatement at the parameter draws of tests/param_draws.py -- the values at which
test_oracle_param_pins.py pins the restatement against OpenCV -- on every entry path a frame can take:

* MOG2: host call, process_dev, submit / wait, a group of 3 streams fed different input, process_batch_dev with T = 3
  on one stream (frame by frame on the T == 1 kernel) and T = 8 on a group of 2 (the temporal-fusion kernel), and the
  pipeline; masks, background images and the exported mixture state, on a tile-aligned and a ragged geometry;
* ASBL, DPZivkovic, the four DP models and SigmaDelta: host, device, a group of 2 and batches of 4;
* the pipeline and the stream pool with the plugin's threshold off and an erode / dilate chain, where the reference
  cleans the grey-level mask and DetectNewBlob thresholds afterwards."""
import numpy as np
import pytest

from conftest import stress_sequence
from param_draws import MOG2_FRAMES, alphas_per_frame, asbl_draws, dp_draws, mog2_draws, scene, segments

pytestmark = pytest.mark.gpu

MOG2 = mog2_draws()
MOG2_PATHS = ["host", "dev", "submit", "group3", "batch_T3", "group2_batch_T8", "pipeline"]


def mog2_geometry(name):
    """(h, w): 32 x 64 = 32 whole state tiles, or 23 x 37 (ragged)."""
    return (32, 64) if sorted(MOG2).index(name) % 2 == 0 else (23, 37)


def mog2_streams(name, S, h, w):
    seed = sum(map(ord, name))
    return [scene(np.random.default_rng(seed + s), MOG2_FRAMES, h, w) if s % 2 == 0 else
            stress_sequence(MOG2_FRAMES, h, w, seed=seed + s) for s in range(S)]


def mog2_expected(oracle, d, frames):
    o = oracle.MixtureOfGaussianV2BGS(enableThreshold=bool(d["enableThreshold"]), threshold=d["threshold"], **d["model"])
    out = []
    for a, f in zip(alphas_per_frame(d), frames):
        o.alpha = a
        out.append(o.process(f))
    return out, o


def check_mog2_state(planes, nm, o, what):
    assert np.array_equal(nm, o.nmodes), what
    for m in range(5):
        live = o.nmodes > m
        assert np.array_equal(planes[m * 5][live], o.gmm[:, m, 0][live]), (what, m)
        assert np.array_equal(planes[m * 5 + 1][live], o.gmm[:, m, 1][live]), (what, m)
        for c in range(3):
            assert np.array_equal(planes[m * 5 + 2 + c][live], o.mean[:, m, c][live]), (what, m, c)


@pytest.mark.parametrize("path", MOG2_PATHS)
@pytest.mark.parametrize("name", sorted(MOG2))
def test_mog2_parameter_space_on_every_path(oracle, name, path):
    import torch
    import tracking_b200 as tb
    d = MOG2[name]
    h, w = mog2_geometry(name)
    S = {"group3": 3, "group2_batch_T8": 2}.get(path, 1)
    streams = mog2_streams(name, S, h, w)
    exp = [mog2_expected(oracle, d, fr) for fr in streams]
    kw = dict(d["model"], enableThreshold=d["enableThreshold"], threshold=d["threshold"])
    alphas = alphas_per_frame(d)

    def check(s, t, fg, bg):
        efg, ebg = exp[s][0][t]
        assert np.array_equal(fg, efg), (name, path, s, t, int((fg != efg).sum()))
        assert np.array_equal(bg, ebg), (name, path, s, t, int((bg != ebg).sum()))

    if path == "pipeline":
        from tracking_b200.pipeline import ForegroundPipeline
        pipe = ForegroundPipeline(5, nstreams=1, morph=(), **kw)
        d_bg = torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda")
        d_mask = torch.zeros((h, w), dtype=torch.uint8, device="cuda")
        d_lab = torch.zeros((h, w), dtype=torch.int32, device="cuda")
        for t, f in enumerate(streams[0]):
            pipe.set("alpha", alphas[t])
            d_in = torch.from_numpy(f).cuda()
            pipe.process_dev(d_in.data_ptr(), w, h, d_mask.data_ptr(), d_bg.data_ptr(), d_lab.data_ptr())
            torch.cuda.synchronize()
            check(0, t, d_mask.cpu().numpy(), d_bg.cpu().numpy())
            assert np.array_equal(d_lab.cpu().numpy(), oracle.ccl8(exp[0][0][t][0], True)[1]), (name, t)
        check_mog2_state(*pipe.export_mog2_state(), exp[0][1], (name, path))
        pipe.close()
        return

    p = tb.MixtureOfGaussianV2BGS(nstreams=S, **kw)
    if path == "host":
        for t, f in enumerate(streams[0]):
            p.set("alpha", alphas[t])
            check(0, t, *p.process(f))
    elif path == "submit":
        fg, bg = np.zeros((h, w), np.uint8), np.zeros((h, w, 3), np.uint8)
        for t, f in enumerate(streams[0]):
            p.set("alpha", alphas[t])
            assert p.submit(np.ascontiguousarray(f), fg, bg) == (True, True)
            p.wait()
            check(0, t, fg, bg)
    elif path in ("dev", "group3"):
        d_fg = torch.zeros((S, h, w), dtype=torch.uint8, device="cuda")
        d_bg = torch.zeros((S, h, w, 3), dtype=torch.uint8, device="cuda")
        for t in range(MOG2_FRAMES):
            p.set("alpha", alphas[t])
            d_in = torch.from_numpy(np.stack([fr[t] for fr in streams])).cuda()
            p.process_dev(d_in.data_ptr(), w, h, d_fg.data_ptr(), d_bg.data_ptr())
            fg, bg = d_fg.cpu().numpy(), d_bg.cpu().numpy()
            for s in range(S):
                check(s, t, fg[s], bg[s])
    else:
        T = 3 if path == "batch_T3" else 8
        for t0, n, a in segments(d, T):
            p.set("alpha", a)
            d_in = torch.from_numpy(np.stack([np.stack(fr[t0:t0 + n]) for fr in streams])).cuda()
            d_fg = torch.zeros((S, n, h, w), dtype=torch.uint8, device="cuda")
            d_bg = torch.zeros((S, n, h, w, 3), dtype=torch.uint8, device="cuda")
            p.process_batch_dev(d_in.data_ptr(), n, w, h, d_fg.data_ptr(), d_bg.data_ptr())
            fg, bg = d_fg.cpu().numpy(), d_bg.cpu().numpy()
            for s in range(S):
                for k in range(n):
                    check(s, t0 + k, fg[s, k], bg[s, k])
    for s in range(S):
        check_mog2_state(*p.export_state(s), exp[s][1], (name, path, s))
    assert p.frame_count == MOG2_FRAMES
    p.close()


def test_mog2_alpha_switch_on_one_context_restarts_the_automatic_rate(oracle):
    """0.05 -> 1.0 (re-initialises) -> -1 (automatic rate counted from the re-initialisation) -> 0.05, on one context
    fed through the host call, device calls and batches in turn; also a reset in the middle."""
    import torch
    import tracking_b200 as tb
    h, w = 24, 40
    frames = stress_sequence(40, h, w, seed=21)
    sched = [0.05] * 6 + [1.0] * 3 + [-1.0] * 12 + [0.05] * 7 + [-1.0] * 12
    p = tb.MixtureOfGaussianV2BGS(enableThreshold=0, history=20)
    o = oracle.MixtureOfGaussianV2BGS(enableThreshold=False, history=20)
    t, was_reset = 0, False
    while t < len(frames):
        T = min(1 + t % 4, len(frames) - t)
        T = next((k for k in range(1, T) if sched[t + k] != sched[t]), T)        # a batch has one alpha
        p.set("alpha", sched[t])
        exp = []
        for k in range(T):
            o.alpha = sched[t + k]
            exp.append(o.process(frames[t + k]))
        if T == 1 and t % 2:
            got = [p.process(frames[t])]
        else:
            d_in = torch.from_numpy(np.stack(frames[t:t + T])).cuda()
            d_fg = torch.zeros((T, h, w), dtype=torch.uint8, device="cuda")
            d_bg = torch.zeros((T, h, w, 3), dtype=torch.uint8, device="cuda")
            p.process_batch_dev(d_in.data_ptr(), T, w, h, d_fg.data_ptr(), d_bg.data_ptr())
            got = list(zip(d_fg.cpu().numpy(), d_bg.cpu().numpy()))
        for k in range(T):
            assert np.array_equal(got[k][0], exp[k][0]) and np.array_equal(got[k][1], exp[k][1]), t + k
        t += T
        if t >= 30 and not was_reset:   # reset: the model and its frame counter start again
            was_reset = True
            p.reset()
            o = oracle.MixtureOfGaussianV2BGS(enableThreshold=False, history=20)
    check_mog2_state(*p.export_state(), o, "switch")
    p.close()


# ---- ASBL, DPZivkovic, DP models, SigmaDelta ----------------------------------------------------------------------

OTHER = [("AdaptiveSelectiveBackgroundLearning", kw) for kw in asbl_draws()[:10]] + dp_draws()


@pytest.mark.parametrize("geometry", [(16, 128), (13, 37)], ids=["aligned", "ragged"])
@pytest.mark.parametrize("i", range(len(OTHER)), ids=lambda i: "%s-%d" % (OTHER[i][0], i))
def test_other_plugins_parameter_space(oracle, i, geometry):
    """Host, device, a group of 2 with different input and batches of 4, against one restatement per stream."""
    import torch
    import tracking_b200 as tb
    cls, kw = OTHER[i]
    h, w = geometry
    n = 14
    fr = [scene(np.random.default_rng(100 + i), n, h, w), stress_sequence(n, h, w, seed=200 + i)]
    exp = []
    for s in range(2):
        o = getattr(oracle, cls)(**kw)
        exp.append([o.process(f) for f in fr[s]])
    bgc = 1 if cls == "AdaptiveSelectiveBackgroundLearning" else 3
    bgshape = (h, w) if bgc == 1 else (h, w, 3)

    def check(s, t, fg, bg, what):
        efg, ebg = exp[s][t]
        assert (fg is None) == (efg is None), (cls, kw, what, s, t)
        if efg is not None:
            assert np.array_equal(fg, efg), (cls, kw, what, s, t, int((fg != efg).sum()))
        if ebg is not None and bg is not None:
            assert np.array_equal(bg, ebg), (cls, kw, what, s, t)

    p = getattr(tb, cls)(**kw)
    for t, f in enumerate(fr[0]):
        check(0, t, *p.process(f), "host")
    p.close()
    for S, T in ((1, 1), (2, 1), (2, 4)):
        p = getattr(tb, cls)(nstreams=S, **kw)
        for t0 in range(0, n, T):
            k = min(T, n - t0)
            d_in = torch.from_numpy(np.stack([np.stack(fr[s][t0:t0 + k]) for s in range(S)])).cuda()
            d_fg = torch.zeros((S, k, h, w), dtype=torch.uint8, device="cuda")
            d_bg = torch.zeros((S, k) + bgshape, dtype=torch.uint8, device="cuda")
            if T == 1:
                fv, bv = p.process_dev(d_in.data_ptr(), w, h, d_fg.data_ptr(), d_bg.data_ptr())
                first = 0 if fv else 1
            else:
                first, bv = p.process_batch_dev(d_in.data_ptr(), k, w, h, d_fg.data_ptr(), d_bg.data_ptr())
            fg, bg = d_fg.cpu().numpy(), d_bg.cpu().numpy()
            for s in range(S):
                for j in range(k):
                    ok = j >= first
                    check(s, t0 + j, fg[s, j] if ok else None, bg[s, j] if ok and bv else None, (S, T))
        p.close()


# ---- pipeline / pool: threshold off, clean-up chain ---------------------------------------------------------------

RAW_CHAINS = {"open": (("erode", 1), ("dilate", 1)), "dilate2_erode2": (("dilate", 2), ("erode", 2))}
RAW_PLUGINS = {"mog2_shadows": (5, {}), "fd": (0, {}), "abl": (6, {"alpha": 0.2})}


def reference_blobs(oracle, raw, chain, zero_border):
    """The reference's order: erode / dilate on the raw grey-level mask, then DetectNewBlob's > 128 and labelling."""
    clean = raw
    for op, it in chain:
        clean = oracle.morph(clean, op, it)
    return oracle.ccl8(clean, zero_border)


def check_components(comps, n, st, ext, what):
    assert len(comps) == n, what
    for c, row, e in zip(comps, st, ext):
        assert (c["x"], c["y"], c["x"] + c["w"] - 1, c["y"] + c["h"] - 1, c["area"], c["first_index"]) == \
            tuple(int(v) for v in row), what
        assert c["external"] == int(e), what


@pytest.mark.parametrize("zero_border", [0, 1])
@pytest.mark.parametrize("chain", sorted(RAW_CHAINS))
@pytest.mark.parametrize("plugin", sorted(RAW_PLUGINS))
def test_pipeline_raw_mask_with_chain_labels_as_the_reference(oracle, clips, plugin, chain, zero_border):
    import torch
    import tracking_b200 as tb
    from tracking_b200.pipeline import ForegroundPipeline
    aid, kw = RAW_PLUGINS[plugin]
    clip = clips["video_clip"][:16]
    h, w = clip.shape[1:3]
    S = 2
    pipe = ForegroundPipeline(aid, nstreams=S, morph=RAW_CHAINS[chain], enableThreshold=0, zeroBorder=zero_border, **kw)
    os_ = [oracle.ALGOS[aid](enableThreshold=False, **kw) for _ in range(S)]
    d_lab = torch.zeros((S, h, w), dtype=torch.int32, device="cuda")
    d_mask = torch.zeros((S, h, w), dtype=torch.uint8, device="cuda")
    grey = False
    for t in range(len(clip)):
        frames = np.stack([clip[t], clip[(3 * t + 5) % len(clip)]])
        d_in = torch.from_numpy(frames).cuda()
        # the cleaned mask of this combination is grey-level: refused, and the model is not advanced
        with pytest.raises(tb.BgsbError):
            pipe.process_dev(d_in.data_ptr(), w, h, d_mask.data_ptr(), None, d_lab.data_ptr())
        valid, _ = pipe.process_dev(d_in.data_ptr(), w, h, None, None, d_lab.data_ptr())
        torch.cuda.synchronize()
        raws = [os_[s].process(frames[s])[0] for s in range(S)]
        assert valid == (raws[0] is not None), t
        if raws[0] is None:
            continue
        for s in range(S):
            grey |= bool(((raws[s] > 0) & (raws[s] < 255)).any())
            n, lab, st, ext = reference_blobs(oracle, raws[s], RAW_CHAINS[chain], bool(zero_border))
            assert np.array_equal(d_lab[s].cpu().numpy(), lab), (plugin, chain, t, s)
            check_components(pipe.components(s), n, st, ext, (plugin, chain, t, s))
        with pytest.raises(tb.BgsbError):
            pipe.rect_moments([(0, 0, w, h)], 0)
    assert grey                        # the raw masks did hold values between 0 and 255
    pipe.close()


def test_pool_raw_mask_with_chain(oracle, clips):
    """The stream pool inherits the pipeline's order (tables only: masks are refused in this combination)."""
    from tracking_b200 import capi
    from tracking_b200.streams import StreamPool
    clip = clips["video_clip"]
    h, w = clip.shape[1:3]
    chain, ring, S = RAW_CHAINS["open"], 2, 3
    pool = StreamPool(capi.ALGO_MOG2, S, w, h, devices=[0], ring=ring, morph=chain, enableThreshold=0)
    os_ = [oracle.MixtureOfGaussianV2BGS(enableThreshold=False) for _ in range(S)]
    frame_of = lambda s, t: clip[(t * (1 + s) + 7 * s) % len(clip)]
    for t in range(10):
        slot = t % ring
        for s in range(S):
            pool.frame_buffer(s, slot)[...] = frame_of(s, t)
        pool.submit(slot, False)
        assert pool.wait(slot)
        for s in range(S):
            raw, _ = os_[s].process(frame_of(s, t))
            n, lab, st, ext = reference_blobs(oracle, raw, chain, True)
            check_components(pool.components(s, slot), n, st, ext, (t, s))
    pool.close()
