"""Every kernel form the launch routers choose from, checked by name against the oracle.

The routers (launch_simple / launch_asbl in simple_bgs.cu, launch_sigma_delta / launch_dp_simple in dp_simple.cu,
launch_mog2_t1 / launch_mog2_fused in mog2_t1.cu) pick a specialised kernel from the pixel count, the number of streams,
the frames per launch, the history state and the alignment of the caller's pointers.  All forms are meant to be
bit-exact, so a parity test alone cannot tell which one it checked.  Each row below therefore

  1. compares masks, background images and (where exposed) component tables with oracle/restate.py, bit for bit;
  2. cuts every caller buffer out of a larger allocation at the row's byte offset, with 0xA5 guard bytes on both
     sides, and checks after every call that no guard byte changed;
  3. records the CUDA kernels of the steady-state calls with torch.profiler and requires the set of library kernel
     names to equal the row's expected set (for a routing boundary this is the fallback form, so the fast form must
     not run).

The CPU-only inventory check requires every __global__ kernel of tracking_b200/csrc to be the expected kernel of some row.
"""
import collections
import glob
import os
import re
import warnings

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SENTINEL = 0xA5
GUARD = 64                 # guard bytes in front of the row's offset and behind the buffer (torch blocks are 512-aligned)

KERNEL_DECL = re.compile(r"__global__\s+(?:void\s+)?(?:__launch_bounds__\([^)]*\)\s*)?(?:void\s+)?(\w+)\s*\(")
KERNEL_NAME = re.compile(r"\w+_kernel")


def library_kernels():
    names = set()
    for path in sorted(glob.glob(os.path.join(ROOT, "tracking_b200", "csrc", "*.cu"))):
        with open(path) as f:
            names.update(KERNEL_DECL.findall(f.read()))
    return names


# kernels outside the plugin routers, run by existing tests
EXEMPT = {"synth_kernel": "tests/test_gpu_bgs.py::test_synth_generator_matches_numpy_twin",
          "synth_churn_kernel": "tests/test_gpu_bgs.py::test_churn_generator_matches_numpy_twin_and_keeps_modes_live"}

GPU_ONLY_KEYS = {"retainInput", "quietGroups", "ablTable", "kernelVariant"}


# ---------------------------------------------------------------------------------------------------------------------
# helpers

class Guarded:
    """`n` bytes at byte offset `off` inside a larger uint8 device allocation; everything around them is SENTINEL."""

    def __init__(self, n, off):
        import torch
        self.n, self.off = n, off
        self.base = torch.full((GUARD + off + n + GUARD,), SENTINEL, dtype=torch.uint8, device="cuda")
        self.view = self.base[GUARD + off:GUARD + off + n]
        assert self.view.data_ptr() % 16 == off % 16

    @property
    def ptr(self):
        return self.view.data_ptr()

    def put(self, arr):
        import torch
        self.view.copy_(torch.from_numpy(np.ascontiguousarray(arr).reshape(-1).view(np.uint8)))

    def get(self, shape, dtype=np.uint8):
        return self.view.cpu().numpy().view(dtype).reshape(shape)

    def check(self, what):
        b = self.base.cpu().numpy()
        head, tail = b[:GUARD + self.off], b[GUARD + self.off + self.n:]
        bad = np.flatnonzero(head != SENTINEL).tolist() + [GUARD + self.off + self.n + i for i in np.flatnonzero(tail != SENTINEL)]
        assert not bad, "%s: guard bytes changed at allocation offsets %s" % (what, bad[:8])


def profiled(fn, full_names=None):
    """Run fn() under the CUDA profiler; -> (Counter of library kernel names launched, fn's result).
    full_names: a list that receives the profiler's full (templated) name of every library kernel launch."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    known = library_kernels()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)           # "Profiler clears events at the end of each cycle"
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out = fn()
            torch.cuda.synchronize()
        events = prof.events()
    seen = collections.Counter()
    for e in events:
        if e.device_type == torch.autograd.DeviceType.CUDA:
            m = KERNEL_NAME.search(e.name)
            if m and m.group(0) in known:
                seen[m.group(0)] += 1
                if full_names is not None:
                    full_names.append(e.name)
    return seen, out


def last_template_arg(full_name, kernel):
    m = re.search(re.escape(kernel) + r"<([^>]*)>", full_name)
    return m.group(1).split(",")[-1].strip() if m else None


def scene(n, h, w, seed):
    """noisy static scene (+-6) crossed by a bright and a dark block, sudden re-lighting on every fifth frame"""
    rng = np.random.default_rng(seed)
    base = rng.integers(20, 236, (h, w, 3)).astype(np.int16)
    frames = []
    for t in range(n):
        f = base + rng.integers(-6, 7, (h, w, 3))
        if t % 5 == 4:
            f += 30
        y, x = (3 * t) % max(h - 8, 1), (7 * t) % max(w - 12, 1)
        f[y:y + 8, x:x + 12] = (250, 240, 10)
        f[(y + h // 2) % h:(y + h // 2) % h + 5, (x + w // 3) % w:(x + w // 3) % w + 9] //= 3
        frames.append(np.clip(f, 0, 255).astype(np.uint8))
    return frames


def oracle_kw(kw):
    out = {}
    for k, v in kw.items():
        if k in GPU_ONLY_KEYS:
            continue
        out["gray_variant" if k == "grayVariant" else k] = bool(v) if k.startswith("enable") else v
    return out


# ---------------------------------------------------------------------------------------------------------------------
# plugin rows: device entry point (bgsb_process_batch_dev), batches of T frames per stream, [S][T][h][w][3] layouts

class Row:
    """frames: byte offset of the frame buffers, or a tuple of offsets taken in turn by successive calls (under
    retainInput the previous buffers are the history, so this sets the history's alignment apart from the frames').
    prof: which calls are profiled -- "steady" (from call `skip` on), "first", "all", or a set of call indices.
    forms: kernel -> its last template argument in every profiled launch (e.g. WMV's quiet-shortcut flag).
    set_at: call index -> parameters changed on the plugin and the oracle before that call."""

    def __init__(self, id, aid, expect, h=64, w=512, S=1, T=1, n=5, kw=None, retain=0, bg=True, last=False,
                 frames=0, fg=0, bgo=0, prof="steady", skip=2, count=None, forms=None, set_at=None):
        self.id, self.aid, self.expect = id, aid, set(expect)
        self.h, self.w, self.S, self.T, self.n = h, w, S, T, n
        self.kw = dict(kw or {})
        if retain:
            self.kw["retainInput"] = 1
        self.bg, self.last = bg, last
        self.off = dict(frames=frames, fg=fg, bg=bgo)
        self.frame_offs = frames if isinstance(frames, tuple) else (frames,)
        self.prof, self.skip, self.count = prof, skip, count or {}
        self.forms, self.set_at = forms or {}, set_at or {}

    def profiled_call(self, b):
        if isinstance(self.prof, (set, frozenset)):
            return b in self.prof
        return (self.prof == "steady" and b >= self.skip) or (self.prof == "first" and b == 0) or self.prof == "all"

    def __repr__(self):
        return self.id


def run_row(oracle, r):
    import tracking_b200 as tb
    h, w, S, T, npx = r.h, r.w, r.S, r.T, r.h * r.w
    bgch = tb.ALGOS[r.aid].BG_CHANNELS
    seqs = [scene(r.n * T, h, w, seed=100 * r.aid + 7 * s + h) for s in range(S)]
    p = tb.ALGOS[r.aid](nstreams=S, **r.kw)
    os_ = [oracle.ALGOS[r.aid](**oracle_kw(r.kw)) for _ in range(S)]
    fg = Guarded(S * T * npx, r.off["fg"])
    nbg = S * (1 if r.last else T) * npx * bgch
    bg = Guarded(nbg, r.off["bg"]) if r.bg else None
    bufs = []                      # frame buffers stay alive and untouched: under retainInput they are the history
    seen, full = collections.Counter(), []
    for b in range(r.n):
        for k, v in r.set_at.get(b, {}).items():
            p.set(k, v)
            for o in os_:
                setattr(o, k, v)
        fr = Guarded(S * T * npx * 3, r.frame_offs[b % len(r.frame_offs)])
        fr.put(np.stack([np.stack(seqs[s][b * T:(b + 1) * T]) for s in range(S)]))
        bufs.append(fr)
        fg.view.fill_(SENTINEL)            # outputs of an earlier call cannot stand in for this call's
        if bg:
            bg.view.fill_(SENTINEL)

        def call():
            return p.process_batch_dev(fr.ptr, T, w, h, fg.ptr, bg.ptr if bg else None, bg_last_only=r.last)
        if r.profiled_call(b):
            got, (first, bgv) = profiled(call, full)
            seen.update(got)
        else:
            first, bgv = call()
        for g in bufs:
            g.check("%s frames" % r.id)
        fg.check("%s fg" % r.id)
        if bg:
            bg.check("%s bg" % r.id)
        out_fg = fg.get((S, T, h, w))
        out_bg = bg.get((S, 1 if r.last else T) + ((h, w, 3) if bgch == 3 else (h, w))) if bg else None
        for s in range(S):
            for t in range(T):
                ofg, obg = os_[s].process(seqs[s][b * T + t])
                where = (r.id, b, s, t)
                if ofg is None:
                    assert t < first and (out_fg[s, t] == SENTINEL).all(), where
                else:
                    assert t >= first and np.array_equal(out_fg[s, t], ofg), ("mask",) + where
                if bg and obg is not None and (not r.last or t == T - 1):
                    assert bgv, where
                    assert np.array_equal(out_bg[s, 0 if r.last else t], obg), ("background",) + where
    p.close()
    assert set(seen) == r.expect, "%s: kernels %s, expected %s" % (r.id, dict(seen), sorted(r.expect))
    for k, c in r.count.items():
        assert seen[k] == c, "%s: %s launched %d times, expected %d" % (r.id, k, seen[k], c)
    for k, arg in r.forms.items():
        args = {last_template_arg(n, k) for n in full if KERNEL_NAME.search(n).group(0) == k}
        assert args == {arg}, "%s: %s launched as <..., %s>, expected <..., %s>" % (r.id, k, sorted(args), arg)


FD, SFD, WMM, WMV, MOG2, ABL, ASBL = 0, 1, 2, 3, 5, 6, 7
AMED, DPZ, MEAN, WREN, PRATI, SD = 9, 11, 12, 13, 14, 35

ROWS = [
    # FrameDifference: whole 512-pixel chunks, 16-byte aligned frames / fg / history -> warp-coalesced kernel
    Row("fd_coalesced_64x512", FD, {"fd_coalesced_kernel"}, skip=1),
    Row("fd_coalesced_96x1024_S3_T3", FD, {"fd_coalesced_kernel"}, h=96, w=1024, S=3, T=3, n=3, skip=1),
    Row("fd_coalesced_64x512_S3_T3", FD, {"fd_coalesced_kernel"}, S=3, T=3, n=3, skip=1),
    Row("fd_coalesced_retain_96x1024", FD, {"fd_coalesced_kernel"}, h=96, w=1024, retain=1, skip=1),
    Row("fd_coalesced_retain_64x512_T3", FD, {"fd_coalesced_kernel"}, T=3, n=3, retain=1, skip=1),
    Row("fd_per_thread_frames+1", FD, {"fd_kernel"}, frames=1, skip=1),
    Row("fd_per_thread_96x1024_fg+1", FD, {"fd_kernel"}, h=96, w=1024, fg=1, skip=1),
    # retainInput: frame buffers at +8 and +0 in turn; the calls profiled (1, 3) read aligned frames and the previous
    # buffer, at +8, as their history
    Row("fd_per_thread_retain_history+8", FD, {"fd_kernel"}, frames=(8, 0), retain=1, prof={1, 3}),
    Row("fd_per_thread_528px", FD, {"fd_kernel"}, h=4, w=132, skip=1),
    Row("fd_per_thread_warmup_frame", FD, {"fd_kernel"}, n=2, prof="first"),
    # StaticFrameDifference
    Row("sfd_coalesced_64x512", SFD, {"sfd_coalesced_kernel"}, skip=1),
    Row("sfd_coalesced_S3", SFD, {"sfd_coalesced_kernel"}, S=3, skip=1),
    Row("sfd_coalesced_T4_bg_per_frame", SFD, {"sfd_coalesced_kernel"}, T=4, n=3, skip=1),
    Row("sfd_coalesced_T4_bg_last_only", SFD, {"sfd_coalesced_kernel"}, T=4, n=3, last=True, skip=1),
    Row("sfd_coalesced_no_bg", SFD, {"sfd_coalesced_kernel"}, bg=False, skip=1),
    Row("sfd_coalesced_raw", SFD, {"sfd_coalesced_kernel"}, kw=dict(enableThreshold=0), skip=1),
    Row("sfd_coalesced_thresholded", SFD, {"sfd_coalesced_kernel"}, kw=dict(enableThreshold=1, threshold=9), skip=1),
    Row("sfd_coalesced_gray1", SFD, {"sfd_coalesced_kernel"}, kw=dict(grayVariant=1), skip=1),
    Row("sfd_per_thread_first_frame", SFD, {"sfd_kernel"}, n=2, prof="first"),
    Row("sfd_per_thread_bg+4", SFD, {"sfd_kernel"}, bgo=4, skip=1),
    Row("sfd_per_thread_ragged", SFD, {"sfd_kernel"}, h=37, w=53, skip=1),
    # WeightedMovingMean: bulk-copy kernel once two history images exist
    Row("wmm_bulk_S1", WMM, {"wmm_bulk_kernel"}),
    Row("wmm_bulk_S1_raw", WMM, {"wmm_bulk_kernel"}, kw=dict(enableThreshold=0)),
    Row("wmm_bulk_S3_retain", WMM, {"wmm_bulk_kernel"}, S=3, retain=1),
    Row("wmm_bulk_S1_retain_no_bg_raw", WMM, {"wmm_bulk_kernel"}, retain=1, bg=False, kw=dict(enableThreshold=0)),
    Row("wmm_bulk_S3_no_bg_gray1", WMM, {"wmm_bulk_kernel"}, S=3, bg=False, kw=dict(grayVariant=1)),
    # frame buffers at +1, +0, +0 in turn: calls 2 and 5 read aligned frames with the older history at +1, call 4 with
    # the newer one at +1 (calls 0 and 1 are warm-up frames, remembered only)
    Row("wmm_per_thread_retain_history+1", WMM, {"wmm_kernel"}, retain=1, frames=(1, 0, 0), n=6, prof={2, 4, 5}),
    Row("wmm_bulk_retain_aligned_history", WMM, {"wmm_bulk_kernel"}, retain=1, frames=(16, 0, 32), n=6, prof={2, 3, 4, 5}),
    # WeightedMovingVariance
    Row("wmv_bulk_S1", WMV, {"wmv_bulk_kernel"}),
    # (retainInput: the warm-up frames launch nothing, so the bound table is built by the first launch, frame 2)
    Row("wmv_bulk_S3_retain", WMV, {"wmv_bulk_kernel"}, S=3, retain=1, n=6, skip=3),
    # (as WMM's row; the bound table is built by the first launch, call 2)
    Row("wmv_per_thread_retain_history+1", WMV, {"wmv_bound_table_kernel", "wmv_kernel"}, retain=1, frames=(1, 0, 0), n=6,
        prof={2, 4, 5}, count={"wmv_bound_table_kernel": 1}, forms={"wmv_kernel": "true"}),
    # last template argument of wmv_kernel: the quiet-group shortcut (threshold on and "quietGroups" 1)
    Row("wmv_per_thread_quiet_frames+1", WMV, {"wmv_kernel"}, frames=1, forms={"wmv_kernel": "true"}),
    Row("wmv_per_thread_raw", WMV, {"wmv_kernel"}, kw=dict(enableThreshold=0), forms={"wmv_kernel": "false"}),
    Row("wmv_per_thread_quiet_off", WMV, {"wmv_kernel"}, kw=dict(quietGroups=0), forms={"wmv_kernel": "false"}),
    Row("wmv_bound_table_weighted", WMV, {"wmv_bound_table_kernel", "wmv_kernel", "wmv_bulk_kernel"}, n=4, prof="all",
        count={"wmv_bound_table_kernel": 1}, forms={"wmv_kernel": "true"}),
    # unweighted (0.3 each): the bound of range 0 is already above threshold 15, so no range is quiet: no bulk launch
    Row("wmv_bound_table_unweighted", WMV, {"wmv_bound_table_kernel", "wmv_kernel"}, n=4, prof="all",
        kw=dict(enableWeight=0), count={"wmv_bound_table_kernel": 1}, forms={"wmv_kernel": "false"}),
    # AdaptiveBackgroundLearning
    Row("abl_bulk_table3", ABL, {"abl_bulk_kernel"}, kw=dict(ablTable=3)),
    Row("abl_lut_coalesced_64x512", ABL, {"abl_lut_coalesced_kernel"}),
    Row("abl_lut_coalesced_ragged", ABL, {"abl_lut_coalesced_kernel"}, h=37, w=53),
    Row("abl_lut_table2", ABL, {"abl_lut_kernel"}, kw=dict(ablTable=2)),
    Row("abl_lut_below_512px", ABL, {"abl_lut_kernel"}, h=13, w=29),
    Row("abl_lut_bg+1", ABL, {"abl_lut_kernel"}, bgo=1),
    Row("abl_arithmetic_table0", ABL, {"abl_kernel"}, kw=dict(ablTable=0)),
    Row("abl_lut_build_on_first_frame", ABL, {"abl_lut_build_kernel", "abl_lut_radius_kernel", "abl_lut_coalesced_kernel"},
        n=2, prof="first", kw=dict(alpha=0.3)),
    # alpha changed before call 2: the table is rebuilt once, for that call only
    Row("abl_lut_rebuild_on_alpha_change", ABL, {"abl_lut_build_kernel", "abl_lut_radius_kernel", "abl_lut_coalesced_kernel"},
        n=4, prof={2, 3}, set_at={2: {"alpha": 0.2}}, count={"abl_lut_build_kernel": 1, "abl_lut_radius_kernel": 1}),
    # AdaptiveSelectiveBackgroundLearning (gray model; learning phase ends after two frames)
    Row("asbl_fused16", ASBL, {"asbl_fused16_kernel"}, h=48, w=64, kw=dict(learningFrames=2)),
    Row("asbl_fused16_S3", ASBL, {"asbl_fused16_kernel"}, h=48, w=64, S=3, kw=dict(learningFrames=2)),
    Row("asbl_fused_w68", ASBL, {"asbl_fused_kernel"}, h=48, w=68, kw=dict(learningFrames=2)),
    Row("asbl_fused_frames+4", ASBL, {"asbl_fused_kernel"}, h=48, w=64, frames=4, kw=dict(learningFrames=2)),
    Row("asbl_two_pass_w66", ASBL, {"asbl_diff_kernel", "asbl_update_kernel"}, h=48, w=66, kw=dict(learningFrames=2)),
    Row("asbl_two_pass_frames+1", ASBL, {"asbl_diff_kernel", "asbl_update_kernel"}, h=48, w=64, frames=1,
        kw=dict(learningFrames=2)),
    # SigmaDelta
    Row("sd_coalesced", SD, {"sigma_delta_coalesced_kernel"}, bg=False, skip=1),
    Row("sd_coalesced_S3", SD, {"sigma_delta_coalesced_kernel"}, S=3, bg=False, skip=1),
    Row("sd_4px_fg+1", SD, {"sigma_delta_kernel"}, fg=1, bg=False, skip=1),
    Row("sd_4px_frames+1", SD, {"sigma_delta_kernel"}, frames=1, bg=False, skip=1),
    Row("sd_4px_ragged", SD, {"sigma_delta_kernel"}, h=37, w=53, bg=False, skip=1),
    Row("sd_initialiser_frames+1", SD, {"sigma_delta_kernel"}, frames=1, bg=False, n=2, prof="first"),
    # DPAdaptiveMedian (model updated every second frame)
    Row("amed_coalesced", AMED, {"dps_median_coalesced_kernel"}, bg=False, kw=dict(samplingRate=2), skip=1),
    Row("amed_coalesced_S3", AMED, {"dps_median_coalesced_kernel"}, S=3, bg=False, kw=dict(samplingRate=2), skip=1),
    Row("amed_4px_fg+1", AMED, {"dps_median_kernel"}, fg=1, bg=False, kw=dict(samplingRate=2), skip=1),
    Row("amed_4px_frames+1", AMED, {"dps_median_kernel"}, frames=1, bg=False, kw=dict(samplingRate=2), skip=1),
    Row("amed_4px_ragged", AMED, {"dps_median_kernel"}, h=37, w=53, bg=False, kw=dict(samplingRate=2), skip=1),
    # MOG2
    Row("mog2_t1_frames+1", MOG2, {"mog2_t1_kernel"}, h=33, w=64, frames=1, skip=1),
    Row("mog2_t1_fg+1", MOG2, {"mog2_t1_kernel"}, h=33, w=64, fg=1, skip=1),
    Row("mog2_t1_bg+1", MOG2, {"mog2_t1_kernel"}, h=33, w=64, bgo=1, skip=1),
    Row("mog2_t1_group_odd_px", MOG2, {"mog2_t1_kernel"}, h=33, w=41, S=3, skip=1),
    Row("mog2_fused_T8_all+1", MOG2, {"mog2_fused_kernel"}, h=33, w=41, T=8, n=3, frames=1, fg=1, bgo=1, skip=1),
    Row("mog2_restatement_variant1", MOG2, {"mog2_kernel"}, h=33, w=41, kw=dict(kernelVariant=1), skip=1),
    # alpha >= 1 re-initialises the model on every frame: batches run one frame (and one stream) per launch
    Row("mog2_reinit_T8_per_frame", MOG2, {"mog2_t1_kernel"}, h=33, w=41, T=8, n=3, kw=dict(alpha=1.5), skip=1),
    Row("mog2_reinit_T8_group_per_frame", MOG2, {"mog2_t1_kernel"}, h=33, w=41, S=2, T=8, n=3, kw=dict(alpha=1.0), skip=1),
]

# DPMean / DPWrenGA / DPPratiMediod / DPZivkovicAGMM: frame and mask pointers off the 4-byte grid (the v12 / v4 word
# paths fall back to bytes), and a 3-stream group whose per-stream strides are odd
_DP = {MEAN: ({"dps_float_kernel"}, {}), WREN: ({"dps_float_kernel"}, {}), DPZ: ({"dpz_kernel"}, {}),
       PRATI: ({"prati_subtract_kernel", "prati_update_kernel"}, dict(historySize=3, samplingRate=1))}
for _aid, (_exp, _kw) in _DP.items():
    _skip = 3 if _aid == PRATI else 1
    for _name, _o in (("frames+1", dict(frames=1)), ("frames+2", dict(frames=2)), ("frames+4", dict(frames=4)),
                      ("fg+1", dict(fg=1))):
        ROWS.append(Row("dp%d_%s" % (_aid, _name), _aid, _exp, h=32, w=40, n=6, bg=False, kw=_kw, skip=_skip, **_o))
    ROWS.append(Row("dp%d_S3_odd_px" % _aid, _aid, _exp, h=33, w=41, S=3, n=6, bg=False, kw=_kw, skip=_skip))


@pytest.mark.gpu
@pytest.mark.parametrize("row", ROWS, ids=repr)
def test_kernel_route(oracle, row):
    run_row(oracle, row)


# ---------------------------------------------------------------------------------------------------------------------
# pipeline (plugin -> morphology -> labelling), morphology and CCL entry points

PIPE_CHAIN = (("erode", 1), ("dilate", 1))
CCL_CHAIN = {"ccl_pack_kernel", "ccl_merge_kernel", "ccl_roots_kernel", "ccl_label_tile_kernel", "ccl_background_kernel"}
MORPH_CCL = {"morph_kernel"} | CCL_CHAIN
# the pipeline's morphology kernel packs the mask and creates the labeller's nodes: no pack launch
PIPE_STREAM = {"mog2_t1_stream_kernel"} | MORPH_CCL - {"ccl_pack_kernel"}
PIPE_GROUP = {"mog2_t1_kernel"} | MORPH_CCL - {"ccl_pack_kernel"}
PIPE_PHASES = PIPE_STREAM - {"ccl_background_kernel"} | {"ccl_background_phase_kernel", "ccl_gather_kernel"}
MOMENTS = {"rect_moments_kernel", "rect_moments_bits_kernel"}


def check_components(comps, exp):
    en, est, eext = exp
    assert len(comps) == en
    for c, st_, e in zip(comps, est, eext):
        assert (c["x"], c["y"], c["x"] + c["w"] - 1, c["y"] + c["h"] - 1, c["area"], c["first_index"]) == \
            tuple(int(v) for v in st_)
        assert c["external"] == int(e)


def run_pipeline(oracle, h, w, S, frames_off, expect, n=3, **params):
    """MOG2 pipeline on S streams; outputs mask, labels and (chainCtas) the gathered tables.  -> Counter of kernels."""
    import torch
    from tracking_b200 import capi
    from tracking_b200.pipeline import ForegroundPipeline
    seqs = [scene(n, h, w, seed=900 + s) for s in range(S)]
    pipe = ForegroundPipeline(MOG2, nstreams=S, morph=PIPE_CHAIN, **params)
    os_ = [oracle.MixtureOfGaussianV2BGS() for _ in range(S)]
    mask = Guarded(S * h * w, 0)
    lab = Guarded(S * h * w * 4, 0)
    rows = 64
    tab = Guarded(S * (rows + 1) * 32, 0)
    seen = collections.Counter()
    for t in range(n):
        fr = Guarded(S * h * w * 3, frames_off)
        fr.put(np.stack([seqs[s][t] for s in range(S)]))

        def call():
            v, _ = pipe.process_dev(fr.ptr, w, h, mask.ptr, None, lab.ptr)
            if "chainCtas" in params:
                capi.check(capi.lib().bgsb_pipeline_tables_dev(pipe._h, tab.ptr, rows, None))
            return v
        if t >= 1:
            got, valid = profiled(call)
            seen.update(got)
        else:
            valid = call()
            torch.cuda.synchronize()
        assert valid
        for g in (fr, mask, lab, tab):
            g.check("pipeline")
        m, lb = mask.get((S, h, w)), lab.get((S, h, w), np.int32)
        tb_ = tab.get((S, rows + 1, 8), np.int32)
        for s in range(S):
            ofg, _ = os_[s].process(seqs[s][t])
            clean = ofg
            for op, it in PIPE_CHAIN:
                clean = oracle.morph(clean, op, it)
            en, elab, est, eext = oracle.ccl8(clean, True)
            assert np.array_equal(m[s], clean), ("mask", t, s)
            assert np.array_equal(lb[s], elab), ("labels", t, s)
            comps = pipe.components(s)
            check_components(comps, (en, est, eext))
            if "chainCtas" in params:
                assert tb_[s, 0, 0] == en
                k = min(en, rows)
                keys = ("label", "first_index", "x", "y", "w", "h", "area", "external")
                assert tb_[s, 1:1 + k].tolist() == [[c[q] for q in keys] for c in comps[:k]], ("tables", t, s)
            if t == n - 1 and s == 0:
                rects = [(c["x"], c["y"], c["w"], c["h"]) for c in comps[:4]] + [(0, 0, w, h)]
                got, mom = profiled(lambda: pipe.rect_moments(rects, 0))
                assert set(got) == {"rect_moments_bits_kernel"}, dict(got)
                for rc, mm in zip(rects, mom):
                    assert mm == oracle.rect_moments(clean, rc), rc
    pipe.close()
    assert set(seen) == expect, "kernels %s, expected %s" % (dict(seen), sorted(expect))


@pytest.mark.gpu
def test_pipeline_1080p_streams_kernel(oracle):
    """Bit-packed pipeline masks on whole 64-pixel tiles with 16-byte aligned frames: the persistent stream kernel."""
    run_pipeline(oracle, 1080, 1920, 2, 0, PIPE_STREAM)


@pytest.mark.gpu
def test_pipeline_frames_off_16_bytes_take_the_group_kernel(oracle):
    run_pipeline(oracle, 64, 128, 2, 8, PIPE_GROUP)


@pytest.mark.gpu
def test_pipeline_plain_background_launches_and_gathered_tables(oracle):
    """"chainCtas": the labeller's background pass as four plain launches; tables gathered on the device."""
    run_pipeline(oracle, 64, 128, 2, 0, PIPE_PHASES, chainCtas=64, forceBackgroundPass=1)


@pytest.mark.gpu
@pytest.mark.parametrize("h,w,S,mask_off,lab_off", [(97, 131, 2, 1, 4), (64, 128, 2, 3, 4), (64, 128, 3, 1, 4),
                                                    (64, 128, 2, 0, 0)])
def test_morph_and_ccl_dev_at_offsets(oracle, h, w, S, mask_off, lab_off):
    """blobs.morph_dev and ConnectedComponents.label_batch_dev on masks off the 16-byte grid (the `vec` gates of
    morph.cu / ccl.cu) and labels that are int32- but not 16-byte aligned; then moments over the byte mask."""
    from tracking_b200 import blobs
    rng = np.random.default_rng(h * w + mask_off)
    masks = ((rng.random((S, h, w)) < 0.35) * 255).astype(np.uint8)
    src = Guarded(S * h * w, mask_off)
    dst = Guarded(S * h * w, mask_off)
    lab = Guarded(S * h * w * 4, lab_off)
    src.put(masks)
    cc = blobs.ConnectedComponents(w, h, max_images=S)

    def call():
        blobs.morph_dev(src.ptr, w, h, S, PIPE_CHAIN, dst.ptr)
        cc.label_batch_dev(dst.ptr, w, h, S, True, lab.ptr)
    got, _ = profiled(call)
    assert set(got) == MORPH_CCL, dict(got)
    for g in (src, dst, lab):
        g.check("morph/ccl")
    clean, lb = dst.get((S, h, w)), lab.get((S, h, w), np.int32)
    for s in range(S):
        exp = masks[s]
        for op, it in PIPE_CHAIN:
            exp = oracle.morph(exp, op, it)
        assert np.array_equal(clean[s], exp), s
        en, elab, est, eext = oracle.ccl8(exp, True)
        assert np.array_equal(lb[s], elab), s
        check_components(cc.components(s), (en, est, eext))
    rects = [(0, 0, w, h), (3, 2, w // 2, h // 3)]
    got, mom = profiled(lambda: cc.rect_moments(rects))
    assert set(got) == {"rect_moments_kernel"}, dict(got)
    for rc, mm in zip(rects, mom):
        assert mm == oracle.rect_moments(clean[0], rc), rc
    cc.close()


# ---------------------------------------------------------------------------------------------------------------------
# host boundary: bgsb_process into cv::Mat ROIs (row strides wider than the image)

HOST_KW = {PRATI: dict(historySize=3, samplingRate=1), AMED: dict(samplingRate=2), ASBL: dict(learningFrames=2)}


@pytest.mark.gpu
@pytest.mark.parametrize("aid", [FD, SFD, WMM, WMV, MOG2, ABL, ASBL, AMED, DPZ, MEAN, WREN, PRATI, SD])
def test_host_call_into_padded_rois(oracle, aid):
    import ctypes as C
    import tracking_b200 as tb
    from tracking_b200 import capi
    h, w = 37, 53
    frames = scene(7, h, w, seed=aid)
    kw = HOST_KW.get(aid, {})
    p, o = tb.ALGOS[aid](**kw), oracle.ALGOS[aid](**oracle_kw(kw))
    ch = tb.ALGOS[aid].BG_CHANNELS
    fg_stride, bg_stride = w + 13, ch * w + 7
    fg = np.full((h, fg_stride), SENTINEL, np.uint8)
    bg = np.full((h, bg_stride), SENTINEL, np.uint8)
    fv, bv = C.c_int(0), C.c_int(0)
    for t, f in enumerate(frames):
        capi.check(capi.lib().bgsb_process(p._h, f.ctypes.data, w, h, w * 3, fg.ctypes.data, fg_stride,
                                           bg.ctypes.data, bg_stride, C.byref(fv), C.byref(bv)))
        assert (fg[:, w:] == SENTINEL).all() and (bg[:, ch * w:] == SENTINEL).all(), ("padding", t)
        ofg, obg = o.process(f)
        assert bool(fv.value) == (ofg is not None) and bool(bv.value) == (obg is not None), t
        if ofg is not None:
            assert np.array_equal(fg[:, :w], ofg), ("mask", t)
        if obg is not None:
            assert np.array_equal(bg[:, :ch * w].reshape(obg.shape), obg), ("background", t)
    p.close()


# ---------------------------------------------------------------------------------------------------------------------
# CPU: every kernel of the library has a routed parity row



def test_every_kernel_has_a_routed_parity_row():
    kernels = library_kernels()
    assert len(kernels) >= 43
    covered = PIPE_STREAM | PIPE_GROUP | PIPE_PHASES | MORPH_CCL | MOMENTS
    for r in ROWS:
        covered |= r.expect
    assert covered <= kernels, "rows expect kernels that do not exist: %s" % sorted(covered - kernels)
    for name, test in EXEMPT.items():
        assert name in kernels
        path, fn = test.split("::")
        with open(os.path.join(ROOT, path)) as f:
            assert "def %s(" % fn in f.read(), test
    missing = kernels - covered - set(EXEMPT)
    assert not missing, "kernels without a routed parity row: %s" % sorted(missing)
