"""MOG2 on constructed model states at every decision boundary of its update (tests/mog2_edges.py), on every kernel
route, bit for bit against the C oracle.

Each route imports the fixture's state (bgsb_mog2_import_state) into the plugin and the same state into the oracle
object, runs the fixture's eight frames (one per call, or as batches) and compares the raw or thresholded mask and the
background image of every frame, then the exported state (mode counts and live slots).  The routes:

    t1             process_dev, one stream                      mog2_t1_kernel
    group3_t1      process_dev, a group of 3                    mog2_t1_kernel (group form)
    fused_T8       process_batch_dev T = 8, per-frame images    mog2_fused_kernel
    fused_T8_last  process_batch_dev T = 8, bg_last_only        mog2_fused_kernel
    group2_T8      process_batch_dev T = 8, a group of 2        mog2_fused_kernel
    batch_T3       process_batch_dev T = 3, 3, 2 (frame by frame on the T == 1 kernel)
    host_banded    process, "hostBands" 3 on 352 x 1024         mog2_t1_kernel
    pipeline       ForegroundPipeline.process_dev, 2 streams, 64 x 128, no chain, packed mask
                                                                mog2_t1_stream_kernel
    variant1       "kernelVariant" 1, process_batch_dev T = 8  mog2_kernel

The pipeline learns its geometry from its first frame, so it runs one frame before the import; the import replaces
everything that frame did (state, mode counts and the frame counter).  The pipeline's mask is the packed, thresholded
one: it runs with enableThreshold = 1 (threshold 127 where the parameter set has the threshold off, which keeps
shadow and foreground apart).

Which kernel each route ran is checked by name with torch.profiler in a child process (late in a long session the
profiler has been seen to deliver only part of a call's kernel records).
"""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

import mog2_edges as E
from test_gpu_param_space import check_mog2_state

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROUTES = {"t1": ("main", 1, "mog2_t1_kernel"), "group3_t1": ("main", 3, "mog2_t1_kernel"),
          "fused_T8": ("main", 1, "mog2_fused_kernel"), "fused_T8_last": ("main", 1, "mog2_fused_kernel"),
          "group2_T8": ("main", 2, "mog2_fused_kernel"), "batch_T3": ("main", 1, "mog2_t1_kernel"),
          "host_banded": ("banded", 1, "mog2_t1_kernel"), "pipeline": ("aligned", 2, "mog2_t1_stream_kernel"),
          "variant1": ("main", 1, "mog2_kernel")}


@functools.lru_cache(maxsize=48)
def fixture(pname, kind, S):
    return E.layout(E.params(pname), kind, S)


def route_params(route, pname):
    p = E.params(pname)
    if route == "pipeline" and not p["enableThreshold"]:
        p.update(enableThreshold=1, threshold=127)
    return p


def where(lay, s, bad):
    """group names of the mismatching pixels (flat indices)"""
    names = {i: lay["groups"][gi]["name"] for ss, i, gi, mi, tags in lay["where"] if ss == s}
    return sorted({names.get(int(i), "filler") for i in np.flatnonzero(bad)})[:12]


def expected(oracle, lay, p, S):
    h, w = lay["h"], lay["w"]
    out, objs = [], []
    for s in range(S):
        o = E.oracle_with_state(oracle, p, lay["planes"][s], lay["nmodes"][s], h, w)
        out.append([o.process(lay["frames"][s, t]) for t in range(E.T)])
        objs.append(o)
    return out, objs


def plugin(p, S, **extra):
    import tracking_b200 as tb
    kw = E.model_kwargs(p)
    kw.update(extra)
    return tb.MixtureOfGaussianV2BGS(nstreams=S, **kw)


def run_route(oracle, route, pname, calls=None):
    """calls: a list that receives (what, zero-argument callable) of one kernel-running call, for the profiler"""
    import torch
    kind, S, _ = ROUTES[route]
    p = route_params(route, pname)
    lay = fixture(pname, kind, S)
    h, w, T = lay["h"], lay["w"], E.T
    frames = lay["frames"]
    exp, objs = expected(oracle, lay, p, S)

    def check(s, t, fg, bg, what=""):
        efg, ebg = exp[s][t]
        bad = fg.reshape(-1) != efg.reshape(-1)
        assert not bad.any(), (route, pname, s, t, "mask", what, int(bad.sum()), where(lay, s, bad))
        if bg is not None:
            badb = (bg.reshape(-1, 3) != ebg.reshape(-1, 3)).any(1)
            assert not badb.any(), (route, pname, s, t, "background", what, int(badb.sum()), where(lay, s, badb))

    def check_state(export):
        for s in range(S):
            planes, nm = export(s)
            bad = nm != objs[s].nmodes
            assert not bad.any(), (route, pname, s, "nmodes", where(lay, s, bad))
            check_mog2_state(planes, nm, objs[s], (route, pname, s))

    if route == "pipeline":
        from tracking_b200 import capi
        from tracking_b200.pipeline import ForegroundPipeline
        kw = E.model_kwargs(p)
        pipe = ForegroundPipeline(5, nstreams=S, morph=(), **kw)
        d_mask = torch.zeros((S, h, w), dtype=torch.uint8, device="cuda")
        d_bg = torch.zeros((S, h, w, 3), dtype=torch.uint8, device="cuda")
        d_in = torch.from_numpy(np.ascontiguousarray(frames[:, 0])).cuda()
        pipe.process_dev(d_in.data_ptr(), w, h, d_mask.data_ptr(), d_bg.data_ptr())
        torch.cuda.synchronize()
        for s in range(S):
            pl = np.ascontiguousarray(lay["planes"][s])
            nm = np.ascontiguousarray(lay["nmodes"][s])
            capi.check(capi.lib().bgsb_mog2_import_state(pipe.bgs_handle, s, w, h, lay["nframes"],
                                                         pl.ctypes.data_as(capi.f32p), nm.ctypes.data_as(capi.u8p)))
        for t in range(T):
            d_in = torch.from_numpy(np.ascontiguousarray(frames[:, t])).cuda()
            call = lambda d_in=d_in: (pipe.process_dev(d_in.data_ptr(), w, h, d_mask.data_ptr(), d_bg.data_ptr()),  # noqa: E731
                                      torch.cuda.synchronize())
            if calls is not None and t == 1:
                calls.append((route, call))
                break
            call()
            m, b = d_mask.cpu().numpy(), d_bg.cpu().numpy()
            for s in range(S):
                check(s, t, m[s], b[s])
        if calls is None:
            check_state(pipe.export_mog2_state)
        return pipe

    extra = {"kernelVariant": 1} if route == "variant1" else {}
    if route == "host_banded":
        extra.update(hostBands=3, trace=1)
    plug = plugin(p, S, **extra)
    for s in range(S):
        plug.import_state(lay["planes"][s], lay["nmodes"][s], w, h, lay["nframes"], s)
    if route == "host_banded":
        for t in range(T):
            call = lambda t=t: plug.process(frames[0, t])             # noqa: E731
            if calls is not None:
                calls.append((route, call))
                return plug
            fg, bg = call()
            assert plug.trace_last()["bands"] == 3
            check(0, t, fg, bg)
    elif route in ("t1", "group3_t1"):
        d_fg = torch.zeros((S, h, w), dtype=torch.uint8, device="cuda")
        d_bg = torch.zeros((S, h, w, 3), dtype=torch.uint8, device="cuda")
        for t in range(T):
            d_in = torch.from_numpy(np.ascontiguousarray(frames[:, t])).cuda()
            call = lambda d_in=d_in: plug.process_dev(d_in.data_ptr(), w, h, d_fg.data_ptr(), d_bg.data_ptr())  # noqa: E731
            if calls is not None:
                calls.append((route, call))
                return plug
            call()
            fg, bg = d_fg.cpu().numpy(), d_bg.cpu().numpy()
            for s in range(S):
                check(s, t, fg[s], bg[s])
    else:
        segs = [(0, 3), (3, 3), (6, 2)] if route == "batch_T3" else [(0, T)]
        last = route == "fused_T8_last"
        for t0, n in segs:
            d_in = torch.from_numpy(np.ascontiguousarray(frames[:, t0:t0 + n])).cuda()
            d_fg = torch.zeros((S, n, h, w), dtype=torch.uint8, device="cuda")
            d_bg = torch.zeros((S, 1 if last else n, h, w, 3), dtype=torch.uint8, device="cuda")
            call = lambda d_in=d_in, n=n, d_fg=d_fg, d_bg=d_bg: plug.process_batch_dev(  # noqa: E731
                d_in.data_ptr(), n, w, h, d_fg.data_ptr(), d_bg.data_ptr(), bg_last_only=last)
            if calls is not None:
                calls.append((route, call))
                return plug
            call()
            fg, bg = d_fg.cpu().numpy(), d_bg.cpu().numpy()
            for s in range(S):
                for k in range(n):
                    if last:
                        check(s, t0 + k, fg[s, k], bg[s, 0] if k == n - 1 else None)
                    else:
                        check(s, t0 + k, fg[s, k], bg[s, k])
    check_state(plug.export_state)
    assert plug.frame_count == lay["nframes"] + T
    return plug


@pytest.mark.parametrize("pname", sorted(E.PARAMS))
@pytest.mark.parametrize("route", sorted(ROUTES))
def test_mog2_edges_on_every_route(oracle, route, pname):
    run_route(oracle, route, pname).close()


def kernel_rows():
    """the body of test_each_route_runs_its_kernel, in a fresh process"""
    from oracle import restate
    from test_gpu_kernel_routes import profiled
    restate.build()
    for route, (_, _, kernel) in sorted(ROUTES.items()):
        calls = []
        obj = run_route(restate, route, "defaults", calls)
        (what, call), = calls
        seen, _ = profiled(call)
        assert set(seen) & {"mog2_t1_kernel", "mog2_fused_kernel", "mog2_t1_stream_kernel", "mog2_kernel"} == {kernel}, \
            (route, dict(seen))
        obj.close()
    print("ok kernel rows")


def test_each_route_runs_its_kernel():
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_gpu_mog2_edges as m; m.kernel_rows()"
            % (ROOT, os.path.join(ROOT, "tests")))
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-6000:]
    assert "ok kernel rows" in res.stdout, res.stdout


def test_import_refuses_more_than_five_modes(oracle):
    """A mode count above K = 5 is refused with BGSB_ERR_ARG before anything changes; the context keeps its state.
    Then a valid import runs one frame against the oracle (the refused state never reaches a kernel)."""
    import tracking_b200 as tb
    p = E.params()
    lay = fixture("defaults", "main", 1)
    h, w = lay["h"], lay["w"]
    plug = plugin(p, 1)
    plug.import_state(lay["planes"][0], lay["nmodes"][0], w, h, lay["nframes"])
    before = plug.export_state()
    count = plug.frame_count
    for bad in (6, 255):
        nm = lay["nmodes"][0].copy()
        nm[len(nm) // 2] = bad
        with pytest.raises(tb.BgsbError) as e:
            plug.import_state(lay["planes"][0] + 1, nm, w, h, lay["nframes"] + 5)
        assert e.value.code == 1, bad
        after = plug.export_state()
        assert np.array_equal(after[1], before[1]) and np.array_equal(after[0], before[0]), bad
        assert plug.frame_count == count
    # a refused import of another geometry leaves the geometry alone too
    nm = np.full((h + 2) * (w + 2), 7, np.uint8)
    with pytest.raises(tb.BgsbError):
        plug.import_state(np.zeros((25, nm.size), np.float32), nm, w + 2, h + 2, 3)
    assert plug.state_bytes() // 101 == h * w
    plug.import_state(lay["planes"][0], lay["nmodes"][0], w, h, lay["nframes"])
    o = E.oracle_with_state(oracle, p, lay["planes"][0], lay["nmodes"][0], h, w)
    fg, bg = plug.process(lay["frames"][0, 0])
    efg, ebg = o.process(lay["frames"][0, 0])
    assert np.array_equal(fg, efg) and np.array_equal(bg, ebg)
    check_mog2_state(*plug.export_state(), o, "after the refused imports")
    plug.close()
