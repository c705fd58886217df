"""TEST INFRASTRUCTURE ONLY - constructed MOG2 model states that sit on the decision boundaries of the update.

Every decision of cv::BackgroundSubtractorMOG2's per-pixel update (oracle/c/bgs_oracle.c, orc_mog2_apply and
orc_mog2_background) is a float32 comparison that a natural sequence almost never lands on.  This module builds, for each
decision, a GROUP of pixels that differ by one float32 ulp in one state field (or by one input byte) and fall on opposite
sides of that decision; where an exact tie exists the group also holds the tie pixel.  The values come from a bisection
over the float32 bit patterns of the field, evaluated by `step`, a numpy float32 copy of the oracle's operation order
(each numpy float32 scalar operation rounds once, like the library's -fmad=false code); tests/test_mog2_edge_fixture.py
checks the copy against the C oracle and the groups against their observables.

GPU-only routing edges (the fast path's eligibility guards in tracking_b200/csrc/mog2_t1.cu) change nothing in the
oracle; their groups straddle the guard so that the pixel is taken by the fast path on one side and by the generic
routine on the other.  The normalised weights the guards `wn <= 8` / `t2 <= 8` look at are <= 1 after the
renormalisation, so of the `<= 8` guards only the total weight `tw` has a reachable edge (imported weights that do not
sum to 1); a weight near the top of the float range covers what the `wt0 <= 4` guard protects (the reciprocal of the
fast path flushes below 2^-126).

`layout(params, kind, nstreams)` places the groups into frames:

* "main" (ragged: odd h and w): every member at an even and an odd pixel, single-mode members in an all-single-mode
  warp (64-pixel state tile, `lean`) and in a mixed one, every member in a 4-warp CTA (256 pixels) whose other pixels
  are all slow (mode count 0) and in one whose other pixels are all fast, one member of every group in the ragged
  last tile;
* "aligned" (64 x 128, whole tiles): the even / odd and lean / mixed placements only (the pipeline's stream kernel);
* "banded" (352 x 1024, three 128-row host bands): the even / odd / lean / mixed placements on both sides of each
  band boundary, and the lone CTAs.

Stream s of a group gets the groups in a rotated order, so different cases sit in different streams.
"""
from __future__ import annotations

import numpy as np

K = 5
T = 8
F = np.float32
EPS = F(1.1920929e-07)

DEFAULTS = dict(alpha=0.05, varThreshold=16.0, varThresholdGen=9.0, backgroundRatio=0.9, varInit=15.0, varMin=4.0,
                varMax=75.0, complexityReductionThreshold=0.05, shadowThreshold=0.5, detectShadows=1, shadowValue=127,
                history=500, enableThreshold=0, threshold=15, nframes=100)
MODEL_KEYS = ("varThreshold", "varThresholdGen", "backgroundRatio", "varInit", "varMin", "varMax",
              "complexityReductionThreshold", "shadowThreshold", "detectShadows", "shadowValue", "history")

# named parameter sets: the routes run at each
PARAMS = {
    "defaults": {},
    "no_shadows": dict(detectShadows=0),
    "thr_template": dict(enableThreshold=1, threshold=15),
    "tg_over_tb": dict(varThreshold=9.0, varThresholdGen=16.0),
    "ct_half": dict(complexityReductionThreshold=0.5),
    "alpha_1e-4": dict(alpha=float(F(1e-4))),
    "alpha_below_1e-4": dict(alpha=float(np.nextafter(F(1e-4), F(0)))),
    "alpha_0": dict(alpha=0.0),
    "alpha_auto": dict(alpha=-1.0, nframes=40, history=100),
    "varmin_over_varmax": dict(varMin=20.0, varMax=10.0),
    "tb_nonpositive": dict(backgroundRatio=0.0),
}


def params(name="defaults"):
    p = dict(DEFAULTS)
    p.update(PARAMS[name] if isinstance(name, str) else name)
    return p


def model_kwargs(p):
    """the plugin's / oracle's keyword arguments of parameter set p (alpha, thresholds and the model's own keys)"""
    kw = {k: p[k] for k in MODEL_KEYS}
    kw.update(alpha=p["alpha"], enableThreshold=p["enableThreshold"], threshold=p["threshold"])
    return kw


def learning_rate(p, t):
    """learning rate of frame t after the import (operator(): ++nframes, then the automatic rule)"""
    nf = p["nframes"] + t + 1
    if p["alpha"] >= 0 and nf > 1:
        return p["alpha"]
    return 1.0 / min(2 * nf, p["history"])


# ---------------------------------------------------------------------------------------------------------------------
# numpy float32 copy of orc_mog2_apply + orc_mog2_background for one pixel, recording every comparison it makes

def _rint_u8(x):
    r = np.rint(F(x))
    return 0 if not r > 0 else (255 if r > 255 else int(r))


def step(n, g, x, p, lr, cmp=None):
    """One frame of one pixel.  n: mode count, g: float32 [K, 5] (w, var, b, g, r), modified in place; x: 3 input
    bytes.  -> (n, raw, bg, bg_unrounded).  cmp (dict) receives key -> (lhs, rhs, outcome) of every comparison."""
    cmp = {} if cmp is None else cmp
    Tb, Tg, TB = F(p["varThreshold"]), F(p["varThresholdGen"]), F(p["backgroundRatio"])
    vmin0, vmax0 = F(p["varMin"]), F(p["varMax"])
    varMin, varMax = (vmin0, vmax0) if vmin0 < vmax0 else (vmax0, vmin0)
    aT = F(lr)
    a1 = F(1) - aT
    prune = F(-lr * float(F(p["complexityReductionThreshold"])))
    nprune = -prune
    d = [F(v) for v in x]
    bg = fits = False
    tw = F(0)
    m = 0
    while m < n:
        w = a1 * g[m, 0] + prune
        swaps = 0
        if not fits:
            var = g[m, 1]
            dD = [g[m, 2 + c] - d[c] for c in range(3)]
            dist2 = dD[0] * dD[0] + dD[1] * dD[1] + dD[2] * dD[2]
            cmp["tw<TB", m] = (tw, TB, tw < TB)
            cmp["bg", m] = (dist2, Tb * var, dist2 < Tb * var)
            if tw < TB and dist2 < Tb * var:
                bg = True
            cmp["fit", m] = (dist2, Tg * var, dist2 < Tg * var)
            if dist2 < Tg * var:
                fits = True
                w = w + aT
                if m == 0:                      # the fast path's range guards on the matched dominant mode
                    cmp["wt0>=1e-4"] = (w, F(1e-4), w >= F(1e-4))
                    cmp["wt0<=4"] = (w, F(4), w <= F(4))
                k = aT / w
                for c in range(3):
                    g[m, 2 + c] = g[m, 2 + c] - k * dD[c]
                vn = var + k * (dist2 - var)
                cmp["varMin"] = (vn, varMin, vn > varMin)
                vn = vn if vn > varMin else varMin
                cmp["varMax"] = (vn, varMax, vn < varMax)
                vn = vn if vn < varMax else varMax
                g[m, 1] = vn
                for j in range(m, 0, -1):
                    cmp["sort", j] = (w, g[j - 1, 0], w < g[j - 1, 0])
                    if w < g[j - 1, 0]:
                        break
                    swaps += 1
                    g[[j, j - 1]] = g[[j - 1, j]]
        cmp["prune", m] = (w, nprune, w < nprune)
        if w < nprune:
            w = F(0)
            n -= 1
        g[m - swaps, 0] = w
        tw = tw + w
        m += 1
    cmp["tw<=8"] = (tw, F(8), tw <= F(8))
    inv = F(1) / tw if abs(tw) > EPS else F(0)
    for m in range(n):
        g[m, 0] = g[m, 0] * inv
    if not fits and aT > 0:
        if n == K:
            m = K - 1
        else:
            m = n
            n += 1
        if n == 1:
            g[m, 0] = F(1)
        else:
            g[m, 0] = aT
            for j in range(n - 1):
                g[j, 0] = g[j, 0] * a1
        g[m, 2:] = d
        g[m, 1] = F(p["varInit"])
        for j in range(n - 1, 0, -1):
            cmp["new", j] = (aT, g[j - 1, 0], aT < g[j - 1, 0])
            if aT < g[j - 1, 0]:
                break
            g[[j, j - 1]] = g[[j - 1, j]]
    raw = 0
    if not bg:
        raw = 255
        if p["detectShadows"] and _shadow(d, n, g, p, cmp):
            raw = int(p["shadowValue"])
    acc = [F(0)] * 3
    t2 = F(0)
    for m in range(n):
        w = g[m, 0]
        acc = [acc[c] + w * g[m, 2 + c] for c in range(3)]
        t2 = t2 + w
        cmp["t2>TB", m] = (t2, TB, t2 > TB)
        if t2 > TB:
            break
    inv = F(1) / t2 if abs(t2) > EPS else F(0)
    pre = [acc[c] * inv for c in range(3)]
    return n, raw, tuple(_rint_u8(v) for v in pre), tuple(pre)


def _shadow(d, n, g, p, cmp):
    Tb, TB, tau = F(p["varThreshold"]), F(p["backgroundRatio"]), F(p["shadowThreshold"])
    tW = F(0)
    for m in range(n):
        num = den = F(0)
        for c in range(3):
            num = num + d[c] * g[m, 2 + c]
            den = den + g[m, 2 + c] * g[m, 2 + c]
        cmp["den==0", m] = (den, F(0), den == 0)
        if den == 0:
            return False
        cmp["num<=den", m] = (num, den, num <= den)
        cmp["num>=tau*den", m] = (num, tau * den, num >= tau * den)
        if num <= den and num >= tau * den:
            a = num / den
            e = F(0)
            for c in range(3):
                dd = a * g[m, 2 + c] - d[c]
                e = e + dd * dd
            cmp["e", m] = (e, Tb * g[m, 1] * a * a, e < Tb * g[m, 1] * a * a)
            if e < Tb * g[m, 1] * a * a:
                return True
        tW = tW + g[m, 0]
        cmp["tW>TB", m] = (tW, TB, tW > TB)
        if tW > TB:
            return False
    return False


def run(member, p, frames=T):
    """step() over the member's input sequence -> list per frame of (n, raw, bg, pre, cmp, state copy)"""
    n, g, xs = member["n"], member["g"].copy(), member["x"]
    out = []
    for t in range(frames):
        cmp = {}
        n, raw, bg, pre = step(n, g, xs[t], p, learning_rate(p, t), cmp)
        out.append((n, raw, bg, pre, cmp, g.copy()))
    return out


def observe(kind, n, raw, bg, gmm, mean, p):
    """the discrete result a group's decision shows in: gmm [K][2] and mean [K][3] of the pixel after the frame"""
    if kind == "raw":
        return int(raw)
    if kind == "nmodes":
        return int(n)
    if kind == "modes":
        return int(n), tuple(int(np.rint(v)) for v in mean[:n, 0]), tuple(bool(v == 0) for v in gmm[:n, 0])
    if kind == "slot4":
        return tuple(float(v) for v in mean[4])
    if kind == "clamp":
        lo, hi = sorted((F(p["varMin"]), F(p["varMax"])))
        return bool(gmm[0, 1] == lo), bool(gmm[0, 1] == hi)
    if kind == "bg":
        return tuple(int(v) for v in bg)
    raise KeyError(kind)


def observe_step(kind, r, p):
    n, raw, bg, _, _, g = r
    return observe(kind, n, raw, bg, g[:, :2], g[:, 2:], p)


# ---------------------------------------------------------------------------------------------------------------------
# groups

def _bits(v):
    return int(np.array(v, np.float32).view(np.int32))


def _flt(i):
    return F(np.array(i, np.int32).view(np.float32))


def _outcome(member, p, frame, key):
    r = run(member, p, frame + 1)[frame][4]
    return r[key][2] if key in r else None


def _tie(member, p, frame, key):
    r = run(member, p, frame + 1)[frame][4]
    return key in r and r[key][0] == r[key][1]


def straddle(make, lo, hi, p, frame, key, grid=40):
    """Bisect the float32 bit patterns of a positive field in [lo, hi] for the adjacent pair of values on which the
    comparison `key` of frame `frame` comes out differently (a coarse grid first: outside a window the comparison may
    not be reached at all).  make(value) -> member.  -> (members, index of the tie member or None): the pair, plus the
    pixel one ulp beyond a tie; None if no flip lies in [lo, hi]."""
    a0, b0 = _bits(F(lo)), _bits(F(hi))
    pts = sorted(set(int(v) for v in np.linspace(a0, b0, grid)))
    outs = [_outcome(make(_flt(i)), p, frame, key) for i in pts]
    for j in range(len(pts) - 1):
        if outs[j] is not None and outs[j + 1] is not None and outs[j] != outs[j + 1]:
            a, b, oa = pts[j], pts[j + 1], outs[j]
            break
    else:
        return None
    while b - a > 1:
        c = (a + b) // 2
        oc = _outcome(make(_flt(c)), p, frame, key)
        if oc is None:
            return None
        if oc == oa:
            a = c
        else:
            b = c
    vals = [_flt(a), _flt(b)]
    tie = None
    if _tie(make(vals[0]), p, frame, key):
        vals.insert(0, _flt(a - 1))
        tie = 1
    elif _tie(make(vals[1]), p, frame, key):
        vals.append(_flt(b + 1))
        tie = 1
    return [make(v) for v in vals], tie


def straddle_byte(make, p, frame, key):
    """the same over an input byte 0..255 (no ties: the members differ by one grey level)"""
    outs = [_outcome(make(v), p, frame, key) for v in range(256)]
    for v in range(255):
        if outs[v] is not None and outs[v + 1] is not None and outs[v] != outs[v + 1]:
            tie = 0 if _tie(make(v), p, frame, key) else (1 if _tie(make(v + 1), p, frame, key) else None)
            return [make(v), make(v + 1)], tie
    return None


def pixel(modes, x, xs=None):
    """member: modes [(w, var, b, g, r)], input x (every frame) or xs (per frame)"""
    g = np.zeros((K, 5), np.float32)
    for i, md in enumerate(modes):
        g[i] = md
    seq = np.array(xs if xs is not None else [x] * T, np.uint8)
    return dict(n=len(modes), g=g, x=seq)


X = (100, 120, 140)
FAR = (10, 250, 30)


def _with(modes, i, j, v):
    modes = [list(md) for md in modes]
    modes[i][j] = v
    return modes


def groups(p):
    """-> list of dict(name, decision, observable, frame, members, tie, single): the groups at parameter set p; a decision
    the parameters make unreachable (e.g. no new mode at alpha 0) yields no group"""
    out = []
    Tb, Tg, TB = p["varThreshold"], p["varThresholdGen"], p["backgroundRatio"]

    def add(name, decision, obs, found, frame=0):
        if found is None:
            return
        members, tie = found
        if obs != "route":                  # the decision must show in the observable at its frame, and not before
            seen = [[observe_step(obs, r, p) for r in run(m, p, frame + 1)] for m in members]
            if seen[0][frame] == seen[-1][frame] and tie is not None and seen[0][frame] != seen[tie][frame]:
                members, seen = members[:tie + 1], seen[:tie + 1]        # the tie alone is on the other side
            if seen[0][frame] == seen[-1][frame] or seen[0][:frame] != seen[-1][:frame]:
                return
        out.append(dict(name=name, decision=decision, observable=obs, frame=frame, members=members, tie=tie,
                        single=all(m["n"] <= 1 for m in members)))

    def var_search(base, slot, x, key, guess, frame=0):
        make = lambda v: pixel(_with(base, slot, 1, v), x)                    # noqa: E731
        return straddle(make, F(guess * 0.5), F(guess * 2), p, frame, key)

    off = (112, 120, 140)                         # dist2 = 144 to X
    # background test dist2 < Tb*var on slot 0 (slot 0 alone) and on slots 1 / 2 under a running tw < TB
    add("bg_slot0", "bg", "raw", var_search([(1.0, 9.0) + off], 0, X, ("bg", 0), 144 / Tb))
    add("bg_slot1", "bg", "raw", var_search([(0.45, 15.0) + FAR, (0.4, 9.0) + off], 1, X, ("bg", 1), 144 / Tb))
    add("bg_slot2", "bg", "raw", var_search([(0.4, 15.0) + FAR, (0.3, 15.0) + (200, 10, 10), (0.3, 9.0) + off], 2, X,
                                            ("bg", 2), 144 / Tb))
    # the running tw < TB gate: slot 1 is background by its distance, slot 0's decayed weight straddles TB
    if TB > 0:
        make = lambda v: pixel([(v, 15.0) + FAR, (0.05, 100.0) + X], X)      # noqa: E731
        add("bg_tw_gate", "bg", "raw", straddle(make, F(TB * 0.5), F(TB * 2 + 1), p, 0, ("tw<TB", 1)))
    # fit dist2 < Tg*var on slot 0, slot 1 (the other side: no mode fits)
    add("fit_slot0", "fit", "nmodes", var_search([(1.0, 16.0) + off], 0, X, ("fit", 0), 144 / Tg))
    add("fit_slot1", "fit", "nmodes", var_search([(0.6, 15.0) + FAR, (0.4, 16.0) + off], 1, X, ("fit", 1), 144 / Tg))
    add("fit_slot0_multi", "fit", "nmodes", var_search([(0.7, 16.0) + off, (0.3, 15.0) + FAR], 0, X, ("fit", 0), 144 / Tg))

    # prune w < -prune: the pruned slot's weight is searched; slot 0 only when it does not fit
    lr = learning_rate(p, 0)
    nprune = float(lr * float(F(p["complexityReductionThreshold"])))
    a1 = 1 - lr
    wguess = (2 * nprune) / a1 if a1 > 0 else 0.01
    if nprune > 0:
        for nm in range(2, 6):
            spread = [(0.5 - 0.05 * i, 15.0) + (20 + 40 * i, 60, 60) for i in range(nm)]
            fitting = [list(md) for md in spread]
            fitting[0] = [0.6, 15.0, *X]           # slot 0 explains the input: the fast path's candidates
            for slot in ([nm - 1, max(1, nm - 2)] if nm > 2 else [1]):
                make = lambda v, s=slot, base=fitting: pixel(_with(base, s, 0, v), X)           # noqa: E731
                tag = "last" if slot == nm - 1 else "middle"
                add("prune_%s_n%d" % (tag, nm), ("prune", slot), "nmodes",
                    straddle(make, F(wguess * 0.25), F(wguess * 4), p, 0, ("prune", slot)))
            if nm >= 4:
                # two slots at once: slot 1 is far under the threshold, slot 2 straddles it (the walk's bound is the live
                # count, so a prune hides the last slot from the walk: slot 2 is the last one visited at n = 4)
                two = _with(fitting, 1, 0, 0.0)
                make = lambda v, base=two: pixel(_with(base, 2, 0, v), X)                      # noqa: E731
                add("prune_two_n%d" % nm, ("prune", 2), "nmodes",
                    straddle(make, F(wguess * 0.25), F(wguess * 4), p, 0, ("prune", 2)))
            make = lambda v, base=spread: pixel(_with(base, 0, 0, v), X)       # noqa: E731  slot 0, no mode fits
            add("prune_slot0_n%d" % nm, ("prune", 0), "modes",
                straddle(make, F(wguess * 0.25), F(wguess * 4), p, 0, ("prune", 0)))

    # sort tie of the matched mode with its predecessor: slot 1 matches (mean == input), slot 0's weight is searched
    make = lambda v: pixel([(v, 15.0) + FAR, (0.4, 15.0) + X], X)                              # noqa: E731
    add("sort_match", ("sort", 1), "modes", straddle(make, F(0.3), F(0.9), p, 0, ("sort", 1)))
    make = lambda v: pixel([(0.5, 15.0) + FAR, (v, 15.0) + (200, 10, 10), (0.2, 15.0) + X], X)  # noqa: E731
    add("sort_match_slot2", ("sort", 2), "modes", straddle(make, F(0.05), F(0.5), p, 0, ("sort", 2)))
    # sort tie of a new mode with its predecessor: alphaT == renormalised weight * alpha1 of the last slot
    if lr > 0:
        for nm in (2, 4, 5):
            base = [(0.9 - 0.1 * i, 15.0) + (20 + 40 * i, 60, 60) for i in range(nm)]
            s = nm - 1 if nm < K else K - 2
            make = lambda v, base=base, s=s: pixel(_with(base, s, 0, v), FAR)                   # noqa: E731
            key = ("new", s + 1)
            add("sort_new_n%d" % nm, key, "modes", straddle(make, F(lr * 0.2), F(lr * 5), p, 0, key))
    # new mode into a full list (slot 4 replaced) or not (slot 0 fits).  A new mode into n = 0 in a context that is
    # not fresh: the layouts' slow filler pixels; none at alpha 0: every pixel that fits no mode at that parameter set.
    full = [(0.3 - 0.05 * i, 15.0) + (20 + 40 * i, 60, 60) for i in range(K)]
    add("new_full", ("fit", 0), "slot4", straddle_byte(lambda b: pixel(full, (b, 60, 60)), p, 0, ("fit", 0)))
    # variance clamp at varMin / varMax (varMin > varMax swaps them): the matched mode's variance is searched
    lo, hi = sorted((p["varMin"], p["varMax"]))
    near = (101, 120, 140)                                    # dist2 = 1
    make = lambda v: pixel([(1.0, v) + near], X)                                              # noqa: E731
    add("clamp_varmin", "varMin", "clamp", straddle(make, F(lo * 0.5), F(lo * 2), p, 0, "varMin"))
    far_ok = (100 + int(np.sqrt(hi * Tg * 0.6)), 120, 140)
    make = lambda v: pixel([(1.0, v) + far_ok], X)                                            # noqa: E731
    add("clamp_varmax", "varMax", "clamp", straddle(make, F(hi * 0.5), F(hi * 2), p, 0, "varMax"))

    # shadow test: not background (slot 0 far in distance, small variance), input a scaled copy of the mean
    sh = (0.95, 1.0, 100.0, 100.0, 100.0)
    if p["detectShadows"]:
        # den == 0: slot 0's mean blue is searched around 2^-75, where its square leaves the subnormal range
        make = lambda v: pixel([(0.3, 1.0, v, 0.0, 0.0), (0.65, 1.0, 100.0, 100.0, 100.0)], (60, 60, 60))  # noqa: E731
        add("shadow_den0", ("den==0", 0), "raw", straddle(make, F(2.0 ** -77), F(2.0 ** -72), p, 0, ("den==0", 0)))
        add("shadow_num_tau", ("num>=tau*den", 0), "raw",
            straddle_byte(lambda b: pixel([sh], (b, 50, 50)), p, 0, ("num>=tau*den", 0)))
        # num <= den on slot 1, whose background test the running weight gates off (slot 0's decayed weight >= TB
        # while its renormalised weight leaves the shadow walk going)
        make = lambda b: pixel([(1.0, 1.0) + FAR, (0.2, 0.2, 100.0, 100.0, 100.0)], (b, 99, 100))  # noqa: E731
        add("shadow_num_den", ("num<=den", 1), "raw", straddle_byte(make, p, 0, ("num<=den", 1)))
        make = lambda v: pixel([(0.95, v, 100.0, 100.0, 100.0)], (70, 60, 60))                 # noqa: E731
        add("shadow_e", ("e", 0), "raw", straddle(make, F(0.05), F(20.0), p, 0, ("e", 0)))
        # the tW > TB stop: slot 0 is not a shadow, slot 1 is; slot 0's weight decides whether slot 1 is reached
        if TB > 0:
            make = lambda v: pixel([(v, 1.0) + FAR, (0.05, 1.0, 100.0, 100.0, 100.0)], (60, 60, 60))  # noqa: E731
            add("shadow_tW_stop", ("tW>TB", 0), "raw", straddle(make, F(TB * 0.5), F(TB * 2 + 1), p, 0, ("tW>TB", 0)))

    # background image: t2 > TB after slot 0 / 1 / 2, colours apart so the blend shows
    if TB > 0:
        for s in range(3):
            base = [(0.3, 15.0) + X, (0.3, 15.0) + (20, 60, 60), (0.3, 15.0) + (200, 10, 10), (0.1, 15.0) + (0, 0, 250)][:s + 2]
            base = [list(md) for md in base]
            make = lambda v, base=base, s=s: pixel(_with(base, s, 0, v), X)                     # noqa: E731
            add("bg_t2_slot%d" % s, ("t2>TB", s), "bg", straddle(make, F(0.01), F(4.0), p, 0, ("t2>TB", s)))
    # a background colour at k + 0.5 (half-even): slot 0 alone, weight 1, mean searched around 100.5 / 101.5
    for k0 in (100.5, 101.5):
        make = lambda v: pixel([(1.0, 15.0, v, 120.0, 140.0)], (int(k0), 120, 140))        # noqa: E731
        found = _rounding(make, F(k0), p)
        add("bg_half_%d" % int(k0), "round", "bg", found)

    # GPU-only routing edges
    if lr > 0:
        make = lambda v: pixel([(v, 15.0) + X], X)                                              # noqa: E731
        add("route_wt0_1e-4", "wt0>=1e-4", "route", straddle(make, F(1e-7), F(1e-3), p, 0, "wt0>=1e-4"))
        add("route_wt0_4", "wt0<=4", "route", straddle(make, F(3.0), F(6.0), p, 0, "wt0<=4"))
        make = lambda v: pixel([(v, 15.0) + X, (0.5, 15.0) + FAR], X)                           # noqa: E731
        add("route_wt0_4_multi", "wt0<=4", "route", straddle(make, F(3.0), F(6.0), p, 0, "wt0<=4"))
        make = lambda v: pixel([(1.0, 15.0) + X, (v, 15.0) + FAR], X)                           # noqa: E731
        add("route_tw_8", "tw<=8", "route", straddle(make, F(4.0), F(12.0), p, 0, "tw<=8"))
        big = F(2.0 ** 127)
        add("route_wt0_huge", "wt0<=4", "route",
            _fixed([pixel([(1.0, 15.0) + X], X), pixel([(big, 15.0) + X], X), pixel([(F(3.0e38), 15.0) + X], X)]))

    # batch cases: a boundary crossed at frame k = 1..7 of an 8-frame batch
    if nprune > 0 and lr > 0:
        for k in range(1, T):
            # the last slot's weight decays to the prune threshold at frame k (slot 0 matches every frame)
            make = lambda v: pixel([(0.9, 15.0) + X, (v, 15.0) + FAR], X)                      # noqa: E731
            add("batch_prune_k%d" % k, ("prune", 1), "nmodes", straddle(make, F(nprune * 0.5), F(0.6), p, k,
                                                                         ("prune", 1)), frame=k)
            # a single-mode pixel gets its second mode at frame k: the input's blue byte walks off the mode
            xs = lambda b, k=k: [X] * k + [(b, 120, 140)] * (T - k)                           # noqa: E731
            add("batch_second_mode_k%d" % k, ("fit", 0), "nmodes",
                straddle_byte(lambda b, k=k: pixel([(1.0, 15.0) + X], None, xs(b)), p, k, ("fit", 0)), frame=k)
            # slot 1 (matched every frame) overtakes slot 0 at frame k
            make = lambda v: pixel([(v, 15.0) + FAR, (0.3, 15.0) + X], X)                      # noqa: E731
            add("batch_sort_k%d" % k, ("sort", 1), "modes", straddle(make, F(0.3), F(0.9), p, k, ("sort", 1)), frame=k)
            # slot 0 (matched every frame) grows past backgroundRatio at frame k: the background image drops slot 1
            if TB > 0:
                make = lambda v: pixel([(v, 15.0) + X, (0.1, 15.0) + (20, 60, 60)], X)          # noqa: E731
                add("batch_bg_rule_k%d" % k, ("t2>TB", 0), "bg", straddle(make, F(0.05), F(4.0), p, k,
                                                                            ("t2>TB", 0)), frame=k)
    return out


def _fixed(members):
    return members, None


def _rounding(make, v0, p):
    """members whose background colour's unrounded value sits just below, at and just above v0 (a k + 0.5)"""
    a, b = _bits(F(v0 - 2)), _bits(F(v0 + 2))
    val = lambda i: run(make(_flt(i)), p, 1)[0][3][0]          # noqa: E731
    while b - a > 1:
        c = (a + b) // 2
        if val(c) < v0:
            a = c
        else:
            b = c
    if val(b) != v0:
        return [make(_flt(a)), make(_flt(b))], None
    return [make(_flt(a)), make(_flt(b)), make(_flt(b + 1))], 1


# ---------------------------------------------------------------------------------------------------------------------
# layouts

TILE, CTA = 64, 256
GEOMETRY = {"main": None, "aligned": (64, 128), "banded": (352, 1024)}
BAND_ROWS = 128                  # hostBands 3 on 352 rows: three bands of 128 rows


def _fast(single):
    """a pixel the fast path takes: slot 0 explains the input"""
    return pixel([(1.0, 15.0) + X] if single else [(0.95, 15.0) + X, (0.05, 15.0) + FAR], X)


def _slow():
    return pixel([], X)           # no mode: a new one is created (generic routine)


def _tiles_dense(members):
    """members [(member, ident)]: each at an even and an odd pixel of mixed tiles, single-mode members also of lean
    tiles; every other pixel of these CTAs is slow"""
    def fill(items, lean):
        tiles, cur = [], []
        for item in items:
            for parity in (0, 1):
                if len(cur) % 2 != parity:
                    cur.append((_slow(), None))
                cur.append(item)
                if len(cur) >= TILE - 2:
                    tiles.append(cur)
                    cur = []
        if cur:
            tiles.append(cur)
        out = []
        for t in tiles:
            t = t + [(_slow(), None)] * (TILE - len(t))
            if not lean:
                t[-1] = (pixel([(0.5, 15.0) + FAR, (0.5, 15.0) + (200, 10, 10)], X), None)   # 2 modes, slow too
            out.append(t)
        return out
    tiles = fill(members, False) + fill([it for it in members if it[0]["n"] <= 1], True)
    while len(tiles) % 4:
        tiles.append([(_slow(), None)] * TILE)
    return tiles


def _tiles_lone(members):
    """every member alone in a CTA of fast pixels; rotates over the four warps and both parities"""
    tiles = []
    for j, (mem, ident) in enumerate(members):
        single = mem["n"] <= 1
        cta = [[(_fast(single or w != j % 4), None) for _ in range(TILE)] for w in range(4)]
        cta[j % 4][(2 * j + j // 4) % TILE] = (mem, ident)
        tiles += cta
    return tiles


def layout(p, kind="main", nstreams=1):
    """-> dict(h, w, planes [S][25][npx] f32, nmodes [S][npx] u8, nframes, frames [S][T][h][w][3] u8, where, groups)
    where: list of (stream, pixel index, group index, member index, tags)"""
    gs = groups(p)
    S = nstreams
    out = dict(groups=gs, nframes=p["nframes"], where=[])
    planes_s, nm_s, frames_s = [], [], []
    for s in range(S):
        order = list(range(len(gs)))
        r = (s * 7) % max(len(gs), 1)
        order = order[r:] + order[:r]
        members = [(m, (gi, mi)) for gi in order for mi, m in enumerate(gs[gi]["members"])]
        dense = _tiles_dense(members)
        dense_tags = ["crowded"] * len(dense)
        if kind == "aligned":
            tiles, tags = dense, dense_tags
        else:
            lone = _tiles_lone(members)
            tiles, tags = dense + lone, dense_tags + ["lone"] * len(lone)
        cells = [c for t in tiles for c in t]
        ctags = [tg for t, tg in zip(tiles, tags) for _ in t]
        if kind == "main":
            tail = [(gs[gi]["members"][(gi + s) % len(gs[gi]["members"])], (gi, (gi + s) % len(gs[gi]["members"])))
                    for gi in order][:TILE - 1]
            w = 65
            body = len(cells)
            # pad so that the tail lands in the ragged last tile and the frame has odd h and w
            h = (body + TILE + w - 1) // w
            h += 1 - h % 2
            while (h * w) % TILE < len(tail) or h * w - len(tail) < body:
                h += 2
            npx = h * w
            pad = npx - body - len(tail)
            cells = cells + [(_fast(True), None)] * pad + tail
            ctags = ctags + ["pad"] * pad + ["ragged"] * len(tail)
        else:
            h, w = GEOMETRY[kind]
            npx = h * w
            if kind == "aligned":
                assert len(cells) <= npx, (len(cells), npx)
                cells += [(_fast(True), None)] * (npx - len(cells))
                ctags += ["pad"] * (npx - len(ctags))
            else:
                # a copy of the dense tiles ending at and one starting at each band boundary, the lone CTAs after
                nd = len(dense) * TILE
                new, ntag = [], []
                for b in (BAND_ROWS * w, 2 * BAND_ROWS * w):
                    start = b - nd
                    fill_ = start - len(new)
                    new += [(_fast(True), None)] * fill_
                    ntag += ["pad"] * fill_
                    dc = [c for t in dense for c in t]
                    new += dc + dc
                    ntag += ["band_before"] * nd + ["band_after"] * nd
                rest = cells[nd:]
                new += rest
                ntag += ctags[nd:]
                assert len(new) <= npx, (len(new), npx)
                cells = new + [(_fast(True), None)] * (npx - len(new))
                ctags = ntag + ["pad"] * (npx - len(ntag))
        planes = np.zeros((5 * K, npx), np.float32)
        nm = np.zeros(npx, np.uint8)
        frames = np.zeros((T, npx, 3), np.uint8)
        tile_n = {}
        for i, (mem, ident) in enumerate(cells):
            planes[:, i] = mem["g"].reshape(-1)
            nm[i] = mem["n"]
            frames[:, i] = mem["x"]
        for i, (mem, ident) in enumerate(cells):
            tile_n[i // TILE] = max(tile_n.get(i // TILE, 0), mem["n"])
        for i, (mem, ident) in enumerate(cells):
            if ident is None:
                continue
            tg = {ctags[i], "even" if i % 2 == 0 else "odd", "lean" if tile_n[i // TILE] <= 1 else "mixed"}
            out["where"].append((s, i, ident[0], ident[1], tg))
        planes_s.append(planes)
        nm_s.append(nm)
        frames_s.append(frames.reshape(T, h, w, 3))
    out.update(h=h, w=w, planes=np.stack(planes_s), nmodes=np.stack(nm_s), frames=np.stack(frames_s))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# the C oracle on an imported state

def oracle_with_state(restate, p, planes, nmodes, h, w):
    """restate.MixtureOfGaussianV2BGS holding planes [25][npx] / nmodes [npx] as if it had seen p["nframes"] frames"""
    o = restate.MixtureOfGaussianV2BGS(**model_kwargs(p))
    npx = h * w
    o.shape = (h, w)
    o.gmm = np.ascontiguousarray(planes.reshape(K, 5, npx)[:, :2].transpose(2, 0, 1), np.float32)
    o.mean = np.ascontiguousarray(planes.reshape(K, 5, npx)[:, 2:].transpose(2, 0, 1), np.float32)
    o.nmodes = np.array(nmodes, np.uint8)
    o.nframes = p["nframes"]
    return o


def members_frame(gs):
    """every member of every group side by side in one 1 x n frame -> (planes, nmodes, frames [T][1][n][3], index)
    index[(group, member)] = pixel"""
    cells = [(gi, mi, m) for gi, g in enumerate(gs) for mi, m in enumerate(g["members"])]
    n = len(cells)
    planes = np.zeros((5 * K, n), np.float32)
    nm = np.zeros(n, np.uint8)
    frames = np.zeros((T, 1, n, 3), np.uint8)
    index = {}
    for i, (gi, mi, m) in enumerate(cells):
        planes[:, i] = m["g"].reshape(-1)
        nm[i] = m["n"]
        frames[:, 0, i] = m["x"]
        index[gi, mi] = i
    return planes, nm, frames, index
