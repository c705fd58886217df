"""The constructed MOG2 states of tests/mog2_edges.py really sit on the decisions they are named for (CPU only).

For every group the C oracle (oracle/c/bgs_oracle.c) must give its first and its last member different results in the
group's observable, at the frame the group names and not before; the routing groups, which the oracle cannot tell
apart, must straddle the fast path's guard in the fixture's float32 copy of the oracle, which in turn must equal the
oracle bit for bit.  The number of exact ties found must not drop, and every group must appear in every placement the
GPU tests rely on."""
import numpy as np
import pytest

import mog2_edges as E

# exact ties the bisection finds at each parameter set (a later edit may find more, never fewer)
MIN_TIES = {"defaults": 51, "tg_over_tb": 50, "ct_half": 47, "alpha_1e-4": 49, "varmin_over_varmax": 51}


def oracle_run(oracle, p, gs):
    planes, nm, frames, index = E.members_frame(gs)
    o = E.oracle_with_state(oracle, p, planes, nm, 1, nm.size)
    per_frame = []
    for t in range(E.T):
        _, bg, raw = o.process(frames[t], want_raw=True)
        per_frame.append((o.nmodes.copy(), raw[0].copy(), bg[0].copy(), o.gmm.copy(), o.mean.copy()))
    return per_frame, index


@pytest.mark.parametrize("name", sorted(E.PARAMS))
def test_float32_copy_equals_the_oracle(oracle, name):
    p = E.params(name)
    gs = E.groups(p)
    per_frame, index = oracle_run(oracle, p, gs)
    for (gi, mi), i in index.items():
        for t, (n, raw, bg, _, _, g) in enumerate(E.run(gs[gi]["members"][mi], p)):
            on, oraw, obg, og, om = per_frame[t]
            what = (gs[gi]["name"], mi, t)
            assert n == on[i] and raw == oraw[i] and bg == tuple(obg[i].tolist()), what
            assert np.array_equal(g[:n, :2], og[i, :n]) and np.array_equal(g[:n, 2:], om[i, :n]), what


@pytest.mark.parametrize("name", sorted(E.PARAMS))
def test_every_group_straddles_its_decision(oracle, name):
    p = E.params(name)
    gs = E.groups(p)
    per_frame, index = oracle_run(oracle, p, gs)
    for gi, g in enumerate(gs):
        k, last = g["frame"], len(g["members"]) - 1
        if g["observable"] == "route":
            outs = [E.run(m, p, k + 1)[k][4][g["decision"]][2] for m in g["members"]]
            assert outs[0] != outs[-1], g["name"]
            continue
        obs = [[E.observe(g["observable"], r[0][index[gi, mi]], r[1][index[gi, mi]], r[2][index[gi, mi]],
                        r[3][index[gi, mi]], r[4][index[gi, mi]], p) for r in per_frame] for mi in (0, last)]
        assert obs[0][k] != obs[1][k], (g["name"], obs[0][k])
        if g["observable"] != "bg" or k:
            assert obs[0][:k] == obs[1][:k], (g["name"], "crossed before frame", k)


def test_groups_and_ties_do_not_drop():
    for name, n in MIN_TIES.items():
        gs = E.groups(E.params(name))
        assert sum(g["tie"] is not None for g in gs) >= n, name
    names = {g["name"] for g in E.groups(E.params())}
    for want in ("bg_slot0", "bg_slot1", "bg_slot2", "bg_tw_gate", "fit_slot0", "fit_slot1", "sort_match", "sort_new_n2",
                 "sort_new_n5", "new_full", "clamp_varmin", "clamp_varmax", "shadow_den0", "shadow_num_tau",
                 "shadow_num_den", "shadow_e", "shadow_tW_stop", "bg_t2_slot0", "bg_t2_slot1", "bg_t2_slot2",
                 "bg_half_100", "bg_half_101", "route_wt0_4", "route_tw_8", "route_wt0_huge"):
        assert want in names, want
    for nm in range(2, 6):
        assert {"prune_last_n%d" % nm, "prune_slot0_n%d" % nm} <= names, nm
        if nm > 2:
            assert "prune_middle_n%d" % nm in names
        if nm > 3:
            assert "prune_two_n%d" % nm in names
    for k in range(1, E.T):
        assert {"batch_prune_k%d" % k, "batch_second_mode_k%d" % k, "batch_sort_k%d" % k,
                "batch_bg_rule_k%d" % k} <= names, k
    assert "route_wt0_1e-4" in {g["name"] for g in E.groups(E.params("alpha_1e-4"))}
    assert "route_wt0_1e-4" in {g["name"] for g in E.groups(E.params("alpha_below_1e-4"))}


def placements(lay):
    seen = {}
    for s, i, gi, mi, tags in lay["where"]:
        seen.setdefault((s, gi), set()).update(tags)
    return seen


def test_every_group_in_every_placement():
    p = E.params()
    gs = E.groups(p)
    main = E.layout(p, "main", 2)
    assert main["h"] % 2 == 1 and main["w"] % 2 == 1
    seen = placements(main)
    for gi, g in enumerate(gs):
        tags = seen[0, gi]
        need = {"even", "odd", "mixed", "crowded", "lone"} | ({"lean"} if g["single"] else set())
        if not g["name"].startswith("batch"):
            need.add("ragged")
        assert need <= tags, (g["name"], need - tags)
    # a group sits at different pixels in different streams
    first = {(s, gi): i for s, i, gi, mi, tags in reversed(main["where"])}
    assert sum(first[0, gi] != first[1, gi] for gi in range(len(gs))) == len(gs)
    # the ragged last tile holds members, and the frame ends inside a tile
    npx = main["h"] * main["w"]
    assert npx % E.TILE and any(i >= npx - npx % E.TILE for s, i, gi, mi, tags in main["where"])
    seen = placements(E.layout(p, "aligned", 2))
    for gi, g in enumerate(gs):
        need = {"even", "odd", "mixed"} | ({"lean"} if g["single"] else set())
        assert need <= seen[0, gi] and need <= seen[1, gi], g["name"]
    band = E.layout(p, "banded", 1)
    seen = placements(band)
    for gi, g in enumerate(gs):
        assert {"band_before", "band_after", "lone", "even", "odd"} <= seen[0, gi], g["name"]
    rows = {i // band["w"] for s, i, gi, mi, tags in band["where"]}
    for b in (E.BAND_ROWS, 2 * E.BAND_ROWS):
        assert b - 1 in rows and b in rows
