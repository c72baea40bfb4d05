"""The build-variant table (tests/build_variants.py) without a GPU: the mirror of the launchers' dispatch agrees with values
worked out by hand from k1_k7_lmpc.cu, and SHAPES reaches every variant and both sides of every size threshold."""
import numpy as np
import pytest

from tests import build_variants as bv


def _labels(shapes):
    return [bv.build_dispatch(s.make()) for s in shapes]


def test_shapes_hit_the_labels_they_record():
    for s, got in zip(bv.SHAPES, _labels(bv.SHAPES)):
        for key, want in s.expect.items():
            assert got[key] == want, (s.name, key, got[key], want)


def test_shapes_cover_every_label():
    seen = {k: set() for k in bv.LABELS}
    for got in _labels(bv.SHAPES):
        for k in bv.LABELS:
            seen[k].add(got[k])
    for k, labels in bv.LABELS.items():
        assert seen[k] == set(labels), (k, set(labels) - seen[k])


def test_shapes_cover_shared_and_per_instance_hessians_for_every_q_and_ef_variant():
    seen = set()
    for got in _labels(bv.SHAPES):
        seen.add(("q", got["q"], got["shared"]))
        seen.add(("ef", got["ef"], got["shared"]))
    for key in ("q", "ef"):
        for label in bv.LABELS[key]:
            for shared in (False, True):
                assert (key, label, shared) in seen, (key, label, shared)


def test_shapes_straddle_every_threshold_by_one_step():
    """each threshold has two shapes, one on each side, that differ only by one step of N (or of nu for K1)"""
    for thr in bv.THRESHOLDS:
        pair = [s for s in bv.SHAPES if s.across == thr]
        assert len(pair) >= 2, thr
        a, b = pair[0].make(), pair[1].make()
        step = "nu" if thr[0] == "k1" else "N"
        assert b[step] == a[step] + 1, (thr, a[step], b[step])
        same = [k for k in ("nx", "nu", "N", "initial_state") if k != step]
        assert all(a.get(k) == b.get(k) for k in same), thr
        assert len(a["costs"]) == len(b["costs"]) and len(a["constraints"]) == len(b["constraints"]), thr
        key, lo, hi = thr
        assert bv.build_dispatch(a)[key] == lo and bv.build_dispatch(b)[key] == hi, thr


def test_every_cost_and_constraint_kind_is_in_the_table():
    costs, cstrs, n1, eq, subset, infs = set(), set(), False, False, False, False
    for s in bv.SHAPES:
        bp = s.make()
        n1 |= bp["N"] == 1
        for c in bp["costs"]:
            mat = c.get("M") if c.get("M") is not None else c["N"]
            rows = np.asarray(mat).shape[-2]
            costs.add((c.get("M") is not None, c.get("N") is not None, rows > 1))
        for c in bp["constraints"]:
            cstrs.add((c["kind"], c.get("E") is not None, c.get("G") is not None))
            eq |= c.get("is_ineq", True) is False
            if c["kind"] == "trajectory_bound":
                lo, up = np.asarray(c["lower"]), np.asarray(c["upper"])
                subset |= 0 < np.isfinite(lo).sum() < lo.size and 0 < np.isfinite(up).sum() < up.size
            if c["kind"] == "control_bound":
                lo, up = np.asarray(c["lower"]), np.asarray(c["upper"])
                infs |= bool(np.isneginf(lo).any() and (up == bv.DBL_MAX).any() and (lo == -bv.DBL_MAX).any())
    for m, n in ((True, False), (False, True), (True, True)):
        for multi in (False, True):
            assert (m, n, multi) in costs, (m, n, multi)
    for kind in (("trajectory", True, False), ("control", False, True), ("mixed", True, True)):
        assert kind in cstrs, kind
    assert ("trajectory_bound", False, False) in cstrs and ("control_bound", False, False) in cstrs
    assert n1 and eq and subset and infs


def _c2(N):
    return bv.c2_like(N)


def test_mirror_agrees_with_hand_arithmetic():
    d = bv.build_dispatch
    # Q: C2-like tiled at N = 73, staged untiled at 74
    assert d(bv.c2_like(73))["q"] == "tiled" and d(bv.c2_like(74))["q"] == "staged"
    assert bv.edge(_c2, "q", 2) == 73
    # C5-like: Q staged at 78 and unstaged at 79; K7 staged at 98 and unstaged at 99
    assert d(bv.c5_like(78))["q"] == "staged" and d(bv.c5_like(79))["q"] == "unstaged"
    assert d(bv.c5_like(98))["k7"] == "staged" and d(bv.c5_like(99))["k7"] == "unstaged"
    # initial state, nx = 2, nu = 1: J in shared memory at N = 167, in the workspace at 168
    assert d(bv.c4_like(167), smem_optin=232448)["schur"] == "smem" and d(bv.c4_like(168), smem_optin=232448)["schur"] == "ws"
    assert d(bv.c4_like(64))["schur"] == "small" and d(bv.c4_like(65))["schur"] == "smem"
    # K1: per = nx^2 + nx nu + nx
    for (nx, nu), want in {(2, 1): "g8", (2, 5): "g16", (1, 15): "g32", (4, 3): "g32", (5, 1): "cta",
                           (16, 2): "cta_strided"}.items():
        assert d(bv.every_kind(nx, nu, 3, 2))["k1"] == want, (nx, nu)
    assert not d(bv.c2_like(10))["shared"] and d(bv.c2_like(10, shared=True))["shared"]
    assert not d(bv.c4_like(10))["shared"]


@pytest.mark.parametrize("s", bv.SHAPES, ids=[s.name for s in bv.SHAPES])
def test_oracle_builds_every_shape(s):
    """every problem of the table is well formed for the oracle (its build runs; the solve is left to the GPU tests)"""
    from copra_b200 import workloads as wl
    from oracle import pyoracle as po
    bp = s.make()
    o = po.lmpc(wl.instance(bp, bp["batch"] - 1), solve=False)
    assert o["Q"].shape == (o["sizes"]["nvar"],) * 2
