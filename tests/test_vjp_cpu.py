"""Sensitivities of LMPC solutions without a GPU: the dense numpy adjoint reference (tests/vjp_reference.py) against central
differences of the CPU oracle, the host-side refusals of copra_b200_lmpc_vjp and its exported symbols."""
import ctypes as C

import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from tests import vjp_reference as vr


def test_one_dimensional_adjoint():
    # min 1/2 x^2 - 5x, x <= 1 with L = x: dL/db = 1, dL/dc = 0
    o = dict(Q=np.eye(1), Aeq=np.zeros((0, 1)), Aineq=np.ones((1, 1)), iact=np.array([1]), Psi=np.zeros((2, 1)),
             Phi=np.zeros((2, 1)))
    adj = vr.adjoint(o, dcontrol=np.ones(1))
    assert adj["bineq"][0] == pytest.approx(1.0, abs=1e-15)
    assert adj["c"][0] == pytest.approx(0.0, abs=1e-15)


CASES = [("c1", lambda: wl.c1(), [0]), ("c2", lambda: wl.c2(batch=8), [3]), ("c3", lambda: wl.c3(batch=4), [0, 3]),
         ("c3_walk", lambda: wl.c3_walk(batch=4), [1, 2]), ("c2_floor", lambda: vr.c2_floor(8), [1, 5])]


@pytest.mark.parametrize("name,make,idx", CASES, ids=[c[0] for c in CASES])
def test_reference_matches_central_differences(name, make, idx):
    bp = make()
    rng = np.random.default_rng(11)
    checked = 0
    for i in idx:
        inst = wl.instance(bp, i)
        o = vr.solve(inst)
        assert o["fail"] == 0
        dcontrol = rng.normal(size=o["control"].shape)
        dtraj = rng.normal(size=o["trajectory"].shape)
        adj = vr.adjoint(o, dcontrol, dtraj)
        act = set(o["iact"].tolist())
        for key in vr.vector_keys(inst):
            delta = vr.random_direction(inst, rng, [key])
            if not np.any(delta[key]):
                continue
            scale = max(1.0, np.abs(vr.get_vector(inst, key)).max())
            # the largest step that keeps the active set: the oracle's own rounding is divided by h
            for h in (1e-2 * scale, 1e-3 * scale, 1e-4 * scale):
                ends = [vr.solve(vr.with_vectors(inst, {key: vr.get_vector(inst, key) + sgn * h * delta[key]}))
                        for sgn in (1.0, -1.0)]
                if all(set(e["iact"].tolist()) == act and e["fail"] == 0 for e in ends):
                    break
            else:
                continue  # the active set moved: the map is not affine across [theta - h delta, theta + h delta]
            fd = (vr.loss(ends[0], dcontrol, dtraj) - vr.loss(ends[1], dcontrol, dtraj)) / (2.0 * h)
            ref = vr.directional(inst, adj, delta)
            mag = max(abs(fd), abs(ref), 1e-3 * np.abs(dcontrol).sum())
            assert abs(fd - ref) <= 1e-5 * mag, (name, i, key, fd, ref)
            checked += 1
    assert checked >= 3


def test_vjp_exports():
    lib = capi.load()
    for name in ("copra_b200_lmpc_vjp", "copra_b200_multi_lmpc_vjp"):
        assert name in capi.EXPORTS
        getattr(lib, name)


def test_vjp_refuses_without_a_solve():
    lib = capi.load()
    out = capi.VjpOut()
    # null handle / null output description
    assert lib.copra_b200_lmpc_vjp(None, None, None, capi.HOST, C.byref(out)) == -1
    with pytest.raises(capi.CopraB200Error) as e:
        _bare_engine().lmpc_vjp()
    assert e.value.code == -5


def _bare_engine():
    eng = capi.Engine.__new__(capi.Engine)  # no device handle: only the host-side bookkeeping
    eng._last_bp = None
    eng.solve_count = 0
    return eng


def test_vjp_lengths():
    nx, plen, clen = capi.vjp_lengths(wl.c3_walk(batch=2))
    assert nx == 6 and plen == [2 * 161, 2] and clen == [4 * 160]
    nx, plen, clen = capi.vjp_lengths(wl.c2(batch=2))
    assert nx == 2 and plen == [2, 1] and clen == [2, 1]
