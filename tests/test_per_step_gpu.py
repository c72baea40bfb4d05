"""Per-step references and limits (COPRA_B200_PER_STEP) and the receding-horizon retarget on the GPU: parity with the
oracle on copra's autoSpan'd full-size form, the structured kernels kept, and retarget bitwise a full build."""
import os
import subprocess

import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from oracle import pyoracle as po
from tests.test_gpu_parity import STAGES, _kkt_ok
from tests.util import active_set, rel_err, x_err

pytestmark = pytest.mark.gpu

E_ARG, E_UNSUPPORTED, E_STATE = -1, -4, -5
RESULTS = ("control", "trajectory", "x", "status", "iters", "nact", "iact")


def tile_per_step(bp):
    """the same problem with every step-size vector (except a TargetCost's) given per step: repeated at every step"""
    N = bp["N"]
    out = dict(bp, costs=[], constraints=[])
    for c in bp["costs"]:
        c = dict(c)
        if c["kind"] != "target":
            steps = N + 1 if c["kind"] == "trajectory" else N
            p = np.asarray(c["p"], dtype=np.float64)
            c.update(p=np.tile(p, (1,) * (p.ndim - 1) + (steps,)), per_step=True)
        out["costs"].append(c)
    for c in bp["constraints"]:
        c = dict(c)
        steps = N + 1 if c["kind"] in ("trajectory", "trajectory_bound") else N
        for k in ("f", "lower", "upper"):
            if c.get(k) is not None:
                v = np.asarray(c[k], dtype=np.float64)
                c[k] = np.tile(v, (1,) * (v.ndim - 1) + (steps,))
        c["per_step"] = True
        out["constraints"].append(c)
    return out


def _every_kind(initial_state, batch=3, N=9, seed=5):
    """every per-step kind (three costs, row constraints of each kind, an equality among them, both bounds) next to step-size
    ones"""
    rng = np.random.default_rng(seed)
    nx, nu = 2, 1
    wave = lambda steps, rows: 0.2 * np.sin(np.arange(steps * rows) * 0.7)  # noqa: E731
    up = np.tile([2.0, 1.0], N + 1) + np.repeat(0.05 * np.arange(N + 1), 2)
    lo = np.tile([-np.inf, 3.0], N + 1) + np.repeat(0.1 * np.arange(N + 1), 2)  # quirk Q1: a finite lower bound reads x <= lower
    bp = dict(name="per-step", nx=nx, nu=nu, N=N, batch=batch, initial_state=initial_state,
              A=np.array([[1.0, 0.1], [0.0, 1.0]]), B=np.array([[0.005], [0.1]]), d=np.array([0.01, -0.02]),
              x0=np.array([0.3, -1.0]) + 0.1 * np.arange(batch)[:, None],
              costs=[dict(kind="trajectory", M=np.eye(2), p=rng.normal(size=(batch, 2 * (N + 1))) * 0.3, w=np.array([1.5, 0.7]),
                          per_step=True),
                     dict(kind="target", M=np.eye(2), p=np.ones(2), w=np.array([2.0, 3.0])),
                     dict(kind="control", N=np.eye(1), p=0.4 + wave(N, 1), w=np.array([0.1]), per_step=True),
                     dict(kind="mixed", M=np.ones((1, 2)), N=np.ones((1, 1)), p=0.3 + wave(N, 1), w=np.array([0.3]), per_step=True),
                     dict(kind="mixed", M=np.ones((1, 2)), N=np.ones((1, 1)), p=np.array([0.1]), w=np.array([0.2]))],
              constraints=[dict(kind="trajectory", E=np.eye(2), f=np.tile([50.0, 40.0], N + 1) + wave(N + 1, 2), per_step=True),
                           dict(kind="trajectory", E=np.array([[1.0, 0.5]]), f=0.8 + wave(N + 1, 1), per_step=True),
                           dict(kind="control", G=np.eye(1), f=20.0 + wave(N, 1), per_step=True),
                           dict(kind="control", G=np.array([[-1.0]]), f=np.full((batch, N), 0.02) + 0.01 * np.arange(N), per_step=True),
                           dict(kind="mixed", E=np.array([[0.0, 1.0]]), G=np.array([[1.0]]), f=-0.5 + wave(N, 1), is_ineq=False,
                                per_step=True),
                           dict(kind="mixed", E=np.ones((2, 2)), G=np.ones((2, 1)), f=60.0 + wave(N, 2), per_step=True),
                           dict(kind="mixed", E=np.ones((1, 2)), G=np.ones((1, 1)), f=np.array([60.0])),
                           dict(kind="trajectory_bound", lower=lo, upper=up, per_step=True),
                           dict(kind="control_bound", lower=np.full(N, -1.0) - 0.01 * np.arange(N),
                                upper=np.full((batch, N), 1.5) + 0.02 * np.arange(N), per_step=True)])
    if initial_state:
        bp.update(R=np.array([[2.0, 0.1], [0.1, 1.0]]), r=np.array([0.1, -0.2]), x0lb=bp["x0"] - np.array([0.1, 0.5]),
                  x0ub=bp["x0"] + np.array([0.1, 0.5]))
    return bp


@pytest.mark.parametrize("initial_state", [False, True])
def test_per_step_entries_match_spanned_oracle(engine, initial_state):
    """per-step costs and constraints of every kind against the oracle given the same problem as copra's autoSpan'd
    full-size entries (block-diagonal matrices, full-length vectors)"""
    bp = _every_kind(initial_state)
    hb = capi.HostBatch(bp)
    out = engine.lmpc_run(hb)
    stages = {k: engine.download(hb, k) for k in STAGES}
    span = wl.spanned(bp)
    for i in range(bp["batch"]):
        o = po.lmpc(wl.instance(span, i))
        for k in STAGES:
            assert rel_err(stages[k][i], o[k]) <= 1e-10, (k, i, rel_err(stages[k][i], o[k]))
        assert out["status"][i] == o["fail"] == 0
        assert x_err(out["x"][i], o["x"]) <= 1e-6
        assert active_set(out["iact"][i], out["nact"][i]) == active_set(o["iact"])
    assert engine.hessian_is_shared() == (not initial_state)


@pytest.mark.parametrize("make", [lambda: wl.c2(batch=96), lambda: wl.c3(batch=64), lambda: wl.c5(batch=8)], ids=["c2", "c3", "c5"])
def test_tiled_vectors_are_step_size_entries_bit_for_bit(engine, make):
    """per-step vectors that repeat the step-size vector run the same kernels to the same bits (C2: gi_small; C3: thin
    solver, shared factor; C5: thin solver, per-instance factors)"""
    bp = make()
    ref = engine.lmpc_run(bp)
    solver, shared = engine.last_solver(), engine.hessian_is_shared()
    got = engine.lmpc_run(tile_per_step(bp))
    assert engine.last_solver() == solver and engine.hessian_is_shared() == shared
    for k in ("control", "trajectory", "iact", "iters", "status"):
        assert np.array_equal(got[k], ref[k]), k


def test_c3_walk_keeps_the_fast_path(engine):
    bp = wl.c3_walk(batch=592)
    hb = capi.HostBatch(bp)
    out = engine.lmpc_run(hb)
    assert engine.last_solver() == "gt_factor_kernel + gi_thin_kernel"
    assert engine.hessian_is_shared()
    assert (out["status"] == 0).all()
    assert _kkt_ok(bp, hb, engine, out, range(0, 592, 37)) <= 1e-8
    E = bp["constraints"][0]["E"]
    f = bp["constraints"][0]["f"].reshape(592, 160, 4)
    zmp = np.einsum("bri,bki->bkr", E, out["trajectory"].reshape(592, 161, 6)[:, :160])
    assert np.all(zmp <= f + 1e-6)  # inside each step's own box


def test_c3_walk_matches_spanned_oracle(engine):
    bp = wl.c3_walk(batch=16)
    hb = capi.HostBatch(bp)
    out = engine.lmpc_run(hb)
    stages = {k: engine.download(hb, k) for k in STAGES}
    span = wl.spanned(bp)
    for i in range(16):
        o = po.lmpc(wl.instance(span, i))
        for k in STAGES:
            assert rel_err(stages[k][i], o[k]) <= 1e-10, (k, i, rel_err(stages[k][i], o[k]))
        assert out["status"][i] == o["fail"] == 0
        assert x_err(out["x"][i], o["x"]) <= 1e-6
        assert active_set(out["iact"][i], out["nact"][i]) == active_set(o["iact"])


def _shift(bp, out, ticks=1):
    """a later tick of a receding horizon: every per-step vector advanced by `ticks` steps (its last step repeated), x0
    halfway between the current one and the solved state `ticks` steps on (a state exactly on a limit would leave the
    step-0 rows, which no control reaches, infeasible by rounding)"""
    nx, N = bp["nx"], bp["N"]
    nxt = dict(bp, x0=0.5 * (np.asarray(bp["x0"]) + out["trajectory"][:, ticks * nx:(ticks + 1) * nx]))

    def adv(v, rows):
        v = np.asarray(v, dtype=np.float64)
        tail = np.tile(v[..., -rows:], (1,) * (v.ndim - 1) + (ticks,))
        return np.concatenate([v[..., ticks * rows:], tail], axis=-1)

    nxt["costs"] = [dict(c, p=adv(c["p"], c["M"].shape[0] if c.get("M") is not None else c["N"].shape[0])) if c.get("per_step") else c
                    for c in bp["costs"]]
    cs = []
    for c in bp["constraints"]:
        c = dict(c)
        if c.get("per_step"):
            rows = nx if c["kind"] == "trajectory_bound" else (bp["nu"] if c["kind"] == "control_bound" else
                                                                 np.asarray(c["E"] if c.get("E") is not None else c["G"]).shape[-2])
            for k in ("f", "lower", "upper"):
                if c.get(k) is not None:
                    c[k] = adv(c[k], rows)
        cs.append(c)
    nxt["constraints"] = cs
    return nxt


def _nan_matrices(bp):
    """the same problem with every matrix (and d, w) replaced by NaN: retarget must not read them"""
    nan = lambda a: np.full(np.shape(a), np.nan)  # noqa: E731
    out = dict(bp, A=nan(bp["A"]), B=nan(bp["B"]), d=nan(bp["d"]))
    out["costs"] = [dict(c, **{k: nan(c[k]) for k in ("M", "N", "w") if c.get(k) is not None}) for c in bp["costs"]]
    out["constraints"] = [dict(c, **{k: nan(c[k]) for k in ("E", "G") if c.get(k) is not None}) for c in bp["constraints"]]
    return out


def _same(a, b):
    for k in RESULTS:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("make", [lambda: tile_per_step(wl.c2(batch=64)), lambda: wl.c3_walk(batch=256)], ids=["c2", "c3_walk"])
def test_retarget_is_a_full_build_bitwise(make):
    eng = capi.Engine(0)
    try:
        bp = make()
        first = eng.lmpc_run(bp)
        one = _shift(bp, first)
        two = _shift(one, first, ticks=2)
        r1 = eng.lmpc_retarget(one)   # small solver: stores the factor cache
        r2 = eng.lmpc_retarget(_nan_matrices(two))  # ... and loads it; the matrices in the problem are ignored
        assert not np.array_equal(r1["control"], first["control"])
        full1 = eng.lmpc_run(one)
        full2 = eng.lmpc_run(two)
        _same(r1, full1)
        _same(r2, full2)
        assert (r2["status"] == 0).all()
    finally:
        eng.close()


def test_warm_started_retarget_matches_cold():
    eng = capi.Engine(0)
    try:
        bp = wl.c3_walk(batch=256)
        first = eng.lmpc_run(bp)
        nxt = _shift(bp, first)
        cold = eng.lmpc_retarget(nxt)
        eng.set_warm_start(True)
        eng.lmpc_run(bp)  # the seed: the active sets at the previous tick
        warm = eng.lmpc_retarget(nxt)
        assert (warm["status"] == 0).all()
        for i in range(256):
            assert active_set(warm["iact"][i], warm["nact"][i]) == active_set(cold["iact"][i], cold["nact"][i]), i
        assert np.abs(warm["control"] - cold["control"]).max() <= 1e-8
    finally:
        eng.close()


def _code(fn):
    with pytest.raises(capi.CopraB200Error) as e:
        fn()
    return e.value.code


def test_retarget_errors():
    eng = capi.Engine(0)
    try:
        bp = tile_per_step(wl.c2(batch=8, N=12))
        assert _code(lambda: eng.lmpc_retarget(bp)) == E_STATE
        first = eng.lmpc_run(bp)
        nxt = _shift(bp, first)
        bad_n = tile_per_step(wl.c2(batch=8, N=13))
        bad_rows = dict(nxt, costs=[nxt["costs"][0], dict(nxt["costs"][1], N=np.eye(1).repeat(2, 0), w=np.ones(2),
                                                                p=np.tile(nxt["costs"][1]["p"], 2))])
        bad_kind = dict(nxt, constraints=[nxt["constraints"][0], dict(nxt["constraints"][1], kind="trajectory_bound",
                                                                     lower=np.full(26, -np.inf), upper=np.full(26, 9.0))])
        bad_count = dict(nxt, costs=nxt["costs"][:1])
        bad_full = dict(nxt, costs=[nxt["costs"][0], dict(nxt["costs"][1], per_step=False, p=np.array([2.0]))])
        lo = np.array(nxt["constraints"][0]["lower"], dtype=float)
        lo[1::2] = -50.0  # a finite lower bound at every step where the build had none
        bad_pattern = dict(nxt, constraints=[dict(nxt["constraints"][0], lower=lo), nxt["constraints"][1]])
        for bad in (bad_n, bad_rows, bad_kind, bad_count, bad_full):
            assert _code(lambda: eng.lmpc_retarget(bad)) == E_ARG
        lo2 = np.full_like(lo, -np.inf)
        lo2[5] = 0.0  # differs across steps: refused by the plan itself
        assert _code(lambda: eng.lmpc_retarget(dict(nxt, constraints=[dict(nxt["constraints"][0], lower=lo2), nxt["constraints"][1]]))) == E_ARG
        assert _code(lambda: eng.lmpc_retarget(bad_pattern)) == E_ARG
        # the resident build is still usable
        _same(eng.lmpc_retarget(nxt), eng.lmpc_run(nxt))
        # initial-state and full-size builds
        eng.lmpc_run(tile_per_step(wl.c4(batch=4)))
        assert _code(lambda: eng.lmpc_retarget(tile_per_step(wl.c4(batch=4)))) == E_UNSUPPORTED
        dense = wl.spanned(wl.c3_walk(batch=2))
        eng.lmpc_run(dense)
        assert _code(lambda: eng.lmpc_retarget(dense)) == E_UNSUPPORTED
        # per-step TARGET cost, and a per-step bound whose pattern changes over the steps
        tgt = dict(bp, costs=[dict(bp["costs"][0], per_step=True), bp["costs"][1]])
        assert _code(lambda: eng.lmpc_run(tgt)) == E_ARG
        assert _code(lambda: eng.lmpc_run(dict(bp, constraints=[dict(bp["constraints"][0], lower=lo2), bp["constraints"][1]]))) == E_ARG
    finally:
        eng.close()


def test_sharded_per_step_run_and_retarget_match_single_device(engine):
    bp = wl.c3_walk(batch=301)
    s = engine.sizes(capi.HostBatch(bp))
    single = engine.lmpc_run(bp)
    nxt = _shift(bp, single)
    single_rt = engine.lmpc_retarget(nxt)
    m = capi.MultiEngine([0, 0])
    try:
        _same(m.lmpc_run(bp, s), single)
        assert [hi - lo for _, lo, hi in m.shards()] == [151, 150]
        _same(m.lmpc_retarget(nxt, s), single_rt)
    finally:
        m.close()


def test_cpp_facade_per_step_and_retarget():
    """BatchedLMPC with per-step descriptors and retarget() against per-instance copra::LMPC on autoSpan'd full-size entries"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "tests", "cpp", "test_per_step")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
