"""The build kernels (K1 condensing, K2-K4 assembly, K4' Schur block, K7 results) at every variant their launchers dispatch
to, both sides of every size threshold and past every grid-stride boundary (tests/build_variants.py), against the oracle:
Phi / Psi / xi bit for bit, the QP to 1e-10, the Schur block against an iteratively refined reference, K7 against an
extended-precision evaluation from the GPU's own solution, and the kernel names under torch.profiler."""
import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from oracle import pyoracle as po
from tests import build_variants as bv
from tests.test_gpu_parity import STAGES
from tests.test_per_step_gpu import RESULTS, tile_per_step
from tests.util import rel_err, zeros_preserved

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
IDS = [s.name for s in bv.SHAPES]
INITIAL = [s for s in bv.SHAPES if s.make().get("initial_state")]
SHARED = [s for s in bv.SHAPES if bv.build_dispatch(s.make())["shared"]]
EF_PAIR = [s for s in bv.SHAPES if s.across == ("ef", "staged", "unstaged") and not bv.hessian_shared(s.make())]


@pytest.fixture(scope="module")
def built(engine):
    """shape -> its problem, the GPU's results and every downloaded stage, and the oracle of its sampled instances (each shape
    is built and solved once per module)"""
    cache = {}

    def get(shape):
        if shape.name not in cache:
            bp = shape.make()
            hb = capi.HostBatch(bp)
            out = engine.lmpc_run(hb)
            stages = {k: engine.download(hb, k) for k in STAGES}
            oracle = {i: po.lmpc(wl.instance(bp, i)) for i in bv.sample(bp)}
            cache[shape.name] = dict(bp=bp, out=out, stages=stages, oracle=oracle, shared=engine.hessian_is_shared())
        return cache[shape.name]
    return get


@pytest.mark.parametrize("shape", bv.SHAPES, ids=IDS)
def test_stages_match_oracle(built, shape):
    """Phi, Psi, xi bitwise (DESIGN section 4); Q, c, rows and bounds to 1e-10 with structural zeros kept (the initial-state
    Q to 1e-9: Cholesky Schur block vs the oracle's LU inverse, quirk Q7); the solve's status"""
    r = built(shape)
    bp, st, out = r["bp"], r["stages"], r["out"]
    assert r["shared"] == bv.build_dispatch(bp)["shared"]
    for i, o in r["oracle"].items():
        for k in ("Phi", "Psi", "xi"):
            assert np.array_equal(st[k][i], o[k]), (shape.name, i, k, np.abs(st[k][i] - o[k]).max())
        for k in STAGES[3:]:
            tol = 1e-9 if (k == "Q" and bp.get("initial_state")) else 1e-10
            e = rel_err(st[k][i], o[k])
            assert e <= tol, (shape.name, i, k, e)
            assert zeros_preserved(st[k][i], o[k]), (shape.name, i, k, "structural zeros")
        assert out["status"][i] == o["fail"], (shape.name, i, out["status"][i], o["fail"])


@pytest.mark.parametrize("shape", INITIAL, ids=[s.name for s in INITIAL])
def test_schur_block_against_refined_reference(built, shape):
    """the top-left block R + E Qb^-1 E' of the initial-state Hessian, from the GPU's own Qb and E, against Qb Y = E' solved in
    float64 with three steps of extended-precision iterative refinement: within 32 nU u cond2(Qb), relative"""
    r = built(shape)
    bp = r["bp"]
    nx = bp["nx"]
    for i in r["oracle"]:
        Q = r["stages"]["Q"][i]
        Qb, E = Q[nx:, nx:], Q[:nx, nx:]
        R = wl.instance(bp, i)["R"]
        R = np.zeros((nx, nx)) if R is None else R
        Y = np.linalg.solve(Qb, E.T)
        Ql, El = Qb.astype(np.longdouble), E.T.astype(np.longdouble)
        for _ in range(3):
            Y = Y + np.linalg.solve(Qb, (El - Ql @ Y.astype(np.longdouble)).astype(float))
        ref = R.astype(np.longdouble) + E.astype(np.longdouble) @ Y.astype(np.longdouble)
        err = float(np.abs(Q[:nx, :nx] - ref).max() / np.abs(ref).max())
        kappa = np.linalg.cond(Qb)
        bound = 32 * Qb.shape[0] * U * kappa
        print("%s #%d: cond2(Qb) %.3e  error %.3e  bound %.3e" % (shape.name, i, kappa, err, bound))
        assert err <= bound, (shape.name, i, err, bound, kappa)


@pytest.mark.parametrize("shape", bv.SHAPES, ids=IDS)
def test_results_against_extended_precision(built, shape):
    """K7 on the GPU's own solution: control is the tail of x bit for bit, and trajectory = Phi x0 + Psi U + xi (x0 from the
    solution in initial-state mode) within (k + 2) u sum|terms| of its extended-precision value, k the row's products"""
    r = built(shape)
    bp, out = r["bp"], r["out"]
    nx, nu = bp["nx"], bp["nu"]
    off = nx if bp.get("initial_state") else 0
    for i, o in r["oracle"].items():
        x = out["x"][i]
        assert np.array_equal(out["control"][i], x[off:]), (shape.name, i)
        x0 = x[:nx] if off else np.asarray(wl.instance(bp, i)["x0"], float)
        Phi, Psi, xi = (o[k].astype(np.longdouble) for k in ("Phi", "Psi", "xi"))
        ref = Phi @ x0.astype(np.longdouble) + Psi @ x[off:].astype(np.longdouble) + xi
        terms = np.abs(Phi) @ np.abs(x0) + np.abs(Psi) @ np.abs(x[off:]) + np.abs(xi)
        k = nx + (np.arange(Phi.shape[0]) // nx) * nu
        err = np.abs(out["trajectory"][i].astype(np.longdouble) - ref)
        bad = np.flatnonzero(err > (k + 2) * U * terms)
        assert bad.size == 0, (shape.name, i, bad[:5], float(err[bad[0]]), float(terms[bad[0]]))


@pytest.mark.parametrize("shape", SHARED, ids=[s.name for s in SHARED])
def test_shared_and_per_instance_hessian_agree_bitwise(engine, built, shape):
    """the batch-invariant assembly (one Q and one E per cost from instance 0's tables) and the per-instance one (the same w
    given per instance) give the same Q and c bit for bit"""
    r = built(shape)
    bp = r["bp"]
    assert r["shared"]
    tiled = dict(bp, costs=[dict(c, w=np.tile(np.asarray(c["w"], float), (bp["batch"], 1))) for c in bp["costs"]])
    hb = capi.HostBatch(tiled)
    engine.lmpc_build(hb)
    assert not engine.hessian_is_shared()
    assert bv.build_dispatch(tiled)["q"] == bv.build_dispatch(bp)["q"] and bv.build_dispatch(tiled)["ef"] == bv.build_dispatch(bp)["ef"]
    for k in ("Q", "c"):
        assert np.array_equal(engine.download(hb, k), r["stages"][k]), (shape.name, k)


def _retargeted(bp):
    """the same problem with new x0 and new vectors (p, f, finite bounds), varying along each vector"""
    def bump(v, scale):
        v = np.asarray(v, dtype=np.float64)
        ramp = scale * (1.0 + 0.01 * np.arange(v.shape[-1]))
        return np.where(np.isfinite(v), v + ramp, v)
    out = dict(bp, x0=0.9 * np.asarray(bp["x0"]) + 0.01)
    out["costs"] = [dict(c, p=bump(c["p"], 0.05)) for c in bp["costs"]]
    cs = []
    for c in bp["constraints"]:
        c = dict(c)
        for k, s in (("f", 0.02), ("lower", -0.1), ("upper", 0.1)):
            if c.get(k) is not None:
                c[k] = bump(c[k], s)
        cs.append(c)
    out["constraints"] = cs
    return out


@pytest.mark.parametrize("per_step", [False, True], ids=["step-size", "per-step"])
@pytest.mark.parametrize("shape", EF_PAIR, ids=[s.name for s in EF_PAIR])
def test_retarget_is_a_fresh_build_bitwise(engine, shape, per_step):
    """copra_b200_lmpc_retarget (K2a vectors, K2c f alone, K4) on either K2c variant: every stage and result equals a fresh
    lmpc_run of the new problem bit for bit"""
    bp = shape.make()
    if per_step:
        bp = tile_per_step(bp)
    assert bv.build_dispatch(bp)["ef"] == shape.expect["ef"]
    first = engine.lmpc_run(bp)
    hb = capi.HostBatch(_retargeted(bp))
    rt = engine.lmpc_retarget(hb)
    rt_st = {k: engine.download(hb, k) for k in STAGES}
    full = engine.lmpc_run(hb)
    for k in STAGES:
        assert np.array_equal(rt_st[k], engine.download(hb, k)), (shape.name, k)
    for k in RESULTS:
        assert np.array_equal(rt[k], full[k]), (shape.name, k)
    assert not np.array_equal(rt["control"], first["control"])


def test_kernel_names_match_the_mirror(engine):
    """each shape on either side of a threshold, run under torch.profiler: the kernels the mirror names ran and their
    alternatives did not (the group width, staged vs unstaged Q and where J lives are arguments of one kernel: those rest
    on the mirror and the CPU test)"""
    from torch.profiler import ProfilerActivity, profile
    for shape in [s for s in bv.SHAPES if s.across is not None]:
        bp = shape.make()
        hb = capi.HostBatch(bp)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            engine.lmpc_run(hb)
            engine.synchronize()
        names = {e.name for e in prof.events()}
        assert any("k1_condense" in n for n in names), (shape.name, "no kernel activity recorded", sorted(names)[:10])
        want = bv.build_dispatch(bp)
        for key, table in bv.KERNELS.items():
            expect = table[want[key]]
            if expect:
                assert any(expect in n for n in names), (shape.name, key, want[key], expect)
            for other in set(table.values()) - {expect, None}:
                assert not any(other in n for n in names), (shape.name, key, want[key], other)
