"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same inputs.
Tolerances are BASELINE.json's: condensed matrices 1e-10 relative, decision variables 1e-6,
identical active set."""
import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from oracle import pyoracle as po
from tests.util import active_set, active_set_excused, rel_err, x_err, zeros_preserved

pytestmark = pytest.mark.gpu

STAGES = ("Phi", "Psi", "xi", "Q", "c", "Aeq", "beq", "Aineq", "bineq", "lb", "ub")


def check_batch(engine, bp, instances=None, tol_mat=1e-10, tol_x=1e-6):
    hb = capi.HostBatch(bp)
    out = engine.lmpc_run(hb)
    stages = {k: engine.download(hb, k) for k in STAGES}
    idx = range(bp["batch"]) if instances is None else instances
    worst = {}
    for i in idx:
        o = po.lmpc(wl.instance(bp, i))
        for k in STAGES:
            e = rel_err(stages[k][i], o[k])
            worst[k] = max(worst.get(k, 0.0), e)
            assert e <= tol_mat, (bp["name"], i, k, e)
            assert zeros_preserved(stages[k][i], o[k]), (bp["name"], i, k, "structural zeros")
        assert out["status"][i] == o["fail"], (bp["name"], i, out["status"][i], o["fail"])
        if o["fail"] == 0:
            assert x_err(out["x"][i], o["x"]) <= tol_x, (bp["name"], i, "x", x_err(out["x"][i], o["x"]))
            # identical as sets; rows that differ must be weakly active at the optimum (counted, SURVEY.md 7)
            worst["excused_rows"] = worst.get("excused_rows", 0) + active_set_excused(active_set(out["iact"][i], out["nact"][i]), o)
            assert x_err(out["control"][i], o["control"]) <= tol_x
            assert x_err(out["trajectory"][i], o["trajectory"]) <= 1e-6  # scaled by max(1, |ref|): a trajectory may be ~0
            worst["x"] = max(worst.get("x", 0.0), x_err(out["x"][i], o["x"]))
            worst["iter_diff"] = max(worst.get("iter_diff", 0), abs(int(out["iters"][i][0]) - o["iter"][0]))
    print(bp["name"], {k: float("%.2e" % v) for k, v in worst.items()})
    return worst


def test_ka1_raw_qp(engine):
    """reference fixture `Problem` (tests/systems.h:11-38) through the raw-QP entry (B200Solver path)"""
    import json, os
    ka = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ka_problem.json")))
    r = engine.solve_qp_batch(ka["Q"], ka["c"], ka["Aeq"], ka["beq"], ka["Aineq"], ka["bineq"], ka["XL"], ka["XU"])
    assert r["status"][0] == 0
    assert np.abs(r["x"][0] - np.array(ka["x"])).max() < 1e-12
    assert active_set(r["iact"][0], r["nact"][0]) == set(ka["iact"])
    assert tuple(r["iters"][0]) == tuple(ka["iter"])


def test_random_qps_vs_oracle(engine):
    rng = np.random.default_rng(7)
    drops = 0
    for trial in range(40):
        n = int(rng.integers(2, 25))
        meq = int(rng.integers(0, max(1, n // 3)))
        m = int(rng.integers(0, 2 * n))
        B = 8
        L = rng.normal(size=(B, n, n))
        Q = L @ np.swapaxes(L, 1, 2) + 0.1 * np.eye(n)
        c = rng.normal(size=(B, n))
        Aeq = rng.normal(size=(B, meq, n))
        xf = rng.normal(size=(B, n))  # a feasible point
        beq = np.einsum("bij,bj->bi", Aeq, xf)
        Aineq = rng.normal(size=(B, m, n))
        bineq = np.einsum("bij,bj->bi", Aineq, xf) + rng.uniform(0.0, 1.0, size=(B, m))
        lb = xf - rng.uniform(0.1, 2.0, size=(B, n))
        ub = xf + rng.uniform(0.1, 2.0, size=(B, n))
        lb[rng.uniform(size=(B, n)) < 0.3] = -np.inf
        ub[rng.uniform(size=(B, n)) < 0.3] = np.finfo(float).max
        r = engine.solve_qp_batch(Q, c, Aeq if meq else None, beq if meq else None, Aineq if m else None,
                                  bineq if m else None, lb, ub)
        for b in range(B):
            o = po.quadprog(Q[b], c[b], Aeq[b], beq[b], Aineq[b], bineq[b], lb[b], ub[b])
            assert r["status"][b] == o["fail"], (trial, b)
            if o["fail"] == 0:
                assert x_err(r["x"][b], o["x"]) < 1e-8, (trial, b, x_err(r["x"][b], o["x"]))
                assert active_set(r["iact"][b], r["nact"][b]) == active_set(o["iact"]), (trial, b)
                assert tuple(r["iters"][b]) == o["iter"], (trial, b, r["iters"][b], o["iter"])
                drops += o["iter"][1]
    assert drops > 0  # the drop path was exercised


def test_infeasible_and_not_pd(engine):
    Q = np.eye(2)
    r = engine.solve_qp_batch(Q, np.zeros(2), None, None, np.array([[1.0, 0.0], [-1.0, 0.0]]), np.array([-1.0, -1.0]),
                              np.full(2, -np.inf), np.full(2, np.inf))
    assert r["status"][0] == 1  # x0 <= -1 and x0 >= 1
    r = engine.solve_qp_batch(np.array([[1.0, 2.0], [2.0, 1.0]]), np.zeros(2), None, None, None, None,
                              np.full(2, -1.0), np.full(2, 1.0))
    assert r["status"][0] == 2


@pytest.mark.parametrize("cost", ["target", "trajectory"])
def test_c1_reference_fixture(engine, cost):
    """configs[0]: BoundedSystem, N=300 (tests/TestLMPC.cpp:36-157) -- also checks the properties the
    reference test asserts."""
    bp = wl.c1(cost)
    check_batch(engine, bp)
    out = engine.lmpc_run(bp)
    traj, u = out["trajectory"][0], out["control"][0]
    assert abs(-1.0 - traj[-1]) <= 1e-3          # CHECK_LE(|xd(1) - vel.tail|, 0.001)
    assert traj[0::2].max() <= 0.0 + 1e-12       # pos <= x0(0)
    assert traj[1::2].max() <= 0.0 + 1e-6        # vel <= xUpper(1) + 1e-6
    assert u.max() <= 200.0 + 1e-6               # u <= uUpper + 1e-6


def test_c2(engine):
    check_batch(engine, wl.c2(batch=96))


def test_c3(engine):
    """64 instances against the oracle (thin solver: shared factor, Toeplitz rows)"""
    w = check_batch(engine, wl.c3(batch=64))
    assert w.get("excused_rows", 0) == 0 and w["iter_diff"] == 0


def test_c3_cluster_kernel(engine):
    """the same shape through the latency-oriented cluster kernel (what a handful of instances use: 4 clusters of at most 8
    CTAs cover the batch twice over on 148 SMs)"""
    check_batch(engine, wl.c3(batch=4))
    assert engine.last_solver() == "gi_cluster_kernel"


def test_c4_initial_state(engine):
    check_batch(engine, wl.c4(batch=24))


def test_c5(engine):
    """8 instances against the oracle (thin solver, per-instance factors, n = 800)"""
    check_batch(engine, wl.c5(batch=8))


def test_c5_single_cta_kernel():
    """the same shape with one CTA per instance (what batches of many waves use): the planner gives each instance a cluster
    only while the batch is at most 16 instances per SM, so 17 instances on one SM take the single-CTA kernel"""
    eng = capi.Engine(0, sm_limit=1)
    try:
        check_batch(eng, wl.c5(batch=17), instances=range(4))
        assert eng.last_solver() == "gt_factor_kernel + gi_thin_kernel"
    finally:
        eng.close()


def test_c5_hybrid_cluster_queue(engine):
    """longest-first queue whose head (batch / 16 = 5 instances) is solved by whole clusters and whose tail by single CTAs:
    every placement gives the same iterates (identical counts and active sets, x to rounding) as the all-single-CTA run (80
    instances on 4 SMs), and the oracle's on a sample"""
    bp = wl.c5(batch=80)
    want = ("status", "iters", "control", "iact", "nact")
    hyb = engine.lmpc_run(bp, want=want)
    assert "thin" in engine.last_solver()
    eng = capi.Engine(0, sm_limit=4)
    try:
        solo = eng.lmpc_run(bp, want=want)
        assert "thin" in eng.last_solver()
    finally:
        eng.close()
    assert np.array_equal(hyb["status"], solo["status"]) and np.array_equal(hyb["iters"], solo["iters"])
    assert np.array_equal(hyb["iact"], solo["iact"])
    assert np.abs(hyb["control"] - solo["control"]).max() <= 1e-9
    heavy = np.argsort(-hyb["iters"].sum(axis=1))[:2]
    for i in list(heavy) + [0, 79]:
        o = po.lmpc(wl.instance(bp, int(i)))
        assert x_err(hyb["control"][i], o["control"]) < 1e-6
        assert active_set(hyb["iact"][i]) == active_set(o["iact"]) and tuple(hyb["iters"][i]) == tuple(o["iter"])


def test_c5_general_kernel(engine):
    """C5's QP (n = 800, more than the cluster kernel holds) through the raw-QP entry, whose planner sends it to the
    single-CTA general kernel"""
    bp = wl.c5(batch=1)
    hb = capi.HostBatch(bp)
    engine.lmpc_run(hb)
    st = {k: engine.download(hb, k) for k in STAGES}
    o = po.lmpc(wl.instance(bp, 0))
    for k in STAGES:
        assert rel_err(st[k][0], o[k]) <= 1e-10, (k, rel_err(st[k][0], o[k]))
        assert zeros_preserved(st[k][0], o[k]), (k, "structural zeros")
    eq = st["Aeq"].shape[1] > 0
    r = engine.solve_qp_batch(st["Q"], st["c"], st["Aeq"] if eq else None, st["beq"] if eq else None, st["Aineq"], st["bineq"],
                              st["lb"], st["ub"])
    assert engine.last_solver() == "gi_batch_kernel"
    assert r["status"][0] == o["fail"] == 0
    # LMPC mode: the decision variables are the controls
    assert x_err(r["x"][0], o["x"]) <= 1e-6 and x_err(r["x"][0], o["control"]) <= 1e-6
    excused = active_set_excused(active_set(r["iact"][0], r["nact"][0]), o)
    assert tuple(r["iters"][0]) == tuple(o["iter"]), (r["iters"][0], o["iter"])
    print(bp["name"], {"excused_rows": excused})


# ---- committed golden fixtures (tests/golden/make_golden.py) -------------------------------------------
def _golden_cases():
    import json, os
    here = os.path.dirname(__file__)
    z = np.load(os.path.join(here, "golden", "small_cases.npz"))
    probs = json.load(open(os.path.join(here, "golden", "small_cases_problems.json")))
    from tests.test_oracle import _revive
    for name, prob in probs.items():
        yield name, _revive(prob), {k.split("/", 1)[1]: z[k] for k in z.files if k.startswith(name + "/")}


@pytest.mark.parametrize("name,prob,gold", list(_golden_cases()), ids=[n for n, _, _ in _golden_cases()])
def test_gpu_matches_committed_goldens(engine, name, prob, gold):
    """every cost / constraint kind, LMPC and InitialStateLMPC, against vectors committed in tests/golden"""
    bp = dict(prob, batch=1, name=name)
    hb = capi.HostBatch(bp)
    out = engine.lmpc_run(hb)
    for k in STAGES:
        got = engine.download(hb, k)[0]
        tol = 1e-9 if (k == "Q" and prob.get("initial_state")) else 1e-10  # Schur block: Cholesky vs LU inverse (quirk Q7)
        assert rel_err(got, gold[k]) <= tol, (name, k, rel_err(got, gold[k]))
    assert out["status"][0] == 0
    assert x_err(out["x"][0], gold["x"]) <= 1e-6
    assert active_set(out["iact"][0], out["nact"][0]) == active_set(gold["iact"])
    assert rel_err(out["trajectory"][0], gold["trajectory"]) <= 1e-8


# ---- BASELINE.json full sizes through size-independent properties ----------------------------------------
def _kkt_ok(bp, hb, engine, out, idx):
    from oracle import copra_numpy as cn
    st = {k: engine.download(hb, k) for k in ("Q", "c", "Aeq", "beq", "Aineq", "bineq", "lb", "ub")}
    worst = 0.0
    for i in idx:
        kkt = cn.kkt_residuals(st["Q"][i], st["c"][i], st["Aeq"][i], st["beq"][i], st["Aineq"][i], st["bineq"][i], st["lb"][i],
                               st["ub"][i], out["x"][i], out["iact"][i][: out["nact"][i]])
        worst = max(worst, kkt["stationarity"], kkt["primal"], kkt["dual"], kkt["complementarity"])
    return worst


def test_full_size_c2_properties(engine):
    """configs[1] at full batch: all solved, KKT on a sample, and shard equivalence (two half batches give
    bit-identical results to the full batch: instances are independent, SURVEY.md 8e)"""
    bp = wl.c2(batch=4096)
    hb = capi.HostBatch(bp)
    out = engine.lmpc_run(hb)
    assert (out["status"] == 0).all()
    assert _kkt_ok(bp, hb, engine, out, range(0, 4096, 257)) <= 1e-8
    halves = [engine.lmpc_run(wl.shard(bp, r, 2)[0]) for r in range(2)]
    assert np.array_equal(np.concatenate([h["control"] for h in halves]), out["control"])
    assert np.array_equal(np.concatenate([h["iact"] for h in halves]), out["iact"])
    # terminal velocity reaches the target within the reference test's tolerance where the bound allows it
    assert np.all(out["trajectory"][:, 1::2].max(axis=1) <= 1e-6)


def test_full_size_c4_drop_path(engine):
    """configs[3]: InitialStateLMPC, 50 drops per instance (SURVEY.md 8d) -- KKT + x0 inside its box"""
    bp = wl.c4(batch=2048)
    hb = capi.HostBatch(bp)
    out = engine.lmpc_run(hb)
    assert (out["status"] == 0).all()
    assert out["iters"][:, 1].min() >= 40
    assert _kkt_ok(bp, hb, engine, out, range(0, 2048, 199)) <= 1e-8
    x0 = out["x"][:, :2]
    assert np.all(x0 >= bp["x0lb"] - 1e-9) and np.all(x0 <= bp["x0ub"] + 1e-9)


def test_c3_sample_properties(engine):
    bp = wl.c3(batch=64)
    hb = capi.HostBatch(bp)
    out = engine.lmpc_run(hb)
    assert (out["status"] == 0).all()
    assert _kkt_ok(bp, hb, engine, out, range(0, 64, 9)) <= 1e-8
    # ZMP stays inside its box at every step (the MixedConstraint rows)
    E, f = bp["constraints"][0]["E"], bp["constraints"][0]["f"]
    traj = out["trajectory"].reshape(64, 161, 6)[:, :160]
    zmp = np.einsum("bri,bki->bkr", E, traj)
    assert np.all(zmp <= f[:, None, :] + 1e-6)


def test_edge_cases(engine):
    # horizon 1, batch 1; no constraints at all (only the DBL_MAX default bounds, quirk Q4)
    bp = wl.c2(batch=1, N=1)
    o = po.lmpc(wl.instance(bp, 0))
    out = engine.lmpc_run(bp)
    assert out["status"][0] == o["fail"] and x_err(out["x"][0], o["x"]) < 1e-9
    bp = wl.c2(batch=3, N=7)
    bp["constraints"] = []
    out = engine.lmpc_run(bp)
    for i in range(3):
        o = po.lmpc(wl.instance(bp, i))
        assert out["nact"][i] == 0 and x_err(out["x"][i], o["x"]) < 1e-9 and tuple(out["iters"][i]) == o["iter"]
    # infeasible instance inside a batch is reported per instance, the others still solve
    bp = wl.c2(batch=4, N=10)
    up = np.array(bp["constraints"][1]["upper"], dtype=float)
    bp["constraints"].append(dict(kind="control", G=np.array([[-1.0]]), f=np.array([-1e6])))  # u >= 1e6 vs u <= ~200
    out = engine.lmpc_run(bp)
    assert (out["status"] == 1).all()
    # argument errors surface as COPRA_B200_E_ARG (std::domain_error in the facade)
    bad = wl.c2(batch=2)
    bad["N"] = 0
    with pytest.raises(capi.CopraB200Error) as e:
        engine.lmpc_run(bad)
    assert e.value.code == -1


def test_condense_entry(engine):
    bp = wl.c5(batch=3, N=9)
    Phi, Psi, xi = engine.condense(bp["A"], bp["B"], bp["d"], 9)
    for i in range(3):
        P, S, x = po.condense(bp["A"][i], bp["B"][i], bp["d"][i], 9)
        assert np.array_equal(Phi[i], P) and np.array_equal(Psi[i], S) and np.array_equal(xi[i], x)  # bit-exact


def test_cpp_facade_reference_scenarios():
    """the reference's test scenarios (tests/TestLMPC.cpp, TestSolvers.cpp, TestLMPC_InitialState.cpp) against
    the C++ facade on the GPU"""
    import os, subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "tests", "cpp", "test_facade")
    r = subprocess.run([exe, "gpu"], capture_output=True, text=True, timeout=600)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


def test_dgemm_dmma_primitive(engine):
    """the tensor-core FP64 GEMM behind full-size assembly: NN (TMA-fed when aligned) and TN, ragged and tiny shapes"""
    rng = np.random.default_rng(11)
    for (M, N, K, ta) in [(64, 64, 16, False), (128, 96, 64, False), (130, 70, 37, False), (5, 3, 2, False), (301, 300, 602, False),
                          (64, 64, 16, True), (77, 33, 129, True), (300, 300, 602, True), (1, 50, 602, True),
                          # even leading dimensions: the tensor-map TMA pipeline, ragged in every direction
                          (130, 70, 38, False), (258, 130, 50, False), (2, 2, 2, False), (66, 34, 130, True), (322, 966, 320, True),
                          (320, 966, 320, False)]:
        A = rng.normal(size=(3, K, M) if ta else (3, M, K))
        B = rng.normal(size=(3, K, N))
        C0 = rng.normal(size=(3, M, N))
        got = engine.dgemm(A, B, C0, alpha=0.7, beta=-1.3, trans_a=ta)
        want = 0.7 * (np.swapaxes(A, 1, 2) if ta else A) @ B - 1.3 * C0
        assert np.abs(got - want).max() <= 1e-12 * max(1.0, np.abs(want).max()), (M, N, K, ta, np.abs(got - want).max())
        got = engine.dgemm(A, B, trans_a=ta)
        want = (np.swapaxes(A, 1, 2) if ta else A) @ B
        assert np.abs(got - want).max() <= 1e-12 * max(1.0, np.abs(want).max()), (M, N, K, ta)


def _span_m(M, steps, add_cols=0):
    M = np.atleast_2d(np.asarray(M, float))
    out = np.zeros((M.shape[0] * steps, M.shape[1] * (steps + add_cols)))
    for i in range(steps):
        out[i * M.shape[0]:(i + 1) * M.shape[0], i * M.shape[1]:(i + 1) * M.shape[1]] = M
    return out


@pytest.mark.parametrize("initial_state", [False, True])
def test_full_size_entries_match_oracle(engine, initial_state):
    """full-size (autoSpan'd) costs and constraints -- the dense `fullSizeEntry_` branches of the reference
    (src/costFunctions.cpp:65-71,141-146,197-203; src/constraints.cpp:68-73,122-126,199-204,297-299,346-351) --
    evaluated by the DMMA GEMM path, mixed with step-size entries, against the oracle"""
    nx, nu, N = 2, 1, 9
    rng = np.random.default_rng(5)
    A = np.array([[1.0, 0.1], [0.0, 1.0]])
    B = np.array([[0.005], [1.0]])
    probs = []
    for b in range(3):
        M, Nm = np.eye(2), np.eye(1)
        w_t = rng.uniform(0.5, 2.0, 2 * (N + 1))
        prob = dict(nx=nx, nu=nu, N=N, initial_state=initial_state, A=A, B=B, d=np.array([0.01, -0.02]), x0=np.array([0.3, -1.0]) + 0.1 * b,
                    costs=[dict(kind="trajectory", M=_span_m(M, N + 1), p=np.tile([0.1, 0.2], N + 1) + 0.01 * b, w=w_t),
                           dict(kind="target", M=np.eye(2), p=np.ones(2), w=np.array([2.0, 3.0])),
                           dict(kind="control", N=_span_m(Nm, N), p=np.full(N, 0.4), w=np.full(N, 0.1)),
                           dict(kind="mixed", M=_span_m(np.ones((1, 2)), N, 1), N=_span_m(np.ones((1, 1)), N), p=np.full(N, 0.3), w=np.full(N, 0.3)),
                           dict(kind="mixed", M=np.ones((1, 2)), N=np.ones((1, 1)), p=np.array([0.1]), w=np.array([0.2]))],
                    constraints=[dict(kind="trajectory", E=_span_m(np.eye(2), N + 1), f=np.tile([50.0, 40.0], N + 1)),
                                 dict(kind="control", G=_span_m(np.eye(1), N), f=np.full(N, 20.0)),
                                 dict(kind="mixed", E=_span_m(np.array([[0.0, 1.0]]), N, 1), G=_span_m(np.array([[1.0]]), N), f=np.full(N, -0.5), is_ineq=False),
                                 dict(kind="mixed", E=np.ones((1, 2)), G=np.ones((1, 1)), f=np.array([60.0])),
                                 dict(kind="trajectory_bound", lower=np.full(nx * (N + 1), -np.inf), upper=np.tile([2.0, 1.0], N + 1)),
                                 dict(kind="control_bound", lower=np.full(N, -1.0), upper=np.full(N, 1.5))])
        if initial_state:
            prob.update(R=np.array([[2.0, 0.1], [0.1, 1.0]]), r=np.array([0.1, -0.2]), x0lb=prob["x0"] - np.array([0.1, 0.5]),
                        x0ub=prob["x0"] + np.array([0.1, 0.5]))
        probs.append(prob)
    # batch them (every array gets a leading batch axis)
    def stack(key, sub=None, idx=None):
        return np.stack([(p[key] if sub is None else p[sub][idx][key]) for p in probs])
    bp = dict(name="full-size", nx=nx, nu=nu, N=N, batch=3, initial_state=initial_state, A=A, B=B, d=probs[0]["d"], x0=stack("x0"),
              costs=[dict(c, p=stack("p", "costs", i), w=stack("w", "costs", i)) for i, c in enumerate(probs[0]["costs"])],
              constraints=probs[0]["constraints"])
    if initial_state:
        bp.update(R=probs[0]["R"], r=probs[0]["r"], x0lb=stack("x0lb"), x0ub=stack("x0ub"))
    hb = capi.HostBatch(bp)
    out = engine.lmpc_run(hb)
    stages = {k: engine.download(hb, k) for k in STAGES}
    for i, prob in enumerate(probs):
        o = po.lmpc(prob)
        for k in STAGES:
            assert rel_err(stages[k][i], o[k]) <= 1e-10, (k, i, rel_err(stages[k][i], o[k]))
        assert out["status"][i] == o["fail"] == 0
        assert x_err(out["x"][i], o["x"]) <= 1e-6
        assert active_set(out["iact"][i], out["nact"][i]) == active_set(o["iact"])


def test_batch_larger_than_grid_limit_is_chunked(engine):
    """batches > 65535 instances are processed in chunks by copra_b200_lmpc_run; results equal the small-batch ones"""
    base = wl.c2(batch=8, N=6)
    reps = 8200  # 65600 instances
    big = dict(base, batch=8 * reps)
    for k in ("A", "B", "d", "x0"):
        big[k] = np.tile(base[k], (reps,) + (1,) * (np.asarray(base[k]).ndim - 1))
    big["costs"] = [dict(c, p=np.tile(c["p"], (reps, 1)) if np.asarray(c["p"]).ndim == 2 else c["p"]) for c in base["costs"]]
    big["constraints"] = [dict(c, upper=np.tile(c["upper"], (reps, 1)) if np.asarray(c["upper"]).ndim == 2 else c["upper"])
                          for c in base["constraints"]]
    small = engine.lmpc_run(base)
    out = engine.lmpc_run(big, want=("control", "status", "nact"))
    assert (out["status"] == 0).all()
    assert np.array_equal(out["control"].reshape(reps, 8, -1), np.broadcast_to(small["control"], (reps,) + small["control"].shape))


def test_receding_horizon_resolve(engine):
    """SURVEY 8f N1: new x0 on a resident build (K4 + K5..K7 only) equals a full run with that x0, bit for bit"""
    bp = wl.c2(batch=64)
    first = engine.lmpc_run(bp)
    x0_new = np.array(bp["x0"]) + np.array([0.0, 0.3])
    again = engine.lmpc_resolve(x0_new, first["sizes"])
    full = engine.lmpc_run(dict(bp, x0=x0_new))
    assert (again["status"] == 0).all()
    assert np.array_equal(again["control"], full["control"]) and np.array_equal(again["iact"], full["iact"])
    assert np.array_equal(again["trajectory"], full["trajectory"])
    assert not np.array_equal(again["control"], first["control"])


def test_small_solver_residency_variants():
    """gi_small_kernel keeps S and the general rows in shared memory or in global memory (L2) depending on how many
    instances fit an SM; every variant runs the same algorithm (same pivots, same active sets; the compiler may
    contract a*b+c*d differently per instantiation, so x agrees to rounding, not bit for bit)"""
    rng = np.random.default_rng(11)
    cases = []
    for n, meq, m in ((7, 2, 9), (24, 3, 31), (51, 5, 60), (64, 0, 33)):
        B = 6
        L = rng.normal(size=(B, n, n))
        Q = L @ np.swapaxes(L, 1, 2) + 0.1 * np.eye(n)
        c = rng.normal(size=(B, n))
        Aeq = rng.normal(size=(B, meq, n))
        xf = rng.normal(size=(B, n))
        beq = np.einsum("bij,bj->bi", Aeq, xf)
        Aineq = rng.normal(size=(B, m, n))
        bineq = np.einsum("bij,bj->bi", Aineq, xf) + rng.uniform(0.0, 1.0, size=(B, m))
        lb = xf - rng.uniform(0.1, 2.0, size=(B, n))
        ub = xf + rng.uniform(0.1, 2.0, size=(B, n))
        cases.append((Q, c, Aeq if meq else None, beq if meq else None, Aineq, bineq, lb, ub))
    bp = wl.c2(batch=48)
    ref = None
    for v in range(3):
        eng = capi.Engine(0, small_variant=v + 1)
        try:
            out = [eng.solve_qp_batch(*cs) for cs in cases]
            mpc = eng.lmpc_run(bp)
        finally:
            eng.close()
        if ref is None:
            ref = (out, mpc)
            for cs, r in zip(cases, out):  # variant 0 against the oracle
                for b in range(cs[0].shape[0]):
                    o = po.quadprog(cs[0][b], cs[1][b], None if cs[2] is None else cs[2][b], None if cs[3] is None else cs[3][b],
                                    cs[4][b], cs[5][b], cs[6][b], cs[7][b])
                    assert r["status"][b] == o["fail"]
                    if o["fail"] == 0:
                        assert x_err(r["x"][b], o["x"]) < 1e-8
                        assert tuple(r["iters"][b]) == o["iter"]
            continue
        for r0, r1 in zip(ref[0], out):
            assert np.array_equal(r0["status"], r1["status"]) and np.array_equal(r0["iact"], r1["iact"])
            assert np.array_equal(r0["iters"], r1["iters"])
            assert np.allclose(r0["x"], r1["x"], rtol=1e-10, atol=1e-12)
        assert np.allclose(ref[1]["control"], mpc["control"], rtol=1e-9, atol=1e-9) and np.array_equal(ref[1]["iact"], mpc["iact"])


@pytest.mark.parametrize("n,meq,m", [(65, 4, 40), (100, 0, 120), (131, 7, 90), (160, 3, 64), (203, 5, 150)])
def test_mid_size_qps_general_and_cluster_kernels(engine, n, meq, m):
    """64 < n: the general kernel (J in shared memory up to ~160 variables; blocked DMMA factorisation, gi_factor.cuh)
    and, past one SM's shared memory, the cluster kernel -- random QPs with equalities, rows and bounds vs the oracle"""
    rng = np.random.default_rng(1000 + n)
    B = 3
    L = rng.normal(size=(B, n, n))
    Q = L @ np.swapaxes(L, 1, 2) / n + 0.5 * np.eye(n)
    c = rng.normal(size=(B, n))
    Aeq = rng.normal(size=(B, meq, n))
    xf = rng.normal(size=(B, n))
    beq = np.einsum("bij,bj->bi", Aeq, xf)
    Aineq = rng.normal(size=(B, m, n))
    bineq = np.einsum("bij,bj->bi", Aineq, xf) + rng.uniform(0.0, 1.0, size=(B, m))
    lb = xf - rng.uniform(0.1, 2.0, size=(B, n))
    ub = xf + rng.uniform(0.1, 2.0, size=(B, n))
    r = engine.solve_qp_batch(Q, c, Aeq if meq else None, beq if meq else None, Aineq, bineq, lb, ub)
    for b in range(B):
        o = po.quadprog(Q[b], c[b], Aeq[b] if meq else None, beq[b] if meq else None, Aineq[b], bineq[b], lb[b], ub[b])
        assert r["status"][b] == o["fail"] == 0
        assert x_err(r["x"][b], o["x"]) < 1e-7, x_err(r["x"][b], o["x"])
        assert active_set(r["iact"][b], r["nact"][b]) == active_set(o["iact"])
        assert tuple(r["iters"][b]) == o["iter"]
