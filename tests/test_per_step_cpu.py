"""Per-step vectors (COPRA_B200_PER_STEP) without a GPU: how HostBatch packs them, the c3_walk workload, and the oracle on its
autoSpan'd full-size form."""
import numpy as np
import pytest

from copra_b200 import capi, workloads as wl
from oracle import pyoracle as po


def _tiny(N=4, batch=3):
    """every per-step kind on a double integrator (nx 2, nu 1)"""
    rng = np.random.default_rng(3)
    return dict(name="tiny", nx=2, nu=1, N=N, batch=batch, initial_state=False,
                A=np.array([[1.0, 0.1], [0.0, 1.0]]), B=np.array([[0.005], [0.1]]), d=np.zeros(2), x0=np.zeros((batch, 2)),
                costs=[dict(kind="trajectory", M=np.eye(2), p=rng.normal(size=(batch, 2 * (N + 1))), w=np.array([1.0, 2.0]),
                            per_step=True),
                       dict(kind="control", N=np.eye(1), p=np.arange(N, dtype=float), w=np.array([0.1]), per_step=True),
                       dict(kind="mixed", M=np.ones((1, 2)), N=np.ones((1, 1)), p=np.zeros(N), w=np.array([0.3]), per_step=True),
                       dict(kind="target", M=np.eye(2), p=np.ones(2), w=np.array([1.0, 1.0]))],
                constraints=[dict(kind="trajectory", E=np.eye(2), f=np.full(2 * (N + 1), 5.0), per_step=True),
                             dict(kind="mixed", E=np.ones((3, 2)), G=np.ones((3, 1)), f=np.full((batch, 3 * N), 4.0), per_step=True),
                             dict(kind="control", G=np.eye(1), f=np.full(N, 3.0), is_ineq=True, per_step=True),
                             dict(kind="trajectory_bound", lower=np.full(2 * (N + 1), -np.inf), upper=np.full(2 * (N + 1), 9.0),
                                  per_step=True),
                             dict(kind="control_bound", lower=np.full(N, -2.0), upper=np.full((batch, N), 2.0), per_step=True)])


def test_host_batch_packs_per_step_entries():
    N, B = 4, 3
    hb = capi.HostBatch(_tiny(N, B))
    c, k = hb.problem.costs, hb.problem.cstrs
    assert [c[i].full_size for i in range(4)] == [capi.PER_STEP] * 3 + [0]
    assert [c[i].rows for i in range(4)] == [2, 1, 1, 2]
    assert c[0].p.stride == 2 * (N + 1) and c[1].p.stride == 0  # batched / shared per-step vectors
    assert c[0].w.stride == 0
    assert [k[i].full_size for i in range(5)] == [capi.PER_STEP] * 5
    assert [k[i].rows for i in range(5)] == [2, 3, 1, 2, 1]
    assert k[1].f.stride == 3 * N and k[0].f.stride == 0
    assert k[4].upper.stride == N and k[4].lower.stride == 0
    # dicts without the key pack exactly as before
    plain = capi.HostBatch(wl.c3(batch=2))
    assert plain.problem.costs[0].full_size == 0 and plain.problem.costs[0].rows == 2
    assert plain.problem.cstrs[0].full_size == 0 and plain.problem.cstrs[0].rows == 4


@pytest.mark.parametrize("where,key,length", [("costs", 0, 9), ("costs", 1, 5), ("constraints", 0, 8), ("constraints", 1, 13),
                                              ("constraints", 3, 8), ("constraints", 4, 5)])
def test_host_batch_rejects_bad_per_step_lengths(where, key, length):
    bp = _tiny(4, 3)
    entry = dict(bp[where][key])
    vec = "p" if where == "costs" else ("lower" if entry["kind"].endswith("bound") else "f")
    entry[vec] = np.zeros(length)
    bp[where][key] = entry
    with pytest.raises(capi.CopraB200Error) as e:
        capi.HostBatch(bp)
    assert e.value.code == -1


def test_c3_walk_is_c3_plus_a_footstep_plan():
    a, b, base = wl.c3_walk(batch=64), wl.c3_walk(batch=64), wl.c3(batch=64)
    for k in ("A", "B", "d", "x0"):
        assert np.array_equal(a[k], base[k]) and np.array_equal(a[k], b[k])
    for x, y, z in zip(a["costs"] + a["constraints"], b["costs"] + b["constraints"], base["costs"] + base["constraints"]):
        for k, v in z.items():
            if k in ("p", "f"):
                continue
            assert np.array_equal(np.asarray(x[k]), np.asarray(v)) and np.array_equal(np.asarray(y[k]), np.asarray(v)), k
    assert np.array_equal(a["costs"][0]["p"], b["costs"][0]["p"])
    assert np.array_equal(a["constraints"][0]["f"], b["constraints"][0]["f"])
    assert not np.array_equal(a["constraints"][0]["f"], wl.c3_walk(batch=64, seed_offset=1)["constraints"][0]["f"])
    # the box is c3's at step 0 and moves later
    f = a["constraints"][0]["f"].reshape(64, 160, 4)
    assert np.array_equal(f[:, 0], base["constraints"][0]["f"])
    assert (np.abs(f[:, -1] - f[:, 0]).max(axis=1) > 0.1).all()
    # c3 itself does not depend on the walk
    assert np.array_equal(wl.c3(batch=64)["constraints"][0]["f"], base["constraints"][0]["f"])
    assert np.array_equal(wl.c3(batch=64)["costs"][0]["p"], base["costs"][0]["p"])


def test_oracle_solves_c3_walk_in_spanned_form():
    bp = wl.spanned(wl.c3_walk(batch=4))
    assert bp["constraints"][0]["E"].shape == (4, 4 * 160, 6 * 161)
    for i in range(4):
        o = po.lmpc(wl.instance(bp, i))
        assert o["fail"] == 0
        # ZMP inside each step's own box
        E, f = bp["constraints"][0]["E"][i], bp["constraints"][0]["f"][i]
        assert (E @ o["trajectory"] <= f + 1e-6).all()
