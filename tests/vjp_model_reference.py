"""TEST INFRASTRUCTURE -- a dense numpy reference for the gradients of one LMPC instance with respect to its dynamics A, B, d
and its row constraints' E and G (copra_b200_lmpc_vjp_model).

Write every active row j in its natural orientation a_j' U = beta_j; a general row is (E x_i + G u_i - f)_l = 0 at its
(step i, line l), x_i = Phi_i x0 + Psi_i U + xi_i.  Differentiating the KKT system QU + c + A_act' lambda = 0, A_act U = beta
with the adjoint (c^ = -v, mu) of tests/vjp_reference gives
    dL/dtheta = c^' (dQ U + dc) + sum_j [lambda_j c^' da_j - mu_j d(a_j' U - beta_j)] + dtraj' dx|_U,
the partial derivative, at fixed U, c^, lambda and mu, of
    Phi = sum_costs sum_i e_i' W t_i + dtraj' x + sum_j [lambda_j (E x^_i + G c^_i)_l - mu_j (E x_i + G u_i - f)_l],
x^ = Psi c^.  With gx_i = dtraj_i + sum_costs M'W t_i - sum_j mu_j E_l', gh_i = sum_costs M'W e_i + sum_j lambda_j E_l',
rho_N = gx_N, rho_i = gx_i + A' rho_{i+1} (rho^ the same from gh):
    dA = sum_{i<N} rho_{i+1} x_i' + rho^_{i+1} x^_i',  dB = sum_{i<N} rho_{i+1} u_i' + rho^_{i+1} c^_i',  dd = sum_{i<N} rho_{i+1},
    dE_l = sum_i lambda_(i,l) x^_i' - mu_(i,l) x_i',  dG_l = sum_i lambda_(i,l) c^_i' - mu_(i,l) u_i',
and rho_0 = dL/dx0.  lambda comes from a dense KKT solve on the oracle's active set.  A trajectory bound's rows are line
selectors (quirk Q1: the lower rows read x <= lower): they enter gx / gh through their multipliers and have no E gradient.
`closed_form` evaluates the above; `directional` evaluates the first line with dQ, dc, da and dbeta central differences of the
oracle's own builds.
"""
import copy

import numpy as np

from copra_b200 import workloads as wl
from tests import vjp_cost_reference as cr
from tests import vjp_reference as vr

SYSTEM = ("A", "B", "d")


def model_keys(inst):
    """("A", 0), ("B", 0), ("d", 0) and ("E", j) / ("G", j) of every row constraint that has them"""
    keys = [(k, 0) for k in SYSTEM]
    for j, c in enumerate(inst["constraints"]):
        keys += [(k, j) for k in ("E", "G") if k in _HAS.get(c["kind"], ())]
    return keys


_HAS = dict(trajectory=("E",), control=("G",), mixed=("E", "G"))


def get_matrix(inst, key):
    kind, j = key
    src = inst if kind in SYSTEM else inst["constraints"][j]
    a = np.asarray(src[kind], float)
    return a if kind == "d" else np.atleast_2d(a)


def with_matrices(inst, mats):
    """copy of `inst` with the entries of `mats` ({("A" | "B" | "d", 0) | ("E" | "G", j): array}) replaced"""
    out = copy.copy(inst)
    out["constraints"] = [dict(c) for c in inst["constraints"]]
    for (kind, j), v in mats.items():
        if kind in SYSTEM:
            out[kind] = v
        else:
            out["constraints"][j][kind] = v
    return out


def general_rows(inst):
    """the general rows [eq | ineq] in the solver's order: lists of (constraint, step, line, E_l or None, G_l or None)"""
    nx, N = inst["nx"], inst["N"]
    eq, ineq = [], []
    for j, c in enumerate(inst["constraints"]):
        if c["kind"] == "control_bound":
            continue
        if c["kind"] == "trajectory_bound":  # up to two selector families: the finite lower lines, then the upper ones
            lo, up = np.asarray(c["lower"], float)[:nx], np.asarray(c["upper"], float)[:nx]
            for lines in ([l for l in range(nx) if lo[l] != -np.inf], [l for l in range(nx) if up[l] != np.inf]):
                for i in range(N + 1):
                    for l in lines:
                        ineq.append((j, i, l, np.eye(nx)[l], None))
            continue
        E = np.atleast_2d(np.asarray(c["E"], float)) if "E" in _HAS[c["kind"]] else None
        G = np.atleast_2d(np.asarray(c["G"], float)) if "G" in _HAS[c["kind"]] else None
        rows = (E if E is not None else G).shape[0]
        dst = ineq if c.get("is_ineq", True) else eq
        for i in range(N + 1 if c["kind"] == "trajectory" else N):
            for l in range(rows):
                dst.append((j, i, l, None if E is None else E[l], None if G is None else G[l]))
    return eq, ineq


def active_system(o):
    """A_act (natural orientation) and beta_act of a solved oracle instance, in iact order"""
    n = o["Q"].shape[0]
    meq, m = o["Aeq"].shape[0], o["Aineq"].shape[0]
    rows, beta = [], []
    for k in np.asarray(o["iact"], int) - 1:
        if k < meq:
            rows.append(o["Aeq"][k]), beta.append(o["beq"][k])
        elif k < meq + m:
            rows.append(o["Aineq"][k - meq]), beta.append(o["bineq"][k - meq])
        else:
            e = np.zeros(n)
            e[(k - meq - m) % n] = 1.0
            rows.append(e), beta.append(o["ub"][k - meq - m] if k - meq - m < n else o["lb"][k - meq - m - n])
    return np.array(rows).reshape(-1, n), np.array(beta)


def forward_multipliers(o):
    """lambda of the forward solve over [eq | ineq | ub | lb] (0 for inactive rows): [Q A'; A 0] [U; lambda] = [-c; beta]"""
    A, beta = active_system(o)
    n, na = o["Q"].shape[0], A.shape[0]
    K = np.block([[o["Q"], A.T], [A, np.zeros((na, na))]])
    sol = np.linalg.solve(K, np.concatenate([-o["c"], beta]))
    lam = np.zeros(o["Aeq"].shape[0] + o["Aineq"].shape[0] + 2 * n)
    lam[np.asarray(o["iact"], int) - 1] = sol[n:]
    return lam


def closed_form(inst, o, adj, dtraj):
    """({key: gradient}, rho_0) of a solved oracle instance `o` (LMPC mode) from its adjoint `adj` and dL/dtrajectory"""
    nx, nu, N = inst["nx"], inst["nu"], inst["N"]
    A = np.asarray(inst["A"], float)
    U = np.asarray(o["control"], float)
    ch = np.asarray(adj["c"], float)
    x = (o["Phi"] @ np.asarray(inst["x0"], float) + o["Psi"] @ U + o["xi"]).reshape(N + 1, nx)
    xh = (o["Psi"] @ ch).reshape(N + 1, nx)
    u, uh = U.reshape(N, nu), ch.reshape(N, nu)
    gx = (np.zeros(x.shape) if dtraj is None else np.asarray(dtraj, float).reshape(N + 1, nx)).copy()
    gh = np.zeros(x.shape)
    for c in inst["costs"]:
        if "M" not in cr.HAS[c["kind"]]:
            continue
        r, w = cr.rows_of(c), cr.weights(c)
        M = np.atleast_2d(np.asarray(c["M"], float))
        Nm = np.atleast_2d(np.asarray(c["N"], float)) if "N" in cr.HAS[c["kind"]] else None
        p = np.asarray(c["p"], float)
        for i in cr.STEPS[c["kind"]](N):
            pi = p[i * r:(i + 1) * r] if c.get("per_step") else p
            e, t = M @ x[i] - pi, M @ xh[i]
            if Nm is not None:
                e, t = e + Nm @ u[i], t + Nm @ uh[i]
            gx[i] += M.T @ (w * t)
            gh[i] += M.T @ (w * e)
    meq = o["Aeq"].shape[0]
    mu = np.concatenate([adj["beq"], adj["bineq"]])
    lam = forward_multipliers(o)
    eq, ineq = general_rows(inst)
    assert len(eq) == meq and len(ineq) == o["Aineq"].shape[0]
    grads = {k: np.zeros(get_matrix(inst, k).shape) for k in model_keys(inst)}
    Psi = o["Psi"]
    for idx, (j, i, l, E, G) in enumerate(eq + ineq):
        # the engine's row order is the oracle's: a_j = E Psi_i + G at block i
        a = np.zeros(Psi.shape[1]) if E is None else E @ Psi[i * nx:(i + 1) * nx]
        if G is not None:
            a[i * nu:(i + 1) * nu] += G
        assert np.allclose(a, o["Aeq"][idx] if idx < meq else o["Aineq"][idx - meq], rtol=1e-12, atol=1e-12)
        m, lm = mu[idx], lam[idx]
        if m == 0.0 and lm == 0.0:
            continue
        if E is not None:
            gx[i] -= m * E
            gh[i] += lm * E
            if ("E", j) in grads:
                grads[("E", j)][l] += lm * xh[i] - m * x[i]
        if G is not None:
            grads[("G", j)][l] += lm * uh[i] - m * u[i]
    rho, rhoh = gx.copy(), gh.copy()
    for i in range(N - 1, -1, -1):
        rho[i] += A.T @ rho[i + 1]
        rhoh[i] += A.T @ rhoh[i + 1]
    grads[("A", 0)] = sum(np.outer(rho[i + 1], x[i]) + np.outer(rhoh[i + 1], xh[i]) for i in range(N))
    grads[("B", 0)] = sum(np.outer(rho[i + 1], u[i]) + np.outer(rhoh[i + 1], uh[i]) for i in range(N))
    grads[("d", 0)] = rho[1:].sum(axis=0)
    return grads, rho[0]


def directional(inst, o, adj, dtraj, delta, h):
    """c^' (dQ U + dc) + sum_j [lambda_j c^' da_j - mu_j (da_j' U - dbeta_j)] + dtraj' (dPhi x0 + dPsi U + dxi) along `delta`
    ({key: array}), with every d. a central difference (step h) of the oracle's builds: exact for d, E and G (the builds are
    affine in each), O(h^2) for A and B"""
    ends = [vr.build(with_matrices(inst, {k: get_matrix(inst, k) + s * h * d for k, d in delta.items()})) for s in (1.0, -1.0)]
    diff = {k: (ends[0][k] - ends[1][k]) / (2.0 * h) for k in ("Q", "c", "Aeq", "beq", "Aineq", "bineq", "Phi", "Psi", "xi")}
    U = np.asarray(o["control"], float)
    ch = np.asarray(adj["c"], float)
    val = float(ch @ (diff["Q"] @ U + diff["c"]))
    if dtraj is not None:
        val += float(np.asarray(dtraj, float) @ (diff["Phi"] @ np.asarray(inst["x0"], float) + diff["Psi"] @ U + diff["xi"]))
    meq = o["Aeq"].shape[0]
    lam = forward_multipliers(o)
    mu = np.concatenate([adj["beq"], adj["bineq"]])
    da = np.vstack([diff["Aeq"].reshape(-1, U.shape[0]), diff["Aineq"].reshape(-1, U.shape[0])])
    db = np.concatenate([diff["beq"], diff["bineq"]])
    for k in np.asarray(o["iact"], int) - 1:
        if k < meq + o["Aineq"].shape[0]:
            val += lam[k] * float(ch @ da[k]) - mu[k] * (float(da[k] @ U) - db[k])
    return val


def dot(grads, delta):
    return float(sum(np.sum(grads[k] * d) for k, d in delta.items()))


def random_direction(inst, rng, keys):
    return {k: rng.normal(size=get_matrix(inst, k).shape) for k in keys}


def c3_g(batch, N=60):
    """C3 (a shorter horizon) whose ZMP MixedConstraint has a non-zero G: each line also bounds a small multiple of the jerk
    along its axis, so that both E and G of the active rows carry gradients"""
    bp = wl.c3(batch=batch, N=N)
    bp["name"] = "C3-G"
    c = bp["constraints"][0]
    G = np.zeros((4, 2))
    G[0, 0], G[1, 0], G[2, 1], G[3, 1] = 1e-4, -1e-4, 2e-4, -2e-4
    bp["constraints"] = [dict(c, G=G)]
    return bp


def c2_two_inputs(batch, N=50):
    """C2 with a second actuator (B' = [B, B]) and two more constraints: a CONTROL equality u1 - u2 = 0 at every step and a
    CONTROL inequality u1 <= 0.3 uUpper, active while the system brakes its fall"""
    bp = wl.c2(batch=batch, N=N)
    bp["name"] = "C2-two-inputs"
    bp["nu"] = 2
    bp["B"] = np.concatenate([bp["B"], bp["B"]], axis=-1)
    tb, cb = bp["constraints"]
    uup = np.asarray(cb["upper"])[:, 0]
    bp["costs"] = [bp["costs"][0], dict(kind="control", N=np.eye(2), p=np.array([2.0, 2.0]), w=np.array([1e-4, 1e-4]))]
    bp["constraints"] = [tb, dict(kind="control_bound", lower=np.full(2, -np.inf), upper=np.stack([uup, uup], axis=1)),
                         dict(kind="control", G=np.array([[1.0, -1.0]]), f=np.zeros(1), is_ineq=False),
                         dict(kind="control", G=np.array([[1.0, 0.0]]), f=(0.3 * uup)[:, None])]
    return bp


def c5_tight(batch, N=60):
    """C5 on a shorter horizon with its TrajectoryConstraint |position| <= 0.51 (was 0.6): every x0 satisfies it, and the
    instances whose reference lies beyond it reach it within the horizon"""
    bp = wl.c5(batch=batch, N=N)
    bp["name"] = "C5-tight"
    bp["constraints"] = [dict(bp["constraints"][0], f=np.full(8, 0.51)), bp["constraints"][1]]
    return bp
