"""TEST INFRASTRUCTURE -- a dense numpy reference for the gradients of one LMPC instance with respect to its cost weights and
matrices (copra_b200_lmpc_vjp_costs).

The cost inputs w, M and N enter the objective only, so with c^ = dL/dc (tests/vjp_reference.adjoint) and the solution U,
    dL/dtheta = c^' (dQ/dtheta U + dc/dtheta).
Per cost, over the steps i it covers, with e_i = M x_i + N u_i - p_i, x^ = Psi c^ and t_i = M x^_i + N c^_i:
    dL/dw_l = sum_i (t_i)_l (e_i)_l,   dL/dM = sum_i W (e_i x^_i' + t_i x_i'),   dL/dN = sum_i W (e_i c^_i' + t_i u_i').
`closed_form` evaluates these; `directional` evaluates c^' (dQ U + dc) with dQ and dc central differences of the oracle's own
builds, which are exact up to rounding because Q and c are at most quadratic in w, M and N.
"""
import copy

import numpy as np

from copra_b200 import workloads as wl
from tests import vjp_reference as vr

STEPS = dict(trajectory=lambda N: range(0, N + 1), target=lambda N: range(N, N + 1), control=lambda N: range(0, N),
             mixed=lambda N: range(0, N))
HAS = dict(trajectory=("M",), target=("M",), control=("N",), mixed=("M", "N"))


def cost_keys(inst):
    """("w", i), ("M", i), ("N", i) of every cost of the instance that has them"""
    keys = []
    for i, c in enumerate(inst["costs"]):
        keys += [("w", i)] + [(k, i) for k in HAS[c["kind"]]]
    return keys


def rows_of(cost):
    if cost.get("per_step"):
        return np.atleast_2d(np.asarray(cost["M"] if cost.get("M") is not None else cost["N"])).shape[0]
    return int(np.asarray(cost["p"]).shape[-1])


def weights(cost):
    r = rows_of(cost)
    w = np.ones(r) if cost.get("w") is None else np.atleast_1d(np.asarray(cost["w"], float))
    return np.tile(w, r // w.shape[0])


def get_matrix(inst, key):
    kind, i = key
    c = inst["costs"][i]
    if kind == "w":
        return weights(c)
    return np.atleast_2d(np.asarray(c[kind], float))


def with_matrices(inst, mats):
    """copy of `inst` with the cost entries of `mats` ({("w" | "M" | "N", i): array}) replaced"""
    out = copy.copy(inst)
    out["costs"] = [dict(c) for c in inst["costs"]]
    for (kind, i), v in mats.items():
        out["costs"][i][kind] = v
    return out


def closed_form(inst, o, adj):
    """{("w" | "M" | "N", i): gradient} of a solved oracle instance `o` (LMPC mode) from its adjoint `adj`"""
    nx, nu, N = inst["nx"], inst["nu"], inst["N"]
    U = np.asarray(o["control"], float)
    ch = np.asarray(adj["c"], float)
    x = o["Phi"] @ np.asarray(inst["x0"], float) + o["Psi"] @ U + o["xi"]
    xh = o["Psi"] @ ch
    out = {}
    for ci, c in enumerate(inst["costs"]):
        r = rows_of(c)
        w = weights(c)
        M = np.atleast_2d(np.asarray(c["M"], float)) if "M" in HAS[c["kind"]] else None
        Nm = np.atleast_2d(np.asarray(c["N"], float)) if "N" in HAS[c["kind"]] else None
        p = np.asarray(c["p"], float)
        gw, gM, gN = np.zeros(r), np.zeros((r, nx)), np.zeros((r, nu))
        for i in STEPS[c["kind"]](N):
            xi_, xhi = x[i * nx:(i + 1) * nx], xh[i * nx:(i + 1) * nx]
            ui, chi = (U[i * nu:(i + 1) * nu], ch[i * nu:(i + 1) * nu]) if i < N else (np.zeros(nu), np.zeros(nu))
            pi = p[i * r:(i + 1) * r] if c.get("per_step") else p
            e, t = -pi.copy(), np.zeros(r)
            if M is not None:
                e += M @ xi_
                t += M @ xhi
            if Nm is not None:
                e += Nm @ ui
                t += Nm @ chi
            gw += t * e
            gM += w[:, None] * (np.outer(e, xhi) + np.outer(t, xi_))
            gN += w[:, None] * (np.outer(e, chi) + np.outer(t, ui))
        out[("w", ci)] = gw
        if M is not None:
            out[("M", ci)] = gM
        if Nm is not None:
            out[("N", ci)] = gN
    return out


def directional(inst, o, adj, delta):
    """c^' (dQ U + dc) along `delta` ({key: array}) with dQ, dc central differences of the oracle's builds.  Any step is
    exact for a function at most quadratic; a step of the entries' own magnitude keeps the rounding of Q and c small."""
    h = 0.5 * max([1.0] + [float(np.abs(get_matrix(inst, k)).max()) for k in delta])
    ends = [vr.build(with_matrices(inst, {k: get_matrix(inst, k) + s * h * d for k, d in delta.items()})) for s in (1.0, -1.0)]
    dQ = (ends[0]["Q"] - ends[1]["Q"]) / (2.0 * h)
    dc = (ends[0]["c"] - ends[1]["c"]) / (2.0 * h)
    return float(adj["c"] @ (dQ @ np.asarray(o["control"], float) + dc))


def dot(grads, delta):
    return float(sum(np.sum(grads[k] * d) for k, d in delta.items()))


def random_direction(inst, rng, keys):
    return {k: rng.normal(size=get_matrix(inst, k).shape) for k in keys}


def mixed(batch, N=50):
    """C2 with a third cost, a MixedCost with both M and N (2 rows): e_i = M x_i + N u_i - p per step i < N"""
    bp = wl.c2(batch=batch, N=N)
    bp["name"] = "C2-mixed"
    bp["costs"] = bp["costs"] + [dict(kind="mixed", M=np.array([[0.5, 1.0], [0.0, 0.2]]), N=np.array([[0.05], [0.1]]),
                                      p=np.asarray(bp["x0"])[:, [1, 1]] * np.array([0.5, 0.1]), w=np.array([1.0, 0.5]))]
    return bp
