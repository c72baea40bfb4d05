"""Which kernel variant each build launcher picks for a problem, restated in Python, and a table of problems that reaches
every variant and both sides of every size threshold.

`build_dispatch` mirrors the launchers of copra_b200/csrc/k1_k7_lmpc.cu (line numbers cited per formula) and the
Hessian-sharing rule of copra_b200/csrc/capi.cu.  `SHAPES` pairs are found by searching with the mirror (`edge`), so a
threshold that moves in the launcher but not here shows up as a profiler-test failure on the GPU, and a table that no
longer straddles a threshold shows up in the CPU test."""
import numpy as np

from copra_b200 import workloads as wl

SMS = 148                # B200 multiprocessors
SMEM_OPTIN = 232448      # B200 cudaDevAttrMaxSharedMemoryPerBlockOptin (227 KB)
GRID_STRIDE = SMS * 8    # grid of the per-instance grid-stride kernels (K1 one CTA per instance, K2a, K4)
DBL_MAX = np.finfo(float).max

LABELS = dict(k1=("g8", "g16", "g32", "cta", "cta_strided"), q=("tiled", "staged", "unstaged"), ef=("staged", "unstaged"),
              k7=("staged", "unstaged"), schur=("none", "small", "smem", "ws"))
# (launcher, label below the threshold, label above it)
THRESHOLDS = (("k1", "g8", "g16"), ("k1", "g16", "g32"), ("k1", "g32", "cta"), ("k1", "cta", "cta_strided"),
              ("q", "tiled", "staged"), ("q", "staged", "unstaged"), ("ef", "staged", "unstaged"), ("k7", "staged", "unstaged"),
              ("schur", "small", "smem"), ("schur", "smem", "ws"))
KERNELS = dict(k1=dict(g8="k1_condense_group_kernel", g16="k1_condense_group_kernel", g32="k1_condense_group_kernel",
                       cta="k1_condense_kernel", cta_strided="k1_condense_kernel"),
               q=dict(tiled="k2_assemble_q_tiled_kernel", staged="k2_assemble_q_kernel", unstaged="k2_assemble_q_kernel"),
               ef=dict(staged="k2_assemble_ef_kernel<true>", unstaged="k2_assemble_ef_kernel<false>"),
               k7=dict(staged="k7_results_kernel<true>", unstaged="k7_results_kernel<false>"),
               schur=dict(none=None, small="k4_schur_small_kernel", smem="k4_schur_kernel", ws="k4_schur_kernel"))

_SPAN = {"trajectory": lambda N: (0, N + 1), "target": lambda N: (N, N + 1), "control": lambda N: (0, N),
         "mixed": lambda N: (0, N)}  # capi.cu:316-319


def _batched(key, a):
    return wl.is_batched(key, a)


def _cost_tables(bp):
    """per step-size cost: (sMGx, sMPhi, sres, rows) as capi.cu:890 sizes them; full-size costs take the GEMM path"""
    nx, nu, N = bp["nx"], bp["nu"], bp["N"]
    out = []
    for c in bp["costs"]:
        mat = c.get("M") if c.get("M") is not None else c.get("N")
        mat = np.asarray(mat)
        if mat.shape[-1] != (nx if c.get("M") is not None else nu):
            continue  # full_size == 1: dense (capi.cu:271-274, k1_k7_lmpc.cu:943)
        rows = mat.shape[-2] if mat.ndim >= 2 else 1
        i0, i1 = _SPAN[c["kind"]](N)
        out.append((rows * nu * (N + 1), rows * nx * (i1 - i0), rows * (i1 - i0), rows))
    return out


def hessian_shared(bp):
    """capi.cu:780-784: one Hessian for the batch when A, B and every cost's M, N, w are shared (LMPC mode, batch > 1)"""
    if bp.get("initial_state") or bp["batch"] <= 1 or _batched("A", bp["A"]) or _batched("B", bp["B"]):
        return False
    for c in bp["costs"]:
        if any(c.get(k) is not None and _batched(k, c[k]) for k in ("M", "N", "w")):
            return False
        if c.get("M") is not None and np.asarray(c["M"]).shape[-1] != bp["nx"]:
            return False
    return True


def build_dispatch(bp, sms=SMS, smem_optin=SMEM_OPTIN):
    """labels of the variants the build launchers pick for batch problem `bp`:
    dict(k1=, q=, ef=, k7=, schur=, shared=)"""
    nx, nu, N = bp["nx"], bp["nu"], bp["N"]
    initial = bool(bp.get("initial_state"))
    nU = nu * N
    nvar = nU + (nx if initial else 0)
    out = {}
    # k1_condense_launch, k1_k7_lmpc.cu:170-180: group width G = 8/16/32 up to per = 32, else one CTA of
    # min(256, per rounded up to a warp) threads, which loops over the entries when per > 256
    per = nx * nx + nx * nu + nx
    if per <= 8:
        out["k1"] = "g8"
    elif per <= 16:
        out["k1"] = "g16"
    elif per <= 32:
        out["k1"] = "g32"
    else:
        out["k1"] = "cta" if min(256, -(-per // 32) * 32) >= per else "cta_strided"
    tabs = _cost_tables(bp)
    # k2k4_assemble_launch, k1_k7_lmpc.cu:942-947: staged when every step-size cost's M A^k B table and weights fit
    # 40 KB, tiled when the nU x nU tile fits next to them in 44 KB
    need = sum(mgx + rows for mgx, _, _, rows in tabs)
    staged = need * 8 <= 40 * 1024
    tiled = staged and (need + nU * nU) * 8 <= 44 * 1024
    out["q"] = "tiled" if tiled else ("staged" if staged else "unstaged")
    # ef_launch, k1_k7_lmpc.cu:911-916: the largest single cost's tables and weights against 40 KB
    if tabs:
        need_ef = max(mgx + mphi + res + rows for mgx, mphi, res, rows in tabs)
        out["ef"] = "staged" if need_ef * 8 <= 40 * 1024 else "unstaged"
    # k7_results_launch, k1_k7_lmpc.cu:1063-1064: the solution and the compact Psi column block against 40 KB
    out["k7"] = "staged" if 8 * (nvar + N * nx * nu) <= 40 * 1024 else "unstaged"
    # K4' Schur block, k1_k7_lmpc.cu:1002 (kSmMaxN = 64, gi_small.cuh:24) and :1012-1015 (odd_ld = n | 1, engine.cuh:20)
    if not initial:
        out["schur"] = "none"
    elif nU <= 64:
        out["schur"] = "small"
    else:
        base = 8 * (2 * nU + 1 + nx * nU)
        with_j = base + 8 * (nU | 1) * nU
        out["schur"] = "smem" if with_j + 1024 <= smem_optin else "ws"
    out["shared"] = hessian_shared(bp)
    return out


def edge(make, key, lo, hi=400):
    """smallest v >= lo whose problem make(v) gets a different `key` label from make(v + 1)"""
    prev = build_dispatch(make(lo))[key]
    for v in range(lo, hi):
        nxt = build_dispatch(make(v + 1))[key]
        if nxt != prev:
            return v
        prev = nxt
    raise ValueError("no %s threshold in [%d, %d]" % (key, lo, hi))


def group_batch(nx, nu):
    """a batch whose last K1 group CTA is ragged (a few instances short of 128 / G) and spans mixed warps"""
    per = nx * nx + nx * nu + nx
    if per > 32:
        return 5
    G = 8 if per <= 8 else (16 if per <= 16 else 32)
    return 2 * (128 // G) + 3


# ---- problem builders ---------------------------------------------------------------------------------------------------
def every_kind(nx, nu, N, batch, shared=True, initial_state=False, seed=0):
    """every step-size cost kind (multi-row M only, nx-row target, N only, single-row M and N) and every constraint kind (E only,
    G only, an equality and an inequality with both, a trajectory bound on a subset of lines, a control bound with +-inf and
    +-DBL_MAX entries).  `shared`: A, B, d, M, N, w without a batch axis (a batch-invariant Hessian in LMPC mode)."""
    rng = np.random.default_rng(seed + 1000 * nx + nu)
    A = np.eye(nx) + 0.05 * np.eye(nx, k=1) + 0.01 * rng.normal(size=(nx, nx))
    B = 0.1 * rng.normal(size=(nx, nu)) + 0.2 * np.eye(nx, nu)
    d = 0.01 * rng.normal(size=nx)
    if not shared:
        A = A + 1e-3 * rng.normal(size=(batch, nx, nx))
        B = B * (1.0 + 0.1 * rng.uniform(size=(batch, 1, 1)))
        d = d + 1e-3 * rng.normal(size=(batch, nx))
    x0 = 0.5 * rng.normal(size=(batch, nx))
    w_ctl = np.full(nu, 0.1) if shared else 0.1 + 0.05 * rng.uniform(size=(batch, nu))
    costs = [dict(kind="trajectory", M=rng.normal(size=(2, nx)), p=0.3 * rng.normal(size=(batch, 2)), w=np.array([1.5, 0.7])),
             dict(kind="target", M=np.eye(nx), p=rng.normal(size=(batch, nx)), w=np.full(nx, 2.0)),
             dict(kind="control", N=np.eye(nu), p=0.1 * np.ones(nu), w=w_ctl),
             dict(kind="mixed", M=0.5 * np.ones((1, nx)), N=np.eye(1, nu), p=np.array([0.2]), w=np.array([0.3])),
             dict(kind="mixed", M=0.2 * rng.normal(size=(2, nx)), N=np.eye(2, nu), p=np.array([0.1, -0.1]), w=np.array([0.4, 0.2]))]
    j = np.arange(nu)
    lo_u = np.where(j % 2 == 0, -np.inf, -50.0)
    lo_u[j % 3 == 2] = -DBL_MAX
    up_u = np.where(j % 2 == 0, 50.0, DBL_MAX)
    lines = np.arange(nx)
    lo_x = np.where(lines == 0, 1e3, -np.inf)   # quirk Q1: a finite lower bound of a trajectory bound reads x <= lower
    up_x = np.where(lines == nx - 1, 1e3, np.inf)
    constraints = [dict(kind="trajectory", E=rng.normal(size=(2, nx)), f=np.full(2, 50.0)),
                   dict(kind="control", G=np.ones((1, nu)), f=np.array([40.0])),
                   dict(kind="mixed", E=0.01 * np.ones((1, nx)), G=np.eye(1, nu), f=0.1 + 0.01 * rng.normal(size=(batch, 1)),
                        is_ineq=False),
                   dict(kind="mixed", E=rng.normal(size=(1, nx)), G=np.ones((1, nu)), f=np.array([30.0])),
                   dict(kind="trajectory_bound", lower=lo_x, upper=up_x),
                   dict(kind="control_bound", lower=lo_u, upper=up_u)]
    bp = dict(name="every-kind nx=%d nu=%d N=%d" % (nx, nu, N), nx=nx, nu=nu, N=N, batch=batch, initial_state=initial_state,
              A=A, B=B, d=d, x0=x0, costs=costs, constraints=constraints)
    if initial_state:
        bp.update(R=2.0 * np.eye(nx) + 0.1, r=0.1 * rng.normal(size=nx), x0lb=x0 - 0.1, x0ub=x0 + 0.1)
    return bp


def c2_like(N, batch=37, shared=False):
    """C2's double integrator (nx = 2, nu = 1; target and control costs, a trajectory bound on one line, a control bound);
    `shared`: every instance has instance 0's mass, so the Hessian is batch-invariant"""
    bp = wl.c2(batch=batch, N=N)
    if shared:
        bp.update(A=bp["A"][0], B=bp["B"][0], d=bp["d"][0])
    bp["name"] = "C2 N=%d%s" % (N, " shared" if shared else "")
    return bp


def c5_like(N, batch=4, shared=False):
    """C5's coupled triple integrators (nx = 12, nu = 4; a 12-row trajectory cost, a 4-row control cost, an 8-row trajectory
    constraint, a control bound); `shared`: instance 0's model and weights for every instance"""
    bp = wl.c5(batch=batch, N=N)
    if shared:
        bp.update(A=bp["A"][0], B=bp["B"][0], d=bp["d"][0])
        bp["costs"] = [dict(bp["costs"][0], w=bp["costs"][0]["w"][0])] + bp["costs"][1:]
    bp["name"] = "C5 N=%d%s" % (N, " shared" if shared else "")
    return bp


def c4_like(N, batch=5):
    """C4: InitialStateLMPC on C2's system (nx = 2, nu = 1)"""
    bp = wl.c4(batch=batch, N=N)
    bp["name"] = "C4 N=%d" % N
    return bp


class Shape:
    """one problem of the table: `make()` builds it, `expect` holds the labels it is meant to hit, and `across` names the
    threshold (launcher, below, above) it straddles together with its partner"""

    def __init__(self, name, make, expect, across=None):
        self.name, self.make, self.expect, self.across = name, make, expect, across

    def __repr__(self):
        return self.name


def _pair(name, make, key, lo, expect_lo, expect_hi, extra=None):
    """the two shapes on each side of the first `key` threshold at or above lo: make(v) and make(v + 1)"""
    v = edge(make, key, lo)
    across = (key, expect_lo, expect_hi)
    e = dict(extra or {})
    return [Shape("%s-%s-%d" % (name, expect_lo, v), lambda v=v: make(v), dict(e, **{key: expect_lo}), across),
            Shape("%s-%s-%d" % (name, expect_hi, v + 1), lambda v=v: make(v + 1), dict(e, **{key: expect_hi}), across)]


def _k1(nx, shared, initial_state=False, N=4):
    return lambda nu: every_kind(nx, nu, N, group_batch(nx, nu), shared=shared, initial_state=initial_state)


SHAPES = (
    # K1: group widths and the CTA kernels, one step of nu on each side (every kind of cost and constraint)
    _pair("k1 nx=2", _k1(2, True), "k1", 1, "g8", "g16")
    + _pair("k1 nx=1", _k1(1, False), "k1", 7, "g16", "g32")
    + _pair("k1 nx=1", _k1(1, True), "k1", 15, "g32", "cta")
    + _pair("k1 nx=15", _k1(15, False, N=3), "k1", 1, "cta", "cta_strided")
    + [Shape("k1 nx=2 nu=5 initial-state", lambda: every_kind(2, 5, 6, group_batch(2, 5), shared=True, initial_state=True),
             dict(k1="g16", schur="small")),
       Shape("k1 nx=4 nu=3 N=1", lambda: every_kind(4, 3, 1, group_batch(4, 3), shared=False), dict(k1="g32")),
       Shape("N=1 shared", lambda: every_kind(2, 1, 1, group_batch(2, 1), shared=True), dict(k1="g8", q="tiled", shared=True)),
       Shape("N=1 initial-state", lambda: every_kind(2, 1, 1, 3, initial_state=True), dict(k1="g8", schur="small"))]
    # Q assembly: tiled | staged (C2, 44 KB) and staged | unstaged (C5, 40 KB), each shared and per instance
    + _pair("q C2", lambda N: c2_like(N), "q", 2, "tiled", "staged", dict(shared=False))
    + _pair("q C2 shared", lambda N: c2_like(N, shared=True), "q", 2, "tiled", "staged", dict(shared=True))
    + _pair("q C5", lambda N: c5_like(N), "q", 17, "staged", "unstaged", dict(shared=False))
    + _pair("q C5 shared", lambda N: c5_like(N, shared=True), "q", 17, "staged", "unstaged", dict(shared=True))
    # K2c: the largest single cost's tables against 40 KB (C5's 12-row trajectory cost)
    + _pair("ef C5", lambda N: c5_like(N), "ef", 2, "staged", "unstaged", dict(shared=False))
    + _pair("ef C5 shared", lambda N: c5_like(N, shared=True), "ef", 2, "staged", "unstaged", dict(shared=True))
    # K7: x and the compact Psi column block against 40 KB (nu > 1; C2 / C4 shapes above cover nu == 1)
    + _pair("k7 C5", lambda N: c5_like(N), "k7", 2, "staged", "unstaged")
    # K4' Schur block: small kernel | J in shared memory | J in the global workspace
    + _pair("schur C4", lambda N: c4_like(N), "schur", 2, "small", "smem")
    + _pair("schur C4", lambda N: c4_like(N), "schur", 66, "smem", "ws")
    # second and third trips of the grid-stride loops (K1 one CTA per instance, K2a, K4, K4' small)
    + [Shape("grid-stride nx=5", lambda: every_kind(5, 1, 3, 2 * GRID_STRIDE + 3, shared=False), dict(k1="cta")),
       Shape("grid-stride initial-state", lambda: c4_like(3, batch=2 * GRID_STRIDE + 3), dict(k1="g8", schur="small"))]
)


def sample(bp):
    """instances compared with the oracle: the first, the last, the first of the last (ragged) K1 group CTA, and those on each
    side of every grid-stride boundary"""
    B = bp["batch"]
    nx, nu = bp["nx"], bp["nu"]
    idx = set(range(B)) if B <= 5 else {0, B - 1}
    per = nx * nx + nx * nu + nx
    if per <= 32:
        ngrp = 128 // (8 if per <= 8 else (16 if per <= 16 else 32))
        idx.add((B - 1) // ngrp * ngrp)
    for k in range(GRID_STRIDE, B, GRID_STRIDE):
        idx.update((k - 1, k))
    return sorted(idx)
