"""Synthetic LMPC workloads C1..C5 (BASELINE.json `configs[0..4]`, definitions in SURVEY.md 8d).

Deterministic: every random draw comes from SplitMix64 seeded with 0xC0B7A000 + 1000*config
(+ `seed_offset`), stepped once per draw, instance-major (SplitMix64 is a dozen lines in any host
language, so C++ callers can regenerate identical batches).

A *batch problem* is a dict:
    nx, nu, N, batch, initial_state,
    A (B,nx,nx) | (nx,nx)  B (B,nx,nu) | (nx,nu)  d (B,nx)|(nx,)  x0 (B,nx)|(nx,)
    costs       = [dict(kind, M, N, p, w)]          arrays carry a leading batch axis when they
    constraints = [dict(kind, E, G, f, lower, upper, is_ineq)]     differ per instance
    R, r, x0lb, x0ub (initial-state mode only)
A cost or constraint with `per_step=True` keeps step-size matrices and holds one vector per step (p, f, lower / upper
of rows x steps entries, step-major: COPRA_B200_PER_STEP); spanned() gives the same problem in copra's autoSpan'd
full-size form.
Matrices are in logical (rows, cols) shape; the C ABI / oracle wrappers do the column-major
conversion.  Reference fixtures cited per config.
"""
import numpy as np

MASK = (1 << 64) - 1
G_ACC = 9.81


class SplitMix64:
    """SplitMix64 stream; uniform() = (u64 >> 11) * 2^-53 in [0, 1)."""

    def __init__(self, seed):
        self.state = seed & MASK

    def u64(self, count):
        idx = np.arange(1, count + 1, dtype=np.uint64)
        with np.errstate(over="ignore"):
            z = np.uint64(self.state) + idx * np.uint64(0x9E3779B97F4A7C15)
            self.state = int(z[-1]) if count else self.state
            z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
            z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
            z = z ^ (z >> np.uint64(31))
        return z

    def uniform(self, lo, hi, shape):
        shape = (shape,) if isinstance(shape, int) else tuple(shape)
        count = int(np.prod(shape)) if shape else 1
        u = (self.u64(count) >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)
        return (lo + (hi - lo) * u).reshape(shape)

    def normal(self, shape):
        """Box-Muller on two uniform streams (u1 drawn first, then u2)."""
        shape = (shape,) if isinstance(shape, int) else tuple(shape)
        u1 = self.uniform(0.0, 1.0, shape)
        u2 = self.uniform(0.0, 1.0, shape)
        return np.sqrt(-2.0 * np.log(1.0 - u1)) * np.cos(2.0 * np.pi * u2)


def _seed(config, seed_offset):
    return 0xC0B7A000 + 1000 * config + seed_offset


def _double_integrator(T, mass):
    """reference tests/systems.h:63-66 (BoundedSystem); `mass` may be an array (batch,)."""
    mass = np.asarray(mass, dtype=np.float64)
    bshape = mass.shape
    A = np.zeros(bshape + (2, 2))
    A[..., 0, 0] = 1.0
    A[..., 0, 1] = T
    A[..., 1, 1] = 1.0
    B = np.zeros(bshape + (2, 1))
    B[..., 0, 0] = 0.5 * T * T / mass
    B[..., 1, 0] = T / mass
    d = np.zeros(bshape + (2,))
    d[..., 0] = (-G_ACC / 2.0) * T * T
    d[..., 1] = -G_ACC * T
    return A, B, d


def c1(cost="target"):
    """configs[0]: exactly the BoundedSystem fixture (tests/systems.h:42-90) with
    TargetCost+ControlCost (tests/TestLMPC.cpp:36-53) or TrajectoryCost (:99-115); batch 1."""
    T, N = 0.005, 300
    A, B, d = _double_integrator(T, 5.0)
    inf = np.inf
    return dict(
        name="C1-%s" % cost, nx=2, nu=1, N=N, batch=1, initial_state=False,
        A=A, B=B, d=d, x0=np.array([0.0, -5.0]),
        costs=[dict(kind=cost, M=np.eye(2), p=np.array([0.0, -1.0]), w=np.array([10.0, 10000.0])),
               dict(kind="control", N=np.eye(1), p=np.array([2.0]), w=np.array([1e-4]))],
        constraints=[dict(kind="trajectory_bound", lower=np.array([-inf, -inf]), upper=np.array([inf, 0.0])),
                     dict(kind="control_bound", lower=np.array([-inf]), upper=np.array([200.0]))])


def c2(batch=4096, seed_offset=0, N=50, T=0.03):
    """configs[1]: double integrator, N=50, T=0.03, per-instance mass/x0/xd/uUpper (SURVEY 8d)."""
    rng = SplitMix64(_seed(2, seed_offset))
    draws = rng.uniform(0.0, 1.0, (batch, 4))  # instance-major
    mass = 4.0 + 2.0 * draws[:, 0]
    v0 = -6.0 + 2.0 * draws[:, 1]
    vd = -1.5 + 1.0 * draws[:, 2]
    uup = 150.0 + 100.0 * draws[:, 3]
    A, B, d = _double_integrator(T, mass)
    inf = np.inf
    x0 = np.stack([np.zeros(batch), v0], axis=1)
    xd = np.stack([np.zeros(batch), vd], axis=1)
    return dict(
        name="C2", nx=2, nu=1, N=N, batch=batch, initial_state=False, A=A, B=B, d=d, x0=x0,
        costs=[dict(kind="target", M=np.eye(2), p=xd, w=np.array([10.0, 10000.0])),
               dict(kind="control", N=np.eye(1), p=np.array([2.0]), w=np.array([1e-4]))],
        constraints=[dict(kind="trajectory_bound", lower=np.array([-inf, -inf]), upper=np.array([inf, 0.0])),
                     dict(kind="control_bound", lower=np.array([-inf]), upper=uup[:, None])])


def c3(batch=16384, seed_offset=0, N=160, T=0.01):
    """configs[2]: walking CoM preview, 3rd-order LIPM, ZMP box as a step-size MixedConstraint."""
    rng = SplitMix64(_seed(3, seed_offset))
    draws = rng.uniform(0.0, 1.0, (batch, 9))
    p0 = -0.02 + 0.04 * draws[:, 0:2]
    v0 = -0.1 + 0.2 * draws[:, 2:4]
    vref = -0.3 + 0.6 * draws[:, 4:6]
    hw = 0.04 + 0.04 * draws[:, 6:8]
    h = 0.75 + 0.10 * draws[:, 8]
    A3 = np.array([[1.0, T, T * T / 2.0], [0.0, 1.0, T], [0.0, 0.0, 1.0]])
    B3 = np.array([T ** 3 / 6.0, T * T / 2.0, T])
    A = np.zeros((6, 6))
    A[0:3, 0:3] = A3
    A[3:6, 3:6] = A3
    B = np.zeros((6, 2))
    B[0:3, 0] = B3
    B[3:6, 1] = B3
    x0 = np.zeros((batch, 6))
    x0[:, 0], x0[:, 1], x0[:, 3], x0[:, 4] = p0[:, 0], v0[:, 0], p0[:, 1], v0[:, 1]
    M = np.zeros((2, 6))
    M[0, 1] = 1.0
    M[1, 4] = 1.0
    E = np.zeros((batch, 4, 6))
    E[:, 0, 0], E[:, 0, 2] = 1.0, -h / G_ACC
    E[:, 1, :] = -E[:, 0, :]
    E[:, 2, 3], E[:, 2, 5] = 1.0, -h / G_ACC
    E[:, 3, :] = -E[:, 2, :]
    f = np.stack([hw[:, 0], hw[:, 0], hw[:, 1], hw[:, 1]], axis=1)
    return dict(
        name="C3", nx=6, nu=2, N=N, batch=batch, initial_state=False, A=A, B=B, d=np.zeros(6), x0=x0,
        costs=[dict(kind="trajectory", M=M, p=vref, w=np.array([1.0, 1.0])),
               dict(kind="control", N=np.eye(2), p=np.zeros(2), w=np.array([1e-4, 1e-4]))],
        constraints=[dict(kind="mixed", E=E, G=np.zeros((4, 2)), f=f)])


def c4(batch=8192, seed_offset=0, N=50, T=0.03):
    """configs[3]: InitialStateLMPC on C2's system, Target+Control cost, control bound, x0 box."""
    rng = SplitMix64(_seed(4, seed_offset))
    draws = rng.uniform(0.0, 1.0, (batch, 4))
    mass = 4.0 + 2.0 * draws[:, 0]
    v0 = -6.0 + 2.0 * draws[:, 1]
    vd = -1.5 + 1.0 * draws[:, 2]
    uup = 150.0 + 100.0 * draws[:, 3]
    A, B, d = _double_integrator(T, mass)
    x0 = np.stack([np.zeros(batch), v0], axis=1)
    xd = np.stack([np.zeros(batch), vd], axis=1)
    delta = np.array([0.1, 0.5])
    R = np.eye(2)
    return dict(
        name="C4", nx=2, nu=1, N=N, batch=batch, initial_state=True, A=A, B=B, d=d, x0=x0,
        costs=[dict(kind="target", M=np.eye(2), p=xd, w=np.array([10.0, 100.0])),
               dict(kind="control", N=np.eye(1), p=np.array([2.0]), w=np.array([1e-2]))],
        constraints=[dict(kind="control_bound", lower=np.array([-np.inf]), upper=uup[:, None])],
        R=R, r=-(x0 @ R.T), x0lb=x0 - delta, x0ub=x0 + delta)


def c5(batch=1024, seed_offset=0, N=200, T=0.01):
    """configs[4]: condensing stress, 4 coupled triple integrators (nx=12, nu=4)."""
    rng = SplitMix64(_seed(5, seed_offset))
    nx, nu = 12, 4
    A3 = np.array([[1.0, T, T * T / 2.0], [0.0, 1.0, T], [0.0, 0.0, 1.0]])
    B3 = np.array([T ** 3 / 6.0, T * T / 2.0, T])
    A0 = np.zeros((nx, nx))
    B0 = np.zeros((nx, nu))
    for k in range(4):
        A0[3 * k:3 * k + 3, 3 * k:3 * k + 3] = A3
        B0[3 * k:3 * k + 3, k] = B3
    per = nx * nx + nx * nu + nx
    nrm = rng.normal((batch, per))
    A = A0 + 1e-3 * nrm[:, :nx * nx].reshape(batch, nx, nx)
    B = B0 + 1e-3 * nrm[:, nx * nx:nx * nx + nx * nu].reshape(batch, nx, nu)
    d = 1e-3 * nrm[:, nx * nx + nx * nu:]
    uni = rng.uniform(0.0, 1.0, (batch, 4 + 4 + 12))
    pos = [0, 3, 6, 9]
    x0 = np.zeros((batch, nx))
    ref = np.zeros((batch, nx))
    x0[:, pos] = -0.5 + uni[:, 0:4]
    ref[:, pos] = -0.8 + 1.6 * uni[:, 4:8]
    w = 1.0 + 99.0 * uni[:, 8:20]
    S = np.zeros((4, nx))
    for k, pcol in enumerate(pos):
        S[k, pcol] = 1.0
    E = np.vstack([S, -S])
    return dict(
        name="C5", nx=nx, nu=nu, N=N, batch=batch, initial_state=False, A=A, B=B, d=d, x0=x0,
        costs=[dict(kind="trajectory", M=np.eye(nx), p=ref, w=w),
               dict(kind="control", N=np.eye(nu), p=np.zeros(nu), w=np.full(nu, 1e-3))],
        constraints=[dict(kind="trajectory", E=E, f=np.full(8, 0.6)),
                     dict(kind="control_bound", lower=np.full(nu, -5.0), upper=np.full(nu, 5.0))])


def c3_walk(batch=16384, seed_offset=0, N=160, T=0.01, tick=0):
    """C3 walking: c3(...) unchanged (same system, weights, E, x0 and draws) plus a footstep plan, so that the ZMP box and
    the velocity reference move over the horizon as in a walking pattern generator.  Per instance, from config 6's stream:
    a step period of 0.4-0.6 s, a step length of 0.10-0.20 m, a lateral offset of 0.02-0.05 m and the phase of the first
    step (0.1 s plus up to one period).  The ZMP box stays centred at 0 until the first step (x0 is feasible at step 0);
    from there its centre advances by one step length per step and alternates sides.  The forward velocity reference ramps
    from 0 to the mean walking speed (step length / period) at the first step and stays there; the lateral one is 0.
    The MixedConstraint's f and the TrajectoryCost's p are per-step entries.  `tick` > 0 is the same plan seen `tick` control
    periods later (the next windows of a receding horizon; x0 stays c3's).  With these draws every instance of the default
    batch solves (status 0)."""
    bp = c3(batch, seed_offset, N, T)
    rng = SplitMix64(_seed(6, seed_offset))
    draws = rng.uniform(0.0, 1.0, (batch, 4))
    period = 0.4 + 0.2 * draws[:, 0]
    length = 0.10 + 0.10 * draws[:, 1]
    lateral = 0.02 + 0.03 * draws[:, 2]
    first = 0.1 + period * draws[:, 3]
    t = (np.arange(N + 1) + tick) * T
    k = np.where(t[None, :] < first[:, None], 0, 1 + np.floor((t[None, :] - first[:, None]) / period[:, None]))  # steps taken
    cx = k * length[:, None]
    cy = np.where(k == 0, 0.0, np.where(k % 2 == 1, 1.0, -1.0)) * lateral[:, None]
    hw = np.asarray(bp["constraints"][0]["f"])[:, [0, 2]]
    f = np.stack([hw[:, :1] + cx, hw[:, :1] - cx, hw[:, 1:] + cy, hw[:, 1:] - cy], axis=2)[:, :N]  # (batch, N, 4)
    speed = length / period
    vref = np.zeros((batch, N + 1, 2))
    vref[:, :, 0] = speed[:, None] * np.minimum(1.0, t[None, :] / first[:, None])
    bp["name"] = "C3-walk"
    bp["costs"][0] = dict(bp["costs"][0], p=vref.reshape(batch, -1), per_step=True)
    bp["constraints"][0] = dict(bp["constraints"][0], f=f.reshape(batch, -1), per_step=True)
    return bp


def _span(M, steps, add_cols=0):
    """block-diagonal copies of the (..., r, c) step matrix M at `steps` steps, `add_cols` zero column blocks appended
    (AutoSpan::spanMatrix)"""
    M = np.asarray(M, dtype=np.float64)
    M = M.reshape(M.shape[:-1] + (1, M.shape[-1])) if M.ndim == 1 else M
    r, c = M.shape[-2:]
    out = np.zeros(M.shape[:-2] + (r * steps, c * (steps + add_cols)))
    for i in range(steps):
        out[..., i * r:(i + 1) * r, i * c:(i + 1) * c] = M
    return out


def spanned(bp):
    """The same batch problem with every per-step entry in copra's full-size form: autoSpan'd block-diagonal matrices,
    weights tiled over the steps, and its full-length vector."""
    N = bp["N"]
    out = dict(bp)
    costs = []
    for c in bp["costs"]:
        c = dict(c)
        if c.pop("per_step", False):
            steps = N + 1 if c["kind"] == "trajectory" else N
            add = 1 if c["kind"] == "mixed" else 0
            if c.get("M") is not None:
                c["M"] = _span(c["M"], steps, add)
            if c.get("N") is not None:
                c["N"] = _span(c["N"], steps)
            w = np.asarray(c["w"], dtype=np.float64)
            c["w"] = np.tile(w, (1,) * (w.ndim - 1) + (steps,))
        costs.append(c)
    cstrs = []
    for c in bp["constraints"]:
        c = dict(c)
        if c.pop("per_step", False) and c["kind"] not in ("trajectory_bound", "control_bound"):
            steps = N + 1 if c["kind"] == "trajectory" else N
            add = 1 if c["kind"] == "mixed" else 0
            if c.get("E") is not None:
                c["E"] = _span(c["E"], steps, add)
            if c.get("G") is not None:
                c["G"] = _span(c["G"], steps)
        cstrs.append(c)
    out["costs"], out["constraints"] = costs, cstrs
    return out


CONFIGS = {"c1": c1, "c2": c2, "c3": c3, "c4": c4, "c5": c5}

# base (un-batched) ndim of every parameter array
_BASE_NDIM = dict(A=2, B=2, d=1, x0=1, R=2, r=1, x0lb=1, x0ub=1, M=2, N=2, E=2, G=2, p=1, w=1, f=1, lower=1, upper=1)


def _pick(key, arr, i):
    if arr is None:
        return None
    arr = np.asarray(arr, dtype=np.float64)
    return arr[i] if arr.ndim > _BASE_NDIM[key] else arr


def is_batched(key, arr):
    return arr is not None and np.asarray(arr).ndim > _BASE_NDIM[key]


def instance(bp, i):
    """Extract instance `i` of a batch problem as a single-instance dict (oracle / facade input)."""
    out = dict(nx=bp["nx"], nu=bp["nu"], N=bp["N"], initial_state=bp.get("initial_state", False))
    for k in ("A", "B", "d", "x0", "R", "r", "x0lb", "x0ub"):
        out[k] = _pick(k, bp.get(k), i)
    out["costs"] = [{k: (_pick(k, v, i) if k in _BASE_NDIM else v) for k, v in c.items()} for c in bp["costs"]]
    out["constraints"] = [{k: (_pick(k, v, i) if k in _BASE_NDIM else v) for k, v in c.items()}
                          for c in bp["constraints"]]
    return out


def take(bp, idx):
    """Sub-batch with the given instance indices (used for sharding and CPU-baseline samples)."""
    idx = np.asarray(idx)
    out = dict(bp)
    out["batch"] = int(idx.shape[0])
    for k in ("A", "B", "d", "x0", "R", "r", "x0lb", "x0ub"):
        if is_batched(k, bp.get(k)):
            out[k] = np.asarray(bp[k])[idx]
    out["costs"] = [{k: (np.asarray(v)[idx] if k in _BASE_NDIM and is_batched(k, v) else v) for k, v in c.items()}
                    for c in bp["costs"]]
    out["constraints"] = [{k: (np.asarray(v)[idx] if k in _BASE_NDIM and is_batched(k, v) else v)
                           for k, v in c.items()} for c in bp["constraints"]]
    return out


def shard(bp, rank, world):
    """Contiguous instance-index shard [rank*ceil(B/W), (rank+1)*ceil(B/W)) (SURVEY.md 8e)."""
    B = bp["batch"]
    per = -(-B // world)
    lo, hi = min(B, rank * per), min(B, (rank + 1) * per)
    return take(bp, np.arange(lo, hi)), (lo, hi)
