"""ctypes binding of the C ABI in include/copra_b200.h (libcopra_b200.so).

This is a thin numpy/torch-pointer adaptor for tests and bench.py; all computation happens in the
sm_100a kernels behind the C ABI.  There is NO CPU fallback: if the shared library is missing or no
CUDA device is usable, construction raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libcopra_b200.so")

HOST, DEVICE = 0, 1
FLAG_NO_REG = 1  # COPRA_B200_FLAG_NO_REG: no 1e-6 I regulariser (single cost evaluation)
FLAG_STABLE_BOUND_PATTERN = 2  # device inputs: the +-inf pattern of trajectory bounds is unchanged since the last build
PER_STEP = 2  # COPRA_B200_PER_STEP: step-size matrices, a vector per step (rows x steps entries, step-major)
COST_KINDS = {"trajectory": 0, "target": 1, "control": 2, "mixed": 3}
CSTR_KINDS = {"trajectory": 0, "control": 1, "mixed": 2, "trajectory_bound": 3, "control_bound": 4}
GET = dict(Phi=0, Psi=1, xi=2, Q=3, c=4, Aeq=5, beq=6, Aineq=7, bineq=8, lb=9, ub=10)

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


class Options(C.Structure):
    _fields_ = [("device", C.c_int), ("stream", C.c_void_p), ("sm_limit", C.c_int), ("small_variant", C.c_int),
                ("reserved", C.c_int * 4)]


class Array(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("stride", C.c_longlong)]


class Cost(C.Structure):
    _fields_ = [("kind", C.c_int), ("rows", C.c_int), ("M", Array), ("N", Array), ("p", Array), ("w", Array), ("full_size", C.c_int)]


class Constraint(C.Structure):
    _fields_ = [("kind", C.c_int), ("rows", C.c_int), ("is_ineq", C.c_int),
                ("E", Array), ("G", Array), ("f", Array), ("lower", Array), ("upper", Array), ("full_size", C.c_int)]


class Problem(C.Structure):
    _fields_ = [("nx", C.c_int), ("nu", C.c_int), ("N", C.c_int), ("batch", C.c_int), ("initial_state", C.c_int),
                ("A", Array), ("B", Array), ("d", Array), ("x0", Array),
                ("ncost", C.c_int), ("costs", C.POINTER(Cost)),
                ("ncstr", C.c_int), ("cstrs", C.POINTER(Constraint)),
                ("R", Array), ("r", Array), ("x0lb", Array), ("x0ub", Array),
                ("memory", C.c_int), ("flags", C.c_int)]


class Sizes(C.Structure):
    _fields_ = [(k, C.c_int) for k in ("X", "nU", "nvar", "meq", "mineq", "q")]


class Results(C.Structure):
    _fields_ = [("control", C.c_void_p), ("trajectory", C.c_void_p), ("x", C.c_void_p), ("status", C.c_void_p),
                ("iters", C.c_void_p), ("nact", C.c_void_p), ("iact", C.c_void_p), ("memory", C.c_int)]


class VjpOut(C.Structure):
    _fields_ = [("x0", C.c_void_p), ("p", C.POINTER(C.c_void_p)), ("f", C.POINTER(C.c_void_p)),
                ("lower", C.POINTER(C.c_void_p)), ("upper", C.POINTER(C.c_void_p))]


class VjpCostOut(C.Structure):
    _fields_ = [("w", C.POINTER(C.c_void_p)), ("M", C.POINTER(C.c_void_p)), ("N", C.POINTER(C.c_void_p))]


class VjpModelOut(C.Structure):
    _fields_ = [("A", C.c_void_p), ("B", C.c_void_p), ("d", C.c_void_p), ("E", C.POINTER(C.c_void_p)),
                ("G", C.POINTER(C.c_void_p))]


class QpVjpOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("Q", "c", "Aeq", "beq", "Aineq", "bineq", "lb", "ub")]


class QpJvpIn(C.Structure):
    _fields_ = [("ndir", C.c_int)] + [(k, Array) for k in ("Q", "c", "Aeq", "beq", "Aineq", "bineq", "lb", "ub")]


class JvpIn(C.Structure):
    _fields_ = [("ndir", C.c_int), ("x0", C.c_void_p), ("p", C.POINTER(C.c_void_p)), ("f", C.POINTER(C.c_void_p)),
                ("lower", C.POINTER(C.c_void_p)), ("upper", C.POINTER(C.c_void_p))]


class VjpInitialOut(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("R", "r", "x0lb", "x0ub")]


class JvpInitialIn(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("R", "r", "x0lb", "x0ub")]


class Timing(C.Structure):
    _fields_ = [(k, C.c_float) for k in ("h2d_ms", "condense_ms", "assemble_ms", "solve_ms", "rollout_ms", "d2h_ms",
                                         "total_ms")] + [("launches", C.c_longlong)]


EXPORTS = ["copra_b200_abi_version", "copra_b200_device_count", "copra_b200_create", "copra_b200_destroy",
           "copra_b200_last_error", "copra_b200_set_stream", "copra_b200_synchronize", "copra_b200_launch_count",
           "copra_b200_last_timing", "copra_b200_condense", "copra_b200_solve_qp_batch", "copra_b200_lmpc_sizes",
           "copra_b200_lmpc_run", "copra_b200_lmpc_build", "copra_b200_lmpc_solve", "copra_b200_lmpc_download",
           "copra_b200_lmpc_results", "copra_b200_dgemm_batch", "copra_b200_lmpc_resolve", "copra_b200_fp64_peaks",
           "copra_b200_lmpc_built_sizes", "copra_b200_last_solver", "copra_b200_hessian_is_shared", "copra_b200_multi_create", "copra_b200_multi_destroy",
           "copra_b200_multi_last_error", "copra_b200_multi_size", "copra_b200_multi_shard", "copra_b200_multi_timing",
           "copra_b200_multi_launch_count", "copra_b200_multi_lmpc_run", "copra_b200_multi_lmpc_resolve",
           "copra_b200_set_warm_start", "copra_b200_get_warm_start", "copra_b200_multi_set_warm_start",
           "copra_b200_lmpc_retarget", "copra_b200_multi_lmpc_retarget", "copra_b200_lmpc_vjp",
           "copra_b200_multi_lmpc_vjp", "copra_b200_lmpc_jvp", "copra_b200_lmpc_feedback_gain",
           "copra_b200_multi_lmpc_jvp", "copra_b200_multi_lmpc_feedback_gain", "copra_b200_lmpc_vjp_costs",
           "copra_b200_multi_lmpc_vjp_costs", "copra_b200_lmpc_vjp_model", "copra_b200_multi_lmpc_vjp_model",
           "copra_b200_qp_vjp", "copra_b200_lmpc_vjp_initial_state", "copra_b200_lmpc_jvp_initial_state",
           "copra_b200_multi_lmpc_vjp_initial_state", "copra_b200_multi_lmpc_jvp_initial_state", "copra_b200_qp_jvp",
           "copra_b200_qp_jacobian"]
VJP_WANT = ("x0", "p", "f", "lower", "upper")
VJP_COST_WANT = ("w", "M", "N")  # gradients with respect to the cost weights and matrices: requested by name only
VJP_MODEL_WANT = ("A", "B", "d", "E", "G")  # ... and to the dynamics and the row constraints' matrices: by name only
QP_VJP_WANT = ("Q", "c", "Aeq", "beq", "Aineq", "bineq", "lb", "ub")  # gradients of a raw QP batch (copra_b200_qp_vjp)
INITIAL_KEYS = ("R", "r", "x0lb", "x0ub")  # initial-state builds: the x0 cost and box (copra_b200_lmpc_vjp_initial_state)
QP_BASE_NDIM = dict(Q=2, c=1, Aeq=2, beq=1, Aineq=2, bineq=1, lb=1, ub=1)
QP_WRT = dict(c=0, beq=1, bineq=2, lb=3, ub=4)  # COPRA_B200_QP_WRT_*: the inputs copra_b200_qp_jacobian differentiates by

_lib = None


class CopraB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("copra_b200 error %d: %s" % (code, msg))
        self.code = code


def load():
    """Load libcopra_b200.so; raises if it has not been built (python __graft_entry__.py / make)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CopraB200Error(-100, "libcopra_b200.so is not built (run `make` or __graft_entry__.build()); "
                                       "there is no CPU fallback")
        lib = C.CDLL(LIB_PATH)
        lib.copra_b200_last_error.restype = C.c_char_p
        lib.copra_b200_last_error.argtypes = [C.c_void_p]
        lib.copra_b200_launch_count.restype = C.c_longlong
        lib.copra_b200_launch_count.argtypes = [C.c_void_p]
        lib.copra_b200_create.argtypes = [C.POINTER(Options), C.POINTER(C.c_void_p)]
        lib.copra_b200_destroy.argtypes = [C.c_void_p]
        lib.copra_b200_destroy.restype = None
        lib.copra_b200_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        lib.copra_b200_synchronize.argtypes = [C.c_void_p]
        lib.copra_b200_last_timing.argtypes = [C.c_void_p, C.POINTER(Timing)]
        lib.copra_b200_condense.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, Array, Array, Array,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        lib.copra_b200_solve_qp_batch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int] + [Array] * 8 + \
            [C.c_void_p] * 5 + [C.c_int]
        lib.copra_b200_lmpc_sizes.argtypes = [C.c_void_p, C.POINTER(Problem), C.POINTER(Sizes)]
        lib.copra_b200_lmpc_run.argtypes = [C.c_void_p, C.POINTER(Problem), C.POINTER(Results)]
        lib.copra_b200_lmpc_build.argtypes = [C.c_void_p, C.POINTER(Problem)]
        lib.copra_b200_lmpc_solve.argtypes = [C.c_void_p, C.POINTER(Results)]
        lib.copra_b200_lmpc_download.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        lib.copra_b200_lmpc_results.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        lib.copra_b200_fp64_peaks.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        lib.copra_b200_lmpc_resolve.argtypes = [C.c_void_p, Array, C.c_int, C.POINTER(Results)]
        lib.copra_b200_lmpc_retarget.argtypes = [C.c_void_p, C.POINTER(Problem), C.POINTER(Results)]
        lib.copra_b200_dgemm_batch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_int,
                                               C.c_longlong, C.c_void_p, C.c_int, C.c_longlong, C.c_double, C.c_void_p, C.c_int,
                                               C.c_longlong, C.c_int, C.c_int]
        lib.copra_b200_lmpc_built_sizes.argtypes = [C.c_void_p, C.POINTER(Sizes)]
        lib.copra_b200_last_solver.argtypes = [C.c_void_p]
        lib.copra_b200_last_solver.restype = C.c_char_p
        lib.copra_b200_hessian_is_shared.argtypes = [C.c_void_p]
        lib.copra_b200_set_warm_start.argtypes = [C.c_void_p, C.c_int]
        lib.copra_b200_get_warm_start.argtypes = [C.c_void_p]
        lib.copra_b200_multi_create.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]
        lib.copra_b200_multi_destroy.argtypes = [C.c_void_p]
        lib.copra_b200_multi_destroy.restype = None
        lib.copra_b200_multi_last_error.argtypes = [C.c_void_p]
        lib.copra_b200_multi_last_error.restype = C.c_char_p
        lib.copra_b200_multi_size.argtypes = [C.c_void_p]
        lib.copra_b200_multi_shard.argtypes = [C.c_void_p, C.c_int, _ip, _ip, _ip]
        lib.copra_b200_multi_timing.argtypes = [C.c_void_p, C.c_int, C.POINTER(Timing), C.POINTER(C.c_double)]
        lib.copra_b200_multi_launch_count.argtypes = [C.c_void_p]
        lib.copra_b200_multi_launch_count.restype = C.c_longlong
        lib.copra_b200_multi_lmpc_run.argtypes = [C.c_void_p, C.POINTER(Problem), C.POINTER(Results)]
        lib.copra_b200_multi_lmpc_resolve.argtypes = [C.c_void_p, Array, C.POINTER(Results)]
        lib.copra_b200_multi_lmpc_retarget.argtypes = [C.c_void_p, C.POINTER(Problem), C.POINTER(Results)]
        lib.copra_b200_multi_set_warm_start.argtypes = [C.c_void_p, C.c_int]
        lib.copra_b200_lmpc_vjp.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(VjpOut)]
        lib.copra_b200_multi_lmpc_vjp.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(VjpOut)]
        lib.copra_b200_lmpc_vjp_costs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(VjpOut),
                                                  C.POINTER(VjpCostOut)]
        lib.copra_b200_multi_lmpc_vjp_costs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(VjpOut),
                                                        C.POINTER(VjpCostOut)]
        lib.copra_b200_lmpc_vjp_model.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(VjpOut),
                                                  C.POINTER(VjpCostOut), C.POINTER(VjpModelOut)]
        lib.copra_b200_multi_lmpc_vjp_model.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(VjpOut),
                                                        C.POINTER(VjpCostOut), C.POINTER(VjpModelOut)]
        lib.copra_b200_qp_vjp.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(QpVjpOut)]
        lib.copra_b200_qp_jvp.argtypes = [C.c_void_p, C.POINTER(QpJvpIn), C.c_int, C.c_void_p]
        lib.copra_b200_qp_jacobian.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        lib.copra_b200_lmpc_jvp.argtypes = [C.c_void_p, C.POINTER(JvpIn), C.c_int, C.c_void_p, C.c_void_p]
        lib.copra_b200_lmpc_feedback_gain.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        lib.copra_b200_multi_lmpc_jvp.argtypes = [C.c_void_p, C.POINTER(JvpIn), C.c_void_p, C.c_void_p]
        lib.copra_b200_multi_lmpc_feedback_gain.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        lib.copra_b200_lmpc_vjp_initial_state.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(VjpOut),
                                                          C.POINTER(VjpInitialOut)]
        lib.copra_b200_multi_lmpc_vjp_initial_state.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(VjpOut),
                                                                C.POINTER(VjpInitialOut)]
        lib.copra_b200_lmpc_jvp_initial_state.argtypes = [C.c_void_p, C.POINTER(JvpIn), C.POINTER(JvpInitialIn), C.c_int,
                                                          C.c_void_p, C.c_void_p]
        lib.copra_b200_multi_lmpc_jvp_initial_state.argtypes = [C.c_void_p, C.POINTER(JvpIn), C.POINTER(JvpInitialIn),
                                                                C.c_void_p, C.c_void_p]
        _lib = lib
    return _lib


def _colmajor(a, base_ndim):
    """logical (..., r, c) -> contiguous buffer holding each instance column-major."""
    a = np.asarray(a, dtype=np.float64)
    if base_ndim == 2:
        a = np.swapaxes(a, -1, -2)
    return np.ascontiguousarray(a)


def _steps(kind, N):
    """steps of the horizon a cost / constraint kind applies to: the length, in steps, of its per-step vector"""
    return N + 1 if kind in ("trajectory", "trajectory_bound") else (1 if kind == "target" else N)


def _rows_of(mat):
    a = np.asarray(mat)
    return int(a.shape[-2]) if a.ndim >= 2 else 1


def _check_per_step(what, vec, rows, steps):
    if np.asarray(vec).shape[-1] != rows * steps:
        raise CopraB200Error(-1, "%s: a per-step vector holds rows x steps = %d x %d entries, got %d"
                             % (what, rows, steps, np.asarray(vec).shape[-1]))


class HostBatch:
    """A batch problem (copra_b200.workloads dict) packed into column-major host buffers + the ctypes
    `Problem` describing them.  Buffers live as long as this object (pin=True: torch pinned memory).
    A cost or constraint dict with `per_step=True` is packed as COPRA_B200_PER_STEP: step-size matrices, and a p / f /
    lower / upper of rows x steps entries (step-major) per instance."""

    _BASE = dict(A=2, B=2, d=1, x0=1, R=2, r=1, x0lb=1, x0ub=1, M=2, N=2, E=2, G=2, p=1, w=1, f=1, lower=1, upper=1)

    def __init__(self, bp, pin=False, device_tensors=None):
        self.bp = bp
        self.keep = []
        self.pin = pin
        self.device = device_tensors  # torch device or None
        self.h2d_bytes = 0
        p = Problem()
        p.nx, p.nu, p.N, p.batch = int(bp["nx"]), int(bp["nu"]), int(bp["N"]), int(bp["batch"])
        p.initial_state = int(bool(bp.get("initial_state", False)))
        p.memory = DEVICE if device_tensors is not None else HOST
        for k in ("A", "B", "d", "x0"):
            setattr(p, k, self._arr(k, bp[k]))
        for k in ("R", "r", "x0lb", "x0ub"):
            if bp.get(k) is not None:
                setattr(p, k, self._arr(k, bp[k]))
        costs = (Cost * max(1, len(bp["costs"])))()
        N_ = int(bp["N"])
        for i, c in enumerate(bp["costs"]):
            costs[i].kind = COST_KINDS[c["kind"]]
            pv = np.asarray(c["p"])
            costs[i].rows = int(pv.shape[-1])
            nx_, nu_ = int(bp["nx"]), int(bp["nu"])
            per_step = bool(c.get("per_step", False))
            if per_step:
                costs[i].rows = _rows_of(c["M"] if c.get("M") is not None else c["N"])
                _check_per_step("cost %d" % i, pv, costs[i].rows, _steps(c["kind"], N_))
            if c.get("M") is not None:
                costs[i].M = self._arr("M", c["M"])
                costs[i].full_size = int(np.asarray(c["M"]).shape[-1] != nx_)
            if c.get("N") is not None:
                costs[i].N = self._arr("N", c["N"])
                costs[i].full_size = int(np.asarray(c["N"]).shape[-1] != nu_) if c.get("M") is None else costs[i].full_size
            if per_step:
                costs[i].full_size = PER_STEP
            costs[i].p = self._arr("p", c["p"])
            w = c.get("w")
            w = np.ones(costs[i].rows) if w is None else np.asarray(w, dtype=np.float64)
            if w.shape[-1] != costs[i].rows:  # CostFunction::weights() tiling (include/costFunctions.h:59-63)
                if costs[i].rows % w.shape[-1] != 0:
                    raise CopraB200Error(-1, "weights badly dimensioned")
                w = np.tile(w, costs[i].rows // w.shape[-1])
            costs[i].w = self._arr("w", w)
        self.keep.append(costs)
        p.ncost, p.costs = len(bp["costs"]), costs
        cstrs = (Constraint * max(1, len(bp["constraints"])))()
        for i, c in enumerate(bp["constraints"]):
            cstrs[i].kind = CSTR_KINDS[c["kind"]]
            cstrs[i].is_ineq = int(bool(c.get("is_ineq", True)))
            per_step = bool(c.get("per_step", False))
            steps = _steps(c["kind"], N_)
            if c["kind"] in ("trajectory_bound", "control_bound"):
                cstrs[i].rows = int(np.asarray(c["lower"]).shape[-1])
                cstrs[i].full_size = int(cstrs[i].rows != (int(bp["nx"]) if c["kind"] == "trajectory_bound" else int(bp["nu"])))
                if per_step:
                    cstrs[i].rows = int(bp["nx"]) if c["kind"] == "trajectory_bound" else int(bp["nu"])
                    cstrs[i].full_size = PER_STEP
                    for k in ("lower", "upper"):
                        _check_per_step("constraint %d %s" % (i, k), c[k], cstrs[i].rows, steps)
                cstrs[i].lower = self._arr("lower", c["lower"])
                cstrs[i].upper = self._arr("upper", c["upper"])
            else:
                cstrs[i].rows = int(np.asarray(c["f"]).shape[-1])
                if c.get("E") is not None:
                    cstrs[i].E = self._arr("E", c["E"])
                    cstrs[i].full_size = int(np.asarray(c["E"]).shape[-1] != int(bp["nx"]))
                if c.get("G") is not None:
                    cstrs[i].G = self._arr("G", c["G"])
                    if c.get("E") is None:
                        cstrs[i].full_size = int(np.asarray(c["G"]).shape[-1] != int(bp["nu"]))
                if per_step:
                    cstrs[i].rows = _rows_of(c["E"] if c.get("E") is not None else c["G"])
                    cstrs[i].full_size = PER_STEP
                    _check_per_step("constraint %d" % i, c["f"], cstrs[i].rows, steps)
                cstrs[i].f = self._arr("f", c["f"])
        self.keep.append(cstrs)
        p.ncstr, p.cstrs = len(bp["constraints"]), cstrs
        self.problem = p

    def _arr(self, key, value):
        base = self._BASE[key]
        a = np.asarray(value, dtype=np.float64)
        if base == 2 and a.ndim == 1:
            a = a.reshape(1, -1) if key in ("M", "N", "E", "G") else a
        batched = a.ndim > base
        buf = _colmajor(a, base)
        size = int(np.prod(buf.shape[1:])) if batched else int(buf.size)
        out = Array()
        if self.device is not None or self.pin:
            import torch
            t = torch.from_numpy(buf.reshape(-1).copy())
            if self.device is not None:
                t = t.to(self.device)
            else:
                t = t.pin_memory()
            self.keep.append(t)
            out.ptr = t.data_ptr()
        else:
            self.keep.append(buf)
            out.ptr = buf.ctypes.data
        out.stride = size if batched else 0
        self.h2d_bytes += buf.nbytes
        return out


def _result_buffers(B, s, want=None):
    """host result arrays for B instances of sizes `s` and the Results struct pointing at those in `want` (default: all)"""
    out = dict(control=np.zeros((B, s["nU"])), trajectory=np.zeros((B, s["X"])), x=np.zeros((B, s["nvar"])),
               status=np.full(B, -1, np.int32), iters=np.zeros((B, 2), np.int32), nact=np.zeros(B, np.int32),
               iact=np.zeros((B, s["nvar"]), np.int32))
    r = Results()
    r.memory = HOST
    for k in out if want is None else want:
        setattr(r, k, out[k].ctypes.data)
    return out, r


class _Memory:
    """Where the arrays of one call live: HOST numpy arrays, or CUDA float64 tensors on the device of its torch inputs (or
    on `device`).  Outputs are allocated the same way.  With tensors the engine runs on its own stream: `run` makes the
    inputs complete before the call (device synchronise) and waits for the engine's stream (`sync`) before the outputs
    are handed back."""

    def __init__(self, *inputs, device=None):
        self.device = next((a.device for a in inputs if hasattr(a, "data_ptr")), device)
        self.kind = HOST if self.device is None else DEVICE
        self.keep = []  # input copies and pointer arrays, alive for the call

    def array(self, a):
        """`a` as a float64 array of this memory"""
        if self.device is None:
            return np.asarray(a, dtype=np.float64)
        import torch
        return torch.as_tensor(a, dtype=torch.float64, device=self.device).detach()

    def buffer(self, a):
        """the pointer to a contiguous float64 copy of `a` kept for the call (None for None)"""
        if a is None:
            return None
        a = self.array(a)
        a = np.ascontiguousarray(a) if self.device is None else a.contiguous()
        self.keep.append(a)
        return self.ptr(a)

    def empty(self, *shape, dtype=np.float64):
        """an output array; the engine writes (or zeroes) every entry of what it is handed"""
        if self.device is None:
            return np.zeros(shape, dtype)
        import torch
        return torch.empty(shape, dtype=getattr(torch, np.dtype(dtype).name), device=self.device)

    def ptr(self, a):
        """the data pointer of `a`, None for None or an empty array"""
        if a is None or 0 in a.shape:
            return None
        return a.ctypes.data if self.device is None else a.data_ptr()

    def pointers(self, arrs):
        """a C array of the pointers of `arrs`, kept for the call"""
        p = (C.c_void_p * max(1, len(arrs)))(*[self.ptr(a) for a in arrs])
        self.keep.append(p)
        return C.cast(p, C.POINTER(C.c_void_p))

    def rowmajor(self, a):
        """(batch, cols, rows) as the engine writes matrices (column-major) -> contiguous (batch, rows, cols)"""
        if a is None:
            return None
        return np.ascontiguousarray(a.transpose(0, 2, 1)) if self.device is None else a.transpose(1, 2).contiguous()

    def run(self, call, sync=None):
        if self.device is None:
            return call()
        import torch
        torch.cuda.synchronize(self.device)
        try:
            return call()
        finally:
            if sync is not None:
                sync()


_MEM = object()  # stands where a single-device entry takes the memory kind; a multi-device entry has no such argument


def vjp_lengths(bp):
    """per-instance lengths of the gradients lmpc_vjp returns: nx, [p of every cost], [(f | lower / upper) of every
    constraint] -- rows, or rows x steps for a per-step entry"""
    plen = [int(np.asarray(c["p"]).shape[-1]) for c in bp["costs"]]
    clen = [int(np.asarray(c["lower"] if c["kind"] in ("trajectory_bound", "control_bound") else c["f"]).shape[-1])
            for c in bp["constraints"]]
    return int(bp["nx"]), plen, clen


def cost_shapes(bp):
    """(rows, has_M, has_N) of every cost: the shapes of the w, M and N gradients lmpc_vjp returns"""
    out = []
    for c in bp["costs"]:
        if c.get("per_step"):
            rows = _rows_of(c["M"] if c.get("M") is not None else c["N"])
        else:
            rows = int(np.asarray(c["p"]).shape[-1])
        out.append((rows, c["kind"] in ("trajectory", "target", "mixed"), c["kind"] in ("control", "mixed")))
    return out


def cstr_shapes(bp):
    """(rows, has_E, has_G) of every constraint: the shapes of the E and G gradients lmpc_vjp returns (0 rows for a bound)"""
    out = []
    for c in bp["constraints"]:
        has_e, has_g = c["kind"] in ("trajectory", "mixed"), c["kind"] in ("control", "mixed")
        rows = _rows_of(c["E"] if has_e else c["G"]) if has_e or has_g else 0
        out.append((rows, has_e, has_g))
    return out


def initial_want(bp):
    """the gradients Engine.initial_state_vjp returns by default: x0 and the vectors, and R, r, x0lb, x0ub where the build
    was given them"""
    return VJP_WANT + tuple(k for k in INITIAL_KEYS if bp.get(k) is not None)


def _vjp_call(bp, B, dcontrol, dtrajectory, want, call, sync=None, initial=False):
    """allocate the wanted gradients (numpy, or torch tensors on the device of the torch cotangents), describe them in a
    VjpOut (and, when w, M or N are wanted, a VjpCostOut; when A, B, d, E or G are, a VjpModelOut) and run
    `call(dcontrol_ptr, dtrajectory_ptr, memory, out, cost_out, model_out)`, cost_out / model_out None unless such gradients
    are wanted.  With `initial` (an initial-state build) it runs `call(dcontrol_ptr, dtrajectory_ptr, memory, out, init_out)`
    instead, init_out a VjpInitialOut for R, r, x0lb and x0ub.  With torch tensors the call runs as _Memory.run orders it."""
    mem = _Memory(dcontrol, dtrajectory)
    nu = int(bp["nu"])
    nx, plen, clen = vjp_lengths(bp)

    def zeros(*shape):  # the engine zeroes every requested gradient on its stream
        return mem.empty(B, *shape)
    bound = [c["kind"] in ("trajectory_bound", "control_bound") for c in bp["constraints"]]
    res = dict(x0=zeros(nx) if "x0" in want else None,
               p=[zeros(k) if "p" in want else None for k in plen],
               f=[zeros(k) if "f" in want and not b else None for k, b in zip(clen, bound)],
               lower=[zeros(k) if "lower" in want and b else None for k, b in zip(clen, bound)],
               upper=[zeros(k) if "upper" in want and b else None for k, b in zip(clen, bound)])
    o = VjpOut(x0=mem.ptr(res["x0"]), **{k: mem.pointers(res[k]) for k in ("p", "f", "lower", "upper")})
    # the engine writes every matrix column-major: allocated as (batch, cols, rows), handed back as (batch, rows, cols)
    co = mo = io = None
    if any(k in want for k in VJP_COST_WANT):
        shapes = cost_shapes(bp)
        res.update(w=[zeros(r) if "w" in want else None for r, _, _ in shapes],
                   M=[zeros(nx, r) if "M" in want and hm else None for r, hm, _ in shapes],
                   N=[zeros(nu, r) if "N" in want and hn else None for r, _, hn in shapes])
        co = VjpCostOut(**{k: mem.pointers(res[k]) for k in VJP_COST_WANT})
    if any(k in want for k in VJP_MODEL_WANT):
        shapes = cstr_shapes(bp)
        res.update(A=zeros(nx, nx) if "A" in want else None, B=zeros(nu, nx) if "B" in want else None,
                   d=zeros(nx) if "d" in want else None,
                   E=[zeros(nx, r) if "E" in want and he else None for r, he, _ in shapes],
                   G=[zeros(nu, r) if "G" in want and hg else None for r, _, hg in shapes])
        mo = VjpModelOut(A=mem.ptr(res["A"]), B=mem.ptr(res["B"]), d=mem.ptr(res["d"]), E=mem.pointers(res["E"]),
                         G=mem.pointers(res["G"]))
    if initial:
        if co is not None or mo is not None:
            raise CopraB200Error(-4, "initial-state builds have no gradients with respect to w, M, N, A, B, d, E or G")
        # R is symmetric: its column-major layout is its logical one
        res.update(R=zeros(nx, nx) if "R" in want else None,
                   **{k: zeros(nx) if k in want else None for k in ("r", "x0lb", "x0ub")})
        io = VjpInitialOut(**{k: mem.ptr(res[k]) for k in INITIAL_KEYS})
    dc, dt = mem.buffer(dcontrol), mem.buffer(dtrajectory)
    mem.run(lambda: call(dc, dt, mem.kind, o, io) if initial else call(dc, dt, mem.kind, o, co, mo), sync)
    for k in ("M", "N", "E", "G"):
        if k in res:
            res[k] = [mem.rowmajor(a) for a in res[k]]
    for k in ("A", "B"):
        if k in res:
            res[k] = mem.rowmajor(res[k])
    return res


def _jvp_call(bp, B, x0, p, f, lower, upper, call, sync=None, init=None):
    """describe the tangents (each (batch, k, len), numpy or CUDA float64 tensors; None = zero) in a JvpIn, allocate dU
    (batch, k, nU) and dtrajectory (batch, k, X) of the same kind and run `call(jvp_in, memory, dU_ptr, dX_ptr)`.  With
    `init` (a dict of the R (batch, k, nx, nx), r, x0lb and x0ub (batch, k, nx) tangents of an initial-state build) it runs
    `call(jvp_in, jvp_initial_in, memory, dU_ptr, dX_ptr)` instead.  With torch tensors the call runs as _Memory.run
    orders it."""
    nx, plen, clen = vjp_lengths(bp)
    bound = [c["kind"] in ("trajectory_bound", "control_bound") for c in bp["constraints"]]
    lists = dict(p=list(p or []), f=list(f or []), lower=list(lower or []), upper=list(upper or []))
    initial = init is not None
    init = dict(init or {})
    R = init.get("R")
    if R is not None and len(R.shape) == 4:  # (batch, k, nx, nx) -> column-major nx x nx per direction
        R = R.transpose(2, 3) if hasattr(R, "data_ptr") else np.swapaxes(np.asarray(R, dtype=np.float64), 2, 3)
        init["R"] = R.reshape(R.shape[0], R.shape[1], nx * nx)
    given = [t for t in [x0] + [t for v in lists.values() for t in v] + list(init.values()) if t is not None]
    if not given:
        raise CopraB200Error(-1, "lmpc_jvp needs at least one tangent")
    k = int(given[0].shape[1]) if len(given[0].shape) == 3 else 0
    mem = _Memory(*given)

    def inp(a, n, what):
        if a is not None and tuple(a.shape) != (B, k, n):
            raise CopraB200Error(-1, "lmpc_jvp: the %s tangent has shape %s, expected (batch, k, len) = %s"
                                 % (what, tuple(a.shape), (B, k, n)))
        return mem.buffer(a)

    t = JvpIn()
    t.ndir = k
    t.x0 = inp(x0, nx, "x0")
    lens = dict(p=plen, f=clen, lower=clen, upper=clen)
    for key, arrs in lists.items():
        n = len(lens[key])
        if len(arrs) > n:
            raise CopraB200Error(-1, "lmpc_jvp: %d %s tangents for %d entries" % (len(arrs), key, n))
        arrs = arrs + [None] * (n - len(arrs))
        if key != "p":
            for j, a in enumerate(arrs):
                if a is not None and bound[j] == (key == "f"):
                    raise CopraB200Error(-1, "lmpc_jvp: constraint %d has no %s vector" % (j, key))
        ptrs = (C.c_void_p * max(1, n))(*[inp(a, lens[key][j], "%s[%d]" % (key, j)) for j, a in enumerate(arrs)])
        mem.keep.append(ptrs)
        setattr(t, key, C.cast(ptrs, C.POINTER(C.c_void_p)))
    ti = JvpInitialIn(**{key: inp(init.get(key), nx * nx if key == "R" else nx, key) for key in INITIAL_KEYS})
    nU, X = int(bp["nu"]) * int(bp["N"]), nx * (int(bp["N"]) + 1)
    du, dx = mem.empty(B, k, nU), mem.empty(B, k, X)
    pu, px = mem.ptr(du), mem.ptr(dx)
    mem.run(lambda: call(t, ti, mem.kind, pu, px) if initial else call(t, mem.kind, pu, px), sync)
    return du, dx


def _gain_call(bp, B, steps, device, call, sync=None):
    """allocate Ku / Kx (numpy, or CUDA tensors on `device`), run `call(steps, Ku_ptr, Kx_ptr, memory)` and return them as
    (batch, nu*steps, nx) and (batch, nx*(steps+1), nx): the engine writes each instance's gain column-major"""
    mem = _Memory(device=device)
    nx, nu = int(bp["nx"]), int(bp["nu"])
    ku, kx = mem.empty(B, nx, max(nu * int(steps), 0)), mem.empty(B, nx, max(nx * (int(steps) + 1), 0))
    mem.run(lambda: call(int(steps), mem.ptr(ku), mem.ptr(kx), mem.kind), sync)
    return mem.rowmajor(ku), mem.rowmajor(kx)


class _Sensitivities:
    """The sensitivities of the resident solve, shared by Engine and MultiEngine.  A subclass runs its C entries through
    `_entry(memory, name, *args)` (copra_b200_<name> or copra_b200_multi_<name>, _MEM where the single-device entry takes
    the memory kind) and names its stream synchronise `_stream_sync`; `_host_only` refuses anything but HOST numpy
    arrays."""

    _host_only = False
    _stream_sync = None

    def _resident(self, name, *inputs, device=None):
        """the problem of the resident build"""
        bp = self._last_bp
        if bp is None:
            raise CopraB200Error(-5, "%s needs a previous lmpc_run / lmpc_retarget on this engine" % name)
        if self._host_only and (device is not None or any(hasattr(t, "data_ptr") for t in inputs)):
            raise CopraB200Error(-1, "the multi-device entry takes HOST numpy arrays (each shard is copied to its own device)")
        return bp

    def lmpc_vjp(self, dcontrol=None, dtrajectory=None, want=VJP_WANT):
        """Vector-Jacobian product of the last solve (copra_b200_lmpc_vjp): dcontrol (batch, nU) = dL/dcontrol and / or
        dtrajectory (batch, X) = dL/dtrajectory, numpy arrays or CUDA float64 tensors.  Returns dict(x0=(batch, nx),
        p=[per cost], f=[per row constraint, None for bounds], lower=/upper=[per bound constraint, None otherwise]), each
        gradient (batch, rows) or (batch, rows x steps) for a per-step entry, of the same kind as the cotangents; a gradient
        not in `want` is None.  Instances whose status is not 0 get zeros.
        With "w", "M" or "N" in `want` (copra_b200_lmpc_vjp_costs, the same KKT solve) it also returns w=[(batch, rows)],
        M=[(batch, rows, nx)] and N=[(batch, rows, nu)] per cost, None where a cost has no such matrix.
        With "A", "B", "d", "E" or "G" in `want` (copra_b200_lmpc_vjp_model, the same KKT solve with the forward solve as a
        second right-hand side) it also returns A=(batch, nx, nx), B=(batch, nx, nu), d=(batch, nx), and E=[(batch, rows, nx)]
        and G=[(batch, rows, nu)] per constraint, None where a constraint has no such matrix (a trajectory bound's selector
        has no gradient)."""
        bp = self._resident("lmpc_vjp", dcontrol, dtrajectory)

        def call(dc, dt, mem, o, co, mo):
            if mo is not None:
                self._entry(mem, "lmpc_vjp_model", dc, dt, _MEM, C.byref(o), co and C.byref(co), C.byref(mo))
            elif co is None:
                self._entry(mem, "lmpc_vjp", dc, dt, _MEM, C.byref(o))
            else:
                self._entry(mem, "lmpc_vjp_costs", dc, dt, _MEM, C.byref(o), C.byref(co))
        return _vjp_call(bp, int(bp["batch"]), dcontrol, dtrajectory, want, call, sync=self._stream_sync)

    def initial_state_vjp(self, dcontrol=None, dtrajectory=None, want=None):
        """Vector-Jacobian product of the last solve of an initial-state build (copra_b200_lmpc_vjp_initial_state): as
        lmpc_vjp, with R=(batch, nx, nx), r=, x0lb=, x0ub=(batch, nx) as well.  x0 receives the multipliers of the x0 bounds
        that defaulted to x0 (zeros when the build was given both x0lb and x0ub).  `want` defaults to x0, the vectors, and
        those of R, r, x0lb and x0ub the build was given; asking for one it was not given raises (E_ARG)."""
        bp = self._resident("initial_state_vjp", dcontrol, dtrajectory)
        return _vjp_call(bp, int(bp["batch"]), dcontrol, dtrajectory, initial_want(bp) if want is None else want,
                         lambda dc, dt, mem, o, io: self._entry(mem, "lmpc_vjp_initial_state", dc, dt, _MEM, C.byref(o),
                                                                C.byref(io)),
                         sync=self._stream_sync, initial=True)

    def lmpc_jvp(self, x0=None, p=None, f=None, lower=None, upper=None):
        """Jacobian-vector product of the last solve (copra_b200_lmpc_jvp) along k tangent directions: x0 (batch, k, nx) and
        lists indexed by cost (p) / constraint (f for row constraints, lower / upper for bounds) of (batch, k, len) tangents,
        len as the matching lmpc_vjp gradient; None entries are zero.  numpy arrays or CUDA float64 tensors.  Returns
        (dcontrol (batch, k, nU), dtrajectory (batch, k, X)) of the same kind.  Instances whose status is not 0 get zeros."""
        bp = self._resident("lmpc_jvp", x0, *(p or []), *(f or []), *(lower or []), *(upper or []))
        return _jvp_call(bp, int(bp["batch"]), x0, p, f, lower, upper,
                         lambda t, mem, du, dx: self._entry(mem, "lmpc_jvp", C.byref(t), _MEM, du, dx),
                         sync=self._stream_sync)

    def initial_state_jvp(self, x0=None, R=None, r=None, x0lb=None, x0ub=None, p=None, f=None, lower=None, upper=None):
        """Jacobian-vector product of the last solve of an initial-state build (copra_b200_lmpc_jvp_initial_state): as
        lmpc_jvp, with tangents R (batch, k, nx, nx), r, x0lb and x0ub (batch, k, nx) as well.  The x0 tangent moves the x0
        bounds the build was not given.  Returns (dcontrol (batch, k, nU), dtrajectory (batch, k, X))."""
        bp = self._resident("initial_state_jvp", x0, R, r, x0lb, x0ub, *(p or []), *(f or []), *(lower or []), *(upper or []))
        return _jvp_call(bp, int(bp["batch"]), x0, p, f, lower, upper,
                         lambda t, ti, mem, du, dx: self._entry(mem, "lmpc_jvp_initial_state", C.byref(t), C.byref(ti), _MEM,
                                                                du, dx),
                         sync=self._stream_sync, init=dict(R=R, r=r, x0lb=x0lb, x0ub=x0ub))

    def lmpc_feedback_gain(self, steps=1, device=None):
        """Local feedback gain of the last solve (copra_b200_lmpc_feedback_gain): (Ku (batch, nu*steps, nx) = dU[:nu*steps]/dx0,
        Kx (batch, nx*(steps+1), nx) = dtrajectory[:nx*(steps+1)]/dx0); numpy, or CUDA tensors on the torch `device`."""
        bp = self._resident("lmpc_feedback_gain", device=device)
        return _gain_call(bp, int(bp["batch"]), steps, device,
                          lambda st, ku, kx, mem: self._entry(mem, "lmpc_feedback_gain", st, ku, kx, _MEM),
                          sync=self._stream_sync)


class Engine(_Sensitivities):
    """One handle == one GPU + one stream (include/copra_b200.h)."""

    def __init__(self, device=0, stream=None, sm_limit=0, small_variant=0):
        self.lib = load()
        opt = Options()
        opt.device, opt.stream, opt.sm_limit, opt.small_variant = int(device), stream, int(sm_limit), int(small_variant)
        self.h = C.c_void_p()
        self.solve_count = 0  # solves run through this object (copra_b200.autograd detects a stale backward with it)
        self._last_bp = None  # the problem of the resident build, for the shapes of lmpc_vjp's gradients
        self._last_qp = None  # the shape (and DEVICE inputs) of the last raw QP batch, for qp_vjp
        rc = self.lib.copra_b200_create(C.byref(opt), C.byref(self.h))
        if rc != 0:
            raise CopraB200Error(rc, "copra_b200_create failed (no usable sm_100 CUDA device? there is no CPU fallback)")

    def close(self):
        if getattr(self, "h", None):
            self.lib.copra_b200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise CopraB200Error(rc, self.lib.copra_b200_last_error(self.h).decode())

    def _entry(self, memory, name, *args):
        """copra_b200_<name> on this engine, `memory` where _MEM stands"""
        self._check(getattr(self.lib, "copra_b200_" + name)(self.h, *[memory if a is _MEM else a for a in args]))

    def _call(self, mem, name, *args):
        """copra_b200_<name> on this engine's stream, ordered against torch's when `mem` is DEVICE memory"""
        mem.run(lambda: self._entry(mem.kind, name, *args), self.synchronize)

    def _stream_sync(self):
        self.synchronize()

    def set_stream(self, stream_ptr):
        self._check(self.lib.copra_b200_set_stream(self.h, C.c_void_p(stream_ptr)))

    def synchronize(self):
        self._check(self.lib.copra_b200_synchronize(self.h))

    def launch_count(self):
        return int(self.lib.copra_b200_launch_count(self.h))

    def timing(self):
        t = Timing()
        self._check(self.lib.copra_b200_last_timing(self.h, C.byref(t)))
        return {k: getattr(t, k) for k, _ in Timing._fields_}

    # ---- K1 ----
    def condense(self, A, B, d, N, want_psi=True):
        """A (batch,nx,nx) | (nx,nx), B, d -> Phi (batch,X,nx), Psi (batch,X,nU), xi (batch,X)."""
        A, B, d = np.asarray(A, float), np.asarray(B, float), np.asarray(d, float)
        batch = A.shape[0] if A.ndim == 3 else (B.shape[0] if B.ndim == 3 else (d.shape[0] if d.ndim == 2 else 1))
        nx, nu = A.shape[-1], B.shape[-1]
        X, nU = nx * (N + 1), nu * N
        keep = []

        def arr(a, base):
            buf = _colmajor(a, base)
            keep.append(buf)
            o = Array()
            o.ptr = buf.ctypes.data
            o.stride = int(np.prod(buf.shape[1:])) if a.ndim > base else 0
            return o

        Phi = np.zeros((batch, nx, X))
        xi = np.zeros((batch, X))
        Psi = np.zeros((batch, nU, X)) if want_psi else None
        self._check(self.lib.copra_b200_condense(self.h, nx, nu, N, batch, arr(A, 2), arr(B, 2), arr(d, 1),
                                                 Phi.ctypes.data, Psi.ctypes.data if want_psi else None,
                                                 xi.ctypes.data, HOST))
        return np.swapaxes(Phi, 1, 2), (np.swapaxes(Psi, 1, 2) if want_psi else None), xi

    # ---- dense assembly primitive (DMMA GEMM) ----
    def dgemm(self, A, B, Cin=None, alpha=1.0, beta=0.0, trans_a=False):
        """C = alpha * op(A) @ B + beta * Cin for arrays with a leading batch axis, logical (rows, cols) shapes."""
        A, B = np.asarray(A, float), np.asarray(B, float)
        batch = A.shape[0]
        M = A.shape[2] if trans_a else A.shape[1]
        K = A.shape[1] if trans_a else A.shape[2]
        N = B.shape[2]
        a, b = _colmajor(A, 2), _colmajor(B, 2)
        c = _colmajor(np.zeros((batch, M, N)) if Cin is None else np.asarray(Cin, float), 2).copy()
        self._check(self.lib.copra_b200_dgemm_batch(self.h, int(trans_a), M, N, K, float(alpha), a.ctypes.data, A.shape[1],
                                                    A.shape[1] * A.shape[2], b.ctypes.data, K, K * N, float(beta), c.ctypes.data, M,
                                                    M * N, batch, HOST))
        return np.swapaxes(c, 1, 2)

    # ---- K5+K6 ----
    def solve_qp_batch(self, Q, c, Aeq, beq, Aineq, bineq, lb, ub):
        """Arrays with a leading batch axis (or shared, without).  Returns dict(x, status, iters, nact, iact).  numpy arrays
        (HOST memory), or CUDA float64 tensors (DEVICE memory: the results are tensors on the same device, and the inputs are
        kept alive on this engine because qp_vjp reads them again)."""
        arrs = dict(Q=Q, c=c, Aeq=Aeq, beq=beq, Aineq=Aineq, bineq=bineq, lb=lb, ub=ub)
        mem = _Memory(*arrs.values())
        arrs = {k: None if a is None else mem.array(a) for k, a in arrs.items()}
        n = arrs["Q"].shape[-1]
        batch = 1
        for k, a in arrs.items():
            if a is not None and a.ndim > QP_BASE_NDIM[k]:
                batch = a.shape[0]

        def given(a):
            return a is not None and 0 not in a.shape
        rows = {k: int(arrs[k].shape[-2]) if given(arrs[k]) else 0 for k in ("Aeq", "Aineq")}
        meq, m = rows["Aeq"], rows["Aineq"]
        cargs = []
        for k in QP_VJP_WANT:
            a, base = arrs[k], QP_BASE_NDIM[k]
            o = Array()
            if given(a) and rows.get(k, 1) > 0:
                o.ptr = mem.buffer(a.swapaxes(-1, -2) if base == 2 else a)  # each instance column-major
                o.stride = int(np.prod(a.shape[1:])) if a.ndim > base else 0
            cargs.append(o)
        self.solve_count += 1
        self._last_qp = None
        x, iters = mem.empty(batch, n), mem.empty(batch, 2, dtype=np.int32)
        status, nact, iact = mem.empty(batch, dtype=np.int32), mem.empty(batch, dtype=np.int32), mem.empty(batch, n, dtype=np.int32)
        self._call(mem, "solve_qp_batch", n, meq, m, batch, *cargs, *[mem.ptr(a) for a in (x, status, iters, nact, iact)], _MEM)
        # DEVICE inputs are read again by qp_vjp: they stay alive until the next raw QP batch
        self._last_qp = dict(n=n, meq=meq, m=m, batch=batch, live=mem.keep if mem.device is not None else None)
        return dict(x=x, status=status, iters=iters, nact=nact, iact=iact)

    def _resident_qp(self, name):
        if getattr(self, "_last_qp", None) is None:
            raise CopraB200Error(-5, "%s needs a previous solve_qp_batch on this engine" % name)
        return self._last_qp

    def qp_vjp(self, dx, want=QP_VJP_WANT):
        """Vector-Jacobian product of the last raw QP batch (copra_b200_qp_vjp): dx (batch, n) = dL/dx, a numpy array or a
        CUDA float64 tensor.  Returns dict(Q=(batch, n, n), c=(batch, n), Aeq=(batch, meq, n), beq=(batch, meq),
        Aineq=(batch, m, n), bineq=(batch, m), lb=(batch, n), ub=(batch, n)) of the same kind as dx, per instance even for
        inputs given shared; a gradient not in `want` is None, and those of absent rows (meq or m = 0) are empty.  dQ is the
        gradient along symmetric perturbations of Q.  Instances whose status is not 0 get zeros."""
        q = self._resident_qp("qp_vjp")
        n, meq, m, B = q["n"], q["meq"], q["m"], q["batch"]
        # the engine writes each instance's matrices column-major: allocated as (batch, cols, rows)
        shapes = dict(Q=(n, n), c=(n,), Aeq=(n, meq), beq=(meq,), Aineq=(n, m), bineq=(m,), lb=(n,), ub=(n,))
        mem = _Memory(dx)
        d = mem.buffer(dx)
        raw = {k: mem.empty(B, *shapes[k]) if k in want else None for k in shapes}
        o = QpVjpOut(**{k: mem.ptr(a) for k, a in raw.items()})
        self._call(mem, "qp_vjp", d, _MEM, C.byref(o))
        return {k: mem.rowmajor(a) if a is not None and a.ndim == 3 else a for k, a in raw.items()}

    def _qp_tangents(self, tangents):
        """check raw-QP tangents against the last batch's shapes: each is (batch, k, *base) or (k, *base) (one tangent for the
        batch), every given one with the same k.  Returns (k, {name: (array, shared)}, device or None)"""
        q = self._resident_qp("qp_jvp")
        n, meq, m, B = q["n"], q["meq"], q["m"], q["batch"]
        base = dict(Q=(n, n), c=(n,), Aeq=(meq, n), beq=(meq,), Aineq=(m, n), bineq=(m,), lb=(n,), ub=(n,))
        given = {k: a for k, a in tangents.items() if a is not None}
        if not given:
            raise CopraB200Error(-1, "qp_jvp: no tangent given")
        mem = _Memory(*given.values())
        ks, out = set(), {}
        for name, a in given.items():
            a = mem.array(a)
            shape, b = tuple(a.shape), base[name]
            if len(shape) == len(b) + 2 and shape[0] == B and shape[2:] == b:
                shared = False
            elif len(shape) == len(b) + 1 and shape[1:] == b:
                shared = True
            else:
                raise CopraB200Error(-1, "qp_jvp: the %s tangent has shape %s, expected (%d, k) + %s or (k,) + %s"
                                     % (name, shape, B, b, b))
            if 0 in b:
                raise CopraB200Error(-1, "qp_jvp: a %s tangent for a batch without those rows" % name)
            ks.add(shape[0] if shared else shape[1])
            out[name] = (a, shared)
        if len(ks) != 1 or min(ks) < 1:
            raise CopraB200Error(-1, "qp_jvp: the tangents disagree on the number of directions k (%s)" % sorted(ks))
        return ks.pop(), out, mem.device

    def qp_jvp(self, Q=None, c=None, Aeq=None, beq=None, Aineq=None, bineq=None, lb=None, ub=None):
        """Jacobian-vector products of the last raw QP batch (copra_b200_qp_jvp) along k tangent directions: each tangent is
        (batch, k, *shape of the input) or (k, *shape) for one tangent shared by the batch, numpy arrays or CUDA float64
        tensors; None is a zero tangent.  Returns xdot (batch, k, n) of the same kind.  Q is read through its symmetric part.
        Instances whose status is not 0 get zeros."""
        k, ts, dev = self._qp_tangents(dict(Q=Q, c=c, Aeq=Aeq, beq=beq, Aineq=Aineq, bineq=bineq, lb=lb, ub=ub))
        q, mem = self._last_qp, _Memory(device=dev)
        t = QpJvpIn()
        t.ndir = k
        for name, (a, shared) in ts.items():
            o = getattr(t, name)
            o.ptr = mem.buffer(a.swapaxes(-1, -2) if QP_BASE_NDIM[name] == 2 else a)  # each direction column-major
            o.stride = 0 if shared else int(np.prod(a.shape[1:]))
        dx = mem.empty(q["batch"], k, q["n"])
        self._call(mem, "qp_jvp", C.byref(t), _MEM, mem.ptr(dx))
        return dx

    def qp_jacobian(self, wrt, device=None):
        """The Jacobian of the last raw QP batch's solutions with respect to one vector input (copra_b200_qp_jacobian): wrt in
        "c", "beq", "bineq", "lb", "ub".  Returns (batch, n, len) -- numpy, or a CUDA tensor on `device`.  dx/dc is symmetric;
        the columns of inactive rows are exactly zero."""
        q = self._resident_qp("qp_jacobian")
        if wrt not in QP_WRT:
            raise CopraB200Error(-1, "qp_jacobian: wrt must be one of %s, got %r" % (sorted(QP_WRT), wrt))
        n = q["n"]
        ln = dict(c=n, beq=q["meq"], bineq=q["m"], lb=n, ub=n)[wrt]
        # the engine writes each instance's n x len Jacobian column-major: allocated as (batch, len, n)
        mem = _Memory(device=device)
        J = mem.empty(q["batch"], ln, n)
        self._call(mem, "qp_jacobian", QP_WRT[wrt], mem.ptr(J), _MEM)
        return mem.rowmajor(J)

    # ---- K1..K7 ----
    def sizes(self, hb):
        s = Sizes()
        self._check(self.lib.copra_b200_lmpc_sizes(self.h, C.byref(hb.problem), C.byref(s)))
        return {k: getattr(s, k) for k, _ in Sizes._fields_}

    def lmpc_run(self, bp_or_hb, want=("control", "trajectory", "x", "status", "iters", "nact", "iact")):
        """Solve a batch problem given as a workloads dict or a prepared HostBatch (HOST memory)."""
        hb = bp_or_hb if isinstance(bp_or_hb, HostBatch) else HostBatch(bp_or_hb)
        s = self.sizes(hb)
        out, r = _result_buffers(hb.problem.batch, s, want)
        self.solve_count += 1
        self._last_bp = None
        self._check(self.lib.copra_b200_lmpc_run(self.h, C.byref(hb.problem), C.byref(r)))
        self._last_bp = hb.bp
        out["sizes"] = s
        return {k: v for k, v in out.items() if k in want or k == "sizes"}

    def last_solver(self):
        return self.lib.copra_b200_last_solver(self.h).decode()

    def hessian_is_shared(self):
        return bool(self.lib.copra_b200_hessian_is_shared(self.h))

    def fp64_peaks(self):
        """measured (DFMA, DMMA) TFLOP/s of this device"""
        a, b = C.c_double(0), C.c_double(0)
        self._check(self.lib.copra_b200_fp64_peaks(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def set_warm_start(self, on=True):
        """SI_warmStart(bool): re-solves seed the previous active sets (shared-factor thin solver only)"""
        self._check(self.lib.copra_b200_set_warm_start(self.h, 1 if on else 0))

    def warm_start(self):
        return bool(self.lib.copra_b200_get_warm_start(self.h))

    def lmpc_resolve(self, x0, sizes):
        """receding-horizon re-solve of the last built batch with new initial states x0 (batch, nx)"""
        x0 = np.ascontiguousarray(np.asarray(x0, dtype=np.float64))
        out, r = _result_buffers(x0.shape[0], sizes)
        a = Array()
        a.ptr, a.stride = x0.ctypes.data, x0.shape[1]
        self.solve_count += 1
        self._check(self.lib.copra_b200_lmpc_resolve(self.h, a, HOST, C.byref(r)))
        return out

    def lmpc_retarget(self, bp_or_hb):
        """receding-horizon step with new x0 and new vectors (p, f, lower / upper) on the resident build; the problem must
        have the resident build's shape, its matrices are ignored (copra_b200_lmpc_retarget)"""
        hb = bp_or_hb if isinstance(bp_or_hb, HostBatch) else HostBatch(bp_or_hb)
        out, r = _result_buffers(hb.problem.batch, self.sizes(hb))
        self.solve_count += 1
        self._check(self.lib.copra_b200_lmpc_retarget(self.h, C.byref(hb.problem), C.byref(r)))
        self._last_bp = hb.bp
        return out

    def lmpc_build(self, hb):
        self._last_bp = None
        self._check(self.lib.copra_b200_lmpc_build(self.h, C.byref(hb.problem)))

    def download(self, hb, what):
        """Assembled stage of the last build in logical (batch, rows, cols) shape."""
        s = self.sizes(hb)
        B, nx = hb.problem.batch, hb.problem.nx
        shapes = dict(Phi=(s["X"], nx), Psi=(s["X"], s["nU"]), xi=(s["X"],), Q=(s["nvar"], s["nvar"]), c=(s["nvar"],),
                      Aeq=(s["meq"], s["nvar"]), beq=(s["meq"],), Aineq=(s["mineq"], s["nvar"]), bineq=(s["mineq"],),
                      lb=(s["nvar"],), ub=(s["nvar"],))
        shp = shapes[what]
        if len(shp) == 2:
            buf = np.zeros((B, shp[1], shp[0]))
        else:
            buf = np.zeros((B, shp[0]))
        if buf.size:
            self._check(self.lib.copra_b200_lmpc_download(self.h, GET[what], buf.ctypes.data, HOST))
        return np.swapaxes(buf, 1, 2) if len(shp) == 2 else buf


class MultiEngine(_Sensitivities):
    """Data-parallel sharder (copra_b200_multi_*): one engine handle + host thread per listed device, the batch split
    into contiguous instance ranges, results gathered by DMA into the caller's buffers.  The sensitivity methods are
    Engine's over the shards of the last run, on HOST numpy arrays holding the whole batch."""

    _host_only = True  # each shard is copied to its own device

    def __init__(self, devices=None):
        self.lib = load()
        self.m = C.c_void_p()
        self._last_bp = None
        if devices is None:
            rc = self.lib.copra_b200_multi_create(None, 0, C.byref(self.m))
        else:
            arr = (C.c_int * len(devices))(*[int(d) for d in devices])
            rc = self.lib.copra_b200_multi_create(arr, len(devices), C.byref(self.m))
        if rc != 0:
            raise CopraB200Error(rc, "copra_b200_multi_create failed (no usable sm_100 CUDA device? there is no CPU fallback)")

    def close(self):
        if getattr(self, "m", None):
            self.lib.copra_b200_multi_destroy(self.m)
            self.m = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise CopraB200Error(rc, self.lib.copra_b200_multi_last_error(self.m).decode())

    def size(self):
        return int(self.lib.copra_b200_multi_size(self.m))

    def launch_count(self):
        return int(self.lib.copra_b200_multi_launch_count(self.m))

    def shards(self):
        out = []
        for g in range(self.size()):
            d, lo, hi = C.c_int(0), C.c_int(0), C.c_int(0)
            self._check(self.lib.copra_b200_multi_shard(self.m, g, C.byref(d), C.byref(lo), C.byref(hi)))
            out.append((d.value, lo.value, hi.value))
        return out

    def timing(self, g):
        t, w = Timing(), C.c_double(0)
        self._check(self.lib.copra_b200_multi_timing(self.m, g, C.byref(t), C.byref(w)))
        d = {k: getattr(t, k) for k, _ in Timing._fields_}
        d["wall_ms"] = w.value
        return d

    def _entry(self, memory, name, *args):
        """copra_b200_multi_<name> over the shards of the last run (HOST arrays only: the entry has no memory argument)"""
        self._check(getattr(self.lib, "copra_b200_multi_" + name)(self.m, *[a for a in args if a is not _MEM]))

    def lmpc_run(self, bp_or_hb, sizes, results=None):
        """`sizes` from Engine.sizes(); `results` an optional prepared ctypes Results (e.g. pinned torch buffers)."""
        hb = bp_or_hb if isinstance(bp_or_hb, HostBatch) else HostBatch(bp_or_hb)
        out, r = (None, results) if results is not None else _result_buffers(hb.problem.batch, sizes)
        self._check(self.lib.copra_b200_multi_lmpc_run(self.m, C.byref(hb.problem), C.byref(r)))
        self._last_bp = hb.bp
        return out

    def set_warm_start(self, on=True):
        self._check(self.lib.copra_b200_multi_set_warm_start(self.m, 1 if on else 0))

    def lmpc_retarget(self, bp_or_hb, sizes):
        """copra_b200_lmpc_retarget on every shard of the last run"""
        hb = bp_or_hb if isinstance(bp_or_hb, HostBatch) else HostBatch(bp_or_hb)
        out, r = _result_buffers(hb.problem.batch, sizes)
        self._check(self.lib.copra_b200_multi_lmpc_retarget(self.m, C.byref(hb.problem), C.byref(r)))
        return out

    def lmpc_resolve(self, x0, sizes):
        x0 = np.ascontiguousarray(np.asarray(x0, dtype=np.float64))
        out, r = _result_buffers(x0.shape[0], sizes)
        a = Array()
        a.ptr, a.stride = x0.ctypes.data, x0.shape[1]
        self._check(self.lib.copra_b200_multi_lmpc_resolve(self.m, a, C.byref(r)))
        return out
