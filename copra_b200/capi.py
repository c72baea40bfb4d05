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


class JvpIn(C.Structure):
    _fields_ = [("ndir", C.c_int), ("x0", C.c_void_p), ("p", C.POINTER(C.c_void_p)), ("f", C.POINTER(C.c_void_p)),
                ("lower", C.POINTER(C.c_void_p)), ("upper", C.POINTER(C.c_void_p))]


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
           "copra_b200_multi_lmpc_vjp_costs", "copra_b200_lmpc_vjp_model", "copra_b200_multi_lmpc_vjp_model"]
VJP_WANT = ("x0", "p", "f", "lower", "upper")
VJP_COST_WANT = ("w", "M", "N")  # gradients with respect to the cost weights and matrices: requested by name only
VJP_MODEL_WANT = ("A", "B", "d", "E", "G")  # ... and to the dynamics and the row constraints' matrices: by name only

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
        lib.copra_b200_lmpc_jvp.argtypes = [C.c_void_p, C.POINTER(JvpIn), C.c_int, C.c_void_p, C.c_void_p]
        lib.copra_b200_lmpc_feedback_gain.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        lib.copra_b200_multi_lmpc_jvp.argtypes = [C.c_void_p, C.POINTER(JvpIn), C.c_void_p, C.c_void_p]
        lib.copra_b200_multi_lmpc_feedback_gain.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
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


def _result_buffers(B, s):
    """host result arrays for B instances of sizes `s` and the Results struct pointing at them"""
    out = dict(control=np.zeros((B, s["nU"])), trajectory=np.zeros((B, s["X"])), x=np.zeros((B, s["nvar"])),
               status=np.full(B, -1, np.int32), iters=np.zeros((B, 2), np.int32), nact=np.zeros(B, np.int32),
               iact=np.zeros((B, s["nvar"]), np.int32))
    r = Results()
    r.memory = HOST
    for k, v in out.items():
        setattr(r, k, v.ctypes.data)
    return out, r


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


def _vjp_call(bp, B, dcontrol, dtrajectory, want, call, sync=None):
    """allocate the wanted gradients (numpy, or torch tensors on the device of the torch cotangents), describe them in a
    VjpOut (and, when w, M or N are wanted, a VjpCostOut; when A, B, d, E or G are, a VjpModelOut) and run
    `call(dcontrol_ptr, dtrajectory_ptr, memory, out, cost_out, model_out)`, cost_out / model_out None unless such gradients
    are wanted.  With torch tensors the engine runs on its own stream:
    the cotangents are complete before the call (device synchronise) and `sync()` waits for the engine's stream before the
    gradients (written, zero-initialised, by the engine itself) and the input copies are handed back."""
    nx, plen, clen = vjp_lengths(bp)
    dev = next((t.device for t in (dcontrol, dtrajectory) if t is not None and hasattr(t, "data_ptr")), None)
    keep = []
    if dev is not None:
        import torch

        def zeros(k):  # the engine zeroes every requested gradient on its stream
            return torch.empty((B, k), dtype=torch.float64, device=dev)

        def ptr(a):
            return a.data_ptr()

        def inp(a):
            if a is None:
                return None
            a = a.detach().to(torch.float64).contiguous()
            keep.append(a)
            return a.data_ptr()
        mem = DEVICE
    else:
        def zeros(k):
            return np.zeros((B, k))

        def ptr(a):
            return a.ctypes.data

        def inp(a):
            if a is None:
                return None
            a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
            keep.append(a)
            return a.ctypes.data
        mem = HOST
    res = dict(x0=zeros(nx) if "x0" in want else None)
    o = VjpOut()
    o.x0 = ptr(res["x0"]) if res["x0"] is not None else None
    kinds = [c["kind"] for c in bp["constraints"]]
    bound = [k in ("trajectory_bound", "control_bound") for k in kinds]
    lists = dict(p=[zeros(k) if "p" in want else None for k in plen],
                 f=[zeros(k) if "f" in want and not b else None for k, b in zip(clen, bound)],
                 lower=[zeros(k) if "lower" in want and b else None for k, b in zip(clen, bound)],
                 upper=[zeros(k) if "upper" in want and b else None for k, b in zip(clen, bound)])
    for key, arrs in lists.items():
        ptrs = (C.c_void_p * max(1, len(arrs)))(*[ptr(a) if a is not None else None for a in arrs])
        keep.append(ptrs)
        setattr(o, key, C.cast(ptrs, C.POINTER(C.c_void_p)))
        res[key] = arrs
    co = None
    if any(k in want for k in VJP_COST_WANT):
        # the engine writes M (rows x nx) and N (rows x nu) column-major: allocated as (batch, cols, rows)
        nu = int(bp["nu"])
        shapes = cost_shapes(bp)
        raw = dict(w=[zeros(r) if "w" in want else None for r, _, _ in shapes],
                   M=[zeros(nx * r).reshape(B, nx, r) if "M" in want and hm else None for r, hm, _ in shapes],
                   N=[zeros(nu * r).reshape(B, nu, r) if "N" in want and hn else None for r, _, hn in shapes])
        co = VjpCostOut()
        for key, arrs in raw.items():
            ptrs = (C.c_void_p * max(1, len(arrs)))(*[ptr(a) if a is not None else None for a in arrs])
            keep.append(ptrs)
            setattr(co, key, C.cast(ptrs, C.POINTER(C.c_void_p)))
    mo = None
    if any(k in want for k in VJP_MODEL_WANT):
        # column-major matrices again: A as (batch, nx, nx) transposed, B (batch, nu, nx), E (batch, nx, rows), G (batch, nu, rows)
        nu = int(bp["nu"])
        shapes = cstr_shapes(bp)
        mraw = dict(A=zeros(nx * nx).reshape(B, nx, nx) if "A" in want else None,
                    B=zeros(nx * nu).reshape(B, nu, nx) if "B" in want else None,
                    d=zeros(nx) if "d" in want else None,
                    E=[zeros(nx * r).reshape(B, nx, r) if "E" in want and he else None for r, he, _ in shapes],
                    G=[zeros(nu * r).reshape(B, nu, r) if "G" in want and hg else None for r, _, hg in shapes])
        mo = VjpModelOut()
        for key in ("A", "B", "d"):
            setattr(mo, key, ptr(mraw[key]) if mraw[key] is not None else None)
        for key in ("E", "G"):
            ptrs = (C.c_void_p * max(1, len(mraw[key])))(*[ptr(a) if a is not None else None for a in mraw[key]])
            keep.append(ptrs)
            setattr(mo, key, C.cast(ptrs, C.POINTER(C.c_void_p)))
    dc, dt = inp(dcontrol), inp(dtrajectory)
    if dev is not None:
        torch.cuda.synchronize(dev)
    try:
        call(dc, dt, mem, o, co, mo)
    finally:
        if dev is not None and sync is not None:
            sync()
    if co is not None:
        res["w"] = raw["w"]
        for key in ("M", "N"):
            res[key] = [None if a is None else (a.transpose(1, 2).contiguous() if dev is not None
                                                else np.ascontiguousarray(a.transpose(0, 2, 1))) for a in raw[key]]

    def logical(a):  # (batch, cols, rows) column-major -> (batch, rows, cols)
        if a is None:
            return None
        return a.transpose(1, 2).contiguous() if dev is not None else np.ascontiguousarray(a.transpose(0, 2, 1))
    if mo is not None:
        res["A"], res["B"], res["d"] = logical(mraw["A"]), logical(mraw["B"]), mraw["d"]
        res["E"], res["G"] = [logical(a) for a in mraw["E"]], [logical(a) for a in mraw["G"]]
    return res


def _jvp_call(bp, B, x0, p, f, lower, upper, call, sync=None):
    """describe the tangents (each (batch, k, len), numpy or CUDA float64 tensors; None = zero) in a JvpIn, allocate dU
    (batch, k, nU) and dtrajectory (batch, k, X) of the same kind and run `call(jvp_in, memory, dU_ptr, dX_ptr)`.  With torch
    tensors the engine runs on its own stream: the tangents are complete before the call (device synchronise) and `sync()`
    waits for the engine's stream before the results are handed back."""
    nx, plen, clen = vjp_lengths(bp)
    kinds = [c["kind"] for c in bp["constraints"]]
    bound = [kd in ("trajectory_bound", "control_bound") for kd in kinds]
    lists = dict(p=list(p or []), f=list(f or []), lower=list(lower or []), upper=list(upper or []))
    given = [x0] + [t for v in lists.values() for t in v]
    given = [t for t in given if t is not None]
    if not given:
        raise CopraB200Error(-1, "lmpc_jvp needs at least one tangent")
    k = int(given[0].shape[1]) if len(given[0].shape) == 3 else 0
    dev = next((t.device for t in given if hasattr(t, "data_ptr")), None)
    if dev is not None:
        import torch
    keep = []

    def inp(a, n, what):
        if a is None:
            return None
        if tuple(a.shape) != (B, k, n):
            raise CopraB200Error(-1, "lmpc_jvp: the %s tangent has shape %s, expected (batch, k, len) = %s"
                                 % (what, tuple(a.shape), (B, k, n)))
        if dev is not None:
            a = a.detach().to(device=dev, dtype=torch.float64).contiguous()
            keep.append(a)
            return a.data_ptr()
        if hasattr(a, "data_ptr"):
            raise CopraB200Error(-1, "lmpc_jvp: numpy and torch tangents cannot be mixed")
        a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
        keep.append(a)
        return a.ctypes.data

    t = JvpIn()
    t.ndir = k
    t.x0 = inp(x0, nx, "x0")
    lens = dict(p=plen, f=clen, lower=clen, upper=clen)
    for key, arrs in lists.items():
        n = len(plen) if key == "p" else len(clen)
        if len(arrs) > n:
            raise CopraB200Error(-1, "lmpc_jvp: %d %s tangents for %d entries" % (len(arrs), key, n))
        arrs = arrs + [None] * (n - len(arrs))
        if key != "p":
            for j, a in enumerate(arrs):
                if a is not None and bound[j] == (key == "f"):
                    raise CopraB200Error(-1, "lmpc_jvp: constraint %d has no %s vector" % (j, key))
        ptrs = (C.c_void_p * max(1, n))(*[inp(a, lens[key][j], "%s[%d]" % (key, j)) for j, a in enumerate(arrs)])
        keep.append(ptrs)
        setattr(t, key, C.cast(ptrs, C.POINTER(C.c_void_p)))
    nU, X = int(bp["nu"]) * int(bp["N"]), nx * (int(bp["N"]) + 1)
    if dev is not None:
        du = torch.empty((B, k, nU), dtype=torch.float64, device=dev)
        dx = torch.empty((B, k, X), dtype=torch.float64, device=dev)
        torch.cuda.synchronize(dev)
        ptr, mem = (lambda a: a.data_ptr()), DEVICE
    else:
        du, dx = np.zeros((B, k, nU)), np.zeros((B, k, X))
        ptr, mem = (lambda a: a.ctypes.data), HOST
    try:
        call(t, mem, ptr(du), ptr(dx))
    finally:
        if dev is not None and sync is not None:
            sync()
    return du, dx


def _gain_call(bp, B, steps, device, call, sync=None):
    """allocate Ku / Kx (numpy, or CUDA tensors on `device`), run `call(steps, Ku_ptr, Kx_ptr, memory)` and return them as
    (batch, nu*steps, nx) and (batch, nx*(steps+1), nx): the engine writes each instance's gain column-major"""
    nx, nu = int(bp["nx"]), int(bp["nu"])
    ru, rx = nu * int(steps), nx * (int(steps) + 1)
    if device is not None:
        import torch
        ku = torch.empty((B, nx, max(ru, 0)), dtype=torch.float64, device=device)
        kx = torch.empty((B, nx, max(rx, 0)), dtype=torch.float64, device=device)
        torch.cuda.synchronize(device)
        try:
            call(int(steps), ku.data_ptr(), kx.data_ptr(), DEVICE)
        finally:
            if sync is not None:
                sync()
        return ku.transpose(1, 2).contiguous(), kx.transpose(1, 2).contiguous()
    ku, kx = np.zeros((B, nx, max(ru, 0))), np.zeros((B, nx, max(rx, 0)))
    call(int(steps), ku.ctypes.data, kx.ctypes.data, HOST)
    return np.ascontiguousarray(ku.transpose(0, 2, 1)), np.ascontiguousarray(kx.transpose(0, 2, 1))


class Engine:
    """One handle == one GPU + one stream (include/copra_b200.h)."""

    def __init__(self, device=0, stream=None, sm_limit=0, small_variant=0):
        self.lib = load()
        opt = Options()
        opt.device, opt.stream, opt.sm_limit, opt.small_variant = int(device), stream, int(sm_limit), int(small_variant)
        self.h = C.c_void_p()
        self.solve_count = 0  # solves run through this object (copra_b200.autograd detects a stale backward with it)
        self._last_bp = None  # the problem of the resident build, for the shapes of lmpc_vjp's gradients
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
        """Arrays with a leading batch axis (or shared, without).  Returns dict(x, status, iters, nact, iact)."""
        Q = np.asarray(Q, float)
        n = Q.shape[-1]
        arrs = dict(Q=(Q, 2), c=(c, 1), Aeq=(Aeq, 2), beq=(beq, 1), Aineq=(Aineq, 2), bineq=(bineq, 1), lb=(lb, 1), ub=(ub, 1))
        batch = 1
        for k, (a, base) in arrs.items():
            if a is not None and np.asarray(a).ndim > base:
                batch = np.asarray(a).shape[0]
        meq = 0 if Aeq is None else np.asarray(Aeq).reshape(-1, np.asarray(Aeq).shape[-2], n).shape[1]
        m = 0 if Aineq is None else np.asarray(Aineq).reshape(-1, np.asarray(Aineq).shape[-2], n).shape[1]
        keep, cargs = [], []
        for k in ("Q", "c", "Aeq", "beq", "Aineq", "bineq", "lb", "ub"):
            a, base = arrs[k]
            o = Array()
            if a is not None and np.asarray(a).size > 0:
                a = np.asarray(a, float)
                buf = _colmajor(a, base)
                keep.append(buf)
                o.ptr = buf.ctypes.data
                o.stride = int(np.prod(buf.shape[1:])) if a.ndim > base else 0
            cargs.append(o)
        x = np.zeros((batch, n))
        status, iters = np.zeros(batch, np.int32), np.zeros((batch, 2), np.int32)
        nact, iact = np.zeros(batch, np.int32), np.zeros((batch, n), np.int32)
        self._check(self.lib.copra_b200_solve_qp_batch(self.h, n, meq, m, batch, *cargs, x.ctypes.data, status.ctypes.data,
                                                       iters.ctypes.data, nact.ctypes.data, iact.ctypes.data, HOST))
        return dict(x=x, status=status, iters=iters, nact=nact, iact=iact)

    # ---- K1..K7 ----
    def sizes(self, hb):
        s = Sizes()
        self._check(self.lib.copra_b200_lmpc_sizes(self.h, C.byref(hb.problem), C.byref(s)))
        return {k: getattr(s, k) for k, _ in Sizes._fields_}

    def lmpc_run(self, bp_or_hb, want=("control", "trajectory", "x", "status", "iters", "nact", "iact")):
        """Solve a batch problem given as a workloads dict or a prepared HostBatch (HOST memory)."""
        hb = bp_or_hb if isinstance(bp_or_hb, HostBatch) else HostBatch(bp_or_hb)
        s = self.sizes(hb)
        B = hb.problem.batch
        out = dict(control=np.zeros((B, s["nU"])), trajectory=np.zeros((B, s["X"])), x=np.zeros((B, s["nvar"])),
                   status=np.full(B, -1, np.int32), iters=np.zeros((B, 2), np.int32), nact=np.zeros(B, np.int32),
                   iact=np.zeros((B, s["nvar"]), np.int32))
        r = Results()
        r.memory = HOST
        for k in want:
            setattr(r, k, out[k].ctypes.data)
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
        B = x0.shape[0]
        out = dict(control=np.zeros((B, sizes["nU"])), trajectory=np.zeros((B, sizes["X"])), x=np.zeros((B, sizes["nvar"])),
                   status=np.full(B, -1, np.int32), iters=np.zeros((B, 2), np.int32), nact=np.zeros(B, np.int32),
                   iact=np.zeros((B, sizes["nvar"]), np.int32))
        r = Results()
        r.memory = HOST
        for k, v in out.items():
            setattr(r, k, v.ctypes.data)
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
        if self._last_bp is None:
            raise CopraB200Error(-5, "lmpc_vjp needs a previous lmpc_run / lmpc_retarget on this engine")
        bp = self._last_bp

        def call(dc, dt, mem, o, co, mo):
            if mo is not None:
                self._check(self.lib.copra_b200_lmpc_vjp_model(self.h, dc, dt, mem, C.byref(o), co and C.byref(co),
                                                               C.byref(mo)))
            elif co is None:
                self._check(self.lib.copra_b200_lmpc_vjp(self.h, dc, dt, mem, C.byref(o)))
            else:
                self._check(self.lib.copra_b200_lmpc_vjp_costs(self.h, dc, dt, mem, C.byref(o), C.byref(co)))
        return _vjp_call(bp, int(bp["batch"]), dcontrol, dtrajectory, want, call, sync=self.synchronize)

    def lmpc_jvp(self, x0=None, p=None, f=None, lower=None, upper=None):
        """Jacobian-vector product of the last solve (copra_b200_lmpc_jvp) along k tangent directions: x0 (batch, k, nx) and
        lists indexed by cost (p) / constraint (f for row constraints, lower / upper for bounds) of (batch, k, len) tangents,
        len as the matching lmpc_vjp gradient; None entries are zero.  numpy arrays or CUDA float64 tensors.  Returns
        (dcontrol (batch, k, nU), dtrajectory (batch, k, X)) of the same kind.  Instances whose status is not 0 get zeros."""
        if self._last_bp is None:
            raise CopraB200Error(-5, "lmpc_jvp needs a previous lmpc_run / lmpc_retarget on this engine")
        bp = self._last_bp
        return _jvp_call(bp, int(bp["batch"]), x0, p, f, lower, upper,
                         lambda t, mem, du, dx: self._check(self.lib.copra_b200_lmpc_jvp(self.h, C.byref(t), mem, du, dx)),
                         sync=self.synchronize)

    def lmpc_feedback_gain(self, steps=1, device=None):
        """Local feedback gain of the last solve (copra_b200_lmpc_feedback_gain): (Ku (batch, nu*steps, nx) = dU[:nu*steps]/dx0,
        Kx (batch, nx*(steps+1), nx) = dtrajectory[:nx*(steps+1)]/dx0); numpy, or CUDA tensors on the torch `device`."""
        if self._last_bp is None:
            raise CopraB200Error(-5, "lmpc_feedback_gain needs a previous lmpc_run / lmpc_retarget on this engine")
        bp = self._last_bp
        return _gain_call(bp, int(bp["batch"]), steps, device,
                          lambda st, ku, kx, mem: self._check(self.lib.copra_b200_lmpc_feedback_gain(self.h, st, ku, kx, mem)),
                          sync=self.synchronize)

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


class MultiEngine:
    """Data-parallel sharder (copra_b200_multi_*): one engine handle + host thread per listed device, the batch split
    into contiguous instance ranges, results gathered by DMA into the caller's buffers."""

    def __init__(self, devices=None):
        self.lib = load()
        self.m = C.c_void_p()
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

    @staticmethod
    def _outputs(B, s):
        return dict(control=np.zeros((B, s["nU"])), trajectory=np.zeros((B, s["X"])), x=np.zeros((B, s["nvar"])),
                    status=np.full(B, -1, np.int32), iters=np.zeros((B, 2), np.int32), nact=np.zeros(B, np.int32),
                    iact=np.zeros((B, s["nvar"]), np.int32))

    def lmpc_run(self, bp_or_hb, sizes, results=None):
        """`sizes` from Engine.sizes(); `results` an optional prepared ctypes Results (e.g. pinned torch buffers)."""
        hb = bp_or_hb if isinstance(bp_or_hb, HostBatch) else HostBatch(bp_or_hb)
        if results is not None:
            self._check(self.lib.copra_b200_multi_lmpc_run(self.m, C.byref(hb.problem), C.byref(results)))
            self._last_bp = hb.bp
            return None
        out = self._outputs(hb.problem.batch, sizes)
        r = Results()
        r.memory = HOST
        for k, v in out.items():
            setattr(r, k, v.ctypes.data)
        self._check(self.lib.copra_b200_multi_lmpc_run(self.m, C.byref(hb.problem), C.byref(r)))
        self._last_bp = hb.bp
        return out

    def lmpc_vjp(self, dcontrol=None, dtrajectory=None, want=VJP_WANT):
        """Engine.lmpc_vjp over the shards of the last run (numpy arrays holding the whole batch)"""
        bp = getattr(self, "_last_bp", None)
        if bp is None:
            raise CopraB200Error(-5, "lmpc_vjp needs a previous lmpc_run on this engine")
        if any(hasattr(t, "data_ptr") for t in (dcontrol, dtrajectory)):
            raise CopraB200Error(-1, "the multi-device entry takes HOST numpy arrays (each shard is copied to its own device)")

        def call(dc, dt, mem, o, co, mo):
            if mo is not None:
                self._check(self.lib.copra_b200_multi_lmpc_vjp_model(self.m, dc, dt, C.byref(o), co and C.byref(co),
                                                                     C.byref(mo)))
            elif co is None:
                self._check(self.lib.copra_b200_multi_lmpc_vjp(self.m, dc, dt, C.byref(o)))
            else:
                self._check(self.lib.copra_b200_multi_lmpc_vjp_costs(self.m, dc, dt, C.byref(o), C.byref(co)))
        return _vjp_call(bp, int(bp["batch"]), dcontrol, dtrajectory, want, call)

    def lmpc_jvp(self, x0=None, p=None, f=None, lower=None, upper=None):
        """Engine.lmpc_jvp over the shards of the last run (numpy arrays holding the whole batch)"""
        bp = getattr(self, "_last_bp", None)
        if bp is None:
            raise CopraB200Error(-5, "lmpc_jvp needs a previous lmpc_run on this engine")
        tangents = [x0] + list(p or []) + list(f or []) + list(lower or []) + list(upper or [])
        if any(hasattr(t, "data_ptr") for t in tangents):
            raise CopraB200Error(-1, "the multi-device entry takes HOST numpy arrays (each shard is copied to its own device)")
        return _jvp_call(bp, int(bp["batch"]), x0, p, f, lower, upper,
                         lambda t, mem, du, dx: self._check(self.lib.copra_b200_multi_lmpc_jvp(self.m, C.byref(t), du, dx)))

    def lmpc_feedback_gain(self, steps=1):
        """Engine.lmpc_feedback_gain over the shards of the last run (numpy arrays holding the whole batch)"""
        bp = getattr(self, "_last_bp", None)
        if bp is None:
            raise CopraB200Error(-5, "lmpc_feedback_gain needs a previous lmpc_run on this engine")
        return _gain_call(bp, int(bp["batch"]), steps, None,
                          lambda st, ku, kx, mem: self._check(self.lib.copra_b200_multi_lmpc_feedback_gain(self.m, st, ku, kx)))

    def set_warm_start(self, on=True):
        rc = self.lib.copra_b200_multi_set_warm_start(self.m, 1 if on else 0)
        if rc:
            raise CopraB200Error("copra_b200_multi_set_warm_start failed (%d)" % rc)

    def lmpc_retarget(self, bp_or_hb, sizes):
        """copra_b200_lmpc_retarget on every shard of the last run"""
        hb = bp_or_hb if isinstance(bp_or_hb, HostBatch) else HostBatch(bp_or_hb)
        out, r = _result_buffers(hb.problem.batch, sizes)
        self._check(self.lib.copra_b200_multi_lmpc_retarget(self.m, C.byref(hb.problem), C.byref(r)))
        return out

    def lmpc_resolve(self, x0, sizes):
        x0 = np.ascontiguousarray(np.asarray(x0, dtype=np.float64))
        out = self._outputs(x0.shape[0], sizes)
        r = Results()
        r.memory = HOST
        for k, v in out.items():
            setattr(r, k, v.ctypes.data)
        a = Array()
        a.ptr, a.stride = x0.ctypes.data, x0.shape[1]
        self._check(self.lib.copra_b200_multi_lmpc_resolve(self.m, a, C.byref(r)))
        return out
