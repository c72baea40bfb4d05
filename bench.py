#!/usr/bin/env python
"""bench.py -- batched LMPC solves/sec (build + QP) on B200, the metric BASELINE.json names.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c3] [--batch B] [--impl reference] [--dump-outputs DIR]

Default workload = BASELINE.json configs[2], the one its metric is quoted on: C3, the walking CoM preview (3rd-order LIPM,
6 states / 2 jerk controls, horizon 160, ZMP mixed inequalities), batch 16384, STRONG-scaled: at N GPUs (one process per GPU
under torchrun) rank r owns the contiguous instance range [r*ceil(B/N), (r+1)*ceil(B/N)) of the SAME 16384 instances.
A *step* is one pass of the hot path (K1 condense -> K2-K4 assemble -> K5/K6 Goldfarb-Idnani solve -> K7 rollout) over that
batch.  There is no collective on the hot path; the only cross-GPU traffic is the final gather of results / timings.

`value`  : whole-job solves/s with the per-instance parameters already resident in HBM, CUDA events per step on the
           launching stream (L2 flushed between steps), max over ranks.
`e2e`    : the same metric through the C ABI with pinned HOST parameter buffers: every step uploads its shard's parameters
           (H2D), runs K1..K7 and gathers control / trajectory / status of ALL instances into rank 0's pinned host buffer
           (N > 1: NCCL gather over NVLink to rank 0's device, then one D2H) inside the timed region.
`roofline`, `cpu_baseline`, `other_configs`: see DESIGN.md "Measurement".
`--impl reference` times the CPU restatement (oracle port) of copra's Eigen + eigen-quadprog path -- the reference itself
cannot be built offline -- on all host threads of this process's affinity mask, same config / metric.
`--dump-outputs DIR` writes what the last timed step returned to the caller (see dump_sample) as DIR/<name>.npy, so that
two builds can be compared output for output: the workloads are seeded, so the same arguments give the same inputs.
"""
import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from copra_b200 import workloads as wl  # noqa: E402

METRIC = "batched LMPC solves/sec (build+QP)"
UNIT = "solves/s"
DEFAULT_BATCH = dict(c1=1, c2=4096, c3=16384, c4=8192, c5=1024)
WORKLOAD_NAME = dict(
    c1="C1: single double-integrator LMPC (tests/systems.h BoundedSystem, N=300), batch 1",
    c2="C2: batch 4096 double-integrator LMPCs, horizon 50, trajectory/control bounds, FP64",
    c3="C3: walking CoM preview (3rd-order LIPM, 6 states/2 jerk controls, horizon 160, ZMP mixed inequalities), "
       "batch 16384 sharded by instance index",
    c4="C4: InitialStateLMPC on the double integrator, target + control costs, batch 8192",
    c5="C5: condensing stress nx=12 nu=4 horizon 200, batch 1024")
# seconds of one oracle solve on one host core (sizing of the bounded CPU samples)
CPU_SECONDS_PER_INSTANCE = dict(c1=0.06, c2=0.0008, c3=0.18, c4=0.0012, c5=1.5)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def shape_of(bp):
    """sizes of one instance's QP without touching a GPU (mirrors copra_b200_lmpc_sizes)"""
    nx, nu, N = bp["nx"], bp["nu"], bp["N"]
    n = nu * N + (nx if bp.get("initial_state") else 0)
    meq = m = 0
    for c in bp["constraints"]:
        k = c["kind"]
        if k == "control_bound":
            continue
        if k == "trajectory_bound":
            lo, up = np.asarray(c["lower"]), np.asarray(c["upper"])
            lo, up = (lo[0], up[0]) if lo.ndim > 1 else (lo, up)
            rows = (int(np.isfinite(lo).sum()) + int(np.isfinite(up).sum())) * (N + 1)
        else:
            r = int(np.asarray(c["f"]).shape[-1])
            rows = r * (N + 1 if k == "trajectory" else N)
        if c.get("is_ineq", True):
            m += rows
        else:
            meq += rows
    return dict(nvar=n, meq=meq, mineq=m, q=meq + m + 2 * n, X=nx * (N + 1), nU=nu * N)


def config_dict(config, bp, total_batch, world):
    """identical in the b200 and the reference arm, so the driver can pair the two lines"""
    sz = shape_of(bp)
    return dict(workload=WORKLOAD_NAME[config], config=config, batch=total_batch, nx=bp["nx"], nu=bp["nu"], horizon=bp["N"],
                n_vars=sz["nvar"], n_ineq_rows=sz["mineq"], n_eq_rows=sz["meq"], q_rows=sz["q"],
                parallelism="instance-sharded x%d (contiguous index ranges), no collective on the hot path" % world,
                l2="flushed between timed steps (256 MiB fill)")


def k6_algorithmic_bytes(sz):
    n, meq, m, q = sz["nvar"], sz["meq"], sz["mineq"], sz["q"]
    return 8 * (n * n + n + (meq + m) * n + (meq + m) + 2 * n) + 8 * n + 4 * q + 12


def k6_algorithmic_flops(sz, iters):
    """F_alg = 2/3 n^3 + I (10 n^2 + 2 n q), I = outer iterations (SURVEY.md 8d / BASELINE.md section 4); vectorised"""
    n, q = sz["nvar"], sz["q"]
    return (2.0 / 3.0) * n ** 3 + np.asarray(iters, dtype=np.float64) * (10.0 * n * n + 2.0 * n * q)


def k6_executed_flops(sz, iters, drops, nact, thin, shared_hessian, batch, shape=None):
    """flops the solver kernels actually issue (estimate from the per-instance iteration / drop / active counts), with
    a = mean active count ~ nact / 2.
    thin solver, general form (per-instance factors: C5): per step-direction pass two triangular mat-vecs (2 n^2), the
    projections on Q1 (4 n a), r = S d1 (2 a^2); per outer iteration the Toeplitz products (m n); per drop two more passes over
    Q1 and S; the factorisation (n^3: Cholesky + inverse) once per DISTINCT Hessian.
    thin solver, shared-factor form (batch-invariant system and Hessian: C3): per pass d1 = P'a over the causal support (n a),
    w = P d1 (2 n a), r = S d1 (2 a^2) and the nx + nu column reads of h (2 (nx + nu) n) -- no mat-vec with the factor; per outer
    iteration the state-space products (2 N nx (L nu / 2 + nx) + 2 m (nx + nu)); one factorisation and three n x n x X GEMMs
    per batch.
    dense solvers (gi_small / cluster / general): the algorithmic count with the implicit bound rows removed."""
    n, m, meq = sz["nvar"], sz["mineq"], sz["meq"]
    it, dr, na = (np.asarray(v, dtype=np.float64) for v in (iters, drops, nact))
    if thin:
        a = 0.5 * na
        if shared_hessian and shape is not None:
            nx, nu, N, X = shape
            per_pass = 3.0 * n * a + 2.0 * a * a + 2.0 * (nx + nu) * n
            prod = 2.0 * N * nx * (8.0 * nu + nx) + 2.0 * (m + meq) * (nx + nu)
            per = (it + dr) * per_pass + it * prod + dr * (4.0 * n * a + 4.0 * a * a)
            return float(per.sum() + float(n) ** 3 + 3.0 * 2.0 * n * n * X)
        per = (it + dr) * (2.0 * n * n + 4.0 * n * a + 2.0 * a * a) + it * (1.0 * (m + meq) * n) + dr * (4.0 * n * a + 4.0 * a * a)
        fac = float(n) ** 3 * (1.0 if shared_hessian else batch)
        return float(per.sum() + fac)
    per = (2.0 / 3.0) * n ** 3 + it * (10.0 * n * n + 2.0 * n * (m + meq))
    return float(per.sum())


FP64_NOMINAL_TFLOPS = 37.0  # nominal B200 FP64 (vector == tensor); MEASURED_PEAKS.json has no FP64 entry: measured live

# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel from the committed `ncu --set full`
# captures under profiles/ (only valid for that exact workload / batch)
NCU_TRAFFIC = {}
try:
    NCU_TRAFFIC = {tuple(k.split(":")): v for k, v in json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).items()}
except Exception:
    pass


class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu)], stdout=open(self.path, "w"),
                                         stderr=subprocess.DEVNULL)
            atexit.register(self.kill)  # an exception before stop() must not leave the sampler running
        except Exception:
            self.proc = None

    def kill(self):
        if self.proc is not None and self.proc.poll() is None:
            self.proc.kill()
            self.proc.wait()

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        try:
            rows = [r.strip().split(", ") for r in open(self.path) if r.strip()]
            os.unlink(self.path)
            sm = [float(r[1]) for r in rows if len(r) >= 9]
            power = [float(r[3]) for r in rows if len(r) >= 9]
            if sm:
                # "under load": samples in the upper half of the power range
                thr = (min(power) + max(power)) / 2.0 if max(power) - min(power) > 50 else -1
                load = [s for s, p in zip(sm, power) if p >= thr] or sm
                out["sm_mhz"] = statistics.median(load)
                out["sm_max_mhz"] = float(rows[0][2])
                out["samples"] = len(sm)
                out["power_w_max"] = max(power)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for k, nm in enumerate(names):
                    if any(r[5 + k].strip().lower().startswith("active") for r in rows if len(r) >= 9):
                        out["reasons"].append(nm)
        except Exception:
            pass
        return out


def make_full_batch(config, batch):
    fn = wl.CONFIGS[config]
    return fn() if config == "c1" else fn(batch=batch, seed_offset=0)


def cpu_sample(bp, max_instances, reps=3, threads=None):
    """oracle port on the host cores, one instance per thread"""
    from oracle import pyoracle as po
    n = min(bp["batch"], max_instances)
    probs = [wl.instance(bp, i) for i in range(n)]
    best = None
    for _ in range(reps):
        r = po.lmpc_batch(probs, threads=threads)
        if best is None or r["wall"] < best["wall"]:
            best = r
    return dict(value=n / best["wall"], cores=best["threads"], n=n, wall=best["wall"],
                p50_ms=float(np.median(best["t_inst"]) * 1e3), ok=int((best["fail"] == 0).sum()))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    config = args.config
    batch = args.batch or DEFAULT_BATCH[config]
    bp = make_full_batch(config, min(batch, 4096) if config != "c1" else 1)
    from oracle import pyoracle as po
    cores = po.hw_threads()
    # bounded sample: the whole --steps/--warmup run stays within a few minutes of CPU time
    per_inst = CPU_SECONDS_PER_INSTANCE[config]
    budget_s = 150.0
    sample = int(budget_s * cores / per_inst / max(1, args.steps + args.warmup))
    sample = max(cores, min(sample, bp["batch"], 2048))
    sample = 1 if config == "c1" else sample
    probs = [wl.instance(bp, i) for i in range(sample)]
    for _ in range(args.warmup):
        po.lmpc_batch(probs)
    times = []
    for _ in range(args.steps):
        r = po.lmpc_batch(probs)
        times.append(r["wall"])
    t = sum(times)
    value = sample * args.steps / t
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * t / args.steps, higher_is_better=True, scaling="strong", vs_baseline=None,
                dtype="f64", data="synthetic", impl="reference",
                config=config_dict(config, bp, batch, args.gpus),
                cpu_baseline=dict(value=value, unit=UNIT, cores=cores, kind="port",
                                  sample="%d instances of %s per step, one instance per host thread (%d threads = "
                                         "sched_getaffinity); CPU restatement (oracle port) of copra's Eigen + eigen-quadprog "
                                         "path, the reference itself cannot be built offline" % (sample, config, cores)),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))
    return 0


class Runner:
    """One rank's engine, device-resident and pinned-host copies of its shard, result buffers and the two step kinds."""

    def __init__(self, torch, capi, dev, local, bp, stream):
        import ctypes as C
        self.torch, self.capi, self.C = torch, capi, C
        self.dev, self.bp = dev, bp
        self.batch = bp["batch"]
        self.eng = capi.Engine(local, stream=stream.cuda_stream)
        self.hb_dev = capi.HostBatch(bp, device_tensors=dev)
        self.hb_dev.problem.flags |= capi.FLAG_STABLE_BOUND_PATTERN  # the resident inputs are never rewritten
        self.hb_host = capi.HostBatch(bp, pin=True)
        self.sz = self.eng.sizes(self.hb_dev)
        sz, b = self.sz, self.batch
        self.d_control = torch.empty(b * sz["nU"], dtype=torch.float64, device=dev)
        self.d_traj = torch.empty(b * sz["X"], dtype=torch.float64, device=dev)
        self.d_status = torch.empty(b, dtype=torch.int32, device=dev)
        self.d_iters = torch.empty(2 * b, dtype=torch.int32, device=dev)
        self.d_nact = torch.empty(b, dtype=torch.int32, device=dev)
        self.d_iact = torch.empty(b * sz["nvar"], dtype=torch.int32, device=dev)
        rd = capi.Results()
        rd.memory = capi.DEVICE
        rd.control, rd.trajectory, rd.status = self.d_control.data_ptr(), self.d_traj.data_ptr(), self.d_status.data_ptr()
        rd.iters, rd.nact, rd.iact = self.d_iters.data_ptr(), self.d_nact.data_ptr(), self.d_iact.data_ptr()
        self.rd = rd
        self.lib = self.eng.lib

    def host_results(self, total):
        """pinned host result buffers for `total` instances (rank 0 holds the whole job's)"""
        torch, sz = self.torch, self.sz
        self.h_control = torch.empty(total * sz["nU"], dtype=torch.float64).pin_memory()
        self.h_traj = torch.empty(total * sz["X"], dtype=torch.float64).pin_memory()
        self.h_status = torch.empty(total, dtype=torch.int32).pin_memory()
        rh = self.capi.Results()
        rh.memory = self.capi.HOST
        rh.control, rh.trajectory, rh.status = self.h_control.data_ptr(), self.h_traj.data_ptr(), self.h_status.data_ptr()
        self.rh = rh
        return self.h_control.numel() * 8 + self.h_traj.numel() * 8 + self.h_status.numel() * 4

    def step_device(self):
        rc = self.lib.copra_b200_lmpc_run(self.eng.h, self.C.byref(self.hb_dev.problem), self.C.byref(self.rd))
        if rc:
            self.eng._check(rc)

    def step_host_to_host(self):
        rc = self.lib.copra_b200_lmpc_run(self.eng.h, self.C.byref(self.hb_host.problem), self.C.byref(self.rh))
        if rc:
            self.eng._check(rc)

    def step_host_to_device(self):
        rc = self.lib.copra_b200_lmpc_run(self.eng.h, self.C.byref(self.hb_host.problem), self.C.byref(self.rd))
        if rc:
            self.eng._check(rc)

    def close(self):
        self.eng.close()


DUMP_BYTES = 64 * 1000 * 1000


def dump_sample(run):
    """float64 host copies of the result arrays copra_b200_lmpc_run filled in its last call (control, trajectory, status,
    iters, nact, iact) for a fixed seeded sample of instances, small enough that the .npy files stay under DUMP_BYTES;
    `instance` holds the sampled instance indices"""
    torch, b = run.torch, run.batch
    bufs = dict(control=run.d_control, trajectory=run.d_traj, status=run.d_status, iters=run.d_iters, nact=run.d_nact,
                iact=run.d_iact)
    per_instance = 8 * (1 + sum(t.numel() // b for t in bufs.values()))
    keep = min(b, (DUMP_BYTES - 128 * (len(bufs) + 1)) // per_instance)  # 128: header of one .npy file
    idx = np.arange(b) if keep == b else np.sort(np.random.default_rng(0).choice(b, keep, replace=False))
    sel = torch.from_numpy(idx).to(run.dev)
    out = dict(instance=idx.astype(np.float64))
    for name, t in bufs.items():
        a = t.view(b, -1).index_select(0, sel).to(torch.float64).cpu().numpy()
        out[name] = a[:, 0] if a.shape[1] == 1 else a
    return out


def time_value(torch, runner, stream, flush, steps, barrier):
    """K timed steps, CUDA events on the launching stream, L2 flushed between steps; per-stage times of every step"""
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    stage = dict(condense_ms=0.0, assemble_ms=0.0, solve_ms=0.0, rollout_ms=0.0)
    barrier()
    wall0 = time.perf_counter()
    for k in range(steps):
        flush.fill_(k & 0xFF)
        starts[k].record(stream)
        runner.step_device()
        stops[k].record(stream)
        tm = runner.eng.timing()  # the library's own CUDA events of this step (synchronises the stream)
        for key in stage:
            stage[key] += tm[key] / steps
    barrier()
    wall1 = time.perf_counter()
    step_ms = [s.elapsed_time(e) for s, e in zip(starts, stops)]
    return step_ms, stage, wall1 - wall0


def measure_single(torch, capi, dev, local, stream, flush, config, batch, steps, warmup, resolve=False):
    """one secondary configuration on ONE GPU: device-resident value, host-buffer e2e, stage split"""
    bp = make_full_batch(config, batch)
    r = Runner(torch, capi, dev, local, bp, stream)
    try:
        d2h = r.host_results(bp["batch"])
        for _ in range(warmup):
            r.step_device()
        torch.cuda.synchronize()
        ok = int((r.d_status == 0).sum().item())
        step_ms, stage, _ = time_value(torch, r, stream, flush, steps, torch.cuda.synchronize)
        r.step_host_to_host()
        torch.cuda.synchronize()
        e0 = time.perf_counter()
        for _ in range(steps):
            r.step_host_to_host()
        torch.cuda.synchronize()
        e1 = time.perf_counter()
        it = r.d_iters.view(-1, 2).cpu().numpy()
        out = dict(workload=WORKLOAD_NAME[config], batch=bp["batch"], steps=steps, value=bp["batch"] * steps / (sum(step_ms) * 1e-3),
                   unit=UNIT, ms_per_step=sum(step_ms) / steps, p50_ms_per_batch=float(np.median(step_ms)),
                   e2e=dict(value=bp["batch"] * steps / (e1 - e0), unit=UNIT, h2d_bytes_per_step=r.hb_host.h2d_bytes,
                            d2h_bytes_per_step=d2h),
                   stage_ms=stage, solved_ok=ok, mean_outer_iterations=float(it[:, 0].mean()), mean_drops=float(it[:, 1].mean()),
                   n_vars=r.sz["nvar"], n_ineq_rows=r.sz["mineq"])
        if resolve and not bp.get("initial_state"):
            # receding-horizon re-solve (SURVEY 8f N1): new x0 on the resident build -- K4 + K5..K7 with the cached factor
            import ctypes as C
            x0 = torch.from_numpy(np.ascontiguousarray(np.asarray(bp["x0"], dtype=np.float64) * 0.97)).to(dev)
            a = capi.Array()
            a.ptr, a.stride = x0.data_ptr(), bp["nx"]
            r.step_device()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            times = []
            for _ in range(steps):
                flush.fill_(3)
                ev0.record(stream)
                rc = r.lib.copra_b200_lmpc_resolve(r.eng.h, a, capi.DEVICE, C.byref(r.rd))
                if rc:
                    r.eng._check(rc)
                ev1.record(stream)
                torch.cuda.synchronize()
                times.append(ev0.elapsed_time(ev1))
            out["resolve"] = dict(value=bp["batch"] * steps / (sum(times) * 1e-3), unit=UNIT, ms_per_step=sum(times) / steps,
                                  ratio_to_full_step=(sum(times) / steps) / out["ms_per_step"],
                                  solved_ok=int((r.d_status == 0).sum().item()),
                                  note="copra_b200_lmpc_resolve: x0 * 0.97, condensing / Q / factor reused")
            if "thin" in r.eng.last_solver() and r.eng.hessian_is_shared():
                # the same re-solve with SI_warmStart(true): seeded with the previous active sets
                r.eng.set_warm_start(True)
                r.step_device()
                times, its = [], None
                for _ in range(steps):
                    flush.fill_(3)
                    ev0.record(stream)
                    rc = r.lib.copra_b200_lmpc_resolve(r.eng.h, a, capi.DEVICE, C.byref(r.rd))
                    if rc:
                        r.eng._check(rc)
                    ev1.record(stream)
                    torch.cuda.synchronize()
                    times.append(ev0.elapsed_time(ev1))
                    if its is None:
                        its = r.d_iters.view(-1, 2).cpu().numpy()
                    r.step_device()  # the seed of the next timed re-solve is again the solve at the original x0
                r.eng.set_warm_start(False)
                out["resolve_warm"] = dict(value=bp["batch"] * steps / (sum(times) * 1e-3), unit=UNIT, ms_per_step=sum(times) / steps,
                                           ratio_to_full_step=(sum(times) / steps) / out["ms_per_step"],
                                           solved_ok=int((r.d_status == 0).sum().item()),
                                           mean_iterations_after_seed=float(its[:, 0].mean()),
                                           note="copra_b200_set_warm_start(1) + copra_b200_lmpc_resolve: x0 * 0.97, seeded with the "
                                                "active sets of the previous solve (same optimum; opt-in, QuadProg itself has no warm start)")
        return out
    finally:
        r.close()


def c1_raw_qp_latency(torch, capi, local, stream, reps=30):
    """C1 through the raw-QP entry B200Solver::SI_solve binds to (copra_b200_solve_qp_batch, batch 1, HOST arrays: the
    1.45 MB H2D of Q / Aineq is inside the call); p50 wall latency"""
    from oracle import pyoracle as po
    bp = wl.c1()
    o = po.lmpc(wl.instance(bp, 0), solve=False)
    eng = capi.Engine(local, stream=stream.cuda_stream)
    try:
        args = [o["Q"][None], o["c"][None], None, None, o["Aineq"][None], o["bineq"][None], o["lb"][None], o["ub"][None]]
        lat = []
        for k in range(reps + 3):
            t0 = time.perf_counter()
            r = eng.solve_qp_batch(*args)
            t1 = time.perf_counter()
            if k >= 3:
                lat.append((t1 - t0) * 1e3)
        return dict(p50_ms=float(np.median(lat)), min_ms=float(min(lat)), status=int(r["status"][0]), iters=int(r["iters"][0][0]),
                    h2d_bytes=int(sum(np.asarray(a).nbytes for a in args if a is not None)),
                    note="python ctypes wrapper overhead (numpy packing of the 720 KB matrices) included")
    finally:
        eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="c3", choices=sorted(wl.CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="instances of the WHOLE job per step (default: the config's batch)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary configurations (other_configs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.dump_outputs and (args.impl != "b200" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        raise SystemExit("--dump-outputs dumps the single-GPU b200 path: use it with --impl b200 on one GPU")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from copra_b200 import capi

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # keep stdout to the ONE JSON line (NCCL prints its version banner there)
        dist.init_process_group("nccl", device_id=dev)

    config = args.config
    total = args.batch or DEFAULT_BATCH[config]
    full = make_full_batch(config, total)
    total = full["batch"]
    bp, (lo, hi) = wl.shard(full, rank, world)  # strong scaling: the same `total` instances, contiguous ranges
    per = -(-total // world)
    if bp["batch"] == 0:
        raise SystemExit("more ranks than instances")

    stream = torch.cuda.Stream(device=dev)  # a real (non-legacy) stream shared by torch events and the engine
    torch.cuda.set_stream(stream)
    run = Runner(torch, capi, dev, local, bp, stream)
    sz, batch = run.sz, run.batch
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up -------------------------------------------------------------------------------------------------
    sampler = ClockSampler(local)
    sampler.start()  # samples clocks / throttle reasons through warm-up, the timed region and the e2e loop
    for _ in range(args.warmup):
        run.step_device()
    torch.cuda.synchronize()
    n_ok = int((run.d_status == 0).sum().item())

    # ---- value: device-resident inputs, CUDA events per step, L2 flushed between steps -----------------------------
    l0 = run.eng.launch_count()
    step_ms, stage, wall_timed = time_value(torch, run, stream, flush, args.steps, barrier)
    launches = run.eng.launch_count() - l0
    dumped = dump_sample(run) if args.dump_outputs else None
    total_ms = sum(step_ms)
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    value = total * args.steps / (total_ms_max * 1e-3)
    iters_np = run.d_iters.view(-1, 2).cpu().numpy().copy()
    nact_np = run.d_nact.cpu().numpy().copy()

    # ---- e2e: pinned host parameters -> H2D -> K1..K7 -> gather of every rank's results into rank 0's pinned buffer -
    d2h_bytes = 0
    if world == 1:
        d2h_bytes = run.host_results(total)

        def e2e_step():
            run.step_host_to_host()
    else:
        if rank == 0:
            d2h_bytes = run.host_results(per * world)
        g_control = torch.empty(per * sz["nU"], dtype=torch.float64, device=dev)
        g_traj = torch.empty(per * sz["X"], dtype=torch.float64, device=dev)
        g_status = torch.full((per,), -1, dtype=torch.int32, device=dev)
        all_control = [torch.empty_like(g_control) for _ in range(world)] if rank == 0 else None
        all_traj = [torch.empty_like(g_traj) for _ in range(world)] if rank == 0 else None
        all_status = [torch.empty_like(g_status) for _ in range(world)] if rank == 0 else None

        def e2e_step():
            run.step_host_to_device()
            g_control[:batch * sz["nU"]].copy_(run.d_control)
            g_traj[:batch * sz["X"]].copy_(run.d_traj)
            g_status[:batch].copy_(run.d_status)
            # the final gather: the only traffic that crosses NVLink
            dist.gather(g_control, all_control, dst=0)
            dist.gather(g_traj, all_traj, dst=0)
            dist.gather(g_status, all_status, dst=0)
            if rank == 0:
                nu_, nx_ = per * sz["nU"], per * sz["X"]
                for w in range(world):
                    run.h_control[w * nu_:(w + 1) * nu_].copy_(all_control[w], non_blocking=True)
                    run.h_traj[w * nx_:(w + 1) * nx_].copy_(all_traj[w], non_blocking=True)
                    run.h_status[w * per:(w + 1) * per].copy_(all_status[w], non_blocking=True)
            torch.cuda.synchronize()

    for _ in range(2):
        e2e_step()
    barrier()
    e0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    torch.cuda.synchronize()
    e1 = time.perf_counter()
    te = torch.tensor([e1 - e0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = total * args.steps / float(te.item())
    ok_host = int((run.h_status == 0).sum().item()) if rank == 0 else 0
    clocks = sampler.stop()

    # ---- per-rank summaries (status counts, timings, iteration statistics): gathered after the timed regions --------
    summary = torch.tensor([float(n_ok), total_ms, float(launches), float(run.hb_host.h2d_bytes), stage["solve_ms"],
                            float(iters_np[:, 0].sum()), float(iters_np[:, 1].sum()), float(batch)], dtype=torch.float64, device=dev)
    if world > 1:
        gathered = [torch.empty_like(summary) for _ in range(world)]
        dist.all_gather(gathered, summary)
        summary_all = torch.stack(gathered).cpu().numpy()
    else:
        summary_all = summary.cpu().numpy()[None, :]

    if rank == 0:
        peak, peak_src = peaks()
        dfma_tf, dmma_tf = run.eng.fp64_peaks()  # measured on this device, outside the timed region
        kernel = run.eng.last_solver()
        thin = "gi_thin_kernel" in kernel
        shared_h = run.eng.hessian_is_shared()
        solve_s = stage["solve_ms"] * 1e-3  # mean K5+K6 time per step of THIS rank (library CUDA events, every timed step)
        b_alg = float(k6_algorithmic_bytes(sz)) * batch
        f_alg = float(k6_algorithmic_flops(sz, iters_np[:, 0]).sum())
        f_exec = k6_executed_flops(sz, iters_np[:, 0], iters_np[:, 1], nact_np, thin, shared_h, batch,
                                   shape=(bp["nx"], bp["nu"], bp["N"], sz["X"]) if np.asarray(bp["A"]).ndim == 2 else None)
        t_hbm, t_fp = b_alg / (peak * 1e9), f_alg / (dfma_tf * 1e12)
        bound = "tensor" if t_fp >= t_hbm else "hbm"
        if bound == "tensor":
            achieved, pk, unit = f_alg / solve_s / 1e12, dfma_tf, "TFLOP/s"
        else:
            achieved, pk, unit = b_alg / solve_s / 1e9, peak, "GB/s"
        step_total = sum(stage.values())
        nx, nu, N, X, nU = bp["nx"], bp["nu"], bp["N"], sz["X"], sz["nU"]
        k1_bytes = 8.0 * (nx * nx + nx * nu + 2 * nx) + 8.0 * (X * nx + N * nx * nu + X)
        # assembly: the SYRK count r n (n+1) + 2 r nx n of every cost (r = stacked rows) + 2 r_c nx n per constraint stack
        k2_flops = 0.0
        for c in full["costs"]:
            rows = int(np.asarray(c["p"]).shape[-1])
            r_ = rows * (N + 1 if c["kind"] == "trajectory" else (1 if c["kind"] == "target" else N))
            k2_flops += r_ * sz["nvar"] * (sz["nvar"] + 1.0) + 2.0 * r_ * nx * sz["nvar"]
        k2_flops += 2.0 * (sz["mineq"] + sz["meq"]) * nx * sz["nvar"]
        line = dict(
            metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
            ms_per_step=total_ms_max / args.steps, higher_is_better=True, scaling="strong", vs_baseline=None,
            dtype="f64", data="synthetic",
            config=config_dict(config, full, total, world),
            p50_ms_per_batch=float(np.median(step_ms)), p50_us_per_solve_amortised=float(np.median(step_ms)) * 1e3 / batch,
            solved_ok=int(summary_all[:, 0].sum()), instances=total, instances_per_rank=[int(v) for v in summary_all[:, 7]],
            stage_ms=stage,
            roofline=dict(
                kernel=kernel + " (K5+K6)", bound=bound, achieved=achieved, peak=pk, unit=unit, frac=achieved / pk,
                traffic=NCU_TRAFFIC.get((config, str(batch))),
                peak_source=("measured live: DFMA-chain microbenchmark copra_b200_fp64_peaks (DMMA.8x8x4 chain: %.1f); "
                             "MEASURED_PEAKS.json has no FP64 entry, nominal %.0f" % (dmma_tf, FP64_NOMINAL_TFLOPS))
                if bound == "tensor" else peak_src,
                pipe="fp64 (DFMA / DMMA.8x8x4; tcgen05 has no f64 kind)",
                t_min_ms=dict(hbm=t_hbm * 1e3, fp64=t_fp * 1e3), t_measured_ms=stage["solve_ms"],
                algorithmic=dict(flops_per_launch=f_alg, bytes_per_launch=b_alg,
                                 formula="F = 2/3 n^3 + I (10 n^2 + 2 n q) per instance, I = its outer iterations; "
                                         "B = 8 (n^2 + n + (meq+m) n + (meq+m) + 2n) + 8n + 4q + 12 (SURVEY.md 8d)"),
                executed_flops_per_launch=f_exec,
                executed_tflops=f_exec / solve_s / 1e12,
                hbm=dict(achieved_gbs=b_alg / solve_s / 1e9, peak_gbs=peak, frac=b_alg / solve_s / 1e9 / peak, peak_source=peak_src),
                mean_outer_iterations=float(iters_np[:, 0].mean()), mean_drops=float(iters_np[:, 1].mean()),
                share_of_step=(stage["solve_ms"] / step_total) if step_total > 0 else None,
                stages=dict(
                    K1_condense=dict(bound="hbm", bytes_per_step=k1_bytes * batch, ms=stage["condense_ms"],
                                     achieved_gbs=k1_bytes * batch / (stage["condense_ms"] * 1e-3) / 1e9 if stage["condense_ms"] > 0 else None,
                                     peak_gbs=peak),
                    K2_K4_assemble=dict(bound="tensor", algorithmic_flops_per_step=k2_flops * batch, ms=stage["assemble_ms"],
                                        achieved_tflops=k2_flops * batch / (stage["assemble_ms"] * 1e-3) / 1e12 if stage["assemble_ms"] > 0 else None,
                                        peak_tflops=dmma_tf,
                                        note="dense SYRK count of the reference; the kernels run the O(N^2) block-Toeplitz recurrence"
                                             + (" and assemble the batch-invariant Hessian once" if shared_h else "")),
                    K7_rollout=dict(ms=stage["rollout_ms"])),
                note="rank 0's shard; `achieved` = algorithmic work / mean K5+K6 device time per step (library CUDA events on the "
                     "launching stream, every timed step)"),
            e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=int(summary_all[:, 3].sum()), d2h_bytes_per_step=d2h_bytes,
                     solved_ok=ok_host,
                     note="pinned host parameters -> H2D per shard -> K1..K7 -> " + ("NCCL gather to rank 0 + " if world > 1 else "")
                          + "D2H of control/trajectory/status of all %d instances into rank 0's pinned buffer" % total),
            gpu_launches=int(summary_all[:, 2].sum()),
            clocks=dict(sm_mhz=clocks["sm_mhz"], sm_max_mhz=clocks["sm_max_mhz"], reasons=clocks["reasons"],
                        samples=clocks["samples"], power_w_max=clocks.get("power_w_max")),
            wall_s_timed_region=wall_timed)
        if not args.no_cpu_baseline and world == 1:
            from oracle import pyoracle as po
            cores = po.hw_threads()
            per_inst = CPU_SECONDS_PER_INSTANCE[config]
            nmax = int(max(cores, min(batch, max(256 if config == "c3" else 0, 6.0 * cores / per_inst))))
            cb = cpu_sample(bp, nmax, reps=2)
            line["cpu_baseline"] = dict(value=cb["value"], unit=UNIT, cores=cb["cores"], kind="port",
                                        sample="first %d instances of the same %s batch, best of 2, one instance per host thread "
                                               "(%d threads = sched_getaffinity); p50 %.3f ms per solve; oracle port of copra's "
                                               "Eigen + eigen-quadprog path" % (cb["n"], config, cb["cores"], cb["p50_ms"]))
        if not args.no_extras and world == 1 and config == "c3":
            extras = {}
            run.close()
            del run
            torch.cuda.empty_cache()
            for cfg, st in (("c2", 20), ("c4", 10), ("c5", 2), ("c1", 20)):
                try:
                    extras[cfg] = measure_single(torch, capi, dev, local, stream, flush, cfg, DEFAULT_BATCH[cfg], st, 3,
                                                 resolve=cfg in ("c2",))
                except Exception as ex:  # a secondary line must never cost the headline
                    extras[cfg] = dict(error=repr(ex))
            try:
                c3r = measure_single(torch, capi, dev, local, stream, flush, "c3", 4096, 3, 3, resolve=True)
                extras["c3_resolve"] = c3r.get("resolve")
                extras["c3_resolve_warm"] = c3r.get("resolve_warm")
            except Exception as ex:
                extras["c3_resolve"] = dict(error=repr(ex))
            try:
                extras["c1_raw_qp_latency"] = c1_raw_qp_latency(torch, capi, local, stream)
            except Exception as ex:
                extras["c1_raw_qp_latency"] = dict(error=repr(ex))
            line["other_configs"] = extras
        if dumped is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dumped.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
