/*
 * copra_b200.h -- C ABI of the B200-native batched linear-MPC engine.
 *
 * This is the drop-in boundary for copra's data-parallel hot path (SURVEY.md 8b).  copra itself has
 * no C ABI: its plug-in point is the C++ virtual class `copra::SolverInterface`
 * (reference include/SolverInterface.h:19-81) selected through `SolverFlag` / `solverFactory`
 * (include/solverUtils.h:34-67, src/solverUtils.cpp:9-34) and driven by `LMPC::solve`
 * (src/LMPC.cpp:79-101).  The C++ facade in include/copra/ mirrors those classes and forwards to the
 * entry points below; every entry point cites the reference interface it replaces.
 *
 * Conventions
 *   - plain C, no exceptions; return 0 = OK, < 0 = argument/CUDA error (text via
 *     copra_b200_last_error); per-instance QP outcomes are reported in `status[]` only
 *     (0 ok / 1 infeasible / 2 Hessian not positive definite == QuadProgDenseSolver::SI_fail,
 *     include/QuadProgSolver.h:21-27).
 *   - all reals are IEEE float64; matrices are column-major with ld == rows (Eigen default).
 *   - every array argument is a (pointer, batch stride) pair; stride 0 = shared by all instances,
 *     otherwise the distance in doubles between consecutive instances.
 *   - `memory` says where ALL array arguments of that call live: COPRA_B200_HOST (copied over PCIe
 *     inside the call) or COPRA_B200_DEVICE (pointers valid on the handle's device; no copies).
 *   - a handle is bound to one CUDA device and one stream and is NOT thread-safe; multi-GPU callers
 *     create one handle per device and shard the batch by instance index (no collective on the path).
 *   - there is no CPU fallback: without a usable CUDA device `copra_b200_create` fails.
 */
#ifndef COPRA_B200_H
#define COPRA_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COPRA_B200_ABI_VERSION 1

typedef struct copra_b200_handle copra_b200_handle;

enum { COPRA_B200_HOST = 0, COPRA_B200_DEVICE = 1 };

/* return codes */
enum {
    COPRA_B200_OK = 0,
    COPRA_B200_E_ARG = -1,     /* bad argument / dimension mismatch (std::domain_error in the facade) */
    COPRA_B200_E_CUDA = -2,    /* CUDA runtime error */
    COPRA_B200_E_NOGPU = -3,   /* no CUDA device: the engine has no CPU fallback */
    COPRA_B200_E_UNSUPPORTED = -4,
    COPRA_B200_E_STATE = -5    /* call order (e.g. download before run) */
};

typedef struct {
    int device;          /* CUDA device ordinal */
    void* stream;        /* cudaStream_t to launch on; NULL = the handle creates its own */
    int sm_limit;        /* 0 = use every SM; otherwise cap the persistent grids (testing) */
    int small_variant;   /* testing: 0 = planner's choice, 1..3 force shared-memory residency variant 0..2 of the small-n
                            kernel (gi_small_kernel) when it fits */
    int reserved[4];
} copra_b200_options;

typedef struct {
    const double* ptr;
    long long stride;    /* doubles between instances; 0 = shared */
} copra_b200_array;

/* A third value of `full_size` (copra_b200_cost, copra_b200_constraint): step-size matrices with a vector that changes
 * from step to step -- the moving ZMP box of a walking pattern generator, the reference trajectory of a tracking MPC.
 *   - `rows` stays the per-step row count (rows of M / N / E / G, nx for a trajectory bound, nu for a control bound) and the
 *     matrices and `w` keep their step-size shapes;
 *   - the vector (p, f, or lower / upper) holds rows x steps entries per instance, step-major: entry i*rows + l is line l at
 *     step i (the layout of AutoSpan::spanVector, include/AutoSpan.h);
 *   - steps = N+1 for TRAJECTORY costs, TRAJECTORY constraints and TRAJECTORY_BOUND; N for CONTROL and MIXED costs and
 *     constraints and for CONTROL_BOUND.  A TARGET cost has one step and rejects it (E_ARG);
 *   - weights stay per row (per-step weights change the Hessian: full-size entries only);
 *   - a per-step TRAJECTORY_BOUND has the same +-inf pattern at every step and in every instance, otherwise E_ARG.
 * The Hessian and the constraint matrices do not depend on these vectors, so such a problem runs on exactly the kernels of the
 * step-size one (shared Hessian and factor, structured thin solver); the autoSpan'd full-size form of the same problem
 * (full_size = 1) does not. */
#define COPRA_B200_PER_STEP 2

/* ---- cost functions: reference include/costFunctions.h:103-219, src/costFunctions.cpp:63-215 ---- */
enum { COPRA_B200_COST_TRAJECTORY = 0, COPRA_B200_COST_TARGET = 1, COPRA_B200_COST_CONTROL = 2, COPRA_B200_COST_MIXED = 3 };
typedef struct {
    int kind;
    int rows;            /* rows of M / N / p / w */
    copra_b200_array M, N, p, w;
    int full_size;       /* 0: step-size entry (M rows x nx, N rows x nu, applied at every step);
                            1: full-size entry (M rows x nx(N+1), N rows x nu*N) -- the `fullSizeEntry_` branch of
                               src/costFunctions.cpp:65-71,141-146,197-203; not allowed for TARGET (:95-97);
                            COPRA_B200_PER_STEP: step-size M / N / w, p with rows x steps entries (see above) */
} copra_b200_cost;

/* ---- constraints: reference include/constraints.h:114-307, src/constraints.cpp:45-367 ---- */
enum {
    COPRA_B200_CSTR_TRAJECTORY = 0,       /* E x_i <= f (or ==), i = 0..N        */
    COPRA_B200_CSTR_CONTROL = 1,          /* G u_i <= f (or ==), i = 0..N-1      */
    COPRA_B200_CSTR_MIXED = 2,            /* E x_i + G u_i <= f, i = 0..N-1      */
    COPRA_B200_CSTR_TRAJECTORY_BOUND = 3, /* lower <= x_i <= upper (+-inf lines skipped; quirk Q1) */
    COPRA_B200_CSTR_CONTROL_BOUND = 4     /* lower <= u_i <= upper -> lb/ub      */
};
typedef struct {
    int kind;
    int rows;            /* rows of E/G/f, or entries of lower/upper */
    int is_ineq;         /* TRAJECTORY/CONTROL/MIXED only */
    copra_b200_array E, G, f, lower, upper;
    int full_size;       /* 1: E rows x nx(N+1), G rows x nu*N, lower/upper with nx(N+1) (trajectory) or nu*N (control)
                               entries -- src/constraints.cpp:68-73,122-126,199-204,297-299,346-351;
                            COPRA_B200_PER_STEP: step-size E / G, f or lower / upper with rows x steps entries (see above) */
} copra_b200_constraint;

/* ---- a batch of LMPC / InitialStateLMPC problems of ONE shape ----
 * replaces: PreviewSystem::system (src/PreviewSystem.cpp:16-55) + LMPC::addCost/addConstraint
 * (src/LMPC.cpp:118-128) for `batch` independent controllers. */
typedef struct {
    int nx, nu, N, batch;
    int initial_state;   /* 0: copra::LMPC, 1: copra::InitialStateLMPC (decision vector [x0; U]) */
    copra_b200_array A, B, d, x0;
    int ncost;
    const copra_b200_cost* costs;
    int ncstr;
    const copra_b200_constraint* cstrs;
    copra_b200_array R, r, x0lb, x0ub; /* initial-state mode; ptr NULL = reference default (R=0,r=0,bounds=x0) */
    int memory;
    int flags;           /* COPRA_B200_FLAG_* */
} copra_b200_problem;

/* LMPC::updateSystem starts every Hessian at 1e-6*I (src/LMPC.cpp:228-229).  The facade sets NO_REG when it
 * evaluates ONE cost function in isolation (CostFunction::Q() getter), where the reference has no such term. */
#define COPRA_B200_FLAG_NO_REG 1
/* DEVICE inputs only: the caller guarantees that the +-inf pattern of every TrajectoryBoundConstraint's lower / upper
 * (which decides the number of inequality rows, include/constraints.h:247-254) is unchanged since the previous build
 * on this handle that used the same pointers, so the engine may skip reading it back.  Without the flag the pattern is
 * re-read from instance 0 on every build. */
#define COPRA_B200_FLAG_STABLE_BOUND_PATTERN 2

typedef struct {
    int X;      /* nx*(N+1) */
    int nU;     /* nu*N     */
    int nvar;   /* nU, or nx+nU in initial-state mode */
    int meq, mineq;
    int q;      /* meq + mineq + 2*nvar : QuadProg's constraint index space */
} copra_b200_sizes;

/* Outputs of a run; every pointer may be NULL.  Instance b occupies [b*len, (b+1)*len). */
typedef struct {
    double* control;     /* nU   per instance : LMPC::control()     (src/LMPC.cpp:284) */
    double* trajectory;  /* X    per instance : LMPC::trajectory()  (src/LMPC.cpp:285) */
    double* x;           /* nvar per instance : SolverInterface::SI_result()            */
    int* status;         /* 1    per instance : SI_fail()                                */
    int* iters;          /* 2    per instance : (outer iterations, constraint drops); [0] == SI_iter() */
    int* nact;           /* 1    per instance : number of active constraints             */
    int* iact;           /* nvar per instance : 1-based active indices in [eq|ineq|upper|lower] space, add order, 0 padded */
    int memory;
} copra_b200_results;

typedef struct {
    float h2d_ms, condense_ms, assemble_ms, solve_ms, rollout_ms, d2h_ms, total_ms;
    long long launches;  /* kernels launched by the last call */
} copra_b200_timing;

/* identifiers for copra_b200_lmpc_download */
enum {
    COPRA_B200_GET_PHI = 0, COPRA_B200_GET_PSI = 1, COPRA_B200_GET_XI = 2,
    COPRA_B200_GET_Q = 3, COPRA_B200_GET_C = 4, COPRA_B200_GET_AEQ = 5, COPRA_B200_GET_BEQ = 6,
    COPRA_B200_GET_AINEQ = 7, COPRA_B200_GET_BINEQ = 8, COPRA_B200_GET_LB = 9, COPRA_B200_GET_UB = 10,
    COPRA_B200_GET_YEQ = 11, COPRA_B200_GET_ZEQ = 12, COPRA_B200_GET_YINEQ = 13, COPRA_B200_GET_ZINEQ = 14,
    /* per-cost E() (nx x nU) and f() (nU) of cost i: COPRA_B200_GET_COST_E + i, COPRA_B200_GET_COST_F + i
     * (CostFunction::E() / f(), include/costFunctions.h:85-87) */
    COPRA_B200_GET_COST_E = 100, COPRA_B200_GET_COST_F = 200
};

/* ---------------------------------------------------------------------------------------------- */
int copra_b200_abi_version(void);
int copra_b200_device_count(void);

int copra_b200_create(const copra_b200_options* opt, copra_b200_handle** out);
void copra_b200_destroy(copra_b200_handle* h);
const char* copra_b200_last_error(const copra_b200_handle* h);
/* rebind the launch stream (e.g. to the caller framework's current stream) */
int copra_b200_set_stream(copra_b200_handle* h, void* cuda_stream);
int copra_b200_synchronize(copra_b200_handle* h);
/* total kernels launched through this handle since creation */
long long copra_b200_launch_count(const copra_b200_handle* h);
int copra_b200_last_timing(const copra_b200_handle* h, copra_b200_timing* t);

/* K1 -- replaces PreviewSystem::updateSystem (src/PreviewSystem.cpp:57-74) for a batch.
 * Outputs (any may be NULL): Phi X x nx, Psi X x nU, xi X per instance, reference layout. */
int copra_b200_condense(copra_b200_handle* h, int nx, int nu, int N, int batch,
    copra_b200_array A, copra_b200_array B, copra_b200_array d,
    double* Phi, double* Psi, double* xi, int memory);

/* K5+K6 -- replaces QuadProgDenseSolver::SI_problem + SI_solve (src/QuadProgSolver.cpp:45-72) and the
 * external Eigen::QuadProgDense::solve / qpgen2 behind it, for a batch of raw QPs
 *   min 1/2 x'Qx + c'x   s.t.  Aeq x = beq,  Aineq x <= bineq,  lb <= x <= ub.
 * Q n x n, Aeq meq x n, Aineq m x n (column-major).  Bounds are handled implicitly but keep
 * QuadProg's row indices (m.. upper, m+n.. lower). */
int copra_b200_solve_qp_batch(copra_b200_handle* h, int n, int meq, int m, int batch,
    copra_b200_array Q, copra_b200_array c, copra_b200_array Aeq, copra_b200_array beq,
    copra_b200_array Aineq, copra_b200_array bineq, copra_b200_array lb, copra_b200_array ub,
    double* x, int* status, int* iters, int* nact, int* iact, int memory);

/* Sensitivities of the last raw QP batch (copra_b200_solve_qp_batch): the vector-Jacobian product of its solutions x with
 * respect to every input, exact on the final active set.  Write the active rows as equalities a_j'x = beta_j in their natural
 * orientation (an Aeq row with beq, an Aineq row with bineq, e_k with ub_k for an upper row and with lb_k for a lower row).  With
 * dx = dL/dx, one adjoint KKT solve per instance, [Q A_act'; A_act 0] [v; mu] = [dx; 0], gives
 *   dL/dc = -v,  dL/dbeta_j = mu_j (dbeq, dbineq, dub, dlb at the row's index; 0 for inactive rows),
 *   dL/dQ = -(v x' + x v') / 2,  dL/da_j = -lambda_j v - mu_j x (the row of dAeq / dAineq; 0 for inactive rows),
 * with lambda the multipliers of the forward solve, [Q A_act'; A_act 0] [x; lambda] = [-c; beta]: the KKT solve takes the
 * forward solve as a second right-hand side only when dAeq or dAineq is wanted.  Q is read as a symmetric matrix, so dQ is the
 * gradient along symmetric perturbations of Q.  A weakly active row gives the one-sided derivative on the final active set.
 * Each gradient has, per instance, the layout copra_b200_solve_qp_batch takes for its input (Q n x n, Aeq meq x n, Aineq
 * m x n, column-major); gradients are per instance even for inputs given with stride 0.  NULL marks a gradient that is not
 * wanted. */
typedef struct {
    double* Q;
    double* c;
    double* Aeq;
    double* beq;
    double* Aineq;
    double* bineq;
    double* lb;
    double* ub;
} copra_b200_qp_vjp_out;
/* `dx` holds n doubles per instance; it and every output pointer live in `memory`.  Instances whose status is not 0 get
 * zeros; a Q or a Gram matrix of the active rows that is not positive definite (linearly dependent active rows) gives NaN.
 * With DEVICE inputs the solve's input arrays are read again: the caller leaves them unchanged until this call.  E_STATE when
 * the last solve on the handle was not a raw QP batch (none yet, or an LMPC build, solve, resolve or retarget since); E_ARG for
 * a NULL dx, or for dAeq / dbeq with meq = 0 or dAineq / dbineq with m = 0; E_UNSUPPORTED when n needs more shared memory per
 * block than the device allows.  A NULL `out` returns 0 after these checks.  Leaves a resident LMPC build, its factor caches
 * and its warm-start seed untouched. */
int copra_b200_qp_vjp(copra_b200_handle* h, const double* dx, int memory, const copra_b200_qp_vjp_out* out);

/* Forward mode on the last raw QP batch: Jacobian-vector products of its solutions x along k tangent directions, exact on the
 * final active set.  With the active rows a_j'x = beta_j written as for copra_b200_qp_vjp and lambda the forward multipliers,
 * one KKT solve per instance with k right-hand sides,
 *   [Q A_act'; A_act 0] [xdot; lambdadot] = [-cdot_eff; bdot_eff],
 *   cdot_eff = cdot + (Qdot + Qdot') x / 2 + sum_active lambda_j adot_j,
 *   bdot_eff_j = bdot_j - adot_j' x (an active Aeq / Aineq row),  ubdot_k / lbdot_k (an active bound row),
 * gives xdot.  Q is read through its symmetric part, as by copra_b200_qp_vjp.  lambda is computed (one more KKT solve with one
 * right-hand side) only when an Aeq or Aineq tangent is given.  A weakly active row gives the one-sided derivative on the final
 * active set. */
typedef struct {
    int ndir;                                      /* k >= 1 tangent directions */
    copra_b200_array Q, c, Aeq, beq, Aineq, bineq, lb, ub;
    /* per instance len x k: the k directions one after the other, each in the layout copra_b200_solve_qp_batch takes for the
     * input (Q n x n, Aeq meq x n, Aineq m x n, column-major); stride in doubles between instances, 0 = one tangent for every
     * instance; ptr NULL = zero tangent */
} copra_b200_qp_jvp_in;
/* `dx` receives n x k doubles per instance (column-major: direction d at d * n); it and the tangents live in `memory`.
 * Instances whose status is not 0 get zeros; a Q or a Gram matrix of the active rows that is not positive definite gives NaN.
 * With DEVICE inputs the solve's input arrays are read again: the caller leaves them unchanged until this call.  E_STATE when
 * the last solve on the handle was not a raw QP batch; E_ARG for a NULL `in`, ndir < 1, a negative stride, Aeq / beq tangents
 * with meq = 0 or Aineq / bineq tangents with m = 0; E_UNSUPPORTED when n needs more shared memory per block than the device
 * allows.  A NULL `dx` returns 0 after these checks.  Leaves a resident LMPC build, its factor caches, its warm-start seed and
 * a later copra_b200_qp_vjp untouched. */
int copra_b200_qp_jvp(copra_b200_handle* h, const copra_b200_qp_jvp_in* in, int memory, double* dx);

/* The Jacobian of the last raw QP batch's solutions x with respect to one vector input: copra_b200_qp_jvp along the columns of
 * the identity on that input (never materialised).  wrt = c gives dx/dc (n x n, the projected inverse Hessian
 * -Z (Z'QZ)^-1 Z' on the active set, symmetric); beq, bineq, lb, ub give n x meq, n x m, n x n, n x n, whose columns of
 * inactive rows are exactly zero.  `J` receives n x len doubles per instance, column-major, in `memory`.  Errors and
 * conventions as copra_b200_qp_jvp; E_ARG for an unknown wrt, or beq with meq = 0 or bineq with m = 0.  A NULL `J` returns 0
 * after the checks. */
enum { COPRA_B200_QP_WRT_C = 0, COPRA_B200_QP_WRT_BEQ = 1, COPRA_B200_QP_WRT_BINEQ = 2, COPRA_B200_QP_WRT_LB = 3,
       COPRA_B200_QP_WRT_UB = 4 };
int copra_b200_qp_jacobian(copra_b200_handle* h, int wrt, double* J, int memory);

/* Dense assembly primitive -- batched FP64 GEMM on the tensor cores (DMMA m8n8k4 fed through shared memory, TMA
 * bulk loads for aligned operands): C[b] = alpha * op(A[b]) * B[b] + beta * C[b], column-major, strides in doubles.
 * It is what full-size (autoSpan'd) entries use for M*Psi, T'WT, E*Psi (src/costFunctions.cpp:65-69,
 * src/constraints.cpp:68-72); exported for callers that assemble their own dense terms. */
int copra_b200_dgemm_batch(copra_b200_handle* h, int transA, int M, int N, int K, double alpha,
    const double* A, int lda, long long strideA, const double* B, int ldb, long long strideB,
    double beta, double* C, int ldc, long long strideC, int batch, int memory);

/* Shape query / validation -- the dimension checks of initializeCost / initializeConstraint
 * (src/costFunctions.cpp:44-193, src/constraints.cpp:45-357); COPRA_B200_E_ARG == std::domain_error. */
int copra_b200_lmpc_sizes(copra_b200_handle* h, const copra_b200_problem* p, copra_b200_sizes* s);

/* K1..K7 -- replaces LMPC::solve (src/LMPC.cpp:79-101) / InitialStateLMPC for `batch` controllers:
 * updateSystem -> makeQPForm -> SI_problem -> SI_solve -> updateResults. */
int copra_b200_lmpc_run(copra_b200_handle* h, const copra_b200_problem* p, const copra_b200_results* r);
/* staged variants: build = K1..K5 (LMPC::updateSystem + makeQPForm), solve = K6+K7 */
int copra_b200_lmpc_build(copra_b200_handle* h, const copra_b200_problem* p);
int copra_b200_lmpc_solve(copra_b200_handle* h, const copra_b200_results* r);
/* Measured FP64 ceilings of this device in TFLOP/s: a DFMA-chain and a DMMA.8x8x4-chain microbenchmark (the
 * denominators of the FP64 roofline in bench.py; SURVEY.md 8d).  Takes a few milliseconds; cached per handle. */
int copra_b200_fp64_peaks(copra_b200_handle* h, double* dfma_tflops, double* dmma_tflops);
/* Receding-horizon re-solve (SURVEY.md 8f N1): only the initial states changed since the last build
 * (PreviewSystem::xInit, include/PreviewSystem.h:52-54, leaves `isUpdated` set so the reference skips
 * updateSystem's condensing too).  Re-runs K4 (c = E'x0 + f, b = z - Y x0) on the resident Phi/Gs/E/f/Y/z and
 * K5..K7; Q, Aeq, Aineq are reused.  LMPC mode only (in initial-state mode x0 is a decision variable). */
int copra_b200_lmpc_resolve(copra_b200_handle* h, copra_b200_array x0, int memory, const copra_b200_results* r);
/* Receding-horizon step with new references and limits: a new x0 and new vectors (every cost's p, every constraint's f /
 * lower / upper; typically per-step entries whose window moved by one tick) on the resident build.
 * `p` must describe the resident build's shape: the same nx, nu, N, batch, the same number, kind, rows, full_size (and
 * is_ineq) of every cost and constraint, and the same trajectory-bound +-inf pattern; a mismatch returns E_ARG and leaves the
 * resident build usable.  Only x0, p, f, lower and upper are read from `p` (and p->memory, p->flags): A, B, d, M, N, w, E,
 * G, R, r, x0lb and x0ub are ignored (they may be NULL) and the resident ones are used.  Re-runs the vector part of K2
 * (res = M xi - p, z = f - E xi, each cost's f), K4 and K5..K7; condensing, Q, E, the constraint matrices, the thin solver's
 * factor, the small solver's factor cache and the warm-start seed are reused, and the results are bitwise those of a full
 * build of the same problem.  E_STATE without a resident build (also after a copra_b200_lmpc_run of more than 65535 instances,
 * which keeps only its last chunk); E_UNSUPPORTED in initial-state mode and for builds with a full-size (full_size = 1) cost,
 * row constraint or trajectory bound, whose vector terms come out of the dense GEMM epilogues (a full-size control bound is
 * fine). */
int copra_b200_lmpc_retarget(copra_b200_handle* h, const copra_b200_problem* p, const copra_b200_results* r);
/* Sensitivities of the last solve: the vector-Jacobian product of (control, trajectory) with respect to x0 and every
 * cost's p and every constraint's f / lower / upper.  On the final active set the solution is an affine function of these
 * vectors, so the product is exact (one adjoint KKT solve per instance, K8).  Gradients are per instance even for inputs
 * given with stride 0; a step-size entry's gradient is the sum over its steps, a per-step entry's has its rows x steps layout.
 * With x0 alone and a unit dcontrol this is a row of the local feedback gain d u / d x0.
 * Instances whose status is not 0 get zero gradients.  NULL pointers (the arrays themselves or their entries) mark gradients
 * that are not wanted; the arrays have ncost / ncstr entries of the resident build. */
typedef struct {
    double* x0;             /* nx per instance */
    double* const* p;       /* [ncost]: rows (x steps for a per-step entry) per instance */
    double* const* f;       /* [ncstr]: rows (x steps) per instance, row constraints */
    double* const* lower;   /* [ncstr]: rows (x steps) per instance, trajectory and control bounds */
    double* const* upper;
} copra_b200_vjp_out;
/* `dcontrol` holds nU doubles per instance (dL/dcontrol), `dtrajectory` X doubles (dL/dtrajectory); either may be NULL.
 * They and every output pointer live in `memory`.  Refers to the last solve on the resident build (run, solve, resolve or
 * retarget): E_STATE without one (also after a copra_b200_lmpc_run of more than 65535 instances); E_UNSUPPORTED in
 * initial-state mode and for builds with a full-size (full_size = 1) cost, row constraint or trajectory bound, as for
 * copra_b200_lmpc_retarget (a full-size control bound is fine).  Leaves the resident build, the factor caches and the
 * warm-start seed untouched. */
int copra_b200_lmpc_vjp(copra_b200_handle* h, const double* dcontrol, const double* dtrajectory, int memory,
    const copra_b200_vjp_out* out);
/* The same vector-Jacobian product, and with it the gradients with respect to every cost's weights and matrices: one adjoint
 * KKT solve serves both (with costs = NULL this is copra_b200_lmpc_vjp).  These inputs enter the objective only, so on the
 * final active set  dL/dtheta = c^' (dQ/dtheta U + dc/dtheta)  with c^ = dL/dc; per cost, with the solution's states x_i and
 * controls u_i, e_i = M x_i + N u_i - p_i, x^ = Psi c^ and t_i = M x^_i + N c^_i over the steps i the cost covers:
 *   dL/dw_l = sum_i (t_i)_l (e_i)_l,  dL/dM = sum_i W (e_i x^_i' + t_i x_i'),  dL/dN = sum_i W (e_i c^_i' + t_i u_i').
 * Gradients are per instance even for inputs given with stride 0.  NULL pointers (the arrays themselves or their entries)
 * mark gradients that are not wanted; `out` may be NULL when only cost gradients are wanted.  With DEVICE inputs, the x0,
 * M, N and w arrays the resident build (or its last retarget / resolve) was given are read again: they must still hold
 * those values.  Preconditions and error codes are those of copra_b200_lmpc_vjp, plus E_ARG for an M entry of a cost
 * without M (CONTROL) or an N entry of a cost without N (TRAJECTORY, TARGET), and E_UNSUPPORTED for a horizon whose
 * 2 nU + 2 X + 2 rows x steps doubles exceed the device's shared memory per block. */
typedef struct {
    double* const* w;   /* [ncost]: rows per instance */
    double* const* M;   /* [ncost]: rows x nx per instance, column-major; must be NULL for a cost without M */
    double* const* N;   /* [ncost]: rows x nu per instance, column-major; must be NULL for a cost without N */
} copra_b200_vjp_cost_out;
int copra_b200_lmpc_vjp_costs(copra_b200_handle* h, const double* dcontrol, const double* dtrajectory, int memory,
    const copra_b200_vjp_out* out /* may be NULL */, const copra_b200_vjp_cost_out* costs);
/* The same products, and with them the gradients with respect to the dynamics A, B, d and every row constraint's E and G
 * (with model = NULL this is copra_b200_lmpc_vjp_costs).  These inputs also move the active rows a_j' U = beta_j, so the
 * multipliers lambda of the forward solve enter: the adjoint KKT solve takes the forward solve as a second right-hand side.
 * With the adjoint (c^ = -v, mu) of copra_b200_lmpc_vjp, the states x_i and controls u_i of the solution, x^ = Psi c^,
 * e_i and t_i of every cost as above, and the active rows j at step i and line l of a constraint (E x_i + G u_i <=/= f):
 *   gx_i = dL/dtrajectory_i + sum_costs M'W t_i - sum_j mu_j E_l',  gh_i = sum_costs M'W e_i + sum_j lambda_j E_l',
 *   rho_N = gx_N, rho_i = gx_i + A' rho_{i+1}, and rho^ the same from gh;
 *   dL/dA = sum_{i<N} rho_{i+1} x_i' + rho^_{i+1} x^_i',  dL/dB = sum_{i<N} rho_{i+1} u_i' + rho^_{i+1} c^_i',
 *   dL/dd = sum_{i<N} rho_{i+1},  dL/dE_l = sum_i lambda_(i,l) x^_i' - mu_(i,l) x_i',  dL/dG_l = sum_i lambda_(i,l) c^_i' -
 *   mu_(i,l) u_i'  (inactive rows have lambda = mu = 0; rho_0 is dL/dx0).
 * A trajectory bound takes part through its multipliers (its E is the engine's line selector; quirk Q1: lower rows are
 * x <= lower) but has no E gradient.  Gradients are per instance even for inputs given with stride 0.  NULL pointers mark
 * gradients that are not wanted; `out` and `costs` may be NULL.  With DEVICE inputs, the E arrays the resident build was
 * given are read again, as are x0, M, N and w: they must still hold those values.  Preconditions and error codes are those
 * of copra_b200_lmpc_vjp_costs, plus E_ARG for an E entry of a constraint without E (CONTROL, bounds) or a G entry of one
 * without G (TRAJECTORY, bounds), and E_UNSUPPORTED for a horizon whose 2 nU + 4 X + 2 (meq + mineq) doubles exceed the
 * device's shared memory per block. */
typedef struct {
    double* A;          /* nx x nx per instance, column-major */
    double* B;          /* nx x nu per instance, column-major */
    double* d;          /* nx per instance */
    double* const* E;   /* [ncstr]: rows x nx per instance, column-major; must be NULL for a constraint without E */
    double* const* G;   /* [ncstr]: rows x nu per instance, column-major; must be NULL for a constraint without G */
} copra_b200_vjp_model_out;
int copra_b200_lmpc_vjp_model(copra_b200_handle* h, const double* dcontrol, const double* dtrajectory, int memory,
    const copra_b200_vjp_out* out /* may be NULL */, const copra_b200_vjp_cost_out* costs /* may be NULL */,
    const copra_b200_vjp_model_out* model);
/* Forward-mode sensitivities of the last solve: the Jacobian-vector product of (control, trajectory) along `ndir` tangent
 * directions of x0 and every cost's p and every constraint's f / lower / upper (one forward KKT solve per instance with
 * ndir right-hand sides, K9; exact on the final active set, as the VJP).  Each tangent holds, per instance, ndir
 * column-major vectors of the length of the matching copra_b200_vjp_out gradient (len x ndir); a step-size entry's tangent
 * moves the value used at every step, a per-step entry's has its rows x steps layout.  NULL pointers (the arrays themselves
 * or their entries) are zero tangents; the arrays have ncost / ncstr entries of the resident build. */
typedef struct {
    int ndir;                    /* k >= 1 tangent directions */
    const double* x0;            /* nx x k per instance */
    const double* const* p;      /* [ncost]: rows (x steps) x k per instance */
    const double* const* f;      /* [ncstr]: row constraints */
    const double* const* lower;  /* [ncstr]: trajectory and control bounds */
    const double* const* upper;
} copra_b200_jvp_in;
/* `dcontrol` receives nU x k doubles per instance (dU), `dtrajectory` X x k (dtrajectory); either may be NULL.  The tangents
 * and both outputs live in `memory`.  Instances whose status is not 0 get zeros; a Hessian or Gram factor that is not
 * positive definite gives NaN.  Preconditions and error codes are those of copra_b200_lmpc_vjp, plus E_ARG for a NULL `in`
 * or ndir < 1.  Leaves the resident build, the factor caches and the warm-start seed untouched. */
int copra_b200_lmpc_jvp(copra_b200_handle* h, const copra_b200_jvp_in* in, int memory, double* dcontrol, double* dtrajectory);
/* The local feedback gain of the last solve, the JVP along the columns of the identity on x0 (the identity is never
 * materialised): Ku = dU[0 : nu*steps] / dx0, (nu*steps) x nx per instance, and Kx = dtrajectory[0 : nx*(steps+1)] / dx0,
 * (nx*(steps+1)) x nx, both column-major; either may be NULL.  A loop running faster than the MPC applies
 * u0 + Ku (x - x0) with steps = 1.  E_ARG for steps outside [1, N]; otherwise as copra_b200_lmpc_jvp. */
int copra_b200_lmpc_feedback_gain(copra_b200_handle* h, int steps, double* Ku, double* Kx, int memory);
/* Sensitivities of the last solve of an initial-state build (copra::InitialStateLMPC, decision vector z = [x0*; U]): the
 * vector-Jacobian product of (control, trajectory) with respect to the vectors of copra_b200_lmpc_vjp and to R, r, x0lb and
 * x0ub.  The trajectory is Phi x0* + Psi U + xi with the optimised x0* (its first nx entries are x0*).  On the final active
 * set, with gbar = [Phi' dL/dtrajectory; dL/dcontrol + Psi' dL/dtrajectory], [Q A'; A 0] [v; mu] = [gbar; 0] and c^ = -v:
 *   dL/dr = c^[0:nx],  dL/dR = (c^_0 x0*' + x0* c^_0') / 2 with c^_0 = c^[0:nx] (R is read through its symmetric part),
 *   dL/dx0lb / dL/dx0ub = mu of the bound rows 0..nx-1, and p, f, lower and upper as copra_b200_lmpc_vjp on c^[nx:] and
 *   the multipliers of the general rows (b = z: no x0 term) and of the control bound rows nx...
 * x0 enters an initial-state build only as the default of an x0 bound that was not given (x0lb = x0ub = x0), so
 * out->x0 receives the sum of the multipliers of those bounds: zeros when both x0lb and x0ub were given.
 * `out` and `init` may be NULL; NULL pointers mark gradients that are not wanted.  Gradients are per instance even for
 * inputs given with stride 0.  Instances whose status is not 0 get zeros; a Hessian (with the default R = 0 it is only
 * semidefinite) or Gram factor that is not positive definite gives NaN.  E_STATE without a solve of the resident build
 * (or after a raw QP batch); E_UNSUPPORTED for an LMPC-mode build (use copra_b200_lmpc_vjp), for a full-size cost, row
 * constraint or trajectory bound (a full-size control bound is fine) and for a problem needing more shared memory per
 * block than the device allows; E_ARG for a gradient of R, r, x0lb or x0ub the build was not given (a NULL array, the
 * reference default).  Gradients with respect to w, M, N, A, B, d, E and G are not available in initial-state mode.
 * Leaves the resident build, the factor caches and the warm-start seed untouched. */
typedef struct {
    double* R;      /* nx x nx per instance, column-major (symmetric) */
    double* r;      /* nx per instance */
    double* x0lb;   /* nx per instance */
    double* x0ub;   /* nx per instance */
} copra_b200_vjp_initial_out;
int copra_b200_lmpc_vjp_initial_state(copra_b200_handle* h, const double* dcontrol, const double* dtrajectory, int memory,
    const copra_b200_vjp_out* out /* x0, p, f, lower, upper; may be NULL */, const copra_b200_vjp_initial_out* init /* may be NULL */);
/* Forward mode of the same: the Jacobian-vector product of (control, trajectory) of the last solve of an initial-state
 * build along in->ndir = k tangent directions of the vectors of copra_b200_jvp_in and of R, r, x0lb and x0ub (nx x nx x k
 * and nx x k per instance; NULL = zero).  cdot = [rdot + sym(Rdot) x0*; sum_costs fdot(pdot)], the bound rows 0..nx-1 move
 * with x0lbdot / x0ubdot, or with in->x0 where that bound defaulted to x0; dtrajectory = Phi zdot[0:nx] + Psi zdot[nx:].
 * Rdot enters through its symmetric part, so this is the exact adjoint of copra_b200_lmpc_vjp_initial_state.
 * `dcontrol` receives nU x k doubles per instance, `dtrajectory` X x k; either may be NULL.  Errors as
 * copra_b200_lmpc_vjp_initial_state (E_ARG for a tangent of R, r, x0lb or x0ub the build was not given), plus E_ARG for a
 * NULL `in` or ndir < 1. */
typedef struct {
    const double* R;     /* nx x nx x k per instance */
    const double* r;     /* nx x k per instance */
    const double* x0lb;  /* nx x k per instance */
    const double* x0ub;  /* nx x k per instance */
} copra_b200_jvp_initial_in;
int copra_b200_lmpc_jvp_initial_state(copra_b200_handle* h, const copra_b200_jvp_in* in, const copra_b200_jvp_initial_in* init /* may be NULL */,
    int memory, double* dcontrol, double* dtrajectory);
/* SolverInterface::SI_warmStart(bool) / SI_warmStart() (include/SolverInterface.h:42-45; QuadProg has none, the reference
 * prints "No warmStart() function for this qp").  Opt-in: with it on, copra_b200_lmpc_resolve seeds every instance with the
 * inequality / bound rows that were active at its previous solve on the resident build, solves that equality-constrained
 * problem in closed form, drops the rows whose multiplier came out negative and lets the dual iterations finish from there:
 * same optimum (the QP is strictly convex), far fewer iterations when the active set moved little.  Takes effect on builds the
 * thin solver runs in its shared-factor form (batch-invariant system and Hessian, n > 64); ignored elsewhere.  `iters` then
 * counts the iterations AFTER the seed. */
int copra_b200_set_warm_start(copra_b200_handle* h, int on);
int copra_b200_get_warm_start(const copra_b200_handle* h);
/* K7 alone -- LMPC::updateResults (src/LMPC.cpp:282-286) for an externally solved QP: `x` holds nvar doubles per
 * instance (the SI_result() of any SolverInterface); control / trajectory as in copra_b200_results. */
int copra_b200_lmpc_results(copra_b200_handle* h, const double* x, double* control, double* trajectory, int memory);
/* assembled stage of the last build, reference layout (LMPC::Q() c() Aeq() ... getters,
 * include/LMPC.h:105-127); `out` must hold batch * size doubles. */
int copra_b200_lmpc_download(copra_b200_handle* h, int what, double* out, int memory);

/* introspection for benchmarks / logs: the K5+K6 kernel(s) the last solve ran ("gi_small_kernel", "gi_cluster_kernel",
 * "gi_batch_kernel", "gt_factor_kernel + gi_thin_kernel") and whether the resident build found the Hessian batch-invariant
 * (A, B and every cost's M, N, w shared: assembled and factored once) */
const char* copra_b200_last_solver(const copra_b200_handle* h);
int copra_b200_hessian_is_shared(const copra_b200_handle* h);
/* sizes of the build resident on the handle (E_STATE without one) */
int copra_b200_lmpc_built_sizes(copra_b200_handle* h, copra_b200_sizes* s);

/* ---- data-parallel sharder (SURVEY.md 8e) ------------------------------------------------------------------------------
 * The batch of independent controllers is split by instance index into contiguous ranges
 * [g*ceil(B/G), (g+1)*ceil(B/G)), one per device; every device has its own engine handle driven by its own host thread,
 * parameters are uploaded per shard and every shard's results are written by DMA into the caller's result buffers (page-lock
 * them for direct DMA).  No collective on the path; results are bit-identical to a single-device run.  HOST arrays only.
 * `devices` NULL / ndev <= 0 = every visible device; a device may be listed more than once (several handles share it). */
typedef struct copra_b200_multi copra_b200_multi;
int copra_b200_multi_create(const int* devices, int ndev, copra_b200_multi** out);
void copra_b200_multi_destroy(copra_b200_multi* m);
const char* copra_b200_multi_last_error(const copra_b200_multi* m);
int copra_b200_multi_size(const copra_b200_multi* m);
/* device ordinal and instance range [lo, hi) of shard g in the last run */
int copra_b200_multi_shard(const copra_b200_multi* m, int g, int* device, int* lo, int* hi);
/* stage timings of shard g's last call and the host wall time of the whole sharded call */
int copra_b200_multi_timing(const copra_b200_multi* m, int g, copra_b200_timing* t, double* wall_ms);
long long copra_b200_multi_launch_count(const copra_b200_multi* m);
/* LMPC::solve for the whole batch (see copra_b200_lmpc_run) / receding-horizon re-solve (see copra_b200_lmpc_resolve) */
int copra_b200_multi_lmpc_run(copra_b200_multi* m, const copra_b200_problem* p, const copra_b200_results* r);
int copra_b200_multi_lmpc_resolve(copra_b200_multi* m, copra_b200_array x0, const copra_b200_results* r);
/* copra_b200_lmpc_retarget on every shard of the last run (same batch) */
int copra_b200_multi_lmpc_retarget(copra_b200_multi* m, const copra_b200_problem* p, const copra_b200_results* r);
/* copra_b200_lmpc_vjp on every shard of the last run; HOST arrays holding the whole batch */
int copra_b200_multi_lmpc_vjp(copra_b200_multi* m, const double* dcontrol, const double* dtrajectory, const copra_b200_vjp_out* out);
/* copra_b200_lmpc_vjp_costs on every shard of the last run; HOST arrays holding the whole batch */
int copra_b200_multi_lmpc_vjp_costs(copra_b200_multi* m, const double* dcontrol, const double* dtrajectory,
    const copra_b200_vjp_out* out, const copra_b200_vjp_cost_out* costs);
/* copra_b200_lmpc_vjp_model on every shard of the last run; HOST arrays holding the whole batch */
int copra_b200_multi_lmpc_vjp_model(copra_b200_multi* m, const double* dcontrol, const double* dtrajectory,
    const copra_b200_vjp_out* out, const copra_b200_vjp_cost_out* costs, const copra_b200_vjp_model_out* model);
/* copra_b200_lmpc_jvp / copra_b200_lmpc_feedback_gain on every shard of the last run; HOST arrays holding the whole batch */
int copra_b200_multi_lmpc_jvp(copra_b200_multi* m, const copra_b200_jvp_in* in, double* dcontrol, double* dtrajectory);
int copra_b200_multi_lmpc_feedback_gain(copra_b200_multi* m, int steps, double* Ku, double* Kx);
/* copra_b200_lmpc_vjp_initial_state / copra_b200_lmpc_jvp_initial_state on every shard of the last run; HOST arrays holding
 * the whole batch */
int copra_b200_multi_lmpc_vjp_initial_state(copra_b200_multi* m, const double* dcontrol, const double* dtrajectory,
    const copra_b200_vjp_out* out, const copra_b200_vjp_initial_out* init);
int copra_b200_multi_lmpc_jvp_initial_state(copra_b200_multi* m, const copra_b200_jvp_in* in, const copra_b200_jvp_initial_in* init,
    double* dcontrol, double* dtrajectory);
/* copra_b200_set_warm_start on every shard's handle */
int copra_b200_multi_set_warm_start(copra_b200_multi* m, int on);

#ifdef __cplusplus
}
#endif
#endif /* COPRA_B200_H */
