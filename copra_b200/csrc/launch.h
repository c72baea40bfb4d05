// launch.h -- host-callable launchers of the sm_100a kernels (internal to libcopra_b200.so).
#pragma once
#include "engine.cuh"
#include <cuda_runtime.h>

namespace cb {

struct GiBatch {
    int n, meq, m, batch;
    DArr Q, c, Aeq, beq, Aineq, bineq, lb, ub;
    double* x;    // n per instance (may be null)
    int* status;  // 1
    int* iters;   // 2
    int* nact;    // 1
    int* iact;    // n
    double* ws;   // global J / S workspace, ws_stride doubles per CTA (may be null if unused)
    long long ws_stride;
    int* counter; // zero-initialised work-queue cursor
    double vsmall;
    int max_iter;
    int j_smem, s_smem, a_smem;
    // gi_small_kernel only -- the factor J = R^-1 of every instance kept across a receding-horizon re-solve (the Hessian does
    // not change with x0): jmode 1 = store J (and jflag = 1 when Q was positive definite) after factoring, 2 = load it instead
    // of factoring (instances whose jflag is 0 factor again), 0 = off.  jcache: ld_vec2(n) * even(n) doubles per instance.
    double* jcache;
    int* jflag;
    int jmode;
};

struct GiPlan {
    int threads, grid, j_smem, s_smem, a_smem;
    int small; // 1: gi_small_kernel (n <= 64, all state in shared memory)
    int cluster; // > 0: gi_cluster_kernel with this cluster size (J distributed over DSMEM)
    size_t smem_bytes;
    long long ws_stride; // doubles per CTA of global workspace
};

// choose threads / smem residency / grid for a (n, meq, m) shape on a device with `sms` SMs; small_variant is
// copra_b200_options::small_variant (0 = the planner's choice)
GiPlan gi_plan(int n, int meq, int m, int batch, int sms, size_t smem_optin, int small_variant);
cudaError_t gi_launch(const GiBatch& B, const GiPlan& plan, cudaStream_t st);
double gi_vsmall();
// cluster path (gi_cluster.cuh): S workspace of odd_ld(n)*n doubles per cluster, sized by the caller
int gi_cluster_max_clusters(const GiPlan& plan);
cudaError_t gi_cluster_launch(const GiBatch& B, const GiPlan& plan, double* Sws, int nclusters, cudaStream_t st);

// K1 .. K7 of the batched LMPC engine.  Each returns the number of kernels it launched (>0) or a
// negative cudaError_t.
int k1_condense_launch(const BuildParams& P, cudaStream_t st);
int k1_psi_fill_launch(const double* Gs, long long sGs, double* Psi, int nx, int nu, int N, int batch, cudaStream_t st);
int k2k4_assemble_launch(const BuildParams& P, double* schur_ws, long long schur_stride, int sms, size_t smem_optin,
    cudaStream_t st);
// batched FP64 tensor-core GEMM (dgemm_dmma.cu): C = alpha op(A) B + beta C, column-major; returns launches or -cudaError
int dgemm_dmma_launch(int transA, int M, int N, int K, double alpha, const double* A, int lda, long long sA, const double* B, int ldb,
    long long sB, double beta, double* C, int ldc, long long sC, int batch, cudaStream_t st);
// measured DFMA / DMMA ceilings (fp64_peak.cu); 0 or -cudaError
int fp64_peaks_measure(int sms, double* scratch, cudaStream_t st, double* dfma_tflops, double* dmma_tflops);
// K3 alone: materialise the step-size rows of Aeq / Aineq (skipped by builds whose solver evaluates them from the tables)
int k3_fill_rows_launch(const BuildParams& P, cudaStream_t st);
// K2 for new per-instance vectors on a resident build: res / z (K2a) and every cost's f (K2c); Q, E, Y, the tables stay
int k2_retarget_launch(const BuildParams& P, int sms, cudaStream_t st);
int k4_finalize_launch(const BuildParams& P, int sms, cudaStream_t st);
int k7_results_launch(const BuildParams& P, const double* x, double* control, double* trajectory, cudaStream_t st);

// K8 / K9 (k8_k9_sens.cu): sensitivities of the last solve, one active-set KKT solve with k right-hand sides per instance, for
// the chunk of instances [b0, b0 + nb).  Buffers marked "chunk" hold nb instances; the others are indexed by the instance
// number in the batch.  SensChunk is what the VJP and the JVP share; per-instance vectors are len x k column-major.
struct SensChunk {
    int n;                           // decision variables (nU: LMPC mode)
    int nm;                          // the largest active-set size of the chunk (the padded width of slab, Y and G)
    int k;                           // right-hand sides: 1 for the VJP (2 with model gradients), the tangent directions for the JVP
    int lds, ldy, ldg;               // leading dimensions of slab / W / V, Y, J_G
    int b0;
    const int* status;
    const int* nact;
    const int* iact;                 // n per instance, 1-based [eq | ineq | upper | lower] indices
    const int* qpd;                  // 1 = the Hessian's factor Jt is valid (positive definite), qpd_stride apart per instance
    int qpd_stride;
    int plen[kMaxCost];              // per instance: each cost's p
    int flen[kMaxFam];               // per family: its constraint's f, or a trajectory bound's lower / upper
    int cblen;                       // the control bound's lower / upper
    double* slab;                    // chunk: lds x (nm + k)   [A_act' | gbar] or [A_act' | -cdot]
    double* Y;                       // chunk: ldy x (nm + k)   Jt' slab = [Y1 | T]
    double* Gf;                      // chunk: (nm + k)^2       Y'Y
    double* Gq;                      // chunk: nm x nm          G with 1 on the padded diagonal
    double* rhs;                     // chunk: nm x k           bdot_act (VJP: 0 | beta), then Y1' T - bdot_act (then VJP: mu | lambda)
    const double* GJ;                // chunk: ldg x nm         R_G^-1
    const int* gpd;                  // chunk: 1 = G positive definite
    double* W;                       // chunk: lds x k          T - Y1 M
    double* V;                       // chunk: lds x k          Jt W (v for the VJP, Udot for the JVP)
};
int sens_gram_launch(const SensChunk& S, int nb, cudaStream_t st);
int sens_solve_launch(const SensChunk& S, int nb, cudaStream_t st);

// K8: the vector-Jacobian product (k = 1); sens_solve leaves the multipliers mu of the active rows (iact order) in rhs.
// k8_cost_grad adds the gradients with respect to each cost's w, M and N from the same v.  With model gradients k = 2: the
// second right-hand side is the forward solve itself (slab column nm + 1 = -c, rhs column 1 = beta of the active rows), so
// rhs column 1 ends up holding the forward multipliers lambda that k8_model_grad needs next to mu.
struct VjpParams : SensChunk {
    const double* dcontrol;          // dL/dU (nU per instance, sdc apart), may be null
    long long sdc;
    const double* dtraj;             // dL/dtrajectory (X per instance, sdt apart), may be null
    long long sdt;
    // outputs (whole batch, zeroed by the caller; null = not wanted)
    double* dx0;                     // nx per instance
    double* dp[kMaxCost];
    double* df[kMaxFam];
    double* dlower;                  // control bound
    double* dupper;
    // cost gradients (k8_cost_grad; whole batch, zeroed by the caller; null = not wanted)
    const double* U;                 // the solution being differentiated, n per instance
    double* dw[kMaxCost];            // rows per instance
    double* dM[kMaxCost];            // rows x nx per instance, column-major
    double* dN[kMaxCost];            // rows x nu per instance, column-major
    // model gradients (k8_model_grad; whole batch, zeroed by the caller; null = not wanted; needs U and k = 2)
    double* dA;                      // nx x nx per instance, column-major
    double* dB;                      // nx x nu per instance, column-major
    double* dd;                      // nx per instance
    double* dE[kMaxFam];             // per row family (not the trajectory-bound selectors): rows x nx per instance, column-major
    double* dG[kMaxFam];             // rows x nu per instance, column-major
};
int k8_gather_launch(const BuildParams& P, const VjpParams& V, int nb, cudaStream_t st);
int k8_adjoint_launch(const BuildParams& P, const VjpParams& V, int nb, cudaStream_t st);
// shared memory of k8_cost_grad for the resident build (the caller checks it against the device's opt-in limit)
size_t k8_cost_grad_smem(const BuildParams& P);
int k8_cost_grad_launch(const BuildParams& P, const VjpParams& V, int nb, cudaStream_t st);
// the same for k8_model_grad
size_t k8_model_grad_smem(const BuildParams& P);
int k8_model_grad_launch(const BuildParams& P, const VjpParams& V, int nb, cudaStream_t st);

// K9: Jacobian-vector products along k tangent directions, or the feedback gain
struct JvpParams : SensChunk {
    int gain;                        // 1: the x0 tangents are the columns of the identity (k = nx), every other tangent zero
    // tangents (whole batch; null = zero)
    const double* tx0;               // nx
    const double* tp[kMaxCost];
    const double* tf[kMaxFam];
    const double* tlower;            // control bound
    const double* tupper;
    // outputs (whole batch, every entry written; null = not wanted)
    double* dcontrol;                // ru x k per instance: the first ru rows of Udot
    int ru;
    double* dtraj;                   // rx x k per instance: the first rx rows of Phi x0dot + Psi Udot
    int rx;
};
int k9_tangent_launch(const BuildParams& P, const JvpParams& J, int nb, cudaStream_t st);
int k9_output_launch(const BuildParams& P, const JvpParams& J, int nb, cudaStream_t st);

} // namespace cb
