// engine.cuh -- device-side descriptors shared by the K1..K7 kernels of the batched LMPC engine.
//
// Everything the reference builds per controller (PreviewSystem + a list of CostFunction /
// Constraint objects, reference include/LMPC.h:166-185) is flattened into "families":
//   cost family      : sum over steps i in [i0,i1) of (T_i U + MPhi_i x0 + res_i)' W (...)
//                      with T_i[:, block j] = M A^(i-1-j) B (j < i), N (j == i), 0 (j > i)
//   constraint family: row block i in [i0,i1):  (E Phi_i) x0 + A_i U  (<=,==)  f - E xi_i
//                      with A_i[:, block j] = E A^(i-1-j) B (j < i), G (j == i), 0 (j > i)
// which covers the four step-size costs (src/costFunctions.cpp:63-215) and the four step-size row
// constraints (src/constraints.cpp:66-315); TrajectoryBoundConstraint becomes up to two selector
// families (lower lines first, then upper lines -- quirk Q1 keeps the lower rows un-negated).
// res_i = M xi_i - p_i and the right-hand side f_i may differ from step to step (COPRA_B200_PER_STEP: pstep / fstep); the
// matrices, hence the Hessian and the rows, may not.
#pragma once
#include <cuda_runtime.h>

namespace cb {

// odd leading dimension => conflict-free shared-memory sweeps along rows and along columns
__host__ __device__ inline int odd_ld(int n) { return (n | 1); }

constexpr int kMaxCost = 8;
constexpr int kMaxFam = 16;

struct DArr { // (pointer, batch stride) on the device
    const double* p;
    long long s;
    __host__ __device__ const double* at(int b) const { return p + (long long)b * s; }
};

struct CostFam {
    int dense;      // 1: full-size entry: M is rows x X, N rows x nU; evaluated by the DMMA GEMM path
    int pstep;      // doubles between the p of consecutive steps (per-step vector, COPRA_B200_PER_STEP); 0 = one p for every step
    double* T;      // dense: rows x nU   T = M Psi (+ N)
    double* WT;     // dense: rows x nU   diag(w) T
    long long sT;
    int rows;       // r
    int i0, i1;     // step range
    int hasM, hasN;
    DArr M, N, p, w;
    // per-instance scratch (device), strides in doubles per instance
    double* MGx;    // r x nu x (N+1): block k+1 = M A^k B, block 0 = N (or 0)
    double* MPhi;   // r x nx x (i1-i0)
    double* res;    // r x (i1-i0)
    double* E;      // nx x nU : this cost's E()
    double* f;      // nU      : this cost's f()
    long long sMGx, sMPhi, sres, sE, sf;
};

struct CstrFam {
    int dense;      // 1: full-size entry (E rows x X, G rows x nU): rows = E Psi + G by the DMMA GEMM path
    int gather;     // 1: rows are copies of Psi/Phi/xi rows fidx[] (full-size TrajectoryBoundConstraint)
    int rows;       // r
    int i0, i1;
    int hasE, hasG;
    int is_eq;
    int row_off;    // first row inside Aeq (is_eq) or Aineq
    int fstep;      // doubles between the f of consecutive steps (per-step vector; nx for a trajectory bound); 0 = one f
    DArr E, G, f;
    const int* fidx; // optional gather of f (TrajectoryBound: line numbers), device, `rows` entries
    double* EGx;    // r x nu x (N+1): block k+1 = E A^k B, block 0 = G (or 0)
    long long sEGx;
};

struct BuildParams {
    int nx, nu, N, batch;
    int X, nU, nvar, meq, mineq;
    int initial_state;
    int ncost, nfam;
    double qdiag;                 // 1e-6 (LMPC::updateSystem) or 0
    DArr A, B, d, x0;
    DArr R, r, x0lb, x0ub;        // initial-state mode (p may be null)
    DArr cb_lower, cb_upper;      // ControlBoundConstraint (p null = none)
    int cb_full;                  // 1: lower/upper hold nU entries (full-size or per-step entry)
    int skip_rows;                // 1: Aeq / Aineq are not materialised by the build (structured solver; filled on demand)
    double* PsiFull;              // X x nU per instance, only materialised when a full-size entry needs it
    // K1 outputs (workspace, per instance)
    double* Phi;   // X x nx
    double* Gs;    // (N*nx) x nu  == Psi[nx:, 0:nu]
    double* xi;    // X
    // assembled QP (per instance)
    double* Q;     // nvar x nvar
    long long sQ;  // doubles between the Hessians of consecutive instances; 0 = batch-invariant Hessian (one copy)
    double* c;     // nvar
    double* Aeq;   // meq x nvar
    double* beq;
    double* Aineq; // mineq x nvar
    double* bineq;
    double* lb;
    double* ub;
    double* Yeq;   // meq x nx    (E Phi_i rows)
    double* zeq;   // meq
    double* Yin;   // mineq x nx
    double* zin;   // mineq
    CostFam cost[kMaxCost];
    CstrFam fam[kMaxFam];
};

} // namespace cb
