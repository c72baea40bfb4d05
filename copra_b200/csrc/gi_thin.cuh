// gi_thin.cuh -- K5+K6 for n > 64: a THROUGHPUT-oriented Goldfarb-Idnani solver, one CTA per instance on one SM.
//
// Same problem, index space, selection / step / drop rules and fail codes as gi_solver.cuh (QuadProgDenseSolver::SI_solve,
// reference src/QuadProgSolver.cpp:54-72, and qpgen2 behind it, SURVEY.md 3.3); what changes is the representation of the
// factorisation, chosen so that the per-instance MUTABLE state is small and the big matrix is read-only:
//
//   qpgen2 / gi_solver.cuh : J = R^-1 Qfull  (n x n, rewritten by every add / drop)           -> 8 n^2 bytes of state
//   here                   : Jt = R^-1       (n x n upper triangular, NEVER modified; one copy per distinct Hessian --
//                                             a single one for the whole batch when the Hessian is batch-invariant)
//                            Q1 = first nact columns of Qfull (n x nact, orthonormal)          -> 8 n nact bytes
//                            S  = (Q1' Jt' N)^-1 (nact x nact)                                 -> 8 nact^2 bytes
//   d  = Jt' a (triangular mat-vec),  d1 = Q1' d,  zt = d - Q1 d1 (= Q2 Q2' d),  z = Jt zt,  r = S d1
//   ADD  : Q1 gains the column zt/|zt|, S the column [-r/|zt| ; 1/|zt|]   (no rotation of anything)
//   DROP : one reflection of Q1 and S whose last column is the dropped row of S (as in gi_solver.cuh)
// In exact arithmetic d1, |d2| = |zt|, z, r and therefore every iterate are those of qpgen2.
//
// Because Jt is read-only it is factored ONCE per distinct Hessian by gt_factor_kernel (blocked DMMA Cholesky + inverse,
// gi_factor.cuh) instead of once per solve, it is shared by every CTA through L2, and a receding-horizon re-solve reuses it.
//
// General rows [Aeq; Aineq] of a step-size LMPC are block-Toeplitz (row of step i, block column j = E A^(i-1-j) B, G at
// j == i; reference src/constraints.cpp:77,142,209-219): their products with x are evaluated straight from the per-family
// r x nu x (N+1) tables in shared memory (a causal convolution), so the m x n matrix is never read by the solver.  A dense
// mode (rows streamed from global memory) serves full-size entries.
#pragma once
#include "common.cuh"
#include "engine.cuh"
#include "gi_solver.cuh"
#include <cooperative_groups.h>
#include <cfloat>
#ifdef GT_PROFILE
#include <cstdio>
#define GT_T(k) do { const long long t1_ = clock64(); gt_acc[k] += t1_ - gt_t0; gt_t0 = t1_; } while (0)
#else
#define GT_T(k) do { } while (0)
#endif

namespace cb {

namespace cg = cooperative_groups;

// Communication policy of the thin solver.
//   GtSolo : one CTA per instance (the throughput configuration: C3).
//   GtClus : one thread-block CLUSTER per instance (the latency configuration for n > 512 with per-instance factors: C5, whose
//            step is the latency of its heaviest instance).  Every heavy stream (the factor, Q1, S, the Toeplitz products) is
//            split over the CTAs; every small vector is REPLICATED: a producer stores its entries at the same shared-memory
//            address of every CTA (DSMEM) with put(), and one cluster barrier publishes them.  All CTAs run the same control
//            flow on bitwise identical replicas, so no decision is ever exchanged.  Q1 and S live in global memory (L2) and are
//            written in disjoint pieces; the cluster barrier (release / acquire at cluster scope) orders those writes too.
//            INTERVAL RULE that makes the remote stores safe: between two consecutive cluster barriers a replicated buffer is
//            either only read or only written through put() -- never both -- because CTAs drift apart by up to one interval
//            (local __syncthreads do not align them).  Hence the cluster barrier after the load phase (no put() may land before
//            a replica is initialised), at the start of a drop (every replica has finished reading r / w of the step update)
//            and after every phase whose outputs are put().
struct GtSolo {
    static constexpr bool multi = false;
    __device__ __forceinline__ int rank() const { return 0; }
    __device__ __forceinline__ int size() const { return 1; }
    __device__ __forceinline__ void sync() const { __syncthreads(); }
    template <class T> __device__ __forceinline__ void put(T* p, T v) const { *p = v; }
};
struct GtClus {
    static constexpr bool multi = true;
    int r, c;
    __device__ __forceinline__ int rank() const { return r; }
    __device__ __forceinline__ int size() const { return c; }
    __device__ __forceinline__ void sync() const { cg::this_cluster().sync(); }
    template <class T> __device__ __forceinline__ void put(T* p, T v) const
    {
        cg::cluster_group g = cg::this_cluster();
        for (int k = 0; k < c; ++k) *g.map_shared_rank(p, k) = v;
    }
};

struct GtLayout {
    size_t oTab, oSS, oX, oXt, oD, oZt, oZ, oAv, oR, oU, oD1, oW, oV, oLb, oUb, oSl, oB, oNorm, oRed, oPart, oQ1; // doubles
    size_t oIact, oRowmap, oRedI, oActive, oSgn, bytes;                                                       // bytes
};

// offsets (doubles) inside the state-space area W.ss
struct GtSS { int oG, oP, oPL, oSt, oSc, oEG, total; };

struct GtFam {
    int rows, i0, i1, is_eq, row_off; // row_off: first row inside Aeq (is_eq) or Aineq
    int tab;                          // offset of this family's table in the shared-memory table area (doubles)
    const double* EGx;                // r x nu x (N+1) per instance: block kk = E A^(kk-1) B (kk >= 1), G | 0 (kk == 0)
    long long sEGx;
    DArr E, G;                        // the family's own r x nx / r x nu blocks (null when absent): used with Dpsi
};

struct GtBatch {
    int n, meq, m, batch;
    int structured, nu, N, nfam, tab_doubles;
    int ldk;            // row length of the transposed tables in shared memory ((N+1) | 1)
    int ld;             // leading dimension of Jt, JtT, Q1 (n rounded up to even: 16-byte aligned columns for 128-bit loads)
    int q1s;            // columns of Q1 held in shared memory (the rest lives in the global workspace)
    double reorth;      // second Gram-Schmidt pass when |zt|^2 < reorth * |d|^2
    GtFam fam[kMaxFam];
    // Batch-invariant system AND Hessian: Dpsi = Jt' Psi' (ld x X, column-major) is formed once per batch by the DMMA GEMM,
    // and d = Jt' a for the step-size row (family, step, line) is  sum_e E[line,e] Dpsi[:, step nx + e] + sum_b G[line,b] Jt'[:, step nu + b]
    // -- nx + nu short column reads instead of a triangular mat-vec over Jt (null: per-instance systems, mat-vec path)
    const double* Dpsi;
    // With them H = Jt Jt' (= Q^-1, ld x n) and Hpsi = Jt Dpsi (= H Psi', ld x X), the SHARED-FACTOR FORM of the pass: the
    // solver stores P = Jt Q1 INSTEAD of Q1 (P' Q P = I) and never touches the factor in the iterations:
    //   h = Jt d = H a (nx + nu column reads of Hpsi / H)      d1 = Q1' d = P' R' Jt' a = P' a      z = Jt zt = h - P d1
    //   |zt|^2 = d' zt = a' z      |d|^2 = a' h      ADD: P gains z / |zt|      DROP: the same reflection, applied to P
    // -- one sweep over P (gt_pass_fused; two for n > 320) and one over S per pass, nothing else.  Null: the general form (Q1, z = Jt zt).
    const double* Hpsi;
    const double* Hm;
    const double* Qs;   // the shared Hessian (n x n), only for the rare second orthogonalisation pass (v = P' Q z)
    int nx, X;
    // State-space evaluation of the general rows (gt_products_ss): row (step i, line) of a step-size family is
    // E s_i + G u_i with s_i = sum_{j<i} A^(i-1-j) B u_j the zero-state response -- O(N (L nu + nx) nx) flops through chunks of
    // L steps instead of the O(m n / 2) convolution.  Phi / Gs: K1's A^k and A^k B blocks of this instance.
    int ss, ssL, ssC, ss_doubles;
    DArr Phi, Gs;
    // shared-memory layout, computed ONCE on the host (gt_layout / gt_ss_layout with the launch's thread count): the kernel reads
    // the offsets from the constant bank instead of re-deriving them wherever a pointer is re-materialised
    GtLayout lay;
    GtSS ssl;
    DArr Jt, JtT;       // R^-1 column-major (entries i <= j of column j) and its transpose (entries j >= i of column i)
    const int* pd;      // 1 = Hessian positive definite, per distinct Hessian
    int pd_stride;      // 0 (shared) or 1
    DArr c, Aeq, beq, Aineq, bineq, lb, ub;
    double* x;
    int *status, *iters, *nact, *iact;
    double* ws;         // per CTA: Q1 (ld x n) then S (n x n, ld n)
    long long ws_stride;
    int* counter;
    double vsmall;
    int max_iter;
    // Scheduling of heavy-tailed batches (iteration counts of C5 range from 10 to > 2000 passes): a PREPASS launch computes,
    // per instance, the number of constraints violated at the unconstrained minimiser (correlation with the work: 0.92) into
    // `prekey`; the solve launch then pulls instances in `order` (descending key: longest first), so the heaviest instance
    // starts at t = 0 instead of wherever the index order put it.  Both null: index order.
    int* prekey;
    int* preidx;
    const int* order;
    const int* warm; // previous active sets (n ints per instance, 1-based, 0-terminated) seeding the shared-factor form; null: cold
    int kheavy; // cluster kernel: queue entries [0, kheavy) are solved by whole clusters, the rest by single CTAs
};

__host__ __device__ inline int gt_even(int n) { return (n + 1) & ~1; }

// `q1s` columns of Q1 (ld doubles each) are placed right after the vectors
__host__ __device__ inline GtLayout gt_layout(int n, int meq, int m, int tab_doubles, int threads, int q1s, int ss_doubles = 0)
{
    GtLayout L;
    const int mg = gt_even(meq + m), np = gt_even(n);
    size_t o = 0;
    L.oTab = o; o += (size_t(tab_doubles) + 1) & ~size_t(1);
    L.oSS = o; o += (size_t(ss_doubles) + 1) & ~size_t(1);
    L.oX = o; o += np;
    L.oXt = o; o += np;
    L.oD = o; o += np;
    L.oZt = o; o += np;
    L.oZ = o; o += np;
    L.oAv = o; o += np;
    L.oR = o; o += np;
    L.oU = o; o += np + 2;
    L.oD1 = o; o += np;
    L.oW = o; o += np;
    L.oV = o; o += np;
    L.oLb = o; o += np;
    L.oUb = o; o += np;
    L.oSl = o; o += mg;
    L.oB = o; o += mg;
    L.oNorm = o; o += mg;
    L.oRed = o; o += 10 * kMaxWarps;
    {
        const size_t trap = (size_t(2 * (threads / 32) + (n + 63) / 64 + 2) << 6) + 2 * size_t(threads);
        const size_t pass = 6 * size_t(threads); // gt_pass_rows: P partials (2T) + S partials (T); twice that for gt_pass_rows2
        L.oPart = o; o += trap > pass ? trap : pass;
    }
    L.oQ1 = o; o += size_t(q1s) * np;
    size_t b = o * sizeof(double);
    L.oIact = b; b += sizeof(int) * size_t(n);
    L.oRowmap = b; b += sizeof(int) * size_t(n);
    L.oRedI = b; b += sizeof(int) * 3 * kMaxWarps;
    L.oActive = b; b += size_t(mg + 2 * n);
    L.oSgn = b; b += size_t(meq > 0 ? meq : 1);
    L.bytes = (b + 15) & ~size_t(15);
    return L;
}

struct GtWork {
    double *tab, *ss, *x, *xt, *d, *zt, *z, *av, *r, *u, *d1, *w, *v, *lb, *ub, *sl, *bv, *norm, *red, *part;
    int *iact, *rowmap, *redi;
    unsigned char* active;
    signed char* sgn;
    double *Q1s, *Q1, *S; // Q1s: columns [0, q1s) in shared memory; Q1: global, column c at Q1 + c * ld (c >= q1s used)
};

__device__ inline GtWork gt_carve(const GtLayout& L, unsigned char* smem, double* ws, int n)
{
    GtWork W;
    double* base = reinterpret_cast<double*>(smem);
    W.tab = base + L.oTab; W.ss = base + L.oSS; W.x = base + L.oX; W.xt = base + L.oXt; W.d = base + L.oD; W.zt = base + L.oZt; W.z = base + L.oZ;
    W.av = base + L.oAv; W.r = base + L.oR; W.u = base + L.oU; W.d1 = base + L.oD1; W.w = base + L.oW; W.v = base + L.oV;
    W.lb = base + L.oLb; W.ub = base + L.oUb; W.sl = base + L.oSl; W.bv = base + L.oB; W.norm = base + L.oNorm;
    W.red = base + L.oRed; W.part = base + L.oPart;
    W.iact = reinterpret_cast<int*>(smem + L.oIact);
    W.rowmap = reinterpret_cast<int*>(smem + L.oRowmap);
    W.redi = reinterpret_cast<int*>(smem + L.oRedI);
    W.active = smem + L.oActive;
    W.sgn = reinterpret_cast<signed char*>(smem + L.oSgn);
    W.Q1s = base + L.oQ1;
    W.Q1 = ws;
    W.S = ws + size_t(gt_even(n)) * n;
    return W;
}

// ---- triangular mat-vecs against the read-only factor ---------------------------------------------------------------
// y = M x restricted to a trapezoid of a column-major matrix: rows are cut into chunks of 64 (a lane owns a PAIR of rows:
// one 128-bit load per column, no predicate, no shuffle), chunk k sums the columns [clo(k), chi(k)).  The (chunk, column
// slice) pairs form a static task list dealt to the warps; partial sums meet in `part` in task order (deterministic).
//   ZMODE : z[i] = sum_{j >= i} Jt[i, j] v[j]      on M = Jt  : clo = 64 k, chi = n      (stored zeros below the diagonal)
//   !ZMODE: d[j] = sum_{i <= j, i < supp} Jt[i, j] a[i]  on M = JtT : clo = 0, chi = min(64 k + 64, supp)
// Contains one __syncthreads; the caller syncs before reading `out`.
// With a cluster the 64-row chunks are dealt to the CTAs in a snake (the work of a chunk is linear in its index), each CTA
// runs the task list of ITS chunks and publishes their rows to every replica.
template <bool ZMODE, class CL>
__device__ __forceinline__ void gt_trap_mv(const CL& cl, const double* __restrict__ M, int ld, int n, int supp, const double* __restrict__ vec,
    double* __restrict__ out, double* __restrict__ part)
{
    const int lane = lane_id(), wp = warp_id(), nw = blockDim.x >> 5;
    const int nc = (n + 63) >> 6, C = cl.size(), me = cl.rank();
    auto clo = [&](int k) { return ZMODE ? (k << 6) : 0; };
    auto chi = [&](int k) { return ZMODE ? n : min(min((k << 6) + 64, supp), n); };
    auto mine = [&](int k) { const int rr = k % (2 * C); return (rr < C ? rr : 2 * C - 1 - rr) == me; };
    int tot = 0;
    for (int k = 0; k < nc; ++k) if (mine(k)) tot += chi(k) - clo(k);
    const int cw = max(64, (((tot + 2 * nw - 1) / (2 * nw)) + 63) & ~63); // columns per task
    int ntask = 0;
    for (int k = 0; k < nc; ++k) if (mine(k)) ntask += (chi(k) - clo(k) + cw - 1) / cw;
    for (int t = wp; t < ntask; t += nw) {
        int k = 0, t0 = 0;
        for (;; ++k) {
            if (!mine(k)) continue;
            const int nt = (chi(k) - clo(k) + cw - 1) / cw;
            if (t < t0 + nt) break;
            t0 += nt;
        }
        const int c0 = clo(k) + (t - t0) * cw, c1 = min(chi(k), c0 + cw);
        const int row = (k << 6) + 2 * lane;
        double2 acc[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) acc[u] = make_double2(0.0, 0.0);
        if (row < ld) {
            const double* mp = M + row + size_t(c0) * ld;
            int j = c0;
            for (; j + 7 < c1; j += 8, mp += 8 * size_t(ld)) {
                double2 a[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) a[u] = __ldg(reinterpret_cast<const double2*>(mp + u * size_t(ld)));
#pragma unroll
                for (int u = 0; u < 8; u += 2) {
                    const double2 x = *reinterpret_cast<const double2*>(vec + j + u);
                    acc[u >> 1].x = fma(a[u].x, x.x, acc[u >> 1].x);
                    acc[u >> 1].y = fma(a[u].y, x.x, acc[u >> 1].y);
                    acc[u >> 1].x = fma(a[u + 1].x, x.y, acc[u >> 1].x);
                    acc[u >> 1].y = fma(a[u + 1].y, x.y, acc[u >> 1].y);
                }
            }
            for (; j < c1; ++j, mp += ld) {
                const double2 a = __ldg(reinterpret_cast<const double2*>(mp));
                const double x = vec[j];
                acc[0].x = fma(a.x, x, acc[0].x);
                acc[0].y = fma(a.y, x, acc[0].y);
            }
        }
        double2 r_;
        r_.x = (acc[0].x + acc[1].x) + (acc[2].x + acc[3].x);
        r_.y = (acc[0].y + acc[1].y) + (acc[2].y + acc[3].y);
        *reinterpret_cast<double2*>(part + (size_t(t) << 6) + 2 * lane) = r_;
    }
    __syncthreads();
    for (int r = threadIdx.x; r < n; r += blockDim.x) {
        const int k = r >> 6;
        if (!mine(k)) continue;
        int t0 = 0;
        for (int kk = 0; kk < k; ++kk) if (mine(kk)) t0 += (chi(kk) - clo(kk) + cw - 1) / cw;
        const int nt = (chi(k) - clo(k) + cw - 1) / cw;
        double sum = 0.0;
        for (int q = 0; q < nt; ++q) sum += part[(size_t(t0 + q) << 6) + (r & 63)];
        cl.put(out + r, sum);
    }
}

// out[c] = Q1[:, c] . vec for c in [0, nact): an 8-lane group per column (128-bit loads, three shuffles per column), head
// columns from shared memory, the rest from the global workspace
template <class CL>
__device__ __forceinline__ void gt_q1_col_dots(const CL& cl, const GtWork& W, int n, int ld, int q1s, int nact, const double* __restrict__ vec,
    double* __restrict__ out, int rows = 1 << 30)
{
    // `rows`: entries of vec past it are zero (the causal support of a step-size row) -- the columns are read only that far
    const int kend = min(ld, (rows + 15) & ~15);
    const int lane = lane_id(), wp = warp_id(), nw = blockDim.x >> 5;
    const int g8 = lane >> 3, l8 = lane & 7;
    (void)n;
    // blocks of four columns are dealt over the CTAs first, then over the warps
    for (int cb = 4 * (cl.rank() + cl.size() * wp); cb < nact; cb += 4 * nw * cl.size()) {
        const int c = cb + g8;
        const bool on = c < nact;
        const double* col = (c < q1s ? W.Q1s : W.Q1) + size_t(on ? c : 0) * ld;
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
        if (on) {
            int k = 2 * l8;
            for (; k + 48 < kend; k += 64) {
                const double2 a0 = *reinterpret_cast<const double2*>(col + k), a1 = *reinterpret_cast<const double2*>(col + k + 16);
                const double2 a2 = *reinterpret_cast<const double2*>(col + k + 32), a3 = *reinterpret_cast<const double2*>(col + k + 48);
                const double2 x0 = *reinterpret_cast<const double2*>(vec + k), x1 = *reinterpret_cast<const double2*>(vec + k + 16);
                const double2 x2 = *reinterpret_cast<const double2*>(vec + k + 32), x3 = *reinterpret_cast<const double2*>(vec + k + 48);
                s0 = fma(a0.y, x0.y, fma(a0.x, x0.x, s0));
                s1 = fma(a1.y, x1.y, fma(a1.x, x1.x, s1));
                s2 = fma(a2.y, x2.y, fma(a2.x, x2.x, s2));
                s3 = fma(a3.y, x3.y, fma(a3.x, x3.x, s3));
            }
            if (k < kend) { // up to three 16-row slices left: one round trip
                const bool h1 = k + 16 < kend, h2 = k + 32 < kend;
                const double2 zero = make_double2(0.0, 0.0);
                const double2 a0 = *reinterpret_cast<const double2*>(col + k);
                const double2 a1 = h1 ? *reinterpret_cast<const double2*>(col + k + 16) : zero;
                const double2 a2 = h2 ? *reinterpret_cast<const double2*>(col + k + 32) : zero;
                const double2 x0 = *reinterpret_cast<const double2*>(vec + k);
                const double2 x1 = h1 ? *reinterpret_cast<const double2*>(vec + k + 16) : zero;
                const double2 x2 = h2 ? *reinterpret_cast<const double2*>(vec + k + 32) : zero;
                s0 = fma(a0.y, x0.y, fma(a0.x, x0.x, s0));
                s1 = fma(a1.y, x1.y, fma(a1.x, x1.x, s1));
                s2 = fma(a2.y, x2.y, fma(a2.x, x2.x, s2));
            }
        }
        double q = (s0 + s1) + (s2 + s3);
        q += __shfl_xor_sync(0xffffffffu, q, 4);
        q += __shfl_xor_sync(0xffffffffu, q, 2);
        q += __shfl_xor_sync(0xffffffffu, q, 1);
        if (on && l8 == 0) cl.put(out + c, q);
    }
}

// out[r] = sum_{c < nact} Q1[r, c] * vec[c]: a thread owns a PAIR of rows (one 128-bit load per column), the column range
// is split over G = T / round32(ld / 2) thread groups whose partial sums meet in `part` (fixed order).  One __syncthreads
// inside when G > 1; the caller syncs before reading `out`.
template <class CL>
__device__ __forceinline__ void gt_q1_row_dots(const CL& cl, const GtWork& W, int ld, int q1s, int nact, const double* __restrict__ vec,
    double* __restrict__ out, double* __restrict__ part)
{
    const int tid = threadIdx.x, T = blockDim.x;
    const int all = ld >> 1, per = (all + cl.size() - 1) / cl.size();          // row pairs: a contiguous slab per CTA
    const int p0 = min(all, cl.rank() * per), pairs = min(all, p0 + per) - p0;
    const int rp = max(32, round32(pairs));
    const int G = max(1, T / rp);
    auto colp = [&](int c) -> const double* { return (c < q1s ? W.Q1s : W.Q1) + size_t(c) * ld + 2 * p0; };
    if (T < rp) { // more row pairs than threads: loop over pairs, all columns per thread (four loads in flight)
        for (int pr = tid; pr < pairs; pr += T) {
            double2 s0 = make_double2(0.0, 0.0), s1 = s0, s2 = s0, s3 = s0;
            int c = 0;
            for (; c + 3 < nact; c += 4) {
                const double2 a0 = *reinterpret_cast<const double2*>(colp(c) + 2 * pr), a1 = *reinterpret_cast<const double2*>(colp(c + 1) + 2 * pr);
                const double2 a2 = *reinterpret_cast<const double2*>(colp(c + 2) + 2 * pr), a3 = *reinterpret_cast<const double2*>(colp(c + 3) + 2 * pr);
                s0.x = fma(a0.x, vec[c], s0.x); s0.y = fma(a0.y, vec[c], s0.y);
                s1.x = fma(a1.x, vec[c + 1], s1.x); s1.y = fma(a1.y, vec[c + 1], s1.y);
                s2.x = fma(a2.x, vec[c + 2], s2.x); s2.y = fma(a2.y, vec[c + 2], s2.y);
                s3.x = fma(a3.x, vec[c + 3], s3.x); s3.y = fma(a3.y, vec[c + 3], s3.y);
            }
            for (; c < nact; ++c) {
                const double2 a0 = *reinterpret_cast<const double2*>(colp(c) + 2 * pr);
                s0.x = fma(a0.x, vec[c], s0.x); s0.y = fma(a0.y, vec[c], s0.y);
            }
            cl.put(out + 2 * (p0 + pr), (s0.x + s1.x) + (s2.x + s3.x));
            cl.put(out + 2 * (p0 + pr) + 1, (s0.y + s1.y) + (s2.y + s3.y));
        }
        return;
    }
    const int g = tid / rp, pr = tid - g * rp;
    double2 s0 = make_double2(0.0, 0.0), s1 = s0, s2 = s0, s3 = s0;
    if (g < G && pr < pairs) {
        int c = g;
        for (; c + 3 * G < nact; c += 4 * G) {
            const double2 a0 = *reinterpret_cast<const double2*>(colp(c) + 2 * pr), a1 = *reinterpret_cast<const double2*>(colp(c + G) + 2 * pr);
            const double2 a2 = *reinterpret_cast<const double2*>(colp(c + 2 * G) + 2 * pr), a3 = *reinterpret_cast<const double2*>(colp(c + 3 * G) + 2 * pr);
            s0.x = fma(a0.x, vec[c], s0.x); s0.y = fma(a0.y, vec[c], s0.y);
            s1.x = fma(a1.x, vec[c + G], s1.x); s1.y = fma(a1.y, vec[c + G], s1.y);
            s2.x = fma(a2.x, vec[c + 2 * G], s2.x); s2.y = fma(a2.y, vec[c + 2 * G], s2.y);
            s3.x = fma(a3.x, vec[c + 3 * G], s3.x); s3.y = fma(a3.y, vec[c + 3 * G], s3.y);
        }
        for (; c < nact; c += G) {
            const double2 a0 = *reinterpret_cast<const double2*>(colp(c) + 2 * pr);
            s0.x = fma(a0.x, vec[c], s0.x); s0.y = fma(a0.y, vec[c], s0.y);
        }
    }
    const double sx = (s0.x + s1.x) + (s2.x + s3.x), sy = (s0.y + s1.y) + (s2.y + s3.y);
    if (G == 1) {
        if (g == 0 && pr < pairs) { cl.put(out + 2 * (p0 + pr), sx); cl.put(out + 2 * (p0 + pr) + 1, sy); } // threads past the last full group idle
        return;
    }
    if (g < G && pr < pairs) {
        part[2 * (g * rp + pr)] = sx;
        part[2 * (g * rp + pr) + 1] = sy;
    }
    __syncthreads();
    if (tid < pairs) {
        double ax = part[2 * tid], ay = part[2 * tid + 1];
        for (int k = 1; k < G; ++k) { ax += part[2 * (k * rp + tid)]; ay += part[2 * (k * rp + tid) + 1]; }
        cl.put(out + 2 * (p0 + tid), ax);
        cl.put(out + 2 * (p0 + tid) + 1, ay);
    }
}

// Q1[:, c] -= wv * cv[c] for c in [0, ncols): a thread owns a pair of rows, the columns are split over the thread groups and
// taken four at a time (four independent 128-bit loads in flight, then four stores)
template <class CL>
__device__ __forceinline__ void gt_q1_rank1(const CL& cl, const GtWork& W, int ld, int q1s, int ncols, const double* __restrict__ wv,
    const double* __restrict__ cv)
{
    const int tid = threadIdx.x, T = blockDim.x;
    const int all = ld >> 1, per = (all + cl.size() - 1) / cl.size();
    const int p0 = min(all, cl.rank() * per), pairs = min(all, p0 + per) - p0;
    const int rp = max(32, round32(pairs));
    const int G = max(1, T / rp);
    auto colp = [&](int c) -> double* { return (c < q1s ? W.Q1s : W.Q1) + size_t(c) * ld + 2 * p0; };
    for (int pr = (T < rp) ? tid : (tid % rp), g = (T < rp) ? 0 : tid / rp; pr < pairs && g < G; pr += (T < rp) ? T : pairs + rp) {
        const double2 w = *reinterpret_cast<const double2*>(wv + 2 * (p0 + pr));
        int c = g;
        for (; c + 3 * G < ncols; c += 4 * G) {
            double2* p0 = reinterpret_cast<double2*>(colp(c) + 2 * pr);
            double2* p1 = reinterpret_cast<double2*>(colp(c + G) + 2 * pr);
            double2* p2 = reinterpret_cast<double2*>(colp(c + 2 * G) + 2 * pr);
            double2* p3 = reinterpret_cast<double2*>(colp(c + 3 * G) + 2 * pr);
            double2 a0 = *p0, a1 = *p1, a2 = *p2, a3 = *p3;
            const double c0 = cv[c], c1 = cv[c + G], c2 = cv[c + 2 * G], c3 = cv[c + 3 * G];
            a0.x = fma(-w.x, c0, a0.x); a0.y = fma(-w.y, c0, a0.y);
            a1.x = fma(-w.x, c1, a1.x); a1.y = fma(-w.y, c1, a1.y);
            a2.x = fma(-w.x, c2, a2.x); a2.y = fma(-w.y, c2, a2.y);
            a3.x = fma(-w.x, c3, a3.x); a3.y = fma(-w.y, c3, a3.y);
            *p0 = a0; *p1 = a1; *p2 = a2; *p3 = a3;
        }
        for (; c < ncols; c += G) {
            double2* p0 = reinterpret_cast<double2*>(colp(c) + 2 * pr);
            double2 a0 = *p0;
            const double c0 = cv[c];
            a0.x = fma(-w.x, c0, a0.x); a0.y = fma(-w.y, c0, a0.y);
            *p0 = a0;
        }
    }
}

// S[rowmap[r], c] -= rv[r] * cv[c] for r in [0, rows) except `skip`, c in [0, ncols): lanes along rows, columns split over
// thread groups, four at a time
template <class CL>
__device__ __forceinline__ void gt_s_rank1(const CL& cl, double* __restrict__ S, size_t lds, const int* __restrict__ rowmap, int rows_all, int skip,
    int ncols, const double* __restrict__ rv, const double* __restrict__ cv)
{
    const int tid = threadIdx.x, T = blockDim.x;
    const int per = (rows_all + cl.size() - 1) / cl.size(), r0 = min(rows_all, cl.rank() * per), rows = min(rows_all, r0 + per) - r0;
    const int rp = max(32, round32(rows));
    const int G = max(1, T / rp);
    rowmap += r0; rv += r0; skip -= r0;
    for (int r = (T < rp) ? tid : (tid % rp), g = (T < rp) ? 0 : tid / rp; r < rows && g < G; r += (T < rp) ? T : rows + rp) {
        if (r == skip) continue;
        double* sr = S + rowmap[r];
        const double ri = rv[r];
        int c = g;
        for (; c + 3 * G < ncols; c += 4 * G) {
            double a0 = sr[size_t(c) * lds], a1 = sr[size_t(c + G) * lds], a2 = sr[size_t(c + 2 * G) * lds], a3 = sr[size_t(c + 3 * G) * lds];
            a0 = fma(-ri, cv[c], a0); a1 = fma(-ri, cv[c + G], a1); a2 = fma(-ri, cv[c + 2 * G], a2); a3 = fma(-ri, cv[c + 3 * G], a3);
            sr[size_t(c) * lds] = a0; sr[size_t(c + G) * lds] = a1; sr[size_t(c + 2 * G) * lds] = a2; sr[size_t(c + 3 * G) * lds] = a3;
        }
        for (; c < ncols; c += G) sr[size_t(c) * lds] = fma(-ri, cv[c], sr[size_t(c) * lds]);
    }
}

// out[r] = sum_{c in [c0,c1)} M[rowof(r) + c*ld] * vec[c], r in [0, rows) -- the S mat-vecs (rows through rowmap).
// Lanes along rows, the column range split over G = T / round32(rows) thread groups; one __syncthreads when G > 1.
template <class CL, class FR>
__device__ __forceinline__ void gt_row_dots(const CL& cl, const double* __restrict__ M, size_t ld, int rows_all, int c0, int c1, FR rowof_all,
    const double* __restrict__ vec, double* __restrict__ out_all, double* __restrict__ part)
{
    const int tid = threadIdx.x, T = blockDim.x;
    const int per = (rows_all + cl.size() - 1) / cl.size(), r0 = min(rows_all, cl.rank() * per), rows = min(rows_all, r0 + per) - r0;
    auto rowof = [&](int r) { return rowof_all(r0 + r); };
    double* out = out_all + r0;
    const int rp = max(32, round32(rows));
    const int G = max(1, T / rp);
    if (G <= 1) {
        for (int r = tid; r < rows; r += T) {
            const double* mr = M + rowof(r);
            double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
            int c = c0;
            for (; c + 3 < c1; c += 4) {
                const double m0 = mr[size_t(c) * ld], m1 = mr[size_t(c + 1) * ld], m2 = mr[size_t(c + 2) * ld], m3 = mr[size_t(c + 3) * ld];
                s0 = fma(m0, vec[c], s0);
                s1 = fma(m1, vec[c + 1], s1);
                s2 = fma(m2, vec[c + 2], s2);
                s3 = fma(m3, vec[c + 3], s3);
            }
            for (; c < c1; ++c) s0 = fma(mr[size_t(c) * ld], vec[c], s0);
            cl.put(out + r, (s0 + s1) + (s2 + s3));
        }
        return;
    }
    const int g = tid / rp, r = tid - g * rp;
    if (g < G && r < rows) {
        const double* mr = M + rowof(r);
        double s0 = 0.0, s1 = 0.0;
        int c = c0 + g;
        for (; c + G < c1; c += 2 * G) {
            const double m0 = mr[size_t(c) * ld], m1 = mr[size_t(c + G) * ld];
            s0 = fma(m0, vec[c], s0);
            s1 = fma(m1, vec[c + G], s1);
        }
        if (c < c1) s0 = fma(mr[size_t(c) * ld], vec[c], s0);
        part[g * rp + r] = s0 + s1;
    }
    __syncthreads();
    if (tid < rows) {
        double s = part[tid];
        for (int k = 1; k < G; ++k) s += part[k * rp + tid];
        cl.put(out + tid, s);
    }
}

// ---- the pass of the shared-factor form (GtBatch::Hpsi) -----------------------------------------------------------------------
// Partial sums of r = S vec over the active rows for gt_pass_fused: lanes along rows, the columns split over GS = T / round32(nact)
// thread groups, group g's sums in partS[g * rs + row] (at most T doubles); gt_s_rows_sum adds the groups up in fixed order.
// Requires nact <= T.  The same arithmetic as the S half of gt_pass_rows, which keeps its inline copy: calling this from there
// too made ptxas spill more in the 2-CTA/SM kernel of FORM 1.
__device__ __forceinline__ void gt_s_rows_part(const GtWork& W, int nact, const double* __restrict__ vec, const double* __restrict__ S,
    size_t lds, double* __restrict__ partS)
{
    const int tid = threadIdx.x, T = blockDim.x;
    const int rs = max(32, round32(nact)), GS = max(1, T / rs);
    const int g = tid / rs, r_ = tid - g * rs;
    if (g < GS && r_ < nact) {
        const size_t cs = size_t(GS) * lds;
        const double* sr = S + W.rowmap[r_] + size_t(g) * lds;
        const double* vp = vec + g;
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
        int c = g;
        for (; c + 3 * GS < nact; c += 4 * GS, sr += 4 * cs, vp += 4 * GS) {
            const double m0 = sr[0], m1 = sr[cs], m2 = sr[2 * cs], m3 = sr[3 * cs];
            s0 = fma(m0, vp[0], s0); s1 = fma(m1, vp[GS], s1); s2 = fma(m2, vp[2 * GS], s2); s3 = fma(m3, vp[3 * GS], s3);
        }
        if (c < nact) {
            const bool h1 = c + GS < nact, h2 = c + 2 * GS < nact;
            const double m0 = sr[0], m1 = h1 ? sr[cs] : 0.0, m2 = h2 ? sr[2 * cs] : 0.0;
            s0 = fma(m0, vp[0], s0); s1 = fma(m1, h1 ? vp[GS] : 0.0, s1); s2 = fma(m2, h2 ? vp[2 * GS] : 0.0, s2);
        }
        partS[g * rs + r_] = (s0 + s1) + (s2 + s3);
    }
}

__device__ __forceinline__ double gt_s_rows_sum(int nact, const double* __restrict__ partS, int i)
{
    const int rs = max(32, round32(nact)), GS = max(1, int(blockDim.x) / rs);
    double s = partS[i];
    for (int k = 1; k < GS; ++k) s += partS[k * rs + i];
    return s;
}

// outw = P vec (a thread per row PAIR, the column range split over G = T / round32(ld / 2) thread groups; P is stored where the
// general form keeps Q1) and, when outr != null, outr = S vec over the active rows (lanes along rows, columns split over
// thread groups); all partial sums meet in `part` in fixed order.  Requires n <= blockDim.x.  ONE __syncthreads inside; the
// caller syncs before reading.
__device__ __forceinline__ void gt_pass_rows(const GtWork& W, int ld, int q1s, int nact, const double* __restrict__ vec,
    double* __restrict__ outw, const double* __restrict__ S, size_t lds, double* __restrict__ outr, double* __restrict__ part)
{
    const int tid = threadIdx.x, T = blockDim.x;
    const int pairs = ld >> 1, rp = max(32, round32(pairs)), G = max(1, T / rp);
    double* partQ = part;
    double* partS = part + 2 * size_t(T);
    {
        const int g = tid / rp, pr = tid - g * rp;
        double2 q0 = make_double2(0.0, 0.0), q1 = q0, q2 = q0, q3 = q0;
        if (g < G && pr < pairs) {
            int c = g;
            // head columns (shared memory), then the global workspace: plain pointer walks, four loads in flight
            for (; c < min(q1s, nact); c += G) {
                const double2 a0 = *reinterpret_cast<const double2*>(W.Q1s + size_t(c) * ld + 2 * pr);
                const double v0 = vec[c];
                q0.x = fma(a0.x, v0, q0.x); q0.y = fma(a0.y, v0, q0.y);
            }
            const size_t cs = size_t(G) * ld;
            const double* cp = W.Q1 + size_t(c) * ld + 2 * pr;
            const double* vp = vec + c;
            for (; c + 3 * G < nact; c += 4 * G, cp += 4 * cs, vp += 4 * G) {
                const double2 a0 = *reinterpret_cast<const double2*>(cp), a1 = *reinterpret_cast<const double2*>(cp + cs);
                const double2 a2 = *reinterpret_cast<const double2*>(cp + 2 * cs), a3 = *reinterpret_cast<const double2*>(cp + 3 * cs);
                const double v0 = vp[0], v1 = vp[G], v2 = vp[2 * G], v3 = vp[3 * G];
                q0.x = fma(a0.x, v0, q0.x); q0.y = fma(a0.y, v0, q0.y);
                q1.x = fma(a1.x, v1, q1.x); q1.y = fma(a1.y, v1, q1.y);
                q2.x = fma(a2.x, v2, q2.x); q2.y = fma(a2.y, v2, q2.y);
                q3.x = fma(a3.x, v3, q3.x); q3.y = fma(a3.y, v3, q3.y);
            }
            if (c < nact) { // up to three columns left: their loads go out together (one round trip, not three)
                const bool h1 = c + G < nact, h2 = c + 2 * G < nact;
                const double2 zero = make_double2(0.0, 0.0);
                const double2 a0 = *reinterpret_cast<const double2*>(cp);
                const double2 a1 = h1 ? *reinterpret_cast<const double2*>(cp + cs) : zero;
                const double2 a2 = h2 ? *reinterpret_cast<const double2*>(cp + 2 * cs) : zero;
                const double v0 = vp[0], v1 = h1 ? vp[G] : 0.0, v2 = h2 ? vp[2 * G] : 0.0;
                q0.x = fma(a0.x, v0, q0.x); q0.y = fma(a0.y, v0, q0.y);
                q1.x = fma(a1.x, v1, q1.x); q1.y = fma(a1.y, v1, q1.y);
                q2.x = fma(a2.x, v2, q2.x); q2.y = fma(a2.y, v2, q2.y);
            }
            *reinterpret_cast<double2*>(partQ + 2 * (g * rp + pr)) = make_double2((q0.x + q1.x) + (q2.x + q3.x), (q0.y + q1.y) + (q2.y + q3.y));
        }
    }
    const int rs = max(32, round32(nact)), GS = max(1, T / rs);
    if (outr) {
        const int g = tid / rs, r_ = tid - g * rs;
        if (g < GS && r_ < nact) {
            const size_t cs = size_t(GS) * lds;
            const double* sr = S + W.rowmap[r_] + size_t(g) * lds;
            const double* vp = vec + g;
            double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
            int c = g;
            for (; c + 3 * GS < nact; c += 4 * GS, sr += 4 * cs, vp += 4 * GS) {
                const double m0 = sr[0], m1 = sr[cs], m2 = sr[2 * cs], m3 = sr[3 * cs];
                s0 = fma(m0, vp[0], s0); s1 = fma(m1, vp[GS], s1); s2 = fma(m2, vp[2 * GS], s2); s3 = fma(m3, vp[3 * GS], s3);
            }
            if (c < nact) {
                const bool h1 = c + GS < nact, h2 = c + 2 * GS < nact;
                const double m0 = sr[0], m1 = h1 ? sr[cs] : 0.0, m2 = h2 ? sr[2 * cs] : 0.0;
                s0 = fma(m0, vp[0], s0); s1 = fma(m1, h1 ? vp[GS] : 0.0, s1); s2 = fma(m2, h2 ? vp[2 * GS] : 0.0, s2);
            }
            partS[g * rs + r_] = (s0 + s1) + (s2 + s3);
        }
    }
    __syncthreads();
    if (tid < pairs) {
        double2 a = *reinterpret_cast<const double2*>(partQ + 2 * tid);
        for (int k = 1; k < G; ++k) {
            const double2 a1 = *reinterpret_cast<const double2*>(partQ + 2 * (k * rp + tid));
            a.x += a1.x; a.y += a1.y;
        }
        *reinterpret_cast<double2*>(outw + 2 * tid) = a;
    }
    if (outr && tid < nact) {
        double s = partS[tid];
        for (int k = 1; k < GS; ++k) s += partS[k * rs + tid];
        outr[tid] = s;
    }
}

// The pass of the shared-factor form in ONE read of P[:, :nact]: d1 = P' y and w = P d1 (P[:, c] d1[c] needs column c only).
// Warp wp owns the columns c = wp, wp + nw, ... in ascending order; lane l holds the rows 2 l + 64 k (k < kFusedKP: one 128-bit
// load each, all issued before the dot) of the current column, forms d1[c] with a fixed butterfly of shuffles and adds
// P[:, c] d1[c] to its own partials of w from the same registers.  Entries of y past `supp` are exact zeros and are skipped by
// the dot; for a bound row (bj >= 0) d1[c] = bsign P[bj, c] comes from the lane that holds row bj and y is not read.
// Behind the one barrier d1 needs, r = S d1 when want_r (gt_s_rows_part).  The nw x ld warp partials of w do not fit in `part`, so
// they meet there in two fixed-order stages: warp wp + nw/2 stores its partial in slot wp before the barrier, warp wp adds its
// own to that slot after it; gt_pass_fused_w sums the nw/2 slots in order.  `part` takes (nw/2) ld doubles of slots and T of
// S partials: (T / 64) ld + T <= 6 T (gt_layout) exactly when ld <= 320, whatever T (a multiple of 64).  Fixed summation order
// throughout, no atomics: deterministic.  Two __syncthreads inside; afterwards gt_pass_fused_w / gt_pass_fused_r read w and r
// straight from `part`, and every thread reads back only the rows it owns before the next barrier.
constexpr int kFusedKP = 5; // ld <= 320: 10 doubles of the column and 10 of w partials per thread, within 64 registers (2 CTAs/SM)

__device__ __forceinline__ void gt_pass_fused(const GtWork& W, int ld, int nact, const double* __restrict__ y, int supp, int bj,
    double bsign, double* __restrict__ d1, const double* __restrict__ S, size_t lds, bool want_r, double* __restrict__ part)
{
    constexpr int KP = kFusedKP;
    const int lane = lane_id(), wp = warp_id(), nw = blockDim.x >> 5, half = nw >> 1;
    double2 w[KP];
#pragma unroll
    for (int u = 0; u < KP; ++u) w[u] = make_double2(0.0, 0.0);
    const int nin = min(KP, (ld - 2 * lane + 63) >> 6);           // chunks of this lane inside the column
    const int ndot = min(nin, (supp + 63) >> 6);                   // ... and inside the support of y
    auto sweep = [&](auto dot) {
        const double* col = W.Q1 + size_t(wp) * ld + 2 * lane;
        double* d1p = d1 + wp;
#pragma unroll 1
        for (int c = wp; c < nact; c += nw, col += size_t(nw) * ld, d1p += nw) {
            double2 p[KP];
#pragma unroll
            for (int u = 0; u < KP; ++u)
                p[u] = (u < nin) ? *reinterpret_cast<const double2*>(col + 64 * u) : make_double2(0.0, 0.0);
            const double s = dot(p);
            if (lane == 0) *d1p = s;
#pragma unroll
            for (int u = 0; u < KP; ++u) { w[u].x = fma(p[u].x, s, w[u].x); w[u].y = fma(p[u].y, s, w[u].y); }
        }
    };
    if (bj >= 0) {
        const int rb = bj - 2 * lane, src = (bj & 63) >> 1; // row bj relative to this lane's first row; the lane that holds it
        sweep([&](const double2 (&p)[KP]) {
            double v = 0.0;
#pragma unroll
            for (int u = 0; u < KP; ++u) {
                v = (rb == 64 * u) ? p[u].x : v;
                v = (rb == 64 * u + 1) ? p[u].y : v;
            }
            return bsign * __shfl_sync(0xffffffffu, v, src);
        });
    } else {
        sweep([&](const double2 (&p)[KP]) {
            double s = 0.0;
#pragma unroll
            for (int u = 0; u < KP; ++u) {
                if (u < ndot) {
                    const double2 a = *reinterpret_cast<const double2*>(y + 2 * lane + 64 * u);
                    s = fma(p[u].y, a.y, fma(p[u].x, a.x, s));
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            return s;
        });
    }
    if (wp >= half) {
        double* slot = part + size_t(wp - half) * ld + 2 * lane;
#pragma unroll
        for (int u = 0; u < KP; ++u)
            if (u < nin) *reinterpret_cast<double2*>(slot + 64 * u) = w[u];
    }
    __syncthreads();
    if (wp < half) {
        double* slot = part + size_t(wp) * ld + 2 * lane;
#pragma unroll
        for (int u = 0; u < KP; ++u) {
            if (u < nin) {
                double2 o = *reinterpret_cast<const double2*>(slot + 64 * u);
                o.x = w[u].x + o.x; o.y = w[u].y + o.y;
                *reinterpret_cast<double2*>(slot + 64 * u) = o;
            }
        }
    }
    if (want_r) gt_s_rows_part(W, nact, d1, S, lds, part + size_t(half) * ld);
    __syncthreads();
}

// w[k] after gt_pass_fused
__device__ __forceinline__ double gt_pass_fused_w(const double* __restrict__ part, int ld, int k)
{
    const int half = blockDim.x >> 6;
    double s = part[k];
    for (int q = 1; q < half; ++q) s += part[size_t(q) * ld + k];
    return s;
}

// r[i] after gt_pass_fused(want_r)
__device__ __forceinline__ double gt_pass_fused_r(const double* __restrict__ part, int ld, int nact, int i)
{
    return gt_s_rows_sum(nact, part + size_t(blockDim.x >> 6) * ld, i);
}

// Two right-hand sides in one sweep (the warm-start seed adds its rows two at a time): out0[c] = P[:, c] . v0, out1[c] = P[:, c] . v1
__device__ __forceinline__ void gt_q1_col_dots2(const GtWork& W, int ld, int q1s, int nact, const double* __restrict__ v0,
    const double* __restrict__ v1, double* __restrict__ out0, double* __restrict__ out1)
{
    const int lane = lane_id(), wp = warp_id(), nw = blockDim.x >> 5;
    const int g8 = lane >> 3, l8 = lane & 7;
    for (int cb = 4 * wp; cb < nact; cb += 4 * nw) {
        const int c = cb + g8;
        const bool on = c < nact;
        const double* col = (c < q1s ? W.Q1s : W.Q1) + size_t(on ? c : 0) * ld;
        double s0 = 0.0, s1 = 0.0, t0 = 0.0, t1 = 0.0;
        if (on) {
            int k = 2 * l8;
            for (; k + 16 < ld; k += 32) {
                const double2 a0 = *reinterpret_cast<const double2*>(col + k), a1 = *reinterpret_cast<const double2*>(col + k + 16);
                const double2 x0 = *reinterpret_cast<const double2*>(v0 + k), x1 = *reinterpret_cast<const double2*>(v0 + k + 16);
                const double2 y0 = *reinterpret_cast<const double2*>(v1 + k), y1 = *reinterpret_cast<const double2*>(v1 + k + 16);
                s0 = fma(a0.y, x0.y, fma(a0.x, x0.x, s0)); s1 = fma(a1.y, x1.y, fma(a1.x, x1.x, s1));
                t0 = fma(a0.y, y0.y, fma(a0.x, y0.x, t0)); t1 = fma(a1.y, y1.y, fma(a1.x, y1.x, t1));
            }
            if (k < ld) {
                const double2 a0 = *reinterpret_cast<const double2*>(col + k);
                const double2 x0 = *reinterpret_cast<const double2*>(v0 + k), y0 = *reinterpret_cast<const double2*>(v1 + k);
                s0 = fma(a0.y, x0.y, fma(a0.x, x0.x, s0)); t0 = fma(a0.y, y0.y, fma(a0.x, y0.x, t0));
            }
        }
        double qa = s0 + s1, qb = t0 + t1;
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) { qa += __shfl_xor_sync(0xffffffffu, qa, o); qb += __shfl_xor_sync(0xffffffffu, qb, o); }
        if (on && l8 == 0) { out0[c] = qa; out1[c] = qb; }
    }
}

// w0 = P v0, w1 = P v1, r0 = S v0, r1 = S v1 in one sweep over P and S (layout and tiling of gt_pass_rows; `part` holds
// 6 * blockDim.x doubles).  ONE __syncthreads inside; the caller syncs before reading.
__device__ __forceinline__ void gt_pass_rows2(const GtWork& W, int ld, int q1s, int nact, const double* __restrict__ v0,
    const double* __restrict__ v1, double* __restrict__ w0, double* __restrict__ w1, const double* __restrict__ S, size_t lds,
    double* __restrict__ r0, double* __restrict__ r1, double* __restrict__ part)
{
    const int tid = threadIdx.x, T = blockDim.x;
    const int pairs = ld >> 1, rp = max(32, round32(pairs)), G = max(1, T / rp);
    double* pQ0 = part;
    double* pQ1 = part + 2 * size_t(T);
    double* pS0 = part + 4 * size_t(T);
    double* pS1 = part + 5 * size_t(T);
    {
        const int g = tid / rp, pr = tid - g * rp;
        if (g < G && pr < pairs) {
            double2 a = make_double2(0.0, 0.0), b2 = a, c2 = a, d2 = a;
            int c = g;
            for (; c + G < nact; c += 2 * G) {
                const double2 p0 = *reinterpret_cast<const double2*>((c < q1s ? W.Q1s : W.Q1) + size_t(c) * ld + 2 * pr);
                const double2 p1 = *reinterpret_cast<const double2*>((c + G < q1s ? W.Q1s : W.Q1) + size_t(c + G) * ld + 2 * pr);
                const double x0 = v0[c], x1 = v0[c + G], y0 = v1[c], y1 = v1[c + G];
                a.x = fma(p0.x, x0, a.x); a.y = fma(p0.y, x0, a.y); b2.x = fma(p1.x, x1, b2.x); b2.y = fma(p1.y, x1, b2.y);
                c2.x = fma(p0.x, y0, c2.x); c2.y = fma(p0.y, y0, c2.y); d2.x = fma(p1.x, y1, d2.x); d2.y = fma(p1.y, y1, d2.y);
            }
            if (c < nact) {
                const double2 p0 = *reinterpret_cast<const double2*>((c < q1s ? W.Q1s : W.Q1) + size_t(c) * ld + 2 * pr);
                const double x0 = v0[c], y0 = v1[c];
                a.x = fma(p0.x, x0, a.x); a.y = fma(p0.y, x0, a.y); c2.x = fma(p0.x, y0, c2.x); c2.y = fma(p0.y, y0, c2.y);
            }
            *reinterpret_cast<double2*>(pQ0 + 2 * (g * rp + pr)) = make_double2(a.x + b2.x, a.y + b2.y);
            *reinterpret_cast<double2*>(pQ1 + 2 * (g * rp + pr)) = make_double2(c2.x + d2.x, c2.y + d2.y);
        }
    }
    const int rs = max(32, round32(nact)), GS = max(1, T / rs);
    {
        const int g = tid / rs, r_ = tid - g * rs;
        if (g < GS && r_ < nact) {
            const double* sr = S + W.rowmap[r_];
            double s0 = 0.0, s1 = 0.0, t0 = 0.0, t1 = 0.0;
            int c = g;
            for (; c + GS < nact; c += 2 * GS) {
                const double m0 = sr[size_t(c) * lds], m1 = sr[size_t(c + GS) * lds];
                s0 = fma(m0, v0[c], s0); s1 = fma(m1, v0[c + GS], s1); t0 = fma(m0, v1[c], t0); t1 = fma(m1, v1[c + GS], t1);
            }
            if (c < nact) { const double m0 = sr[size_t(c) * lds]; s0 = fma(m0, v0[c], s0); t0 = fma(m0, v1[c], t0); }
            pS0[g * rs + r_] = s0 + s1;
            pS1[g * rs + r_] = t0 + t1;
        }
    }
    __syncthreads();
    if (tid < pairs) {
        double2 a = *reinterpret_cast<const double2*>(pQ0 + 2 * tid), b2 = *reinterpret_cast<const double2*>(pQ1 + 2 * tid);
        for (int k = 1; k < G; ++k) {
            const double2 a1 = *reinterpret_cast<const double2*>(pQ0 + 2 * (k * rp + tid)), b1 = *reinterpret_cast<const double2*>(pQ1 + 2 * (k * rp + tid));
            a.x += a1.x; a.y += a1.y; b2.x += b1.x; b2.y += b1.y;
        }
        *reinterpret_cast<double2*>(w0 + 2 * tid) = a;
        *reinterpret_cast<double2*>(w1 + 2 * tid) = b2;
    }
    if (tid < nact) {
        double s = pS0[tid], t = pS1[tid];
        for (int k = 1; k < GS; ++k) { s += pS0[k * rs + tid]; t += pS1[k * rs + tid]; }
        r0[tid] = s;
        r1[tid] = t;
    }
}

// Fused block reduction of a pass: four sums and the step-length arg-min behind ONE barrier (every warp finishes the
// reduction redundantly).  `scr` (5 x kMaxWarps doubles) / `scri` must not be touched by anything else between two barriers.
struct GtPassRed { double dd, zz, za, dn; MinIdx t1; };
__device__ __forceinline__ GtPassRed gt_pass_reduce(double dd, double zz, double za, double dn, MinIdx tc, double* scr, int* scri)
{
    const int lane = lane_id(), wp = warp_id(), nw = (blockDim.x + 31) >> 5;
    dd = warp_sum(dd); zz = warp_sum(zz); za = warp_sum(za); dn = warp_sum(dn);
    tc = warp_argmin(tc);
    if (lane == 0) {
        scr[wp] = dd; scr[kMaxWarps + wp] = zz; scr[2 * kMaxWarps + wp] = za; scr[3 * kMaxWarps + wp] = dn;
        scr[4 * kMaxWarps + wp] = tc.v; scri[wp] = tc.i;
    }
    __syncthreads();
    const bool on = lane < nw;
    GtPassRed r;
    r.dd = warp_sum(on ? scr[lane] : 0.0);
    r.zz = warp_sum(on ? scr[kMaxWarps + lane] : 0.0);
    r.za = warp_sum(on ? scr[2 * kMaxWarps + lane] : 0.0);
    r.dn = warp_sum(on ? scr[3 * kMaxWarps + lane] : 0.0);
    MinIdx t;
    t.v = on ? scr[4 * kMaxWarps + lane] : 0.0;
    t.i = on ? scri[lane] : -1;
    r.t1 = warp_argmin(t);
    return r;
}

// ---- structured general rows -------------------------------------------------------------------------------------------
// sl[row] = sum_{j <= min(i, N-1)} sum_bb T[line, bb, i - j] x[j nu + bb]   for every row (family, step i, line).
// One warp per (4 steps x 4 lines) tile: the lanes split the kk = i - j range -- the tables are stored kk-fastest and x is
// de-interleaved per input (xt[bb N + j]) so that every shared-memory load of a warp is a run of consecutive words -- keep
// 16 accumulators and meet in a 16-shuffle transpose-reduction; fixed summation order (deterministic).
template <class CL>
__device__ __forceinline__ void gt_products(const CL& cl, const GtBatch& B, const GtWork& W)
{
    const int nu = B.nu, N = B.N, ldk = B.ldk;
    const int lane = lane_id(), nw = (blockDim.x >> 5) * cl.size(), wp = warp_id() * cl.size() + cl.rank(); // warps of the whole cluster
    for (int k = threadIdx.x; k < B.n; k += blockDim.x) {
        const int j = k / nu, bb = k - j * nu;
        W.xt[bb * N + j] = W.x[k];
    }
    __syncthreads();
    int task0 = 0;
    for (int fi = 0; fi < B.nfam; ++fi) {
        const GtFam& F = B.fam[fi];
        const int r = F.rows, ns = F.i1 - F.i0;
        const int nsb = (ns + 3) >> 2, nrg = (r + 3) >> 2, ntask = nsb * nrg;
        const double* tab = W.tab + F.tab;
        double* out = W.sl + (F.is_eq ? 0 : B.meq) + F.row_off;
        // tiles are dealt longest first in a snake (round 0: warp 0..nw-1, round 1: warp nw-1..0, ...): the work of a tile
        // grows linearly with its step, so the snake keeps the per-warp totals within one tile of each other
        const int w0 = (wp - task0 % nw + nw) % nw;
        for (int rnd = 0; rnd * nw < ntask; ++rnd) {
            const int t = rnd * nw + ((rnd & 1) ? nw - 1 - w0 : w0);
            if (t >= ntask) continue;
            const int sb = nsb - 1 - t / nrg, rg = t % nrg;
            const int ib = F.i0 + 4 * sb, l0 = 4 * rg;
            const int kk_lo = max(0, ib - (N - 1)), kk_hi = min(ib + 3, F.i1 - 1);
            double acc[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) acc[k] = 0.0;
            // interior lags: every (step, line, lag) of the tile exists -> no predicates; the <= 3 lags past `ib` and ragged
            // tiles (last steps / lines of a family) take the guarded loop
            const bool full = (ib + 3 < F.i1) && (l0 + 3 < r);
            const int kk_in_lo = full ? max(kk_lo, ib + 3 - (N - 1)) : kk_hi + 1, kk_in_hi = full ? min(ib, kk_hi) : kk_hi;
            for (int kk = kk_in_lo + lane; kk <= kk_in_hi; kk += 32) {
                for (int bb = 0; bb < nu; ++bb) {
                    const double* tp = tab + size_t(l0 + r * bb) * ldk + kk;
                    const double* xp = W.xt + bb * N + (ib - kk);
                    const double t0 = tp[0], t1 = tp[ldk], t2 = tp[2 * size_t(ldk)], t3 = tp[3 * size_t(ldk)];
                    const double x0 = xp[0], x1 = xp[1], x2 = xp[2], x3 = xp[3];
                    acc[0] = fma(t0, x0, acc[0]); acc[1] = fma(t1, x0, acc[1]); acc[2] = fma(t2, x0, acc[2]); acc[3] = fma(t3, x0, acc[3]);
                    acc[4] = fma(t0, x1, acc[4]); acc[5] = fma(t1, x1, acc[5]); acc[6] = fma(t2, x1, acc[6]); acc[7] = fma(t3, x1, acc[7]);
                    acc[8] = fma(t0, x2, acc[8]); acc[9] = fma(t1, x2, acc[9]); acc[10] = fma(t2, x2, acc[10]); acc[11] = fma(t3, x2, acc[11]);
                    acc[12] = fma(t0, x3, acc[12]); acc[13] = fma(t1, x3, acc[13]); acc[14] = fma(t2, x3, acc[14]); acc[15] = fma(t3, x3, acc[15]);
                }
            }
            for (int kk = kk_lo + lane; kk <= kk_hi; kk += 32) {
                if (full && kk >= kk_in_lo && kk <= kk_in_hi) continue; // done above
                for (int bb = 0; bb < nu; ++bb) {
                    const double* tp = tab + size_t(l0 + r * bb) * ldk + kk;
                    const double* xp = W.xt + bb * N + (ib - kk);
                    double tv[4], xv[4];
#pragma unroll
                    for (int ll = 0; ll < 4; ++ll) tv[ll] = (l0 + ll < r) ? tp[size_t(ll) * ldk] : 0.0;
#pragma unroll
                    for (int s_ = 0; s_ < 4; ++s_) {
                        const int j = ib + s_ - kk;
                        xv[s_] = (j >= 0 && j < N && ib + s_ < F.i1) ? xp[s_] : 0.0;
                    }
#pragma unroll
                    for (int s_ = 0; s_ < 4; ++s_)
#pragma unroll
                        for (int ll = 0; ll < 4; ++ll) acc[4 * s_ + ll] = fma(tv[ll], xv[s_], acc[4 * s_ + ll]);
                }
            }
            // transpose-reduce: afterwards lane 2e (e = 0..15) holds the total of acc[e]
#pragma unroll
            for (int o = 16, cnt = 16; cnt > 1; o >>= 1, cnt >>= 1) {
                const int half = cnt >> 1;
                const bool up = (lane & o) != 0;
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    if (k < half) {
                        const double send = up ? acc[k] : acc[k + half];
                        const double recv = __shfl_xor_sync(0xffffffffu, send, o);
                        acc[k] = (up ? acc[k + half] : acc[k]) + recv;
                    }
                }
            }
            acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], 1);
            if ((lane & 1) == 0) {
                const int e = lane >> 1, s_ = e >> 2, ll = e & 3;
                if (ib + s_ < F.i1 && l0 + ll < r) cl.put(out + (ib + s_ - F.i0) * r + l0 + ll, acc[0]);
            }
        }
        task0 += ntask;
    }
}

__host__ __device__ inline GtSS gt_ss_layout(int nx, int nu, int N, int L, int C, int eg_doubles)
{
    GtSS s;
    int o = 0;
    s.oG = o; o += L * nx * nu;          // GsL[k][e][bb] = (A^k B)[e, bb], k < L
    s.oP = o; o += (L + 1) * nx * nx;    // PhiL[t] = A^t (column-major nx x nx), t <= L
    s.oPL = o; o += C * nx * nx;         // PhiLL[k] = A^(k L), k < C
    s.oSt = o; o += (N + 1) * nx;        // zero-state response s_i, i = 0..N
    s.oSc = o; o += C * nx;              // chunk-boundary states s_(c L)
    s.oEG = o; o += eg_doubles;          // per family: E (r x nx) then G (r x nu)
    s.total = o;
    return s;
}

// one entry of phase A of gt_products_ss: loc(i1 + 1)[e] = sum_{k < t} (A^k B)[e, :] u_(i1 - k); compile-time input count NU
// (0: run-time): the inner products unroll into 128-bit shared-memory loads and the lag loop advances two pointers
template <int NU>
__device__ __forceinline__ double gt_ss_loc(const double* __restrict__ GsL, const double* __restrict__ x, int nx, int nu, int i1, int e, int t)
{
    const int nxu = nx * nu;
    const double* g = GsL + e * nu;
    const double* u = x + i1 * nu;
    double a0 = 0.0, a1 = 0.0;
    int k = 0;
    for (; k + 1 < t; k += 2, g += 2 * nxu, u -= 2 * nu) {
        if (NU == 2 || NU == 4) {
#pragma unroll
            for (int bb = 0; bb < NU; bb += 2) {
                const double2 g0 = *reinterpret_cast<const double2*>(g + bb), g1 = *reinterpret_cast<const double2*>(g + nxu + bb);
                const double2 u0 = *reinterpret_cast<const double2*>(u + bb), u1 = *reinterpret_cast<const double2*>(u - nu + bb);
                a0 = fma(g0.y, u0.y, fma(g0.x, u0.x, a0));
                a1 = fma(g1.y, u1.y, fma(g1.x, u1.x, a1));
            }
        } else {
            for (int bb = 0; bb < nu; ++bb) { a0 = fma(g[bb], u[bb], a0); a1 = fma(g[nxu + bb], u[bb - nu], a1); }
        }
    }
    if (k < t) for (int bb = 0; bb < nu; ++bb) a0 = fma(g[bb], u[bb], a0);
    return a0 + a1;
}

// Phases A and B of gt_products_ss.  The chunk-boundary states (phase B) are a short serial recurrence over the chunk-end
// responses only, so two warps compute those entries first and run phase B behind a named barrier while the other warps
// finish phase A; everybody meets at the caller's __syncthreads.
template <int NU>
__device__ __forceinline__ void gt_ss_local(const double* __restrict__ GsL, const double* __restrict__ PhiLL, const double* __restrict__ x,
    double* __restrict__ st, double* __restrict__ Sc, int nx, int N, int L, int C, int nu_rt = 0)
{
    const int nu = NU ? NU : nu_rt;
    const int tid = threadIdx.x, T = blockDim.x, nx2 = nx * nx;
    const bool split = T >= 128 && C >= 2;
    const int nend = split ? (C - 1) * nx : 0; // chunk-end entries (steps c L + L, c < C - 1) taken by the first two warps
    if (split && tid < 64) {
        for (int w = tid; w < nend; w += 64) {
            const int c = w / nx, e = w - c * nx, i1 = (c + 1) * L - 1;
            st[(i1 + 1) * nx + e] = gt_ss_loc<NU>(GsL, x, nx, nu, i1, e, L);
        }
        asm volatile("bar.sync 1, 64;" ::: "memory");
    } else {
        const int t0 = split ? tid - 64 : tid, ts = split ? T - 64 : T;
        int i1 = t0 / nx, e = t0 - i1 * nx;
        const int di = ts / nx, de = ts - di * nx;
        for (; i1 < N;) {
            const int t = i1 % L + 1;
            if (!(split && t == L && i1 + 1 <= (C - 1) * L)) st[(i1 + 1) * nx + e] = gt_ss_loc<NU>(GsL, x, nx, nu, i1, e, t);
            i1 += di; e += de;
            if (e >= nx) { e -= nx; ++i1; }
        }
    }
    if (split ? tid < 64 : true) {
        if (!split) __syncthreads();
        // B: chunk-boundary states s_(c L) = sum_{c' < c} A^((c-1-c') L) loc(c' L + L)
        for (int w = tid; w < C * nx; w += (split ? 64 : T)) {
            const int c = w / nx, e = w - c * nx;
            double a0 = 0.0, a1 = 0.0;
            int cp = 0;
            for (; cp + 1 < c; cp += 2) {
                const double* Am = PhiLL + (c - 1 - cp) * nx2 + e;
                const double* le = st + (cp * L + L) * nx;
                for (int f = 0; f < nx; ++f) { a0 = fma(Am[f * nx], le[f], a0); a1 = fma(Am[f * nx - nx2], le[f + L * nx], a1); }
            }
            if (cp < c) {
                const double* Am = PhiLL + (c - 1 - cp) * nx2 + e;
                const double* le = st + (cp * L + L) * nx;
                for (int f = 0; f < nx; ++f) a0 = fma(Am[f * nx], le[f], a0);
            }
            Sc[w] = a0 + a1;
        }
    }
}

// value of every general row through the state-space form (see GtBatch::ss), handed to emit(row in [eq | ineq], value) by
// the thread that formed it; fixed summation order (deterministic)
template <class CL, class EMIT>
__device__ __forceinline__ void gt_products_ss(const CL& cl, const GtBatch& B, const GtWork& W, EMIT emit)
{
    const int nx = B.nx, nu = B.nu, N = B.N, L = B.ssL, C = B.ssC;
    const int tid = threadIdx.x, T = blockDim.x;
    const GtSS& o = B.ssl;
    const double* __restrict__ GsL = W.ss + o.oG;
    const double* __restrict__ PhiL = W.ss + o.oP;
    const double* __restrict__ PhiLL = W.ss + o.oPL;
    double* __restrict__ st = W.ss + o.oSt;
    double* __restrict__ Sc = W.ss + o.oSc;
    const double* __restrict__ EG = W.ss + o.oEG;
    const int nx2 = nx * nx;
    // A: response of each chunk to its own inputs, loc(i) = sum_{k < t} A^k B u_(i-1-k), t = i - c L;  B: boundary states
    switch (nu) {
    case 1: gt_ss_local<1>(GsL, PhiLL, W.x, st, Sc, nx, N, L, C); break;
    case 2: gt_ss_local<2>(GsL, PhiLL, W.x, st, Sc, nx, N, L, C); break;
    case 4: gt_ss_local<4>(GsL, PhiLL, W.x, st, Sc, nx, N, L, C); break;
    default: gt_ss_local<0>(GsL, PhiLL, W.x, st, Sc, nx, N, L, C, nu); break;
    }
    if (tid >= T - nx) st[tid - (T - nx)] = 0.0;
    __syncthreads();
    // C: s_i = loc(i) + A^t s_(c L)
    for (int w = tid + L * nx; w < N * nx; w += T) {
        const int i1 = w / nx, e = w - i1 * nx;
        const int c = i1 / L, t = i1 - c * L + 1; // L is a power of two on the host side
        const double* Am = PhiL + t * nx2 + e;
        const double* sc = Sc + c * nx;
        double a0 = st[(i1 + 1) * nx + e];
        for (int f = 0; f < nx; ++f) a0 = fma(Am[f * nx], sc[f], a0);
        st[(i1 + 1) * nx + e] = a0;
    }
    __syncthreads();
    // D: rows E s_i + G u_i
    int eg = 0;
    for (int fi = 0; fi < B.nfam; ++fi) {
        const GtFam& F = B.fam[fi];
        const int r = F.rows, cnt = r * (F.i1 - F.i0);
        const double* Ef = F.E.p ? EG + eg : nullptr;
        if (F.E.p) eg += r * nx;
        const double* Gf = F.G.p ? EG + eg : nullptr;
        if (F.G.p) eg += r * nu;
        const int row0 = (F.is_eq ? 0 : B.meq) + F.row_off;
        for (int w = tid; w < cnt; w += T) {
            const int si = w / r, line = w - si * r, step = F.i0 + si;
            double a0 = 0.0;
            if (Ef) for (int e = 0; e < nx; ++e) a0 = fma(Ef[line + e * r], st[step * nx + e], a0);
            if (Gf && step < N) for (int bb = 0; bb < nu; ++bb) a0 = fma(Gf[line + bb * r], W.x[step * nu + bb], a0);
            emit(row0 + w, a0);
        }
    }
}

// locate general row `g` (0-based in [eq | ineq]) in the family list: family, step and line
__device__ __forceinline__ void gt_locate(const GtBatch& B, int g, int& fi, int& step, int& line)
{
    const bool iseq = g < B.meq;
    const int lrow = iseq ? g : g - B.meq;
    fi = 0;
    for (int k = 0; k < B.nfam; ++k) {
        const GtFam& F = B.fam[k];
        if ((F.is_eq != 0) == iseq && lrow >= F.row_off && lrow < F.row_off + F.rows * (F.i1 - F.i0)) { fi = k; break; }
    }
    const GtFam& F = B.fam[fi];
    step = F.i0 + (lrow - F.row_off) / F.rows;
    line = (lrow - F.row_off) % F.rows;
}

// table entry (line, input bb, lag kk) of family F in the transposed shared-memory layout
__device__ __forceinline__ double gt_tab(const GtBatch& B, const double* tab, const GtFam& F, int line, int bb, int kk)
{
    return tab[F.tab + size_t(line + F.rows * bb) * B.ldk + kk];
}

// ---- the solver ----------------------------------------------------------------------------------------------------------
// FORM is a compile-time switch so that each kernel carries the code of one form only (less code, fewer spills: +10% on C3):
//   0 general form (per-instance factors)   1 shared-factor form (GtBatch::Hpsi != null), any row path, warm start
//   2 shared-factor form + state-space products, cold start: the C3 hot path
template <int FORM, class CL>
__device__ inline int gt_solve(const CL& cl, const GtBatch& B, const GtWork& W, int b, double vsmall, int max_iter)
{
    const int n = B.n, meq = B.meq, m = B.m, mg = meq + m, q = mg + 2 * n, np = gt_even(n);
    const int tid = threadIdx.x, T = blockDim.x;
    const int ld = B.ld;
    const int q1s = (FORM >= 1) ? 0 : B.q1s; // shared-factor form: P lives in the global workspace only (the host plans q1s = 0)
    const size_t ldn = size_t(n);
    const double* __restrict__ Jt = B.Jt.at(b);
    const double* __restrict__ JtT = B.JtT.at(b);
    double* __restrict__ S = W.S;
    double* scal = W.red + 2 * kMaxWarps;
    const double* gc = B.c.at(b);
    const double* gAeq = B.Aeq.p ? B.Aeq.at(b) : nullptr;
    const double* gAin = B.Aineq.p ? B.Aineq.at(b) : nullptr;
    auto q1col = [&](int c) -> double* { return (c < q1s ? W.Q1s : W.Q1) + size_t(c) * ld; };
    constexpr bool pform = FORM >= 1; // shared-factor form: z = H a - P d1 (see GtBatch::Hpsi)
    // its pass reads P once (gt_pass_fused) up to n = 320; larger n keep the two sweeps (gt_q1_col_dots, then gt_pass_rows)
    [[maybe_unused]] const bool fused = pform && ld <= 64 * kFusedKP;
    const bool use_ss = (FORM == 2) ? true : (B.ss != 0);                // compile-time in the hot kernel: the other row paths vanish
    const bool structured = (FORM == 2) ? true : (B.structured != 0);

    // ---- 0. load ----------------------------------------------------------------------------------------------------------
    if (structured) {
        for (int fi = 0; fi < B.nfam; ++fi) {
            const GtFam& F = B.fam[fi];
            const double* src = F.EGx + (long long)b * F.sEGx;
            const int rn = F.rows * B.nu, cnt = rn * (B.N + 1);
            for (int t = tid; t < cnt; t += T) {
                const int kk = t / rn, rem = t - kk * rn; // rem = line + rows * bb
                W.tab[F.tab + size_t(rem) * B.ldk + kk] = src[t];
            }
        }
    }
    if (use_ss) {
        const int nx = B.nx, nu = B.nu, L = B.ssL, C = B.ssC, Xr = B.X, Nnx = B.N * nx;
        const GtSS& o = B.ssl;
        const double* gPhi = B.Phi.at(b);
        const double* gGs = B.Gs.at(b);
        for (int t = tid; t < L * nx * nu; t += T) { // GsL[(k nx + e) nu + bb] = Gs[(k nx + e) + bb N nx]
            const int bb = t % nu, ke = t / nu;
            W.ss[o.oG + t] = (ke < Nnx) ? gGs[ke + size_t(bb) * Nnx] : 0.0;
        }
        for (int t = tid; t < (L + 1) * nx * nx; t += T) { // PhiL[k][e + f nx] = Phi[(k nx + e) + f X]
            const int k = t / (nx * nx), rem = t - k * nx * nx, f = rem / nx, e = rem - f * nx;
            W.ss[o.oP + t] = (k <= B.N) ? gPhi[(k * nx + e) + size_t(f) * Xr] : 0.0;
        }
        for (int t = tid; t < C * nx * nx; t += T) {
            const int k = t / (nx * nx), rem = t - k * nx * nx, f = rem / nx, e = rem - f * nx;
            W.ss[o.oPL + t] = (k * L <= B.N) ? gPhi[(k * L * nx + e) + size_t(f) * Xr] : 0.0;
        }
        int eg = o.oEG;
        for (int fi = 0; fi < B.nfam; ++fi) {
            const GtFam& F = B.fam[fi];
            if (F.E.p) { const double* src = F.E.at(b); for (int t = tid; t < F.rows * nx; t += T) W.ss[eg + t] = src[t]; eg += F.rows * nx; }
            if (F.G.p) { const double* src = F.G.at(b); for (int t = tid; t < F.rows * nu; t += T) W.ss[eg + t] = src[t]; eg += F.rows * nu; }
        }
    }
    {
        const double* glb = B.lb.at(b);
        const double* gub = B.ub.at(b);
        for (int i = tid; i < np; i += T) {
            const bool in = i < n;
            W.av[i] = in ? -gc[i] : 0.0;
            W.lb[i] = in ? glb[i] : 0.0;
            W.ub[i] = in ? gub[i] : 0.0;
            W.u[i] = 0.0;
            W.x[i] = W.d[i] = W.zt[i] = W.z[i] = W.d1[i] = W.w[i] = W.v[i] = W.r[i] = 0.0;
            if (in) { W.iact[i] = 0; W.rowmap[i] = i; }
        }
        if (tid == 0) W.u[n] = 0.0;
        const double* gbe = meq ? B.beq.at(b) : nullptr;
        const double* gbi = m ? B.bineq.at(b) : nullptr;
        for (int i = tid; i < mg; i += T) W.bv[i] = (i < meq) ? gbe[i] : gbi[i - meq];
        for (int i = tid; i < q; i += T) W.active[i] = 0;
        for (int i = tid; i < meq; i += T) W.sgn[i] = 1;
    }
    cl.sync(); // (cluster: no remote store may land before every replica is initialised)

    int fail = 0, nact = 0, iter0 = 0, iter1 = 0;
    if (B.pd[(long long)b * B.pd_stride] == 0) fail = 2;
    // no finite bound on any variable (the 2n rows QuadProgDenseSolver appends are +-DBL_MAX / +-inf): they can never be
    // violated, so the selection skips them
    bool nobounds;
    {
        int fin = 0;
        for (int i = tid; i < n; i += T) fin |= (W.lb[i] > -DBL_MAX) || (W.ub[i] < DBL_MAX);
        nobounds = __syncthreads_or(fin) == 0;
    }
    if (B.prekey && fail != 0) {
        if (tid == 0 && cl.rank() == 0) { B.prekey[b] = 0; B.preidx[b] = b; }
        return fail;
    }
#ifdef GT_PROFILE
    long long gt_acc[10] = { 0, 0, 0, 0, 0, 0, 0, 0, 0, 0 };
    long long gt_t0 = clock64();
    const long long gt_tstart = gt_t0;
    int gt_reorth = 0;
#endif

    if (fail == 0) {
        // ---- unconstrained minimiser x = Jt Jt' (-c) -------------------------------------------------------------------------
        gt_trap_mv<false>(cl, JtT, ld, n, n, W.av, W.d, W.part);
        // ---- norms of the general rows (the reference's summation order: columns ascending) ---------------------------------
        for (int i = tid; i < mg; i += T) {
            double s = 0.0;
            if (structured) {
                int fi, step, line;
                gt_locate(B, i, fi, step, line);
                const GtFam& F = B.fam[fi];
                const int jmax = min(step, B.N - 1);
                for (int j = 0; j <= jmax; ++j)
                    for (int bb = 0; bb < B.nu; ++bb) {
                        const double v = gt_tab(B, W.tab, F, line, bb, step - j);
                        s += v * v;
                    }
            } else if (i < meq) {
                for (int k = 0; k < n; ++k) { const double v = gAeq[i + size_t(k) * meq]; s += v * v; }
            } else {
                for (int k = 0; k < n; ++k) { const double v = gAin[(i - meq) + size_t(k) * m]; s += v * v; }
            }
            W.norm[i] = sqrt(s);
        }
        cl.sync();
        gt_trap_mv<true>(cl, Jt, ld, n, n, W.d, W.x, W.part);
        cl.sync();
        GT_T(0);

        // ---- the two updates of the factorisation (shared by the iterations and the warm start) --------------------------------
        auto add_column_from = [&](int nvl, double dd, const double* zsrc, const double* rsrc) {
            // ---- add constraint nvl: Q1 gains zt / delta, S the column [-r/delta ; 1/delta] ----------------------
            const double delta = sqrt(dd), inv = 1.0 / delta;
            double* qc = q1col(nact);
            for (int j = tid * cl.size() + cl.rank(); j < np; j += T * cl.size()) qc[j] = (j < n) ? zsrc[j] * inv : 0.0;
            const int newrow = W.rowmap[nact];
            if (cl.rank() == 0) {
                for (int i = tid; i < nact; i += T) {
                    S[W.rowmap[i] + size_t(nact) * ldn] = -rsrc[i] * inv;
                    S[newrow + size_t(i) * ldn] = 0.0;
                }
                if (tid == 0) S[newrow + size_t(nact) * ldn] = inv;
            }
            if (tid == 0) {
                W.iact[nact] = nvl + 1;
                W.active[nvl] = 1;
            }
            ++nact;
            cl.sync();
        };
        auto add_column = [&](int nvl, double dd) { add_column_from(nvl, dd, pform ? W.z : W.zt, W.r); }; // pform: the column of P is z / |zt|
        auto drop_constraint = [&](int p) {
            cl.sync(); // (cluster: every replica has finished reading r / w before the stores below replace them)
                        const int dropped = (tid == 0) ? W.iact[p] - 1 : 0;
            const int prow = W.rowmap[p];
            if (nact > 1) {
                double vv = 0.0;
                for (int k = tid; k < nact; k += T) { const double t_ = S[prow + size_t(k) * ldn]; W.v[k] = t_; vv += t_ * t_; }
                vv = block_sum(vv, W.red);
                const double rho = sqrt(vv);
                const double vl = W.v[nact - 1];
                const double gamma = (vl >= 0.0) ? -rho : rho;
                const double tau = 1.0 / (rho * (rho + fabs(vl)));
                __syncthreads();
                if (tid == 0) W.v[nact - 1] = vl - gamma;
                __syncthreads();
                for (int k = tid; k < nact; k += T) W.d1[k] = tau * W.v[k];
                // Q1 v (all rows of Q1) and S v (active rows), then the two rank-1 updates
                if (pform) {
                    gt_pass_rows(W, ld, q1s, nact, W.v, W.w, S, ldn, W.r, W.part);
                    __syncthreads();
                } else {
                    gt_q1_row_dots(cl, W, ld, q1s, nact, W.v, W.w, W.part);
                    __syncthreads();
                    gt_row_dots(cl, S, ldn, nact, 0, nact, [&](int r_) { return size_t(W.rowmap[r_]); }, W.v, W.r, W.part);
                    cl.sync();
                }
                gt_q1_rank1(cl, W, ld, q1s, nact - 1, W.w, W.d1);
                gt_s_rank1(cl, S, ldn, W.rowmap, nact, p, nact - 1, W.r, W.d1);
                cl.sync();
                if (warp_id() == 0) {
                    const int lane = lane_id();
                    for (int base = p; base < nact - 1; base += 32) {
                        const int k = base + lane;
                        double uu = 0.0; int ia = 0, rm = 0;
                        if (k < nact - 1) { uu = W.u[k + 1]; ia = W.iact[k + 1]; rm = W.rowmap[k + 1]; }
                        __syncwarp();
                        if (k < nact - 1) { W.u[k] = uu; W.iact[k] = ia; W.rowmap[k] = rm; }
                        __syncwarp();
                    }
                    if (lane == 0) W.rowmap[nact - 1] = prow;
                }
                __syncthreads();
            }
            if (tid == 0) {
                W.u[nact - 1] = W.u[nact];
                W.u[nact] = 0.0;
                W.iact[nact - 1] = 0;
                W.active[dropped] = 0;
            }
            --nact;
            ++iter1;
            __syncthreads();
        };

        // ---- warm start (shared-factor form only; opt-in, SolverInterface::SI_warmStart) -------------------------------------------
        // Seed the factorisation with the inequality / bound rows that were active at the previous solve of this instance
        // (B.warm), solve the equality-constrained problem on that set in closed form,
        //     s_i = slack of row i at the unconstrained minimiser,  t = -S' s,  x = x_unc + P t,  u = S t,
        // and repair dual feasibility by dropping rows with a negative multiplier.  What is left is a valid (x, u, active set)
        // triple of the dual method -- x minimises on the active rows, u >= 0 -- so the iterations below continue from it and
        // stop at the same (unique) optimum; a seed row that is linearly dependent on the earlier ones is skipped.
        if (FORM == 1 && B.warm && !B.prekey) {
            const int* wl = B.warm + (long long)b * n;
            for (int k = tid; k < n; k += T) W.d[k] = W.x[k]; // x_unc (W.d is otherwise unused in this form)
            __syncthreads();
            // The seed rows enter TWO at a time: one sweep over P forms both d1 = P'a, one sweep over P and S both w = P d1 and
            // r = S d1; the second row is then made orthogonal to the first new column in closed form:
            //   g = p1'a2 = (z1'a2) / |zt1| ,  z2 = z2' - g p1 ,  |zt2|^2 = a2'z2' - g^2 ,  d1_2 <- [d1_2 ; g] ,  r2 <- [r2 - g r1 / |zt1| ; g / |zt1|]
            // Storage: row 1 uses av / z / w / d1 / r as a regular pass does, row 2 uses xt / zt / v / u / x (x_unc sits in W.d).
            auto seed_normal = [&](int nvl, double* av, double* hz) { // av = signed normal (explicit also for bound rows), hz = H a
                if (nvl < mg) {
                    int fi, step, line;
                    gt_locate(B, nvl, fi, step, line);
                    const GtFam& F = B.fam[fi];
                    const int supp = min(step + 1, B.N) * B.nu;
                    for (int k = tid; k < np; k += T) {
                        const int j = k / B.nu, bb = k - j * B.nu;
                        av[k] = (k < supp) ? -gt_tab(B, W.tab, F, line, bb, step - j) : 0.0;
                    }
                    const double* Ef = F.E.p ? F.E.at(b) : nullptr;
                    const double* Gf = (F.G.p && step < B.N) ? F.G.at(b) : nullptr;
                    const double* dp = B.Hpsi + size_t(step) * B.nx * ld;
                    const double* jp = B.Hm + size_t(step) * B.nu * ld;
                    for (int k = tid; k < n; k += T) {
                        double acc = 0.0;
                        if (Ef) for (int e = 0; e < B.nx; ++e) acc = fma(Ef[line + e * F.rows], __ldg(dp + k + size_t(e) * ld), acc);
                        if (Gf) for (int e = 0; e < B.nu; ++e) acc = fma(Gf[line + e * F.rows], __ldg(jp + k + size_t(e) * ld), acc);
                        hz[k] = -acc;
                    }
                } else {
                    const int j = nvl - mg, bj = j < n ? j : j - n;
                    const double bsign = j < n ? -1.0 : 1.0;
                    const double* hp = B.Hm + size_t(bj) * ld;
                    for (int k = tid; k < np; k += T) av[k] = (k == bj) ? bsign : 0.0;
                    for (int k = tid; k < n; k += T) hz[k] = bsign * __ldg(hp + k);
                }
            };
            auto next_seed = [&](int& wi) -> int { // next usable entry of the previous active set (uniform over the CTA), -1: none
                for (; wi < n; ++wi) {
                    const int id = wl[wi];
                    if (id <= 0) { wi = n; return -1; }
                    const int nvl = id - 1;
                    if (nvl < meq || nvl >= q || W.active[nvl]) continue; // equalities enter through the regular iterations
                    ++wi;
                    return nvl;
                }
                return -1;
            };
            double* scr6 = W.red + 4 * kMaxWarps; // 5 x kMaxWarps doubles: the five sums below
            for (int wi = 0; nact < n;) {
                const int s1 = next_seed(wi);
                if (s1 < 0) break;
                int wi2 = wi;
                int s2 = (nact + 1 < n) ? next_seed(wi2) : -1;
                if (s2 == s1) s2 = -1;
                seed_normal(s1, W.av, W.z);
                if (s2 >= 0) seed_normal(s2, W.xt, W.zt);
                __syncthreads();
                if (nact > 0) {
                    if (s2 >= 0) {
                        gt_q1_col_dots2(W, ld, q1s, nact, W.av, W.xt, W.d1, W.u);
                        __syncthreads();
                        gt_pass_rows2(W, ld, q1s, nact, W.d1, W.u, W.w, W.v, S, ldn, W.r, W.x, W.part);
                    } else {
                        gt_q1_col_dots(cl, W, n, ld, q1s, nact, W.av, W.d1);
                        __syncthreads();
                        gt_pass_rows(W, ld, q1s, nact, W.d1, W.w, S, ldn, W.r, W.part);
                    }
                    __syncthreads();
                }
                // z1 = h1 - w1, z2' = h2 - w2 and the five inner products
                double c11 = 0.0, c12 = 0.0, c22 = 0.0, e1 = 0.0, e2 = 0.0;
                for (int k = tid; k < n; k += T) {
                    const double a1 = W.av[k];
                    double z1 = W.z[k];
                    e1 = fma(a1, z1, e1);
                    if (nact > 0) { z1 -= W.w[k]; W.z[k] = z1; }
                    c11 = fma(a1, z1, c11);
                    if (s2 >= 0) {
                        const double a2 = W.xt[k];
                        double z2 = W.zt[k];
                        e2 = fma(a2, z2, e2);
                        if (nact > 0) { z2 -= W.v[k]; W.zt[k] = z2; }
                        c22 = fma(a2, z2, c22);
                        c12 = fma(a2, z1, c12);
                    }
                }
                {
                    const int lane = lane_id(), wpi = warp_id(), nw = T >> 5;
                    c11 = warp_sum(c11); c12 = warp_sum(c12); c22 = warp_sum(c22); e1 = warp_sum(e1); e2 = warp_sum(e2);
                    if (lane == 0) { scr6[wpi] = c11; scr6[kMaxWarps + wpi] = c12; scr6[2 * kMaxWarps + wpi] = c22; scr6[3 * kMaxWarps + wpi] = e1; scr6[4 * kMaxWarps + wpi] = e2; }
                    __syncthreads();
                    const bool on = lane < nw;
                    c11 = warp_sum(on ? scr6[lane] : 0.0); c12 = warp_sum(on ? scr6[kMaxWarps + lane] : 0.0);
                    c22 = warp_sum(on ? scr6[2 * kMaxWarps + lane] : 0.0); e1 = warp_sum(on ? scr6[3 * kMaxWarps + lane] : 0.0);
                    e2 = warp_sum(on ? scr6[4 * kMaxWarps + lane] : 0.0);
                }
                const bool ok1 = c11 > 1e-10 * e1;
                const int nact0 = nact;
                double g = 0.0, inv1 = 0.0;
                if (ok1) {
                    inv1 = 1.0 / sqrt(c11);
                    g = c12 * inv1;
                    add_column_from(s1, c11, W.z, W.r); // ends with a barrier
                } else __syncthreads();
                if (s2 >= 0) {
                    const double dd2 = ok1 ? c22 - g * g : c22;
                    // row 2 enters in the same round only when the closed-form correction did not cancel most of it; otherwise
                    // it is left for the next round (wi is not advanced past it), where it gets its own exact projection
                    if (dd2 > 1e-10 * e2 && dd2 > 0.25 * c22) {
                        if (ok1) {
                            for (int k = tid; k < n; k += T) W.zt[k] -= (g * inv1) * W.z[k];
                            for (int i = tid; i < nact0; i += T) W.x[i] -= (g * inv1) * W.r[i];
                            if (tid == 0) W.x[nact0] = g * inv1;
                            __syncthreads();
                        }
                        add_column_from(s2, dd2, W.zt, W.x); // ends with a barrier
                        wi = wi2;
                    } else if (dd2 <= 1e-10 * e2 && !(ok1 && dd2 <= 0.25 * c22 && c22 > 1e-10 * e2)) {
                        wi = wi2; // dependent on the rows already in: skipped for good
                    }
                }
            }
            for (int k = tid; k < n; k += T) W.x[k] = W.d[k]; // x_unc back in place (W.x was scratch above)
            if (tid == 0) { W.u[n] = 0.0; }
            for (int k = tid; k < n; k += T) W.u[k] = 0.0;
            __syncthreads();
            if (nact > 0) {
                // slacks of the seeded rows at x_unc (W.x still holds it)
                if (use_ss) gt_products_ss(cl, B, W, [&](int row, double v) { cl.put(W.sl + row, v); });
                else gt_products(cl, B, W);
                __syncthreads();
                for (int i = tid; i < nact; i += T) {
                    const int k = W.iact[i] - 1;
                    double sv;
                    if (k < mg) sv = W.bv[k] - W.sl[k];
                    else { const int j = k - mg, v_ = j < n ? j : j - n; sv = (j < n) ? W.ub[v_] - W.x[v_] : W.x[v_] - W.lb[v_]; }
                    W.zt[i] = sv;
                }
                __syncthreads();
                for (;;) {
                    // t = -S' s : one warp per column of S, lanes along the active rows
                    for (int j = warp_id(); j < nact; j += (T >> 5)) {
                        double acc = 0.0;
                        for (int i = lane_id(); i < nact; i += 32) acc = fma(S[W.rowmap[i] + size_t(j) * ldn], W.zt[i], acc);
                        acc = warp_sum(acc);
                        if (lane_id() == 0) W.d1[j] = -acc;
                    }
                    __syncthreads();
                    gt_pass_rows(W, ld, q1s, nact, W.d1, W.w, S, ldn, W.r, W.part); // w = P t, r = S t
                    __syncthreads();
                    for (int k = tid; k < n; k += T) W.x[k] = W.d[k] + W.w[k];
                    MinIdx worst; worst.v = 0.0; worst.i = -1;
                    for (int i = tid; i < nact; i += T) {
                        const double ui = W.r[i];
                        W.u[i] = ui > 0.0 ? ui : 0.0;
                        if (ui < 0.0) { MinIdx c; c.v = ui; c.i = i; worst = better(worst, c); }
                    }
                    if (tid == 0) W.u[nact] = 0.0;
                    const MinIdx wsel = block_argmin(worst, W.red, W.redi);
                    // a multiplier that is negative only by rounding is clamped above; a really negative one leaves the seed
                    double usc = 0.0;
                    for (int i = tid; i < nact; i += T) usc = fmax(usc, fabs(W.r[i]));
                    usc = block_sum(usc, W.red); // an upper bound of the scale is enough
                    if (wsel.i < 0 || wsel.v > -1e-12 * usc) break;
                    const int p = wsel.i;
                    drop_constraint(p); // shifts u / iact / rowmap; the slacks follow
                    if (warp_id() == 0) {
                        const int lane = lane_id();
                        for (int base = p; base < nact; base += 32) {
                            const int k = base + lane;
                            double sv = 0.0;
                            if (k < nact) sv = W.zt[k + 1];
                            __syncwarp();
                            if (k < nact) W.zt[k] = sv;
                            __syncwarp();
                        }
                    }
                    --iter1; // a repair drop is not an iteration of the method
                    __syncthreads();
                    if (nact == 0) { for (int k = tid; k < n; k += T) W.x[k] = W.d[k]; __syncthreads(); break; }
                }
                __syncthreads();
            }
        }

        // ---- dual active-set iterations ----------------------------------------------------------------------------------------
        for (;;) {
            ++iter0;
            if (iter0 > max_iter) { fail = 3; break; }
            // all slacks; most violated normalised constraint, lowest index on ties
            MinIdx best; best.v = 0.0; best.i = -1;
            int nviol = 0;
            auto consider = [&](int i, double slv) {
                double s;
                if (i < meq) s = double(W.sgn[i]) * (slv - W.bv[i]);
                else if (i < mg) s = W.bv[i] - slv;
                else s = gi_bound_slack(i - mg, n, mg, W.x, W.lb, W.ub, W.active);
                if (fabs(s) < vsmall) s = 0.0;
                if (i < meq) {
                    if (s > 0.0) W.sgn[i] = -W.sgn[i];
                    s = -fabs(s);
                }
                if (W.active[i]) s = 0.0;
                nviol += s < 0.0;
                if (s < 0.0) {
                    const double nrm = (i < mg) ? W.norm[i] : 1.0;
                    MinIdx c; c.v = s / nrm; c.i = i;
                    best = better(best, c);
                }
            };
            // hot kernel: the thread that forms a row judges it at once -- no barrier between the products and the selection
            constexpr bool fused = FORM == 2 && !CL::multi;
            if (mg > 0) {
                if (fused) gt_products_ss(cl, B, W, [&](int row, double v) { W.sl[row] = v; consider(row, v); });
                else if (use_ss) gt_products_ss(cl, B, W, [&](int row, double v) { cl.put(W.sl + row, v); });
                else if (structured) gt_products(cl, B, W);
                else {
                    if (meq) gt_row_dots(cl, gAeq, size_t(meq), meq, 0, n, [](int r_) { return size_t(r_); }, W.x, W.sl, W.part);
                    if (meq && m) __syncthreads();
                    if (m) gt_row_dots(cl, gAin, size_t(m), m, 0, n, [](int r_) { return size_t(r_); }, W.x, W.sl + meq, W.part);
                }
            }
            if (!fused) {
                cl.sync();
                for (int i = tid; i < mg; i += T) consider(i, W.sl[i]);
            }
            GT_T(1);
            if (!nobounds) for (int i = mg + tid; i < q; i += T) consider(i, 0.0);
            // ONE barrier: per-warp winners to a scratch of their own, every warp finishes the arg-min redundantly
            MinIdx sel;
            {
                const MinIdx wbest = warp_argmin(best);
                double* sv = W.red + 9 * kMaxWarps;
                int* si = W.redi + 2 * kMaxWarps;
                if (lane_id() == 0) { sv[warp_id()] = wbest.v; si[warp_id()] = wbest.i; }
                __syncthreads();
                MinIdx t_;
                const bool on = lane_id() < (T >> 5);
                t_.v = on ? sv[lane_id()] : 0.0;
                t_.i = on ? si[lane_id()] : -1;
                sel = warp_argmin(t_);
            }
            if (B.prekey) { // prepass: only the difficulty estimate is wanted
                const double cnt = block_sum(double(nviol), W.red);
                if (tid == 0 && cl.rank() == 0) { B.prekey[b] = int(cnt); B.preidx[b] = b; }
                return 0;
            }
            if (sel.i < 0) break; // optimal
            const int nvl = sel.i;
            // its slack, recomputed by every thread from the published values (equalities: the sign was already turned)
            double s_nvl;
            if (nvl < meq) s_nvl = -fabs(W.sl[nvl] - W.bv[nvl]);
            else if (nvl < mg) s_nvl = W.bv[nvl] - W.sl[nvl];
            else s_nvl = gi_bound_slack(nvl - mg, n, mg, W.x, W.lb, W.ub, W.active);
            GT_T(2);

            // the signed normal a_nvl (quadprog orientation a'x >= b) and d = Jt' a: they do not change at label 55
            int bj = -1, supp = n;
            double bsign = 0.0;
            int hfi = 0, hstep = 0, hline = 0;
            if (nvl < mg) {
                const double sg = (nvl < meq) ? double(W.sgn[nvl]) : -1.0;
                if (structured) {
                    gt_locate(B, nvl, hfi, hstep, hline);
                    const GtFam& F = B.fam[hfi];
                    supp = min(hstep + 1, B.N) * B.nu;
                    for (int k = tid; k < np; k += T) {
                        const int j = k / B.nu, bb = k - j * B.nu;
                        W.av[k] = (k < supp) ? sg * gt_tab(B, W.tab, F, hline, bb, hstep - j) : 0.0;
                    }
                } else if (nvl < meq) {
                    for (int k = tid; k < n; k += T) W.av[k] = sg * gAeq[nvl + size_t(k) * meq];
                } else {
                    for (int k = tid; k < n; k += T) W.av[k] = sg * gAin[(nvl - meq) + size_t(k) * m];
                }
                if (pform) {
                    // d is never formed
                } else if (structured && B.Dpsi) {
                    const GtFam& F = B.fam[hfi];
                    const double* Ef = F.E.p ? F.E.at(b) : nullptr;
                    const double* Gf = (F.G.p && hstep < B.N) ? F.G.at(b) : nullptr;
                    const double* dp = B.Dpsi + size_t(hstep) * B.nx * ld;
                    const double* jp = JtT + size_t(hstep) * B.nu * ld;
                    for (int k = tid; k < n; k += T) {
                        double acc = 0.0;
                        if (Ef) for (int e = 0; e < B.nx; ++e) acc = fma(Ef[hline + e * F.rows], __ldg(dp + k + size_t(e) * ld), acc);
                        if (Gf) for (int e = 0; e < B.nu; ++e) acc = fma(Gf[hline + e * F.rows], __ldg(jp + k + size_t(e) * ld), acc);
                        W.d[k] = sg * acc;
                    }
                } else {
                    __syncthreads();
                    gt_trap_mv<false>(cl, JtT, ld, n, supp, W.av, W.d, W.part);
                }
            } else {
                const int j = nvl - mg;
                if (j < n) { bj = j; bsign = -1.0; }
                else { bj = j - n; bsign = 1.0; }
                // d[j] = bsign * Jt[bj, j] (j >= bj): a contiguous run of the transposed factor
                if (!pform) for (int k = tid; k < n; k += T) W.d[k] = (k >= bj) ? bsign * __ldg(JtT + size_t(bj) * ld + k) : 0.0;
            }
            // shared-factor form: h = Jt d = H a into W.z (reloaded at every pass: z overwrites it)
            auto load_h = [&]() {
                if (bj >= 0) {
                    const double* hp = B.Hm + size_t(bj) * ld;
                    for (int k = tid; k < n; k += T) W.z[k] = bsign * __ldg(hp + k);
                } else {
                    const double sg = (nvl < meq) ? double(W.sgn[nvl]) : -1.0;
                    const GtFam& F = B.fam[hfi];
                    const double* Ef = F.E.p ? F.E.at(b) : nullptr;
                    const double* Gf = (F.G.p && hstep < B.N) ? F.G.at(b) : nullptr;
                    const double* dp = B.Hpsi + size_t(hstep) * B.nx * ld;
                    const double* jp = B.Hm + size_t(hstep) * B.nu * ld;
                    for (int k = tid; k < n; k += T) {
                        double acc = 0.0;
                        if (Ef) for (int e = 0; e < B.nx; ++e) acc = fma(Ef[hline + e * F.rows], __ldg(dp + k + size_t(e) * ld), acc);
                        if (Gf) for (int e = 0; e < B.nu; ++e) acc = fma(Gf[hline + e * F.rows], __ldg(jp + k + size_t(e) * ld), acc);
                        W.z[k] = sg * acc;
                    }
                }
            };
            cl.sync();
            double dnorm2 = 0.0;
            if (!pform) {
                for (int k = tid; k < n; k += T) dnorm2 += W.d[k] * W.d[k];
                dnorm2 = block_sum(dnorm2, W.red);
            }
            GT_T(3);

            for (int pass = 0;; ++pass) { // label 55
                double dd, zz = 0.0, za = 0.0;
                MinIdx t1m;
                if (pform) {
                    // ---- shared-factor form: d1 = P' a ; [w, r] = [P, S] d1 ; z = h - w ; |zt|^2 = a'z ; |d|^2 = a'h -----------------
                    load_h(); // every thread reads back only the entries it wrote: the loads overlap with the sweeps below
                    if (nact > 0 && fused) {
                        gt_pass_fused(W, ld, nact, W.av, supp, bj, bsign, W.d1, S, ldn, true, W.part);
                    } else if (nact > 0) {
                        if (bj >= 0) {
                            for (int c = tid; c < nact; c += T) W.d1[c] = bsign * q1col(c)[bj];
                        } else {
                            gt_q1_col_dots(cl, W, n, ld, q1s, nact, W.av, W.d1, supp);
                        }
                        __syncthreads();
                        gt_pass_rows(W, ld, q1s, nact, W.d1, W.w, S, ldn, W.r, W.part);
                        __syncthreads();
                    }
                    GT_T(4);
                    auto combine = [&](bool first) -> GtPassRed {
                        double a_zz = 0.0, a_za = 0.0, a_dn = 0.0;
                        for (int k = tid; k < n; k += T) {
                            const double ak = (bj >= 0) ? (k == bj ? bsign : 0.0) : W.av[k];
                            double zk = W.z[k];
                            if (first) {
                                a_dn = fma(ak, zk, a_dn); // W.z still holds h
                                if (nact > 0) { zk -= fused ? gt_pass_fused_w(W.part, ld, k) : W.w[k]; W.z[k] = zk; }
                            }
                            a_zz = fma(zk, zk, a_zz); a_za = fma(ak, zk, a_za);
                        }
                        MinIdx tc; tc.v = 0.0; tc.i = -1;
                        for (int i = tid; i < nact; i += T) {
                            if (first && fused) W.r[i] = gt_pass_fused_r(W.part, ld, nact, i);
                            if (W.iact[i] - 1 >= meq && W.r[i] > 0.0) {
                                MinIdx c; c.v = W.u[i] / W.r[i]; c.i = i;
                                tc = better(tc, c);
                            }
                        }
                        return gt_pass_reduce(0.0, a_zz, a_za, a_dn, tc, W.red + 4 * kMaxWarps, W.redi + kMaxWarps);
                    };
                    GtPassRed pr = combine(true);
                    const double dn_ = pr.dn;
                    if (nact > 0 && pr.za < B.reorth * dn_) {
                        // most of d cancelled: second Gram-Schmidt pass, v = Q1' zt = P' (Q z) ; z -= P v ; d1 += v ; r = S d1 again
#ifdef GT_PROFILE
                        ++gt_reorth;
#endif
                        __syncthreads();
                        for (int k = tid; k < n; k += T) {
                            const double* qr = B.Qs + k;
                            double s0 = 0.0, s1 = 0.0;
                            int j = 0;
                            for (; j + 1 < n; j += 2) { s0 = fma(__ldg(qr + size_t(j) * n), W.z[j], s0); s1 = fma(__ldg(qr + size_t(j + 1) * n), W.z[j + 1], s1); }
                            if (j < n) s0 = fma(__ldg(qr + size_t(j) * n), W.z[j], s0);
                            W.zt[k] = s0 + s1;
                        }
                        for (int k = n + tid; k < np; k += T) W.zt[k] = 0.0;
                        __syncthreads();
                        if (fused) {
                            gt_pass_fused(W, ld, nact, W.zt, n, -1, 0.0, W.v, S, ldn, false, W.part);
                            for (int k = tid; k < n; k += T) W.z[k] -= gt_pass_fused_w(W.part, ld, k);
                        } else {
                            gt_q1_col_dots(cl, W, n, ld, q1s, nact, W.zt, W.v);
                            __syncthreads();
                            gt_pass_rows(W, ld, q1s, nact, W.v, W.w, S, ldn, nullptr, W.part);
                            __syncthreads();
                            for (int k = tid; k < n; k += T) W.z[k] -= W.w[k];
                        }
                        for (int k = tid; k < nact; k += T) W.d1[k] += W.v[k];
                        __syncthreads();
                        gt_row_dots(cl, S, ldn, nact, 0, nact, [&](int r_) { return size_t(W.rowmap[r_]); }, W.d1, W.r, W.part);
                        __syncthreads();
                        pr = combine(false);
                    }
                    dd = pr.za; zz = pr.zz; za = pr.za; t1m = pr.t1;
                    GT_T(5);
                } else {
                // d1 = Q1' d ; zt = d - Q1 d1 (second pass when most of d cancelled: "twice is enough")
                dd = dnorm2;
                if (nact > 0) {
                    gt_q1_col_dots(cl, W, n, ld, q1s, nact, W.d, W.d1);
                    cl.sync();
                    gt_q1_row_dots(cl, W, ld, q1s, nact, W.d1, W.w, W.part);
                    cl.sync();
                    double acc = 0.0;
                    for (int k = tid; k < n; k += T) { const double v = W.d[k] - W.w[k]; W.zt[k] = v; acc += v * v; }
                    dd = block_sum(acc, W.red);
                    if (dd < B.reorth * dnorm2) {
#ifdef GT_PROFILE
                        ++gt_reorth;
#endif
                        gt_q1_col_dots(cl, W, n, ld, q1s, nact, W.zt, W.v);
                        cl.sync();
                        gt_q1_row_dots(cl, W, ld, q1s, nact, W.v, W.w, W.part);
                        cl.sync();
                        acc = 0.0;
                        for (int k = tid; k < n; k += T) { const double v = W.zt[k] - W.w[k]; W.zt[k] = v; acc += v * v; }
                        for (int k = tid; k < nact; k += T) W.d1[k] += W.v[k];
                        dd = block_sum(acc, W.red);
                    }
                } else {
                    for (int k = tid; k < n; k += T) W.zt[k] = W.d[k];
                    __syncthreads();
                }
                GT_T(4);
                // z = Jt zt ; r = S d1
                gt_trap_mv<true>(cl, Jt, ld, n, n, W.zt, W.z, W.part);
                __syncthreads(); // `part` is reused; z and r are published by the one cluster barrier below
                if (nact > 0) gt_row_dots(cl, S, ldn, nact, 0, nact, [&](int r_) { return size_t(W.rowmap[r_]); }, W.d1, W.r, W.part);
                cl.sync();
                GT_T(5);
                MinIdx tc; tc.v = 0.0; tc.i = -1;
                for (int i = tid; i < nact; i += T) {
                    if (W.iact[i] - 1 >= meq && W.r[i] > 0.0) {
                        MinIdx c; c.v = W.u[i] / W.r[i]; c.i = i;
                        tc = better(tc, c);
                    }
                }
                t1m = block_argmin(tc, W.red, W.redi);
                for (int j = tid; j < n; j += T) {
                    const double zj = W.z[j];
                    zz += zj * zj;
                    if (bj < 0) za += zj * W.av[j];
                }
                block_sum2(zz, za, W.red);
                }
                const bool t1inf = t1m.i < 0;
                const double t1 = t1m.v;
                const int it1 = t1m.i;
                if (bj >= 0 && !pform) za = bsign * W.z[bj];

                bool do_drop = false;
                if (fabs(zz) <= vsmall) {
                    if (t1inf) { fail = 1; break; }
                    for (int i = tid; i < nact; i += T) W.u[i] -= t1 * W.r[i];
                    if (tid == 0) W.u[nact] += t1;
                    do_drop = true;
                } else {
                    double tt = -s_nvl / za;
                    bool t2min = true;
                    if (!t1inf && t1 < tt) { tt = t1; t2min = false; }
                    for (int j = tid; j < n; j += T) W.x[j] += tt * W.z[j];
                    for (int i = tid; i < nact; i += T) W.u[i] -= tt * W.r[i];
                    if (tid == 0) W.u[nact] += tt;
                    if (t2min) {
                        add_column(nvl, dd);
                        GT_T(6);
                        break; // next outer iteration
                    } else {
                        // partial step: refresh s_nvl at the new x (with the equality sign rule)
                        __syncthreads();
                        double s;
                        if (bj >= 0) {
                            s = (bsign < 0.0) ? W.ub[bj] - W.x[bj] : W.x[bj] - W.lb[bj];
                        } else {
                            double acc = 0.0; // av holds the signed normal, so a'x = av . x
                            for (int k = tid; k < n; k += T) acc += W.av[k] * W.x[k];
                            acc = block_sum(acc, W.red);
                            if (nvl < meq) s = acc - double(W.sgn[nvl]) * W.bv[nvl];
                            else s = acc + W.bv[nvl];
                        }
                        if (nvl < meq) {
                            // the sign flip of an equality changes the orientation of a_nvl, hence of d
                            __syncthreads();
                            if (s > 0.0) {
                                if (tid == 0) W.sgn[nvl] = -W.sgn[nvl];
                                for (int k = tid; k < n; k += T) { W.av[k] = -W.av[k]; W.d[k] = -W.d[k]; }
                            }
                            s = -fabs(s);
                        }
                        s_nvl = s;
                        do_drop = true;
                    }
                }
                if (do_drop) {
                    // ---- drop the it1-th active constraint: reflection with last column ~ row p of S ---------------------------
                    drop_constraint(it1);
                    GT_T(7);
                    continue; // label 55
                }
            }
            if (fail != 0) break;
        }
    }
    __syncthreads();
#ifdef GT_PROFILE
    if (tid == 0 && ((b % 97) == 0 || clock64() - gt_tstart > 60000000LL))
        printf("GTPROF b=%d n=%d iters=%d drops=%d nact=%d reorth=%d | init %lld prod %lld sel %lld normal+Jt'a %lld q1 %lld Jz+S %lld step+add %lld drop %lld\n",
            b, n, iter0, iter1, nact, gt_reorth, gt_acc[0], gt_acc[1], gt_acc[2], gt_acc[3], gt_acc[4], gt_acc[5], gt_acc[6], gt_acc[7]);
#endif
    // ---- results ---------------------------------------------------------------------------------------------------------------
    if (cl.rank() != 0) return fail;
    if (B.x) for (int i = tid; i < n; i += T) B.x[(long long)b * n + i] = (fail == 2) ? 0.0 : W.x[i];
    if (B.iact) for (int i = tid; i < n; i += T) B.iact[(long long)b * n + i] = (i < nact) ? W.iact[i] : 0;
    if (tid == 0) {
        if (B.status) B.status[b] = fail;
        if (B.iters) { B.iters[2LL * b] = iter0; B.iters[2LL * b + 1] = iter1; }
        if (B.nact) B.nact[b] = nact;
    }
    return fail;
}

// ---- host side (k6_thin.cu) ------------------------------------------------------------------------------------------------
struct GtPlan {
    int threads, grid, per_sm, ok, q1s;
    int cluster;         // CTAs per instance (0 / 1: one CTA per instance)
    size_t smem_bytes;
    long long ws_stride; // doubles of global workspace per CTA (Q1 + S)
};
struct GtShape { int n, meq, m, tab_doubles, ldk, ld, ss_doubles, pform, cluster; };
GtPlan gt_plan(const GtShape& s, int batch, int sms, size_t smem_optin);
size_t gt_factor_smem(int n);
// factor `count` Hessians Q (n x n each): Jt / JtT receive count * n * n doubles, pd count flags
cudaError_t gt_factor_launch(DArr Q, int n, int ld, int count, double* Jt, double* JtT, int* pd, int sms, cudaStream_t st);
cudaError_t gt_launch(const GtBatch& B, const GtPlan& plan, cudaStream_t st);
// order = indices sorted by key, descending (stable); `temp` must hold gt_sort_temp_bytes(count) bytes
size_t gt_sort_temp_bytes(int count);
cudaError_t gt_sort_launch(const int* keys, int* keys_sorted, const int* idx, int* order, int count, void* temp, size_t temp_bytes, cudaStream_t st);
cudaError_t gt_psit_fill_launch(const double* Gs, double* PsiT, int nx, int nu, int N, cudaStream_t st);

} // namespace cb
