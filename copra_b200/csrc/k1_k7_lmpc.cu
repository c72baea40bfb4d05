// k1_k7_lmpc.cu -- condensing (K1), QP assembly (K2-K4, K4'), result rollout (K7) for a batch of
// LMPC / InitialStateLMPC controllers.  One CTA per instance unless noted; all instance-major,
// reference (Eigen column-major) layouts.
//
// The block-Toeplitz structure of Psi (Psi_ij = A^(i-1-j) B) is exploited everywhere: only the first
// block column Gs = [B; AB; ...; A^(N-1)B] is produced by K1, every consumer indexes it.  The
// reference multiplies through the structural zeros (src/costFunctions.cpp:73 "Lot of sums of zero
// here"); here Q is produced with O(N^2) block operations by running sums along block diagonals, in
// the SAME accumulation order as the reference (steps ascending), with un-fused multiply/add so the
// condensed matrices agree with the CPU oracle to the last bit where the order is defined.
#include "engine.cuh"
#include "gi_small.cuh"
#include "gi_solver.cuh"
#include "launch.h"

#include <algorithm>
#include <cfloat>

namespace cb {

__device__ __forceinline__ double mul_(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add_(double a, double b) { return __dadd_rn(a, b); }

// ------------------------------------------------------------------------------------------------
// K1: PreviewSystem::updateSystem (reference src/PreviewSystem.cpp:57-74).
// Phi_i = A Phi_{i-1}, G_k = A G_{k-1} (G_0 = B), xi_i = A xi_{i-1} + d.  Sequential in the step index,
// parallel over the nx*nx + nx*nu + nx entries of one step and over instances.
// ------------------------------------------------------------------------------------------------
// A read-only table that is either a slice of the CTA's dynamic shared memory (32-bit offsets, LDS) or a global array.
extern __shared__ double stage_sm[];
template <bool STAGED> struct Tab {
    const double* g;
    int o;
    __device__ __forceinline__ double operator[](int i) const { return STAGED ? stage_sm[o + i] : g[i]; }
    __device__ __forceinline__ Tab shifted(int d) const { return Tab{ g + d, o + d }; }
};
// cooperative copy of `count` doubles into stage_sm at offset `o`
__device__ __forceinline__ void stage_copy(int o, const double* src, int count)
{
    for (int t = threadIdx.x; t < count; t += blockDim.x) stage_sm[o + t] = src[t];
}

__device__ __forceinline__ void dev_condense(const BuildParams& P, double* sm, int b)
{
    const int nx = P.nx, nu = P.nu, N = P.N, X = P.X;
    const int nA = nx * nx, nB = nx * nu, per = nA + nB + nx;
    double* sA = sm;            // nx x nx
    double* cur = sA + nA;      // [Phi | G | xi] current step
    double* nxt = cur + per;
    double* sd = nxt + per;     // nx
    const long long NX = (long long)N * nx;
    {
        const double* A = P.A.at(b);
        const double* Bm = P.B.at(b);
        const double* d = P.d.at(b);
        double* Phi = P.Phi + (long long)b * X * nx;
        double* Gs = P.Gs + (long long)b * NX * nu;
        double* xi = P.xi + (long long)b * X;
        __syncthreads();
        for (int t = threadIdx.x; t < nA; t += blockDim.x) {
            sA[t] = A[t];
            cur[t] = A[t]; // Phi_1 = A (assignment, :59)
            const int r = t % nx, c = t / nx;
            Phi[r + (long long)c * X] = (r == c) ? 1.0 : 0.0; // Phi_0 = I (PreviewSystem::system :51-52)
            Phi[nx + r + (long long)c * X] = A[t];
        }
        for (int t = threadIdx.x; t < nB; t += blockDim.x) {
            cur[nA + t] = Bm[t]; // G_0 = B (:60)
            const int r = t % nx, c = t / nx;
            Gs[r + (long long)c * NX] = Bm[t];
        }
        for (int t = threadIdx.x; t < nx; t += blockDim.x) {
            sd[t] = d[t];
            cur[nA + nB + t] = d[t]; // xi_1 = d (:61)
            xi[t] = 0.0;
            xi[nx + t] = d[t];
        }
        __syncthreads();
        for (int i = 2; i <= N; ++i) {
            for (int t = threadIdx.x; t < per; t += blockDim.x) {
                int r, c;
                const double* src;
                if (t < nA) { r = t % nx; c = t / nx; src = cur + c * nx; }
                else if (t < nA + nB) { r = (t - nA) % nx; c = (t - nA) / nx; src = cur + nA + c * nx; }
                else { r = t - nA - nB; c = 0; src = cur + nA + nB; }
                double s = 0.0;
                for (int k = 0; k < nx; ++k) s = add_(s, mul_(sA[r + k * nx], src[k]));
                if (t < nA) Phi[(long long)i * nx + r + (long long)c * X] = s;
                else if (t < nA + nB) Gs[(long long)(i - 1) * nx + r + (long long)c * NX] = s;
                else { s = add_(s, sd[r]); xi[(long long)i * nx + r] = s; }
                nxt[t] = s;
            }
            __syncthreads();
            double* tmp = cur; cur = nxt; nxt = tmp;
        }
    }
}

__global__ void k1_condense_kernel(const __grid_constant__ BuildParams P)
{
    extern __shared__ double sm[];
    for (int b = blockIdx.x; b < P.batch; b += gridDim.x) dev_condense(P, sm, b);
}

// Small systems (nx^2 + nx nu + nx <= 32): a sub-warp group of G = 8/16/32 lanes per instance, so that a 128-thread
// CTA carries 128/G instances and the N-step power chain synchronises with __syncwarp instead of a block barrier --
// the whole batch is one wave of short latency chains instead of several CTA-per-instance rounds.
__global__ void __launch_bounds__(128) k1_condense_group_kernel(const __grid_constant__ BuildParams P, int G)
{
    extern __shared__ double sm[];
    const int nx = P.nx, nu = P.nu, N = P.N, X = P.X;
    const int nA = nx * nx, nB = nx * nu, per = nA + nB + nx;
    const int grp = threadIdx.x / G, t = threadIdx.x % G, ngrp = blockDim.x / G;
    const int stride = nA + 2 * per + nx;
    double* sA = sm + grp * stride;
    double* cur = sA + nA;
    double* nxt = cur + per;
    double* sd = nxt + per;
    const long long NX = (long long)N * nx;
    const int b = blockIdx.x * ngrp + grp;
    if (b >= P.batch) return; // whole groups leave together; warps of mixed groups keep using __syncwarp on the rest
    const unsigned lane = threadIdx.x & 31;
    const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~unsigned(G - 1)));
    const double* A = P.A.at(b);
    const double* Bm = P.B.at(b);
    const double* d = P.d.at(b);
    double* Phi = P.Phi + (long long)b * X * nx;
    double* Gs = P.Gs + (long long)b * NX * nu;
    double* xi = P.xi + (long long)b * X;
    int r, c, kind; // this lane's entry of [Phi | G | xi]
    if (t < nA) { kind = 0; r = t % nx; c = t / nx; }
    else if (t < nA + nB) { kind = 1; r = (t - nA) % nx; c = (t - nA) / nx; }
    else { kind = 2; r = t - nA - nB; c = 0; }
    if (t < per) {
        if (kind == 0) {
            const double a = A[t];
            sA[t] = a; cur[t] = a;
            Phi[r + (long long)c * X] = (r == c) ? 1.0 : 0.0;
            Phi[nx + r + (long long)c * X] = a;
        } else if (kind == 1) {
            const double v = Bm[t - nA];
            cur[t] = v;
            Gs[r + (long long)c * NX] = v;
        } else {
            const double v = d[r];
            sd[r] = v; cur[t] = v;
            xi[r] = 0.0;
            xi[nx + r] = v;
        }
    }
    __syncwarp(gmask);
    const int srcoff = (kind == 0) ? c * nx : ((kind == 1) ? nA + c * nx : nA + nB);
    for (int i = 2; i <= N; ++i) {
        if (t < per) {
            const double* src = cur + srcoff;
            double s = 0.0;
            for (int k = 0; k < nx; ++k) s = add_(s, mul_(sA[r + k * nx], src[k]));
            if (kind == 0) Phi[(long long)i * nx + r + (long long)c * X] = s;
            else if (kind == 1) Gs[(long long)(i - 1) * nx + r + (long long)c * NX] = s;
            else { s = add_(s, sd[r]); xi[(long long)i * nx + r] = s; }
            nxt[t] = s;
        }
        __syncwarp(gmask);
        double* tmp = cur; cur = nxt; nxt = tmp;
    }
}

int k1_condense_launch(const BuildParams& P, cudaStream_t st)
{
    const int per = P.nx * P.nx + P.nx * P.nu + P.nx;
    if (per <= 32) {
        const int G = per <= 8 ? 8 : (per <= 16 ? 16 : 32);
        const int ngrp = 128 / G;
        const size_t smem = sizeof(double) * size_t(P.nx * P.nx + 2 * per + P.nx) * ngrp;
        k1_condense_group_kernel<<<(P.batch + ngrp - 1) / ngrp, 128, smem, st>>>(P, G);
        cudaError_t e = cudaGetLastError();
        return e == cudaSuccess ? 1 : -int(e);
    }
    const size_t smem = sizeof(double) * size_t(P.nx * P.nx + 2 * per + P.nx);
    int threads = std::min(256, ((per + 31) / 32) * 32);
    int grid = std::min(P.batch, 148 * 8);
    k1_condense_kernel<<<grid, threads, smem, st>>>(P);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 1 : -int(e);
}

// ------------------------------------------------------------------------------------------------
// K1b: materialise Psi (X x nU, reference layout) from the compact first block column.
// Column (j, c) of Psi is [zeros((j+1) nx); Gs[0 : X-(j+1)nx, c]]: a pure HBM-write-bound fill.
// ------------------------------------------------------------------------------------------------
__global__ void k1_psi_fill_kernel(const double* __restrict__ Gs, long long sGs, double* __restrict__ Psi, int nx, int nu, int N, int batch)
{
    const int X = nx * (N + 1), nU = nu * N;
    const long long NX = (long long)N * nx;
    const int b = blockIdx.y;
    const double* g = Gs + (long long)b * sGs;
    double* psi = Psi + (long long)b * X * nU;
    for (int col = blockIdx.x; col < nU; col += gridDim.x) {
        const int j = col / nu, c = col % nu;
        const int shift = (j + 1) * nx;
        const double* src = g + (long long)c * NX;
        double* dst = psi + (long long)col * X;
        for (int row = threadIdx.x; row < X; row += blockDim.x) dst[row] = (row >= shift) ? src[row - shift] : 0.0;
    }
}

int k1_psi_fill_launch(const double* Gs, long long sGs, double* Psi, int nx, int nu, int N, int batch, cudaStream_t st)
{
    const int nU = nu * N;
    int launches = 0;
    for (int b0 = 0; b0 < batch; b0 += 65535) {
        const int nb = std::min(65535, batch - b0);
        dim3 grid(std::min(nU, 64), nb);
        k1_psi_fill_kernel<<<grid, 256, 0, st>>>(Gs + (long long)b0 * sGs, sGs, Psi + (long long)b0 * nx * (N + 1) * nU, nx, nu, N, nb);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return -int(e);
        ++launches;
    }
    return launches;
}

// ------------------------------------------------------------------------------------------------
// K2a: per-family small products (one CTA per instance):
//   cost  : MGx[kk] = M A^(kk-1) B (kk>=1), MGx[0] = N | 0 ; MPhi_i = M Phi_i ; res_i = M xi_i - p
//   cstr  : EGx[kk] likewise with E/G ; Y rows = E Phi_i ; z rows = f - E xi_i
// (reference: tmp = M_*Psi.block(..), M_*Phi.block(..), M_*xi.segment(..)-p_  src/costFunctions.cpp:74-78;
//  E_*Psi.block, E_*Phi.block, f_-E_*xi.segment  src/constraints.cpp:77-81)
// p and f are the only per-step inputs (pstep / fstep > 0: step i reads its own vector).  VEC_ONLY: res and z alone, for a
// retarget of a resident build whose matrices did not change (MGx, MPhi, EGx and Y are kept).
// ------------------------------------------------------------------------------------------------
template <bool VEC_ONLY>
__device__ __forceinline__ void dev_precompute(const BuildParams& P, int b)
{
    const int nx = P.nx, nu = P.nu, N = P.N, X = P.X;
    const long long NX = (long long)N * nx;
    const int tid = threadIdx.x, T = blockDim.x;
    {
        const double* Phi = P.Phi + (long long)b * X * nx;
        const double* Gs = P.Gs + (long long)b * NX * nu;
        const double* xi = P.xi + (long long)b * X;
        for (int ci = 0; ci < P.ncost; ++ci) {
            const CostFam& F = P.cost[ci];
            if (F.dense) continue; // full-size entry: DMMA GEMM path
            const int r = F.rows, ns = F.i1 - F.i0;
            const double* M = F.hasM ? F.M.at(b) : nullptr;
            const double* Nn = F.hasN ? F.N.at(b) : nullptr;
            const double* p = F.p.at(b);
            double* MGx = F.MGx + (long long)b * F.sMGx;
            double* MPhi = F.MPhi + (long long)b * F.sMPhi;
            double* res = F.res + (long long)b * F.sres;
            for (int t = tid; t < r * nu * (N + 1) && !VEC_ONLY; t += T) {
                const int l = t % r, bb = (t / r) % nu, kk = t / (r * nu);
                double s = 0.0;
                if (kk == 0) s = Nn ? Nn[l + bb * r] : 0.0;
                else if (M) {
                    const double* g = Gs + (long long)(kk - 1) * nx + (long long)bb * NX;
                    for (int k = 0; k < nx; ++k) s = add_(s, mul_(M[l + k * r], g[k]));
                }
                MGx[t] = s;
            }
            for (int t = tid; t < r * nx * ns && !VEC_ONLY; t += T) {
                const int l = t % r, sidx = (t / r) % nx, ii = t / (r * nx);
                double s = 0.0;
                if (M) {
                    const double* ph = Phi + (long long)(F.i0 + ii) * nx + (long long)sidx * X;
                    for (int k = 0; k < nx; ++k) s = add_(s, mul_(M[l + k * r], ph[k]));
                }
                MPhi[t] = s;
            }
            for (int t = tid; t < r * ns; t += T) {
                const int l = t % r, ii = t / r;
                const double pl = p[(F.i0 + ii) * F.pstep + l];
                double s = 0.0;
                if (M) {
                    const double* xv = xi + (long long)(F.i0 + ii) * nx;
                    for (int k = 0; k < nx; ++k) s = add_(s, mul_(M[l + k * r], xv[k]));
                    s = add_(s, -pl);
                } else s = -pl;
                res[t] = s;
            }
        }
        for (int fi = 0; fi < P.nfam; ++fi) {
            const CstrFam& F = P.fam[fi];
            if (F.dense || F.gather) continue;
            const int r = F.rows, ns = F.i1 - F.i0;
            const double* E = F.hasE ? F.E.at(b) : nullptr;
            const double* G = F.hasG ? F.G.at(b) : nullptr;
            const double* f = F.f.at(b);
            double* EGx = F.EGx + (long long)b * F.sEGx;
            const int mtot = F.is_eq ? P.meq : P.mineq;
            double* Y = (F.is_eq ? P.Yeq : P.Yin) + (long long)b * mtot * nx;
            double* z = (F.is_eq ? P.zeq : P.zin) + (long long)b * mtot;
            for (int t = tid; t < r * nu * (N + 1) && !VEC_ONLY; t += T) {
                const int l = t % r, bb = (t / r) % nu, kk = t / (r * nu);
                double s = 0.0;
                if (kk == 0) s = G ? G[l + bb * r] : 0.0;
                else if (E) {
                    const double* g = Gs + (long long)(kk - 1) * nx + (long long)bb * NX;
                    for (int k = 0; k < nx; ++k) s = add_(s, mul_(E[l + k * r], g[k]));
                }
                EGx[t] = s;
            }
            for (int t = tid; t < r * nx * ns && !VEC_ONLY; t += T) {
                const int l = t % r, ii = (t / r) % ns, sidx = t / (r * ns);
                double s = 0.0;
                if (E) {
                    const double* ph = Phi + (long long)(F.i0 + ii) * nx + (long long)sidx * X;
                    for (int k = 0; k < nx; ++k) s = add_(s, mul_(E[l + k * r], ph[k]));
                }
                Y[(F.row_off + ii * r + l) + (long long)sidx * mtot] = s;
            }
            for (int t = tid; t < r * ns; t += T) {
                const int l = t % r, ii = t / r;
                const double fl = f[(F.i0 + ii) * F.fstep + (F.fidx ? F.fidx[l] : l)];
                double s = 0.0;
                if (E) {
                    const double* xv = xi + (long long)(F.i0 + ii) * nx;
                    for (int k = 0; k < nx; ++k) s = add_(s, mul_(E[l + k * r], xv[k]));
                }
                z[F.row_off + ii * r + l] = E ? add_(fl, -s) : fl;
            }
        }
    }
}

template <bool VEC_ONLY> __global__ void k2_precompute_kernel(const __grid_constant__ BuildParams P)
{
    for (int b = blockIdx.x; b < P.batch; b += gridDim.x) dev_precompute<VEC_ONLY>(P, b);
}

// ------------------------------------------------------------------------------------------------
// K2b: Hessian block Q = 1e-6 I + sum_costs sum_i T_i' W T_i  (LMPC::updateSystem :228-229 +
// makeQPForm :252-255 + cost update loops).  One thread per (block diagonal dd, a, b) chain walking
// jmax = N-1 .. |dd|; Toeplitz => the entry at jmax is a running sum over kk = i - jmax ascending.
// grid = (chain tiles, batch)
// ------------------------------------------------------------------------------------------------
// `qtile` != null: the chain writes into a dense nU x nU tile in shared memory (written out coalesced by the caller)
// instead of walking a diagonal of Q in global memory with one 32-byte sector per 8-byte store.
__device__ __forceinline__ void dev_q_chain(const BuildParams& P, int b, int ch, const double* const* MG, const double* const* Wt,
    double* qtile)
{
    const int nu = P.nu, N = P.N, nvar = P.nvar;
    const int off = P.initial_state ? P.nx : 0;
    const int a = ch % nu, bb = (ch / nu) % nu, dd = ch / (nu * nu) - (N - 1); // dd = j1 - j2
    const int ad = dd < 0 ? -dd : dd;
    double* Q = P.Q + (long long)b * P.sQ;
    double run[kMaxCost];
    int done[kMaxCost];
    for (int ci = 0; ci < P.ncost; ++ci) {
        run[ci] = 0.0;
        done[ci] = 0;
    }
    // weighted dot of two r-vectors in the reference order: sum_l (ga[l] * w[l]) * gb[l]
    auto wdot = [](const double* ga, const double* w, const double* gb, int r) {
        double s = 0.0;
        for (int l = 0; l < r; ++l) s = add_(s, mul_(mul_(ga[l], w[l]), gb[l]));
        return s;
    };
    const int o1 = dd >= 0 ? 0 : -dd, o2 = dd >= 0 ? dd : 0; // jmax - j1, jmax - j2 (constant along the chain)
    double* qout = qtile ? qtile + ((N - 1 - o1) * nu + a) + (long long)((N - 1 - o2) * nu + bb) * P.nU
                         : Q + (off + (N - 1 - o1) * nu + a) + (long long)(off + (N - 1 - o2) * nu + bb) * nvar;
    const long long qstep = (long long)nu * ((qtile ? P.nU : nvar) + 1); // one block up the diagonal per step
    for (int jmax = N - 1; jmax >= ad; --jmax, qout -= qstep) {
        double val = (dd == 0 && a == bb) ? P.qdiag : 0.0;
        for (int ci = 0; ci < P.ncost; ++ci) {
            const CostFam& F = P.cost[ci];
            if (F.dense) continue; // added afterwards by the GEMM path (Q += T'WT)
            const int r = F.rows, rnu = r * nu;
            // steps i in [max(i0,jmax), i1-1]  <->  kk = i - jmax
            const int kk_hi = F.i1 - 1 - jmax;
            if (kk_hi < 0) continue;
            const double* base_a = MG[ci] + r * (a + nu * o1);
            const double* base_b = MG[ci] + r * (bb + nu * o2);
            double contrib;
            if (F.i0 == 0) {
                // running sum over kk ascending; terms are independent of jmax (Toeplitz), so only
                // the not-yet-included kk in (done, kk_hi] are added at this jmax
                for (int kk = done[ci]; kk <= kk_hi; ++kk) run[ci] = add_(run[ci], wdot(base_a + rnu * kk, Wt[ci], base_b + rnu * kk, r));
                done[ci] = kk_hi + 1;
                contrib = run[ci];
            } else {
                contrib = 0.0;
                for (int kk = max(F.i0 - jmax, 0); kk <= kk_hi; ++kk)
                    contrib = add_(contrib, wdot(base_a + rnu * kk, Wt[ci], base_b + rnu * kk, r));
            }
            val = add_(val, contrib);
        }
        *qout = val;
    }
}

// `staged`: the per-instance M A^k B tables and weights of every step-size cost are first copied to shared memory, so the
// sequential walk down each block diagonal runs at shared-memory instead of L2 latency (host checks that they fit).
__global__ void k2_assemble_q_kernel(const __grid_constant__ BuildParams P, int staged)
{
    extern __shared__ double stage_sm[];
    const int nchain = (2 * P.N - 1) * P.nu * P.nu;
    const int ch = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    const double* MG[kMaxCost];
    const double* Wt[kMaxCost];
    int o = 0;
    for (int ci = 0; ci < P.ncost; ++ci) {
        const CostFam& F = P.cost[ci];
        MG[ci] = F.MGx + (long long)b * F.sMGx;
        Wt[ci] = F.w.at(b);
        if (!staged || F.dense) continue;
        for (int t = threadIdx.x; t < int(F.sMGx); t += blockDim.x) stage_sm[o + t] = MG[ci][t];
        MG[ci] = stage_sm + o;
        o += int(F.sMGx);
        for (int t = threadIdx.x; t < F.rows; t += blockDim.x) stage_sm[o + t] = Wt[ci][t];
        Wt[ci] = stage_sm + o;
        o += F.rows;
    }
    if (staged) __syncthreads();
    if (ch < nchain) dev_q_chain(P, b, ch, MG, Wt, nullptr);
}

// Small Hessians (nU^2 doubles fit shared memory next to the staged cost tables): one CTA per instance assembles Q in a
// shared-memory tile.  Work is balanced by giving every thread the block diagonal dd = p (N - p steps) AND its
// complement dd = p - N (p steps): N steps per thread.  Costs are the outer loop, so their descriptors live in
// registers; every entry still receives  ((qdiag + cost_0) + cost_1) + ...  with each cost's running sum over kk
// ascending -- the reference accumulation order.  The tile is written out coalesced.
__global__ void k2_assemble_q_tiled_kernel(const __grid_constant__ BuildParams P)
{
    const int nu = P.nu, N = P.N, nU = P.nU, nvar = P.nvar;
    const int b = blockIdx.x;
    int mgo[kMaxCost], wto[kMaxCost];
    int o = 0;
    for (int ci = 0; ci < P.ncost; ++ci) {
        const CostFam& F = P.cost[ci];
        mgo[ci] = wto[ci] = 0;
        if (F.dense) continue;
        stage_copy(o, F.MGx + (long long)b * F.sMGx, int(F.sMGx));
        mgo[ci] = o;
        o += int(F.sMGx);
        stage_copy(o, F.w.at(b), F.rows);
        wto[ci] = o;
        o += F.rows;
    }
    const int tile = o;
    for (int idx = threadIdx.x; idx < nU * nU; idx += blockDim.x) stage_sm[tile + idx] = 0.0;
    __syncthreads();
    for (int i = threadIdx.x; i < nU; i += blockDim.x) stage_sm[tile + i * (nU + 1)] = P.qdiag; // LMPC::updateSystem: Q = 1e-6 I
    __syncthreads();
    const int qstep = nu * (nU + 1);
    for (int t = threadIdx.x; t < N * nu * nu; t += blockDim.x) {
        const int a = t % nu, bb = (t / nu) % nu, pidx = t / (nu * nu);
        // virtual chain of exactly N steps: block diagonal dd = pidx for the first N - pidx steps (jmax = N-1 .. pidx),
        // then dd = pidx - N for the remaining pidx steps (jmax = N-1 .. N-pidx): every lane of a warp runs N steps
        const int len0 = N - pidx;
        for (int ci = 0; ci < P.ncost; ++ci) {
            const CostFam& F = P.cost[ci];
            if (F.dense) continue; // added afterwards by the GEMM path (Q += T'WT)
            const int r = F.rows, rnu = r * nu, i0 = F.i0, i1 = F.i1, wo = wto[ci];
            int ga = mgo[ci] + r * a, gb = mgo[ci] + r * (bb + nu * pidx);               // dd = pidx: o1 = 0, o2 = dd
            int qp = tile + ((N - 1) * nu + a) + ((N - 1 - pidx) * nu + bb) * nU;         // its entry at jmax = N-1
            // sum_l (ga[l] * w[l]) * gb[l] in the reference order; straight-line code for the usual 1- and 2-row costs
            auto wdot = [&](int oa, int ob) {
                double sd = add_(0.0, mul_(mul_(stage_sm[oa], stage_sm[wo]), stage_sm[ob]));
                if (r == 1) return sd;
                sd = add_(sd, mul_(mul_(stage_sm[oa + 1], stage_sm[wo + 1]), stage_sm[ob + 1]));
#pragma unroll 1
                for (int l = 2; l < r; ++l) sd = add_(sd, mul_(mul_(stage_sm[oa + l], stage_sm[wo + l]), stage_sm[ob + l]));
                return sd;
            };
            double run = 0.0;
            int kk = 0, jmax = N - 1;
            for (int sidx = 0; sidx < N; ++sidx, --jmax, qp -= qstep) {
                if (sidx == len0) { // switch to dd = pidx - N: o1 = N - pidx, o2 = 0
                    ga = mgo[ci] + r * (a + nu * (N - pidx));
                    gb = mgo[ci] + r * bb;
                    qp = tile + ((pidx - 1) * nu + a) + ((N - 1) * nu + bb) * nU;
                    run = 0.0;
                    kk = 0;
                    jmax = N - 1;
                }
                const int kk_hi = i1 - 1 - jmax;
                if (kk_hi < 0) continue;
                double contrib;
                if (i0 == 0) {
#pragma unroll 1 // one new term per step (two at the first step of an (N+1)-step cost): no unroll cascade
                    for (; kk <= kk_hi; ++kk) run = add_(run, wdot(ga + rnu * kk, gb + rnu * kk));
                    contrib = run;
                } else {
                    contrib = 0.0;
#pragma unroll 1
                    for (int k2 = max(i0 - jmax, 0); k2 <= kk_hi; ++k2) contrib = add_(contrib, wdot(ga + rnu * k2, gb + rnu * k2));
                }
                stage_sm[qp] = add_(stage_sm[qp], contrib);
            }
        }
    }
    __syncthreads();
    const int off = P.initial_state ? P.nx : 0;
    double* Q = P.Q + (long long)b * P.sQ + off + (long long)off * nvar;
    if (off == 0 && nvar == nU) {
        for (int idx = threadIdx.x; idx < nU * nU; idx += blockDim.x) Q[idx] = stage_sm[tile + idx];
    } else {
        for (int idx = threadIdx.x; idx < nU * nU; idx += blockDim.x) {
            const int i = idx % nU, j = idx / nU;
            Q[i + (long long)j * nvar] = stage_sm[tile + idx];
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K2c: per-cost E (nx x nU) and f (nU):  E = sum_i MPhi_i' W T_i, f = sum_i res_i' W T_i
// (src/costFunctions.cpp:77-78,105-106,210-211).  One thread per (s|f, column).  grid = (tiles, batch)
// ------------------------------------------------------------------------------------------------
template <bool STAGED>
__device__ __forceinline__ void dev_ef(const BuildParams& P, int b, int t, int ci, Tab<STAGED> MG, Tab<STAGED> MPhi, Tab<STAGED> res,
    Tab<STAGED> w)
{
    const int nx = P.nx, nu = P.nu, nU = P.nU;
    const int s = t % (nx + 1), col = t / (nx + 1);
    const int j = col / nu, bb = col % nu;
    const CostFam& F = P.cost[ci];
    const int r = F.rows;
    double acc = 0.0;
    {
        const int ibeg = max(F.i0, j);
        Tab<STAGED> g = MG.shifted(r * (bb + nu * (ibeg - j)));
        Tab<STAGED> lhs = (s < nx) ? MPhi.shifted(r * (s + nx * (ibeg - F.i0))) : res.shifted(r * (ibeg - F.i0));
        const int gstep = r * nu, lstep = (s < nx) ? r * nx : r;
        int go = 0, lo = 0;
        for (int i = ibeg; i < F.i1; ++i, go += gstep, lo += lstep) {
            double sum = 0.0;
            if (r == 1) sum = add_(sum, mul_(mul_(lhs[lo], w[0]), g[go]));
            else
                for (int l = 0; l < r; ++l) sum = add_(sum, mul_(mul_(lhs[lo + l], w[l]), g[go + l]));
            acc = add_(acc, sum);
        }
    }
    if (s < nx) F.E[(long long)b * F.sE + s + (long long)col * nx] = acc;
    else F.f[(long long)b * F.sf + col] = acc;
    (void)nU;
}

// grid = (tiles over (nx+1) nU, batch, cost); STAGED: this cost's tables are first copied to shared memory.
// f_all: every instance forms only f (a retarget: E is resident and unchanged)
template <bool STAGED> __global__ void k2_assemble_ef_kernel(const __grid_constant__ BuildParams P, int f_all)
{
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y, ci = blockIdx.z;
    const CostFam& F = P.cost[ci];
    if (F.dense) return;
    // batch-invariant E (sE == 0): instance 0 forms E and its f, every other instance only its nU entries of f
    const bool f_only = (F.sE == 0 && b > 0) || f_all;
    if (f_only) {
        if (blockIdx.x * blockDim.x >= P.nU) return;
        t = (t < P.nU) ? t * (P.nx + 1) + P.nx : (P.nx + 1) * P.nU; // (s, col) = (nx, t)
    }
    Tab<STAGED> MG{ F.MGx + (long long)b * F.sMGx, 0 };
    Tab<STAGED> MPhi{ F.MPhi + (long long)b * F.sMPhi, 0 };
    Tab<STAGED> res{ F.res + (long long)b * F.sres, 0 };
    Tab<STAGED> w{ F.w.at(b), 0 };
    if (STAGED) {
        int o = 0;
        stage_copy(o, MG.g, int(F.sMGx)); MG.o = o; o += int(F.sMGx);
        stage_copy(o, MPhi.g, int(F.sMPhi)); MPhi.o = o; o += int(F.sMPhi);
        stage_copy(o, res.g, int(F.sres)); res.o = o; o += int(F.sres);
        stage_copy(o, w.g, F.rows); w.o = o;
        __syncthreads();
    }
    if (t < (P.nx + 1) * P.nU) dev_ef<STAGED>(P, b, t, ci, MG, MPhi, res, w);
}

// ------------------------------------------------------------------------------------------------
// K3: constraint rows.  A_i[:, block j] = EGx[i-j] (j <= i, j < N), zero otherwise
// (src/constraints.cpp:77,142,209-219,289,302); in initial-state mode the first nx columns are Y
// (src/InitialStateLMPC.cpp:88-101).  One thread per row, coalesced down each column.
// grid = (row tiles over meq+mineq, batch)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void dev_fill_row(const BuildParams& P, int b, int row)
{
    const int nx = P.nx, nu = P.nu, N = P.N, nvar = P.nvar;
    const int off = P.initial_state ? nx : 0;
    const bool iseq = row < P.meq;
    const int lrow = iseq ? row : row - P.meq;
    const int mtot = iseq ? P.meq : P.mineq;
    // find the family (few of them)
    int fi = -1;
    for (int k = 0; k < P.nfam; ++k) {
        const CstrFam& F = P.fam[k];
        if ((F.is_eq != 0) == iseq && lrow >= F.row_off && lrow < F.row_off + F.rows * (F.i1 - F.i0)) { fi = k; break; }
    }
    if (fi < 0) return;
    const CstrFam& F = P.fam[fi];
    double* Aout = (iseq ? P.Aeq : P.Aineq) + (long long)b * mtot * nvar;
    if (off) {
        const double* Y = (iseq ? P.Yeq : P.Yin) + (long long)b * mtot * nx;
        for (int s = 0; s < nx; ++s) Aout[lrow + (long long)s * mtot] = Y[lrow + (long long)s * mtot];
    }
    if (F.dense || F.gather) return; // rows written by the GEMM / gather path
    const int r = F.rows;
    const int i = F.i0 + (lrow - F.row_off) / r, l = (lrow - F.row_off) % r;
    const double* EGx = F.EGx + (long long)b * F.sEGx;
    for (int j = 0; j < N; ++j) {
        const int kk = i - j;
        for (int bb = 0; bb < nu; ++bb) {
            const double v = (kk >= 0) ? EGx[l + r * (bb + nu * kk)] : 0.0;
            Aout[lrow + (long long)(off + j * nu + bb) * mtot] = v;
        }
    }
}

__global__ void k3_fill_rows_kernel(const __grid_constant__ BuildParams P)
{
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row < P.meq + P.mineq) dev_fill_row(P, blockIdx.y, row);
}

// ------------------------------------------------------------------------------------------------
// Full-size (autoSpan'd) entries: epilogues around the DMMA GEMMs (dgemm_dmma.cu).
//   cost : T (rows x nU) holds M Psi; T += N (or T = N); WT = diag(w) T; res = M xi - p (or -p); MPhi = 0 without M
//          (src/costFunctions.cpp:65-71,141-146,197-203)
//   cstr : A rows hold E Psi; A += G (or A = G); z = f - E xi (or f); Y = 0 without E   (src/constraints.cpp:68-73,199-204)
// grid = (element tiles, batch)
// ------------------------------------------------------------------------------------------------
__global__ void k2_dense_cost_epilogue_kernel(const __grid_constant__ BuildParams P, int ci)
{
    const CostFam& F = P.cost[ci];
    const int b = blockIdx.y, R = F.rows, nU = P.nU, nx = P.nx;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)R * nU) return;
    const int r = int(t % R), c = int(t / R);
    double* T = F.T + (long long)b * F.sT;
    double* WT = F.WT + (long long)b * F.sT;
    double v = F.hasM ? T[t] : 0.0;
    if (F.hasN) v = F.hasM ? add_(v, F.N.at(b)[t]) : F.N.at(b)[t];
    T[t] = v;
    WT[t] = mul_(F.w.at(b)[r], v);
    if (c == 0) {
        double* res = F.res + (long long)b * F.sres;
        res[r] = F.hasM ? add_(res[r], -F.p.at(b)[r]) : -F.p.at(b)[r];
        if (!F.hasM) {
            double* MPhi = F.MPhi + (long long)b * F.sMPhi;
            for (int s = 0; s < nx; ++s) MPhi[r + (long long)s * R] = 0.0;
        }
    }
}

__global__ void k3_dense_cstr_epilogue_kernel(const __grid_constant__ BuildParams P, int fi)
{
    const CstrFam& F = P.fam[fi];
    const int b = blockIdx.y, R = F.rows, nU = P.nU, nx = P.nx, nvar = P.nvar;
    const int off = P.initial_state ? nx : 0;
    const int mtot = F.is_eq ? P.meq : P.mineq;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)R * nU) return;
    const int r = int(t % R), c = int(t / R);
    double* Aout = (F.is_eq ? P.Aeq : P.Aineq) + (long long)b * mtot * nvar + F.row_off + (long long)off * mtot;
    double v = F.hasE ? Aout[r + (long long)c * mtot] : 0.0;
    if (F.hasG) v = F.hasE ? add_(v, F.G.at(b)[t]) : F.G.at(b)[t];
    Aout[r + (long long)c * mtot] = v;
    if (c == 0) {
        double* z = (F.is_eq ? P.zeq : P.zin) + (long long)b * mtot + F.row_off;
        z[r] = F.hasE ? add_(F.f.at(b)[r], -z[r]) : F.f.at(b)[r];
        if (!F.hasE) {
            double* Y = (F.is_eq ? P.Yeq : P.Yin) + (long long)b * mtot * nx + F.row_off;
            for (int s = 0; s < nx; ++s) Y[r + (long long)s * mtot] = 0.0;
        }
    }
}

// full-size TrajectoryBoundConstraint: rows are copies of rows fidx[] of Psi / Phi / xi (src/constraints.cpp:288-314)
__global__ void k3_gather_rows_kernel(const __grid_constant__ BuildParams P, int fi)
{
    const CstrFam& F = P.fam[fi];
    const int b = blockIdx.y, R = F.rows, nU = P.nU, nx = P.nx, nu = P.nu, N = P.N, X = P.X, nvar = P.nvar;
    const int off = P.initial_state ? nx : 0;
    const int mtot = F.is_eq ? P.meq : P.mineq;
    const long long NX = (long long)N * nx;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)R * nU) return;
    const int r = int(t % R), col = int(t / R);
    const int idx = F.fidx[r], i = idx / nx, l = idx % nx, j = col / nu, c = col % nu;
    const double* Gs = P.Gs + (long long)b * NX * nu;
    double* Aout = (F.is_eq ? P.Aeq : P.Aineq) + (long long)b * mtot * nvar + F.row_off + (long long)off * mtot;
    Aout[r + (long long)col * mtot] = (i > j) ? Gs[(long long)(i - 1 - j) * nx + l + (long long)c * NX] : 0.0;
    if (col == 0) {
        const double* Phi = P.Phi + (long long)b * X * nx;
        double* Y = (F.is_eq ? P.Yeq : P.Yin) + (long long)b * mtot * nx + F.row_off;
        double* z = (F.is_eq ? P.zeq : P.zin) + (long long)b * mtot + F.row_off;
        for (int s = 0; s < nx; ++s) Y[r + (long long)s * mtot] = Phi[idx + (long long)s * X];
        z[r] = add_(F.f.at(b)[idx], -P.xi[(long long)b * X + idx]);
    }
}

// ------------------------------------------------------------------------------------------------
// K4: c, beq/bineq, lb/ub (+ the E blocks of the initial-state Hessian).  One CTA per instance.
//  LMPC : c = sum_costs (E'x0 + f) ; b = z - Y x0             (src/costFunctions.cpp:81, constraints.cpp:82, LMPC.cpp:252-279)
//  IS   : c = [r; sum f] ; Q_tr = sum E, Q_bl = Q_tr' ; b = z  (src/InitialStateLMPC.cpp:80-121)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void dev_finalize(const BuildParams& P, int b)
{
    const int nx = P.nx, nu = P.nu, nU = P.nU, nvar = P.nvar;
    const int off = P.initial_state ? nx : 0;
    const int tid = threadIdx.x, T = blockDim.x;
    {
        const double* x0 = P.x0.at(b);
        double* c = P.c + (long long)b * nvar;
        double* Q = P.Q + (long long)b * P.sQ;
        for (int col = tid; col < nU; col += T) {
            double acc = 0.0;
            for (int ci = 0; ci < P.ncost; ++ci) {
                const CostFam& F = P.cost[ci];
                const double* E = F.E + (long long)b * F.sE + (long long)col * nx;
                const double fv = F.f[(long long)b * F.sf + col];
                if (P.initial_state) acc = add_(acc, fv);
                else {
                    double s = 0.0;
                    for (int a = 0; a < nx; ++a) s = add_(s, mul_(E[a], x0[a]));
                    acc = add_(acc, add_(s, fv));
                }
            }
            c[off + col] = acc;
            if (P.initial_state) {
                for (int a = 0; a < nx; ++a) {
                    double e = 0.0;
                    for (int ci = 0; ci < P.ncost; ++ci) e = add_(e, P.cost[ci].E[(long long)b * P.cost[ci].sE + a + (long long)col * nx]);
                    Q[a + (long long)(off + col) * nvar] = e;
                    Q[(off + col) + (long long)a * nvar] = e;
                }
            }
        }
        for (int pass = 0; pass < 2; ++pass) {
            const int mtot = pass == 0 ? P.meq : P.mineq;
            const double* Y = (pass == 0 ? P.Yeq : P.Yin) + (long long)b * mtot * nx;
            const double* z = (pass == 0 ? P.zeq : P.zin) + (long long)b * mtot;
            double* bo = (pass == 0 ? P.beq : P.bineq) + (long long)b * mtot;
            for (int row = tid; row < mtot; row += T) {
                if (P.initial_state) bo[row] = z[row];
                else {
                    double s = 0.0;
                    for (int a = 0; a < nx; ++a) s = add_(s, mul_(Y[row + (long long)a * mtot], x0[a]));
                    bo[row] = add_(z[row], -s);
                }
            }
        }
        double* lb = P.lb + (long long)b * nvar;
        double* ub = P.ub + (long long)b * nvar;
        for (int k = tid; k < nU; k += T) {
            lb[off + k] = P.cb_lower.p ? P.cb_lower.at(b)[P.cb_full ? k : k % nu] : -DBL_MAX;
            ub[off + k] = P.cb_upper.p ? P.cb_upper.at(b)[P.cb_full ? k : k % nu] : DBL_MAX;
        }
        if (P.initial_state) {
            for (int k = tid; k < nx; k += T) {
                c[k] = P.r.p ? P.r.at(b)[k] : 0.0;
                lb[k] = P.x0lb.p ? P.x0lb.at(b)[k] : x0[k];
                ub[k] = P.x0ub.p ? P.x0ub.at(b)[k] : x0[k];
            }
        }
    }
}

__global__ void k4_finalize_kernel(const __grid_constant__ BuildParams P)
{
    for (int b = blockIdx.x; b < P.batch; b += gridDim.x) dev_finalize(P, b);
}

// ------------------------------------------------------------------------------------------------
// K4': initial-state Schur block  Q_tl = R + E Qb^-1 E'  (src/InitialStateLMPC.cpp:114-117, quirk Q7).
// The reference inverts Qb with Eigen's LU; Qb is SPD (it contains the 1e-6 I regulariser), so the
// GPU path uses Cholesky: Qb = U'U, J = U^-1, V = E J, Q_tl = R + V V'.  One CTA per instance; J in
// shared memory when it fits, else in the global workspace `ws`.
// ------------------------------------------------------------------------------------------------
__global__ void k4_schur_kernel(const __grid_constant__ BuildParams P, double* ws, long long ws_stride, int j_smem)
{
    extern __shared__ double sm[];
    const int nx = P.nx, nU = P.nU, nvar = P.nvar, ld = odd_ld(nU);
    const int tid = threadIdx.x, T = blockDim.x;
    double* rowbuf = sm;                 // nU + 1
    double* rowk = rowbuf + nU + 1;      // nU
    double* V = rowk + nU;               // nx x nU
    double* Jm = j_smem ? V + (size_t)nx * nU : ws + (long long)blockIdx.x * ws_stride;
    for (int b = blockIdx.x; b < P.batch; b += gridDim.x) {
        double* Q = P.Q + (long long)b * nvar * nvar;
        __syncthreads();
        for (int idx = tid; idx < nU * nU; idx += T) {
            const int i = idx % nU, j = idx / nU;
            Jm[i + (size_t)j * ld] = Q[(nx + i) + (long long)(nx + j) * nvar];
        }
        __syncthreads();
        const bool ok = chol_upper_inplace(Jm, ld, nU, rowbuf);
        if (ok) {
            tri_inverse_upper_inplace(Jm, ld, nU, rowbuf, rowk);
            for (int t = tid; t < nx * nU; t += T) { // V[s,i] = sum_{k<=i} E[s,k] J[k,i]
                const int s = t % nx, i = t / nx;
                double acc = 0.0;
                for (int k = 0; k <= i; ++k) acc += Q[s + (long long)(nx + k) * nvar] * Jm[k + (size_t)i * ld];
                V[t] = acc;
            }
            __syncthreads();
        }
        for (int t = tid; t < nx * nx; t += T) {
            const int s = t % nx, u = t / nx;
            double acc = 0.0;
            if (ok) for (int i = 0; i < nU; ++i) acc += V[s + (size_t)i * nx] * V[u + (size_t)i * nx];
            else acc = CUDART_NAN; // Hessian not PD: the solver will report fail=2 on the NaN pivot
            const double Rv = P.R.p ? P.R.at(b)[t] : 0.0;
            Q[s + (long long)u * nvar] = Rv + acc;
        }
    }
}

// nU <= 64: the same Schur block with the fused Cholesky + inverse sweep of the small solver (gi_small.cuh:
// one rank-1 sweep and two barriers per pivot).  128 threads per instance, 4 instances resident per SM.
__global__ void __launch_bounds__(kSmT, 4) k4_schur_small_kernel(const __grid_constant__ BuildParams P)
{
    extern __shared__ __align__(16) double sm[];
    const int nx = P.nx, nU = P.nU, nvar = P.nvar, n2 = (nU + 1) & ~1, ld = ld_vec2(nU);
    const int tid = threadIdx.x;
    double* Jm = sm;                       // ld x n2
    double* coef = Jm + (size_t)ld * n2;   // n2 + 2
    double* V = coef + 8 * (size_t)(n2 + 2); // nx x nU   (8 scratch vectors of n2 + 2: coefficients / multipliers of 4 pivots)
    for (int b = blockIdx.x; b < P.batch; b += gridDim.x) {
        double* Q = P.Q + (long long)b * nvar * nvar;
        __syncthreads();
        for (int idx = tid; idx < ld * n2; idx += kSmT) {
            const int i = idx % ld, j = idx / ld;
            Jm[idx] = (i < nU && j < nU) ? Q[(nx + i) + (long long)(nx + j) * nvar] : ((i == j && i < n2) ? 1.0 : 0.0);
        }
        __syncthreads();
        double* const coefp[4] = { coef, coef + (n2 + 2), coef + 2 * (n2 + 2), coef + 3 * (n2 + 2) };
        double* const multp[4] = { coef + 4 * (n2 + 2), coef + 5 * (n2 + 2), coef + 6 * (n2 + 2), coef + 7 * (n2 + 2) };
        const bool ok = gs_factor_nb<kSmFacNB>(Jm, ld, nU, n2, coefp, multp);
        if (ok) {
            for (int t = tid; t < nx * nU; t += kSmT) { // V[s,i] = sum_{k<=i} E[s,k] J[k,i]
                const int s = t % nx, i = t / nx;
                double acc = 0.0;
                for (int k = 0; k <= i; ++k) acc += Q[s + (long long)(nx + k) * nvar] * Jm[k + (size_t)i * ld];
                V[t] = acc;
            }
            __syncthreads();
        }
        for (int t = tid; t < nx * nx; t += kSmT) {
            const int s = t % nx, u = t / nx;
            double acc = 0.0;
            if (ok) for (int i = 0; i < nU; ++i) acc += V[s + (size_t)i * nx] * V[u + (size_t)i * nx];
            else acc = CUDART_NAN; // Hessian not PD: the solver will report fail=2 on the NaN pivot
            const double Rv = P.R.p ? P.R.at(b)[t] : 0.0;
            Q[s + (long long)u * nvar] = Rv + acc;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K7: LMPC::updateResults (src/LMPC.cpp:282-286 / InitialStateLMPC.cpp:124-128):
//   control = result (tail), trajectory = Phi x0 + Psi U + xi with Psi applied as the block-Toeplitz
//   convolution sum_{j<i} G_{i-1-j} u_j straight from the compact Gs.  One thread per trajectory row.
// grid = (row tiles over X, batch)
// ------------------------------------------------------------------------------------------------
template <bool STAGED>
__global__ void k7_results_kernel(const __grid_constant__ BuildParams P, const double* __restrict__ xres, double* __restrict__ control,
    double* __restrict__ traj)
{
    const int nx = P.nx, nu = P.nu, N = P.N, X = P.X, nU = P.nU, nvar = P.nvar;
    const int off = P.initial_state ? nx : 0;
    const int NX = N * nx;
    const int b = blockIdx.y;
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    // the solution and the compact Psi column block are read N times per row: keep them in shared memory when they fit
    Tab<STAGED> xr{ xres + (long long)b * nvar, 0 };
    Tab<STAGED> Gs{ P.Gs + (long long)b * NX * nu, nvar };
    if (STAGED) {
        stage_copy(0, xr.g, nvar);
        stage_copy(nvar, Gs.g, NX * nu);
        __syncthreads();
    }
    if (control && row < nU) control[(long long)b * nU + row] = xr[off + row];
    if (!traj || row >= X) return;
    const double* Phi = P.Phi + (long long)b * X * nx;
    const int i = row / nx, r = row % nx;
    double s1 = 0.0;
    for (int a = 0; a < nx; ++a) s1 = add_(s1, mul_(Phi[row + (long long)a * X], P.initial_state ? xr[a] : P.x0.at(b)[a]));
    double s2 = 0.0;
    int go = (i - 1) * nx + r; // G_{i-1-j}[r, :]
    if (nu == 1) { // the common single-input case without the inner-loop bookkeeping
        for (int j = 0; j < i; ++j, go -= nx) s2 = add_(s2, mul_(Gs[go], xr[off + j]));
    } else {
        for (int j = 0; j < i; ++j, go -= nx) {
#pragma unroll 1
            for (int cc = 0; cc < nu; ++cc) s2 = add_(s2, mul_(Gs[go + cc * NX], xr[off + j * nu + cc]));
        }
    }
    traj[(long long)b * X + row] = add_(add_(s1, s2), P.xi[(long long)b * X + row]);
}

// ------------------------------------------------------------------------------------------------
static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

#define CB_CHECK_LAUNCH()                         \
    do {                                          \
        cudaError_t e_ = cudaGetLastError();      \
        if (e_ != cudaSuccess) return -int(e_);   \
        ++launches;                               \
    } while (0)

#define CB_GEMM(...)                                   \
    do {                                               \
        int n_ = dgemm_dmma_launch(__VA_ARGS__);       \
        if (n_ < 0) return n_;                         \
        launches += n_;                                \
    } while (0)

// K2c for every step-size cost (f_all: f alone, see k2_assemble_ef_kernel)
static int ef_launch(const BuildParams& P, int f_all, cudaStream_t st)
{
    size_t need = 0; // largest single cost: its M A^k B, M Phi_i, residual tables and weights
    for (int i = 0; i < P.ncost; ++i)
        if (!P.cost[i].dense)
            need = std::max(need, size_t(P.cost[i].sMGx) + size_t(P.cost[i].sMPhi) + size_t(P.cost[i].sres) + P.cost[i].rows);
    const dim3 grid(ceil_div(f_all ? P.nU : (P.nx + 1) * P.nU, 128), P.batch, P.ncost);
    if (need * sizeof(double) <= 40 * 1024) k2_assemble_ef_kernel<true><<<grid, 128, need * sizeof(double), st>>>(P, f_all);
    else k2_assemble_ef_kernel<false><<<grid, 128, 0, st>>>(P, f_all);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 1 : -int(e);
}

int k2k4_assemble_launch(const BuildParams& P, double* schur_ws, long long schur_stride, int sms, size_t smem_optin, cudaStream_t st)
{
    int launches = 0;
    if (P.batch > 65535) return -int(cudaErrorInvalidValue); // gridDim.y limit: the C API chunks larger batches
    const int pgrid = std::min(P.batch, sms * 8);
    const int nb = P.batch, nx = P.nx, nU = P.nU, X = P.X, nvar = P.nvar;
    const int off = P.initial_state ? nx : 0;
    bool any_dense = false;
    for (int i = 0; i < P.ncost; ++i) any_dense |= P.cost[i].dense && P.cost[i].hasM;
    for (int k = 0; k < P.nfam; ++k) any_dense |= P.fam[k].dense && P.fam[k].hasE;
    k2_precompute_kernel<false><<<pgrid, 128, 0, st>>>(P);
    CB_CHECK_LAUNCH();
    if (any_dense) { // dense M / E blocks multiply the materialised Psi
        int n_ = k1_psi_fill_launch(P.Gs, (long long)P.N * nx * P.nu, P.PsiFull, nx, P.nu, P.N, nb, st);
        if (n_ < 0) return n_;
        launches += n_;
    }
    {
        const int nchain = (2 * P.N - 1) * P.nu * P.nu;
        const int nbq = P.sQ == 0 ? 1 : nb; // batch-invariant Hessian: assembled once from instance 0's tables
        size_t need = 0; // staged tables: M A^k B blocks + weights of every step-size cost
        for (int i = 0; i < P.ncost; ++i) if (!P.cost[i].dense) need += size_t(P.cost[i].sMGx) + P.cost[i].rows;
        const int staged = need * sizeof(double) <= 40 * 1024;
        // small Hessians: one CTA per instance assembles Q in a shared-memory tile and writes it out coalesced
        const size_t tile = size_t(nU) * nU;
        const int tiled = staged && (need + tile) * sizeof(double) <= 44 * 1024;
        if (tiled) {
            const int threads = std::min(256, std::max(32, ceil_div(P.N * P.nu * P.nu, 32) * 32));
            k2_assemble_q_tiled_kernel<<<nbq, threads, (need + tile) * sizeof(double), st>>>(P);
        } else
            k2_assemble_q_kernel<<<dim3(ceil_div(nchain, 128), nbq), 128, staged ? need * sizeof(double) : 0, st>>>(P, staged);
        CB_CHECK_LAUNCH();
    }
    const long long sPsi = (long long)X * nU, sPhi = (long long)X * nx;
    for (int ci = 0; ci < P.ncost; ++ci) { // full-size costs: T = M Psi (+N), Q += T'WT, E = (M Phi)'WT, f = res'WT
        const CostFam& F = P.cost[ci];
        if (!F.dense) continue;
        const int R = F.rows;
        if (F.hasM) {
            CB_GEMM(0, R, nU, X, 1.0, F.M.p, R, F.M.s, P.PsiFull, X, sPsi, 0.0, F.T, R, F.sT, nb, st);
            CB_GEMM(0, R, nx, X, 1.0, F.M.p, R, F.M.s, P.Phi, X, sPhi, 0.0, F.MPhi, R, F.sMPhi, nb, st);
            CB_GEMM(0, R, 1, X, 1.0, F.M.p, R, F.M.s, P.xi, X, (long long)X, 0.0, F.res, R, F.sres, nb, st);
        }
        k2_dense_cost_epilogue_kernel<<<dim3(ceil_div(R * nU, 256), nb), 256, 0, st>>>(P, ci);
        CB_CHECK_LAUNCH();
        CB_GEMM(1, nU, nU, R, 1.0, F.T, R, F.sT, F.WT, R, F.sT, 1.0, P.Q + off + (long long)off * nvar, nvar, P.sQ, nb, st);
        CB_GEMM(1, nx, nU, R, 1.0, F.MPhi, R, F.sMPhi, F.WT, R, F.sT, 0.0, F.E, nx, F.sE, nb, st);
        CB_GEMM(1, 1, nU, R, 1.0, F.res, R, F.sres, F.WT, R, F.sT, 0.0, F.f, 1, F.sf, nb, st);
    }
    if (P.ncost > 0) {
        const int n_ = ef_launch(P, 0, st);
        if (n_ < 0) return n_;
        launches += n_;
    }
    for (int fi = 0; fi < P.nfam; ++fi) { // full-size constraints: rows = E Psi (+G), Y = E Phi, z = f - E xi
        const CstrFam& F = P.fam[fi];
        if (!F.dense && !F.gather) continue;
        const int R = F.rows, mtot = F.is_eq ? P.meq : P.mineq;
        double* Aout = (F.is_eq ? P.Aeq : P.Aineq) + F.row_off + (long long)off * mtot;
        double* Y = (F.is_eq ? P.Yeq : P.Yin) + F.row_off;
        double* z = (F.is_eq ? P.zeq : P.zin) + F.row_off;
        if (F.gather) {
            k3_gather_rows_kernel<<<dim3(ceil_div(R * nU, 256), nb), 256, 0, st>>>(P, fi);
            CB_CHECK_LAUNCH();
            continue;
        }
        if (F.hasE) {
            CB_GEMM(0, R, nU, X, 1.0, F.E.p, R, F.E.s, P.PsiFull, X, sPsi, 0.0, Aout, mtot, (long long)mtot * nvar, nb, st);
            CB_GEMM(0, R, nx, X, 1.0, F.E.p, R, F.E.s, P.Phi, X, sPhi, 0.0, Y, mtot, (long long)mtot * nx, nb, st);
            CB_GEMM(0, R, 1, X, 1.0, F.E.p, R, F.E.s, P.xi, X, (long long)X, 0.0, z, mtot, (long long)mtot, nb, st);
        }
        k3_dense_cstr_epilogue_kernel<<<dim3(ceil_div(R * nU, 256), nb), 256, 0, st>>>(P, fi);
        CB_CHECK_LAUNCH();
    }
    if (P.meq + P.mineq > 0 && !P.skip_rows) {
        k3_fill_rows_kernel<<<dim3(ceil_div(P.meq + P.mineq, 128), nb), 128, 0, st>>>(P);
        CB_CHECK_LAUNCH();
    }
    k4_finalize_kernel<<<pgrid, 128, 0, st>>>(P);
    CB_CHECK_LAUNCH();
    if (P.initial_state && P.nU <= kSmMaxN) {
        const int n2 = (P.nU + 1) & ~1;
        const size_t smem = sizeof(double) * (size_t(ld_vec2(P.nU)) * n2 + 8 * (size_t(n2) + 2) + size_t(P.nx) * P.nU);
        if (smem + 1024 > smem_optin) return -int(cudaErrorInvalidValue);
        cudaError_t e = cudaFuncSetAttribute(k4_schur_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
        if (e != cudaSuccess) return -int(e);
        const int per_sm = int(std::max<size_t>(1, std::min<size_t>(4, (smem_optin + 1024) / (smem + 1024))));
        k4_schur_small_kernel<<<std::min(P.batch, sms * per_sm), kSmT, smem, st>>>(P);
        CB_CHECK_LAUNCH();
    } else if (P.initial_state) {
        const int ld = odd_ld(P.nU);
        size_t base = sizeof(double) * (2 * size_t(P.nU) + 1 + size_t(P.nx) * P.nU);
        size_t withJ = base + sizeof(double) * size_t(ld) * P.nU;
        const int j_smem = withJ + 1024 <= smem_optin ? 1 : 0;
        const size_t smem = j_smem ? withJ : base;
        if (!j_smem && (!schur_ws || schur_stride < (long long)ld * P.nU)) return -int(cudaErrorInvalidValue);
        cudaError_t e = cudaFuncSetAttribute(k4_schur_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
        if (e != cudaSuccess) return -int(e);
        const int threads = P.nU <= 32 ? 128 : (P.nU <= 128 ? 256 : 512);
        const int per_sm = int(std::max<size_t>(1, std::min<size_t>(8, smem_optin / (smem + 1024))));
        const int grid = std::min(P.batch, sms * per_sm);
        k4_schur_kernel<<<grid, threads, smem, st>>>(P, schur_ws, schur_stride, j_smem);
        CB_CHECK_LAUNCH();
    }
    return launches;
}

int k2_retarget_launch(const BuildParams& P, int sms, cudaStream_t st)
{
    if (P.batch > 65535) return -int(cudaErrorInvalidValue);
    int launches = 0;
    k2_precompute_kernel<true><<<std::min(P.batch, sms * 8), 128, 0, st>>>(P);
    CB_CHECK_LAUNCH();
    if (P.ncost > 0) {
        const int n_ = ef_launch(P, 1, st);
        if (n_ < 0) return n_;
        launches += n_;
    }
    return launches;
}

int k3_fill_rows_launch(const BuildParams& P, cudaStream_t st)
{
    if (P.meq + P.mineq == 0) return 0;
    if (P.batch > 65535) return -int(cudaErrorInvalidValue);
    k3_fill_rows_kernel<<<dim3(ceil_div(P.meq + P.mineq, 128), P.batch), 128, 0, st>>>(P);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 1 : -int(e);
}

int k4_finalize_launch(const BuildParams& P, int sms, cudaStream_t st)
{
    k4_finalize_kernel<<<std::min(P.batch, sms * 8), 128, 0, st>>>(P);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 1 : -int(e);
}

int k7_results_launch(const BuildParams& P, const double* x, double* control, double* trajectory, cudaStream_t st)
{
    if (P.batch > 65535) return -int(cudaErrorInvalidValue);
    const int rows = std::max(P.X, P.nU);
    const size_t need = sizeof(double) * (size_t(P.nvar) + size_t(P.N) * P.nx * P.nu);
    const int staged = need <= 40 * 1024;
    const dim3 grid(ceil_div(rows, 128), P.batch);
    if (staged) k7_results_kernel<true><<<grid, 128, need, st>>>(P, x, control, trajectory);
    else k7_results_kernel<false><<<grid, 128, 0, st>>>(P, x, control, trajectory);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 1 : -int(e);
}

} // namespace cb
