// k8_vjp.cu -- K8: vector-Jacobian products of a solved batch of LMPC problems (LMPC mode, decision vector U).
//
// On the final active set the solution is an affine function of every vector input, so one adjoint KKT solve per
// instance gives the whole VJP.  With the active rows written as equalities a_j' U = beta_j (an Aeq row, an Aineq row
// or e_k for either bound, in their natural orientation) and gbar = dL/dU (+ Psi' dL/dtrajectory):
//   [Q A'; A 0] [v; mu] = [gbar; 0]        dL/dc = -v,   dL/dbeta_j = mu_j,   0 for the inactive rows.
// With Q = R'R, Jt = R^-1, Y = Jt' [A' | gbar] = [Y1 | t]:  G = Y1'Y1,  mu = G^-1 Y1' t,  v = Jt (t - Y1 mu).
// The GEMMs (Y, G, v) run on the DMMA kernel of dgemm_dmma.cu and G is factored by gt_factor_kernel; this file holds
// the four per-instance kernels around them:
//   k8_gather   [A_act' | gbar] into a zero-padded n x (nmax+1) slab: structured rows from the E A^k B tables (the
//               indexing of K3's dev_fill_row, so Aineq is never materialised), bound rows as unit vectors
//   k8_gram     G (nmax x nmax, 1 on the padded diagonal) and Y1' t out of the (nmax+1)^2 Gram matrix of Y
//   k8_mu       mu = R_G^-1 R_G^-T (Y1' t) and w = t - Y1 mu
//   k8_adjoint  the transpose of the vector part of K2 / K4 (what a retarget re-runs):
//               dx0 = sum_costs E c^ - Yeq' b^eq - Yin' b^in + Phi' dtraj,  dp_i = -W T_i c^,
//               df / dlower / dupper: b^, lb^, ub^ scattered through the index maps of dev_precompute / dev_finalize
// Instances whose status is not 0 keep an all-zero slab and their (pre-zeroed) gradients; a Hessian or Gram factorisation that
// fails gives NaN gradients instead of silently wrong ones.
#include "active_rows.cuh"
#include "common.cuh"
#include "engine.cuh"
#include "launch.h"

#include <algorithm>

namespace cb {

namespace {

constexpr int kVjpThreads = 256;

__device__ __forceinline__ int vjp_nact(const VjpParams& V, int b) { return V.status[b] == 0 ? V.nact[b] : 0; }

__global__ void __launch_bounds__(kVjpThreads) k8_gather_kernel(const __grid_constant__ BuildParams P, const __grid_constant__ VjpParams V)
{
    const int lb = blockIdx.x, b = V.b0 + lb;
    const int n = V.n, nu = P.nu, N = P.N, nx = P.nx, mg = P.meq + P.mineq, nm = V.nm;
    const long long NX = (long long)N * nx;
    double* slab = V.slab + (long long)lb * V.lds * (nm + 1);
    const int na = vjp_nact(V, b);
    for (long long t = threadIdx.x; t < (long long)V.lds * (nm + 1); t += blockDim.x) slab[t] = 0.0;
    __syncthreads();
    const int* iact = V.iact + (long long)b * n;
    for (int t = threadIdx.x; t < na * n; t += blockDim.x) {
        const int k = t / n, col = t % n;
        slab[col + (long long)k * V.lds] = active_row_entry(P, b, n, nu, mg, iact[k] - 1, col);
    }
    if (V.status[b] != 0) return;
    // gbar = dcontrol + Psi' dtraj, Psi' applied as the transposed block-Toeplitz product over the compact Gs
    const double* Gs = P.Gs + (long long)b * NX * nu;
    for (int col = threadIdx.x; col < n; col += blockDim.x) {
        double g = V.dcontrol ? V.dcontrol[(long long)b * V.sdc + col] : 0.0;
        if (V.dtraj) {
            const int j = col / nu, bb = col % nu;
            const double* dt = V.dtraj + (long long)b * V.sdt;
            double s = 0.0;
            for (int i = j + 1; i <= N; ++i) {
                const double* gcol = Gs + (long long)(i - 1 - j) * nx + (long long)bb * NX;
                for (int a = 0; a < nx; ++a) s += gcol[a] * dt[i * nx + a];
            }
            g += s;
        }
        slab[col + (long long)nm * V.lds] = g;
    }
}

// Gf: (nm+1) x (nm+1) Gram matrix of [Y1 | t] per instance -> Gq (nm x nm, padded diagonal 1) and rhs = Y1' t
__global__ void k8_gram_kernel(const __grid_constant__ VjpParams V)
{
    const int lb = blockIdx.x, b = V.b0 + lb, nm = V.nm, ld = nm + 1;
    const int na = vjp_nact(V, b);
    const double* Gf = V.Gf + (long long)lb * ld * ld;
    double* Gq = V.Gq + (long long)lb * nm * nm;
    for (int t = threadIdx.x; t < nm * nm; t += blockDim.x) {
        const int i = t % nm, j = t / nm;
        Gq[t] = (i < na && j < na) ? Gf[i + (long long)j * ld] : (i == j ? 1.0 : 0.0);
    }
    for (int i = threadIdx.x; i < nm; i += blockDim.x) V.rhs[(long long)lb * nm + i] = i < na ? Gf[i + (long long)nm * ld] : 0.0;
}

// mu = J_G J_G' rhs (J_G = R_G^-1), w = t - Y1 mu.  A Gram matrix that is not positive definite (linearly dependent
// active rows) gives NaN multipliers: the gradients of that instance are NaN rather than silently wrong.
__global__ void __launch_bounds__(kVjpThreads) k8_mu_kernel(const __grid_constant__ VjpParams V)
{
    extern __shared__ double vjp_sm[];
    const int lb = blockIdx.x, b = V.b0 + lb, nm = V.nm, n = V.n;
    const int na = vjp_nact(V, b);
    double* rhs = vjp_sm;     // nm
    double* s = rhs + nm;     // nm
    double* mu = s + nm;      // nm
    const double* Y = V.Y + (long long)lb * V.ldy * (nm + 1);
    if (na > 0) {
        const double* J = V.GJ + (long long)lb * V.ldg * nm;
        const bool ok = V.gpd[lb] != 0;
        for (int i = threadIdx.x; i < nm; i += blockDim.x) rhs[i] = V.rhs[(long long)lb * nm + i];
        __syncthreads();
        for (int j = threadIdx.x; j < na; j += blockDim.x) {
            double acc = 0.0;
            for (int i = 0; i <= j; ++i) acc += J[i + (long long)j * V.ldg] * rhs[i];
            s[j] = acc;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < na; i += blockDim.x) {
            double acc = 0.0;
            for (int j = i; j < na; ++j) acc += J[i + (long long)j * V.ldg] * s[j];
            mu[i] = ok ? acc : CUDART_NAN;
        }
        __syncthreads();
    }
    // a Hessian factor that failed (not positive definite) makes Y meaningless: NaN, as for G
    const bool qok = V.qpd[(long long)b * V.qpd_stride] != 0;
    for (int k = threadIdx.x; k < nm; k += blockDim.x) V.mu[(long long)lb * nm + k] = k < na ? (qok ? mu[k] : CUDART_NAN) : 0.0;
    double* w = V.W + (long long)lb * V.lds;
    for (int r = threadIdx.x; r < V.lds; r += blockDim.x) {
        double acc = 0.0;
        if (r < n && V.status[b] == 0) {
            acc = Y[r + (long long)nm * V.ldy];
            for (int k = 0; k < na; ++k) acc -= Y[r + (long long)k * V.ldy] * mu[k];
            if (!qok) acc = CUDART_NAN;
        }
        w[r] = acc;
    }
}

__global__ void __launch_bounds__(kVjpThreads) k8_adjoint_kernel(const __grid_constant__ BuildParams P, const __grid_constant__ VjpParams V)
{
    extern __shared__ double vjp_sm[];
    __shared__ double red[2 * kMaxWarps];
    const int lb = blockIdx.x, b = V.b0 + lb;
    if (V.status[b] != 0) return; // gradients stay at the zeros they were initialised to
    const int n = V.n, nx = P.nx, nu = P.nu, N = P.N, X = P.X, meq = P.meq, mineq = P.mineq, mg = meq + mineq, nm = V.nm;
    const int na = V.nact[b];
    const int tid = threadIdx.x, T = blockDim.x;
    double* ch = vjp_sm;          // n    c^ = -v
    double* bh = ch + n;          // mg + 2n: b^eq | b^in | ub^ | lb^  (the solver's constraint index space)
    double* tmp = bh + mg + 2 * n; // per-step partials of one cost
    for (int t = tid; t < n; t += T) ch[t] = -V.V[(long long)lb * V.lds + t];
    for (int t = tid; t < mg + 2 * n; t += T) bh[t] = 0.0;
    __syncthreads();
    const int* iact = V.iact + (long long)b * n;
    for (int k = tid; k < na; k += T) bh[iact[k] - 1] = V.mu[(long long)lb * nm + k];
    __syncthreads();
    // dx0 = sum_costs E c^ - Yeq' b^eq - Yin' b^in + Phi' dtraj
    if (V.dx0) {
        const double* Yeq = P.Yeq + (long long)b * meq * nx;
        const double* Yin = P.Yin + (long long)b * mineq * nx;
        const double* Phi = P.Phi + (long long)b * X * nx;
        const double* dt = V.dtraj ? V.dtraj + (long long)b * V.sdt : nullptr;
        for (int s = 0; s < nx; ++s) {
            double acc = 0.0;
            for (int ci = 0; ci < P.ncost; ++ci) {
                const double* E = P.cost[ci].E + (long long)b * P.cost[ci].sE;
                for (int col = tid; col < n; col += T) acc += E[s + (long long)col * nx] * ch[col];
            }
            for (int r = tid; r < meq; r += T) acc -= Yeq[r + (long long)s * meq] * bh[r];
            for (int r = tid; r < mineq; r += T) acc -= Yin[r + (long long)s * mineq] * bh[meq + r];
            if (dt)
                for (int r = tid; r < X; r += T) acc += Phi[r + (long long)s * X] * dt[r];
            acc = block_sum(acc, red);
            if (tid == 0) V.dx0[(long long)b * nx + s] = acc;
        }
    }
    // dp_i = -W T_i c^ with T_i[l, (j, bb)] = MGx[l, bb, i - j] (j <= i); a step-size p receives the sum over its steps
    for (int ci = 0; ci < P.ncost; ++ci) {
        double* out = V.dp[ci];
        if (!out) continue;
        const CostFam& F = P.cost[ci];
        const int r = F.rows, ns = F.i1 - F.i0;
        const double* MG = F.MGx + (long long)b * F.sMGx;
        const double* w = F.w.at(b);
        out += (long long)b * V.plen[ci];
        __syncthreads();
        for (int t = tid; t < r * ns; t += T) {
            const int l = t % r, i = F.i0 + t / r;
            double acc = 0.0;
            for (int j = 0; j <= min(i, N - 1); ++j)
                for (int bb = 0; bb < nu; ++bb) acc += MG[l + r * (bb + nu * (i - j))] * ch[j * nu + bb];
            const double v = -w[l] * acc;
            if (F.pstep) out[(long long)i * F.pstep + l] = v;
            else tmp[t] = v;
        }
        __syncthreads();
        if (!F.pstep)
            for (int l = tid; l < r; l += T) {
                double acc = 0.0;
                for (int ii = 0; ii < ns; ++ii) acc += tmp[ii * r + l];
                out[l] = acc;
            }
    }
    // df (or a trajectory bound's dlower / dupper): b^ through f[i fstep + (fidx ? fidx[l] : l)]
    for (int fi = 0; fi < P.nfam; ++fi) {
        double* out = V.df[fi];
        if (!out) continue;
        const CstrFam& F = P.fam[fi];
        const int r = F.rows, ns = F.i1 - F.i0;
        const double* bf = bh + (F.is_eq ? 0 : meq) + F.row_off;
        out += (long long)b * V.flen[fi];
        if (F.fstep) {
            for (int t = tid; t < r * ns; t += T) {
                const int l = t % r, i = F.i0 + t / r;
                out[(long long)i * F.fstep + (F.fidx ? F.fidx[l] : l)] = bf[t];
            }
        } else {
            for (int l = tid; l < r; l += T) {
                double acc = 0.0;
                for (int ii = 0; ii < ns; ++ii) acc += bf[ii * r + l];
                out[F.fidx ? F.fidx[l] : l] = acc;
            }
        }
    }
    // control bounds: lb[k] = lower[cb_full ? k : k % nu] (dev_finalize)
    for (int side = 0; side < 2; ++side) {
        double* out = side == 0 ? V.dlower : V.dupper;
        if (!out) continue;
        const double* g = bh + mg + (side == 0 ? n : 0);
        out += (long long)b * V.cblen;
        if (V.cblen == n)
            for (int k = tid; k < n; k += T) out[k] = g[k];
        else
            for (int e = tid; e < nu; e += T) {
                double acc = 0.0;
                for (int k = e; k < n; k += nu) acc += g[k];
                out[e] = acc;
            }
    }
}

int launched(cudaError_t e) { return e == cudaSuccess ? 1 : -int(e); }

} // namespace

int k8_gather_launch(const BuildParams& P, const VjpParams& V, int nb, cudaStream_t st)
{
    k8_gather_kernel<<<nb, kVjpThreads, 0, st>>>(P, V);
    return launched(cudaGetLastError());
}

int k8_gram_launch(const VjpParams& V, int nb, cudaStream_t st)
{
    k8_gram_kernel<<<nb, kVjpThreads, 0, st>>>(V);
    return launched(cudaGetLastError());
}

int k8_mu_launch(const VjpParams& V, int nb, cudaStream_t st)
{
    const size_t smem = sizeof(double) * 3 * size_t(std::max(V.nm, 1));
    cudaError_t e = cudaFuncSetAttribute(k8_mu_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return -int(e);
    k8_mu_kernel<<<nb, kVjpThreads, smem, st>>>(V);
    return launched(cudaGetLastError());
}

size_t k8_adjoint_smem(const BuildParams& P)
{
    int tmp = 1;
    for (int ci = 0; ci < P.ncost; ++ci) tmp = std::max(tmp, P.cost[ci].rows * (P.cost[ci].i1 - P.cost[ci].i0));
    return sizeof(double) * (size_t(P.nvar) * 3 + P.meq + P.mineq + tmp);
}

int k8_adjoint_launch(const BuildParams& P, const VjpParams& V, int nb, cudaStream_t st)
{
    const size_t smem = k8_adjoint_smem(P);
    cudaError_t e = cudaFuncSetAttribute(k8_adjoint_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return -int(e);
    k8_adjoint_kernel<<<nb, kVjpThreads, smem, st>>>(P, V);
    return launched(cudaGetLastError());
}

} // namespace cb
