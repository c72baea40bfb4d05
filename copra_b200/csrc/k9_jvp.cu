// k9_jvp.cu -- K9: Jacobian-vector products of a solved batch of LMPC problems (LMPC mode, decision vector U), and the
// local feedback gain dU/dx0 as the JVP along the columns of the identity on x0.
//
// On the final active set the solution is an affine function of every vector input, so the forward KKT system gives the
// exact tangent.  With the active rows written as equalities a_j' U = beta_j (K8's orientation), a tangent direction of the
// inputs gives cdot (the vector part of K2 / K4: sum_costs E' x0dot + fdot, fdot = -sum_i T_i' W pdot_i) and bdot_act (fdot
// at the row's (step, line) minus Y_row x0dot, or the bound's lbdot / ubdot), and
//   [Q A'; A 0] [Udot; lamdot] = [-cdot; bdot_act].
// With Q = R'R, Jt = R^-1, Y = Jt' [A_act' | -cdot] = [Y1 | T]:  G = Y1'Y1,  M = G^-1 (Y1' T - bdot_act),
// Udot = Jt (T - Y1 M),  xdot = Phi x0dot + Psi Udot.  k directions share the gather, the factor of G and every GEMM: the
// right-hand side has k columns where K8's has one.  The GEMMs (Y, G, Udot) run on the DMMA kernel of dgemm_dmma.cu and G
// is factored by gt_factor_kernel, as in K8; this file holds the four per-instance kernels around them:
//   k9_tangent  [A_act' | -cdot_1 .. -cdot_k] into a zero-padded n x (nmax+k) slab (the active rows through K8's gather
//               helper), and bdot_act (nmax x k)
//   k9_gram     G (nmax x nmax, 1 on the padded diagonal) and Y1' T - bdot_act out of the (nmax+k)^2 Gram matrix of Y
//   k9_solve    M = R_G^-1 R_G^-T (Y1' T - bdot_act) and W = T - Y1 M, k right-hand sides in tiles of kDirTile
//   k9_output   the caller's layout: the first ru rows of Udot, and the first rx rows of Phi x0dot + Toeplitz(Gs) Udot
// Every sum runs in a fixed order.  Instances whose status is not 0 get zeros; a Hessian or Gram factorisation that failed
// gives NaN tangents instead of silently wrong ones.
#include "active_rows.cuh"
#include "common.cuh"
#include "engine.cuh"
#include "launch.h"

#include <algorithm>

namespace cb {

namespace {

constexpr int kJvpThreads = 256;
constexpr int kDirTile = 8; // right-hand sides k9_solve keeps in registers per pass over J_G and Y

__device__ __forceinline__ int jvp_nact(const JvpParams& J, int b) { return J.status[b] == 0 ? J.nact[b] : 0; }

// entry s of the x0 tangent of direction d (the identity's column d for the gain)
__device__ __forceinline__ double x0_tangent(const JvpParams& J, int b, int nx, int d, int s)
{
    if (J.gain) return s == d ? 1.0 : 0.0;
    return J.tx0 ? J.tx0[((long long)b * J.k + d) * nx + s] : 0.0;
}

__global__ void __launch_bounds__(kJvpThreads) k9_tangent_kernel(const __grid_constant__ BuildParams P, const __grid_constant__ JvpParams J)
{
    const int lb = blockIdx.x, b = J.b0 + lb;
    const int n = J.n, nu = P.nu, nx = P.nx, mg = P.meq + P.mineq, nm = J.nm, k = J.k;
    double* slab = J.slab + (long long)lb * J.lds * (nm + k);
    const int na = jvp_nact(J, b);
    for (long long t = threadIdx.x; t < (long long)J.lds * (nm + k); t += blockDim.x) slab[t] = 0.0;
    __syncthreads();
    if (J.status[b] != 0) return;
    const int* iact = J.iact + (long long)b * n;
    for (int t = threadIdx.x; t < na * n; t += blockDim.x) {
        const int a = t / n, col = t % n;
        slab[col + (long long)a * J.lds] = active_row_entry(P, b, n, nu, mg, iact[a] - 1, col);
    }
    const bool has_x0 = J.gain || J.tx0;
    // -cdot_d: cdot[col] = sum_costs (sum_s E[s, col] x0dot[s] + fdot[col]),  fdot[(j, bb)] = -sum_{i >= j} sum_l
    // w[l] pdot_i[l] MGx[l, bb, i - j]  (the tangent of dev_ef's f through res_i = M xi_i - p_i)
    for (int t = threadIdx.x; t < n * k; t += blockDim.x) {
        const int col = t % n, d = t / n;
        const int j = col / nu, bb = col % nu;
        double c = 0.0;
        for (int ci = 0; ci < P.ncost; ++ci) {
            const CostFam& F = P.cost[ci];
            if (has_x0) {
                const double* E = F.E + (long long)b * F.sE + (long long)col * nx;
                for (int s = 0; s < nx; ++s) c += E[s] * x0_tangent(J, b, nx, d, s);
            }
            if (!J.tp[ci]) continue;
            const int r = F.rows;
            const double* pd = J.tp[ci] + ((long long)b * k + d) * J.plen[ci];
            const double* MG = F.MGx + (long long)b * F.sMGx;
            const double* w = F.w.at(b);
            double fd = 0.0;
            for (int i = max(F.i0, j); i < F.i1; ++i)
                for (int l = 0; l < r; ++l) fd += w[l] * pd[i * F.pstep + l] * MG[l + r * (bb + nu * (i - j))];
            c -= fd;
        }
        slab[col + (long long)(nm + d) * J.lds] = -c;
    }
    // bdot_act (nm x k): an Aeq / Aineq row's fdot at its (step, line) minus Y_row x0dot; a bound row's lbdot / ubdot
    for (int t = threadIdx.x; t < nm * k; t += blockDim.x) {
        const int a = t % nm, d = t / nm;
        double v = 0.0;
        if (a < na) {
            const int idx = iact[a] - 1;
            if (idx < mg) {
                const bool iseq = idx < P.meq;
                const int lrow = iseq ? idx : idx - P.meq, mtot = iseq ? P.meq : P.mineq;
                int i, l;
                const int fi = active_row_family(P, iseq, lrow, i, l);
                if (fi >= 0 && J.tf[fi]) {
                    const CstrFam& F = P.fam[fi];
                    v = J.tf[fi][((long long)b * k + d) * J.flen[fi] + i * F.fstep + (F.fidx ? F.fidx[l] : l)];
                }
                if (has_x0) {
                    const double* Yr = (iseq ? P.Yeq : P.Yin) + (long long)b * mtot * nx + lrow;
                    for (int s = 0; s < nx; ++s) v -= Yr[(long long)s * mtot] * x0_tangent(J, b, nx, d, s);
                }
            } else {
                const int var = (idx - mg) % n;
                const double* src = (idx - mg) < n ? J.tupper : J.tlower; // upper rows first, then lower rows
                if (src) v = src[((long long)b * k + d) * J.cblen + (J.cblen == n ? var : var % nu)];
            }
        }
        J.rhs[(long long)lb * nm * k + t] = v;
    }
}

// Gf: (nm+k) x (nm+k) Gram matrix of [Y1 | T] per instance -> Gq (nm x nm, padded diagonal 1) and rhs = Y1' T - bdot_act
__global__ void k9_gram_kernel(const __grid_constant__ JvpParams J)
{
    const int lb = blockIdx.x, b = J.b0 + lb, nm = J.nm, k = J.k, ld = nm + k;
    const int na = jvp_nact(J, b);
    const double* Gf = J.Gf + (long long)lb * ld * ld;
    double* Gq = J.Gq + (long long)lb * nm * nm;
    for (int t = threadIdx.x; t < nm * nm; t += blockDim.x) {
        const int i = t % nm, j = t / nm;
        Gq[t] = (i < na && j < na) ? Gf[i + (long long)j * ld] : (i == j ? 1.0 : 0.0);
    }
    double* rhs = J.rhs + (long long)lb * nm * k;
    for (int t = threadIdx.x; t < nm * k; t += blockDim.x) {
        const int i = t % nm, d = t / nm;
        rhs[t] = i < na ? Gf[i + (long long)(nm + d) * ld] - rhs[t] : 0.0;
    }
}

// M = J_G J_G' rhs (J_G = R_G^-1) and W = T - Y1 M for every direction, kDirTile directions per pass.  A Gram matrix that is
// not positive definite (linearly dependent active rows) or a Hessian factor that failed gives NaN, as in K8.
__global__ void __launch_bounds__(kJvpThreads) k9_solve_kernel(const __grid_constant__ JvpParams J)
{
    extern __shared__ double jvp_sm[];
    const int lb = blockIdx.x, b = J.b0 + lb, nm = J.nm, n = J.n, k = J.k;
    const int na = jvp_nact(J, b);
    double* rm = jvp_sm;           // nm x kDirTile: rhs, then M
    double* s = rm + nm * kDirTile; // nm x kDirTile
    const double* Y = J.Y + (long long)lb * J.ldy * (nm + k);
    const double* Jg = J.GJ + (long long)lb * J.ldg * nm;
    const bool ok = na == 0 || J.gpd[lb] != 0;
    const bool qok = J.qpd[(long long)b * J.qpd_stride] != 0;
    const bool live = J.status[b] == 0;
    double* W = J.W + (long long)lb * J.lds * k;
    for (int d0 = 0; d0 < k; d0 += kDirTile) {
        const int kt = min(kDirTile, k - d0);
        __syncthreads(); // the previous tile's M is no longer read
        if (na > 0) {
            for (int t = threadIdx.x; t < nm * kt; t += blockDim.x)
                rm[t] = J.rhs[(long long)lb * nm * k + (long long)d0 * nm + t];
            __syncthreads();
            for (int j = threadIdx.x; j < na; j += blockDim.x) {
                double acc[kDirTile];
#pragma unroll
                for (int dd = 0; dd < kDirTile; ++dd) acc[dd] = 0.0;
                for (int i = 0; i <= j; ++i) {
                    const double g = Jg[i + (long long)j * J.ldg];
#pragma unroll
                    for (int dd = 0; dd < kDirTile; ++dd)
                        if (dd < kt) acc[dd] += g * rm[i + dd * nm];
                }
#pragma unroll
                for (int dd = 0; dd < kDirTile; ++dd)
                    if (dd < kt) s[j + dd * nm] = acc[dd];
            }
            __syncthreads();
            for (int i = threadIdx.x; i < na; i += blockDim.x) {
                double acc[kDirTile];
#pragma unroll
                for (int dd = 0; dd < kDirTile; ++dd) acc[dd] = 0.0;
                for (int j = i; j < na; ++j) {
                    const double g = Jg[i + (long long)j * J.ldg];
#pragma unroll
                    for (int dd = 0; dd < kDirTile; ++dd)
                        if (dd < kt) acc[dd] += g * s[j + dd * nm];
                }
#pragma unroll
                for (int dd = 0; dd < kDirTile; ++dd)
                    if (dd < kt) rm[i + dd * nm] = (ok && qok) ? acc[dd] : CUDART_NAN;
            }
            __syncthreads();
        }
        for (int r = threadIdx.x; r < J.lds; r += blockDim.x) {
            double acc[kDirTile];
#pragma unroll
            for (int dd = 0; dd < kDirTile; ++dd) acc[dd] = 0.0;
            if (r < n && live) {
#pragma unroll
                for (int dd = 0; dd < kDirTile; ++dd)
                    if (dd < kt) acc[dd] = Y[r + (long long)(nm + d0 + dd) * J.ldy];
                for (int a = 0; a < na; ++a) {
                    const double y = Y[r + (long long)a * J.ldy];
#pragma unroll
                    for (int dd = 0; dd < kDirTile; ++dd)
                        if (dd < kt) acc[dd] -= y * rm[a + dd * nm];
                }
            }
#pragma unroll
            for (int dd = 0; dd < kDirTile; ++dd)
                if (dd < kt) W[r + (long long)(d0 + dd) * J.lds] = (r < n && live && !qok) ? CUDART_NAN : acc[dd];
        }
    }
}

// dcontrol = the first ru rows of Udot; dtraj = the first rx rows of Phi x0dot + Psi Udot, Psi applied as the block-Toeplitz
// product over the compact Gs (K7 without xi).  Zeros for an instance whose status is not 0.
__global__ void __launch_bounds__(kJvpThreads) k9_output_kernel(const __grid_constant__ BuildParams P, const __grid_constant__ JvpParams J)
{
    const int lb = blockIdx.x, b = J.b0 + lb, k = J.k;
    const int nx = P.nx, nu = P.nu, X = P.X, NX = P.N * P.nx;
    const bool live = J.status[b] == 0;
    const double* Ud = J.V + (long long)lb * J.lds * k;
    if (J.dcontrol) {
        double* out = J.dcontrol + (long long)b * J.ru * k;
        for (int t = threadIdx.x; t < J.ru * k; t += blockDim.x) {
            const int row = t % J.ru, d = t / J.ru;
            out[t] = live ? Ud[row + (long long)d * J.lds] : 0.0;
        }
    }
    if (!J.dtraj) return;
    double* out = J.dtraj + (long long)b * J.rx * k;
    const double* Phi = P.Phi + (long long)b * X * nx;
    const double* Gs = P.Gs + (long long)b * NX * nu;
    for (int t = threadIdx.x; t < J.rx * k; t += blockDim.x) {
        const int row = t % J.rx, d = t / J.rx;
        const int i = row / nx, r = row % nx;
        double v = 0.0;
        if (live) {
            const double* u = Ud + (long long)d * J.lds;
            double s1 = 0.0;
            for (int a = 0; a < nx; ++a) s1 += Phi[row + (long long)a * X] * x0_tangent(J, b, nx, d, a);
            double s2 = 0.0;
            int go = (i - 1) * nx + r; // G_{i-1-j}[r, :]
            for (int j = 0; j < i; ++j, go -= nx)
                for (int cc = 0; cc < nu; ++cc) s2 += Gs[go + (long long)cc * NX] * u[j * nu + cc];
            v = s1 + s2;
        }
        out[t] = v;
    }
}

int launched(cudaError_t e) { return e == cudaSuccess ? 1 : -int(e); }

} // namespace

int k9_tangent_launch(const BuildParams& P, const JvpParams& J, int nb, cudaStream_t st)
{
    k9_tangent_kernel<<<nb, kJvpThreads, 0, st>>>(P, J);
    return launched(cudaGetLastError());
}

int k9_gram_launch(const JvpParams& J, int nb, cudaStream_t st)
{
    k9_gram_kernel<<<nb, kJvpThreads, 0, st>>>(J);
    return launched(cudaGetLastError());
}

int k9_solve_launch(const JvpParams& J, int nb, cudaStream_t st)
{
    const size_t smem = sizeof(double) * 2 * kDirTile * size_t(std::max(J.nm, 1));
    cudaError_t e = cudaFuncSetAttribute(k9_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return -int(e);
    k9_solve_kernel<<<nb, kJvpThreads, smem, st>>>(J);
    return launched(cudaGetLastError());
}

int k9_output_launch(const BuildParams& P, const JvpParams& J, int nb, cudaStream_t st)
{
    k9_output_kernel<<<nb, kJvpThreads, 0, st>>>(P, J);
    return launched(cudaGetLastError());
}

} // namespace cb
