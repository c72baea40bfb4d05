// k8_k9_sens.cu -- K8 / K9: sensitivities of a solved batch of LMPC problems (LMPC mode, decision vector U): vector-Jacobian
// products (K8), Jacobian-vector products and the local feedback gain dU/dx0 (K9).
//
// On the final active set the solution is an affine function of every vector input, so one KKT solve per instance gives the
// exact sensitivity.  With the active rows written as equalities a_j' U = beta_j (an Aeq row, an Aineq row or e_k for either
// bound, in their natural orientation), Q = R'R and Jt = R^-1, both modes solve
//   [Q A'; A 0] [x; y] = [r; bdot_act]   for k right-hand sides:  Y = Jt' [A_act' | r] = [Y1 | T],  G = Y1'Y1,
//   M = G^-1 (Y1' T - bdot_act),  W = T - Y1 M,  x = Jt W.
// The VJP has k = 1, r = gbar = dL/dU (+ Psi' dL/dtrajectory) and bdot_act = 0: x = v, M = mu, and dL/dc = -v, dL/dbeta_j = mu_j
// (0 for the inactive rows).  The JVP has r = -cdot_d and bdot_act of each tangent direction d (the forward vector part of K2 /
// K4), and x = Udot.  The GEMMs (Y, G, x) run on the DMMA kernel of dgemm_dmma.cu and G is factored by gt_factor_kernel; this
// file holds the per-instance kernels around them:
//   k8_gather   [A_act' | gbar] into a zero-padded n x (nmax+1) slab, bdot_act = 0
//   k9_tangent  [A_act' | -cdot_1 .. -cdot_k] into a zero-padded n x (nmax+k) slab, and bdot_act (nmax x k)
//               (both through sens_gather: structured rows from the E A^k B tables with the indexing of K3's dev_fill_row,
//               so Aineq is never materialised, bound rows as unit vectors)
//   sens_gram   G (nmax x nmax, 1 on the padded diagonal) and Y1' T - bdot_act out of the (nmax+k)^2 Gram matrix of Y
//   sens_solve  M = R_G^-1 R_G^-T (Y1' T - bdot_act) and W = T - Y1 M, k right-hand sides in tiles of kDirTile (1 for k = 1)
//   k8_adjoint  the transpose of the vector part of K2 / K4 (what a retarget re-runs):
//               dx0 = sum_costs E c^ - Yeq' b^eq - Yin' b^in + Phi' dtraj,  dp_i = -W T_i c^,
//               df / dlower / dupper: b^, lb^, ub^ scattered through the index maps of dev_precompute / dev_finalize
//   k8_cost_grad the cost weights and matrices, which enter the objective only: dL/dtheta = c^' (dQ/dtheta U + dc/dtheta).
//               With x^ = Psi c^, the solution's states x_i and controls u_i, e_i = M x_i + N u_i - p_i and
//               t_i = T_i c^ = M x^_i + N c^_i:  dw_l = sum_i t_il e_il,  dM = sum_i W (e_i x^_i' + t_i x_i'),
//               dN = sum_i W (e_i c^_i' + t_i u_i')
//   k8_model_grad the dynamics A, B, d and the row constraints' E, G.  These also move the active rows, so the forward
//               multipliers lambda enter: the VJP then runs with k = 2, the second right-hand side being the forward solve
//               (-c in the slab, beta of the active rows in rhs), which leaves lambda in rhs column 1.  With gx_i = dtraj_i +
//               sum_costs M'W t_i - sum_rows mu_j E_l', gh_i = sum_costs M'W e_i + sum_rows lambda_j E_l' (rows j at step i,
//               line l), rho_N = gx_N, rho_i = gx_i + A' rho_{i+1} and rho^ the same from gh:
//               dA = sum_{i<N} rho_{i+1} x_i' + rho^_{i+1} x^_i',  dB = sum_{i<N} rho_{i+1} u_i' + rho^_{i+1} c^_i',
//               dd = sum_{i<N} rho_{i+1},  dE_l = sum_i lambda_(i,l) x^_i' - mu_(i,l) x_i',  dG_l = sum_i lambda_(i,l) c^_i' -
//               mu_(i,l) u_i'  (rho_0 is dx0)
//   qp_gather / qp_grad  the same VJP for a raw QP batch (copra_b200_qp_vjp): the active rows come from the caller's dense
//               Aeq / Aineq, and dc = -v, dQ = -(v x' + x v') / 2, dbeta_j = mu_j, da_j = -lambda_j v - mu_j x (k = 2 when the
//               Aeq / Aineq gradients are wanted, lambda again from the forward solve as second right-hand side)
//   qp_tangent / qp_output  the JVP of a raw QP batch (copra_b200_qp_jvp, copra_b200_qp_jacobian): r = -cdot_eff with
//               cdot_eff = cdot + sym(Qdot) x + sum_active lambda_j adot_j, bdot_act of a general row bdot_j - adot_j' x, of a
//               bound row lbdot / ubdot, and x = xdot (n x k per instance).  With Aeq / Aineq tangents lambda comes first, from
//               a k = 1 pass on the forward right-hand side (qp_lambda_gather: -c and beta; qp_lambda_store keeps rhs = lambda)
//   k9_output  the caller's layout: the first ru rows of Udot, and the first rx rows of Phi x0dot + Toeplitz(Gs) Udot
// Initial-state mode (copra_b200_lmpc_vjp_initial_state / _jvp_initial_state): the decision vector is z = [x0*; U] (n = nx + nU)
// with the per-instance Hessian of the build, and x0 enters only as the default of a bound that was not given.  The same
// kernels take the branch off = nx: a general row is [Y_row | EGx row] with b = z (no -Y x0 term), gbar = [Phi' dtraj;
// dcontrol + Psi' dtraj], c = [r; sum f], so dr = c^[0:nx], dR = (c^_0 x0*' + x0* c^_0') / 2 (the top-left block of
// -(v z' + z v') / 2), dp / df / the control bounds read c^[nx:] and the bound rows nx.., dx0lb / dx0ub are the multipliers of
// the bound rows 0..nx-1 and dx0 their sum over the bounds that defaulted.  Forward: cdot = [rdot + sym(Rdot) x0*; sum fdot],
// bdot of bound row k < nx is x0lbdot_k / x0ubdot_k (x0dot_k when that bound defaulted), dtraj = Phi zdot[0:nx] + Psi zdot[nx:].
// Every sum runs in a fixed order.  Instances whose status is not 0 get zeros; a Hessian or Gram factorisation that failed
// gives NaN instead of silently wrong results.
#include "common.cuh"
#include "engine.cuh"
#include "launch.h"

#include <algorithm>

namespace cb {

namespace {

constexpr int kSensThreads = 256;
constexpr int kDirTile = 8; // right-hand sides sens_solve keeps in registers per pass over J_G and Y (k > 1)

__device__ __forceinline__ int sens_nact(const SensChunk& S, int b) { return S.status[b] == 0 ? S.nact[b] : 0; }

// the family of general row `lrow` of Aeq (iseq) or Aineq, and its (step, line)
__device__ __forceinline__ int active_row_family(const BuildParams& P, bool iseq, int lrow, int& step, int& line)
{
    for (int k = 0; k < P.nfam; ++k) {
        const CstrFam& F = P.fam[k];
        if ((F.is_eq != 0) == iseq && lrow >= F.row_off && lrow < F.row_off + F.rows * (F.i1 - F.i0)) {
            step = F.i0 + (lrow - F.row_off) / F.rows;
            line = (lrow - F.row_off) % F.rows;
            return k;
        }
    }
    return -1;
}

// entry `col` of general row `idx` (0-based in the solver's [eq | ineq] index space, idx < P.meq + P.mineq) of instance b;
// nu = P.nu
__device__ __forceinline__ double general_row_entry(const BuildParams& P, int b, int nu, int idx, int col)
{
    double v = 0.0;
    const bool iseq = idx < P.meq;
    int i, l;
    const int fi = active_row_family(P, iseq, iseq ? idx : idx - P.meq, i, l);
    if (fi >= 0) {
        const CstrFam& F = P.fam[fi];
        const int j = col / nu, bb = col % nu, kk = i - j;
        if (kk >= 0) v = F.EGx[(long long)b * F.sEGx + l + F.rows * (bb + nu * kk)];
    }
    return v;
}

// entry col < nx of general row idx in initial-state mode: the row's Y = E Phi_i block, resident from the build (K3's
// dev_fill_row copies the same values into Aeq / Aineq)
__device__ __forceinline__ double initial_row_entry(const BuildParams& P, int b, int idx, int col)
{
    const bool iseq = idx < P.meq;
    const int mtot = iseq ? P.meq : P.mineq;
    const double* Y = (iseq ? P.Yeq : P.Yin) + (long long)b * mtot * P.nx;
    return Y[(iseq ? idx : idx - P.meq) + (long long)col * mtot];
}

// zero the lds x (nm + k) slab of chunk instance lb (batch instance b) and write its active rows as the first nact columns:
// row(idx, col) gives entry `col` of general row idx < mg, a bound row (upper rows first, then lower rows) is a unit vector.
// The caller writes the k right-hand-side columns
template <class Row> __device__ __forceinline__ double* sens_gather(const SensChunk& S, int lb, int b, int mg, Row row)
{
    const int n = S.n;
    double* slab = S.slab + (long long)lb * S.lds * (S.nm + S.k);
    const int na = sens_nact(S, b);
    for (long long t = threadIdx.x; t < (long long)S.lds * (S.nm + S.k); t += blockDim.x) slab[t] = 0.0;
    __syncthreads();
    const int* iact = S.iact + (long long)b * n;
    for (int t = threadIdx.x; t < na * n; t += blockDim.x) {
        const int a = t / n, col = t % n, idx = iact[a] - 1;
        slab[col + (long long)a * S.lds] = idx < mg ? row(idx, col) : ((idx - mg) % n == col ? 1.0 : 0.0);
    }
    return slab;
}

// rhs of a VJP (nm x k): a cotangent has bdot_act = 0; the forward solve's right-hand side (k = 2) is beta(idx) of the active
// rows, in their natural orientation
template <class Beta> __device__ __forceinline__ void vjp_rhs(const SensChunk& S, int lb, int b, Beta beta)
{
    const int na = sens_nact(S, b), nm = S.nm;
    const int* iact = S.iact + (long long)b * S.n;
    for (int t = threadIdx.x; t < nm * S.k; t += blockDim.x) {
        const int a = t % nm;
        S.rhs[(long long)lb * nm * S.k + t] = (t >= nm && a < na) ? beta(iact[a] - 1) : 0.0;
    }
}

// beta of row idx in the solver's index space: beq | bineq | ub | lb (per-instance pointers)
__device__ __forceinline__ double active_beta(int idx, int meq, int mg, int n, const double* beq, const double* bineq,
    const double* ub, const double* lb)
{
    return idx < meq ? beq[idx] : idx < mg ? bineq[idx - meq] : idx < mg + n ? ub[idx - mg] : lb[idx - mg - n];
}

__global__ void __launch_bounds__(kSensThreads) k8_gather_kernel(const __grid_constant__ BuildParams P, const __grid_constant__ VjpParams V)
{
    const int lb = blockIdx.x, b = V.b0 + lb;
    const int n = V.n, nu = P.nu, N = P.N, nx = P.nx, nm = V.nm, mg = P.meq + P.mineq, X = P.X;
    const int off = P.initial_state ? nx : 0;
    const long long NX = (long long)N * nx;
    double* slab = sens_gather(V, lb, b, mg, [&](int idx, int col) {
        return col < off ? initial_row_entry(P, b, idx, col) : general_row_entry(P, b, nu, idx, col - off);
    });
    vjp_rhs(V, lb, b, [&](int idx) {
        return active_beta(idx, P.meq, mg, n, P.beq + (long long)b * P.meq, P.bineq + (long long)b * P.mineq,
            P.ub + (long long)b * P.nvar, P.lb + (long long)b * P.nvar);
    });
    if (V.status[b] != 0) return;
    if (V.k == 2)
        for (int col = threadIdx.x; col < n; col += blockDim.x) slab[col + (long long)(nm + 1) * V.lds] = -P.c[(long long)b * P.nvar + col];
    // gbar = dcontrol + Psi' dtraj, Psi' applied as the transposed block-Toeplitz product over the compact Gs; in initial-state
    // mode the first nx entries are Phi' dtraj (x0* enters the trajectory through Phi)
    const double* Gs = P.Gs + (long long)b * NX * nu;
    for (int col = threadIdx.x; col < n; col += blockDim.x) {
        if (col < off) {
            double g = 0.0;
            if (V.dtraj) {
                const double* Phi = P.Phi + (long long)b * X * nx + (long long)col * X;
                const double* dt = V.dtraj + (long long)b * V.sdt;
                for (int r = 0; r < X; ++r) g += Phi[r] * dt[r];
            }
            slab[col + (long long)nm * V.lds] = g;
            continue;
        }
        const int cu = col - off;
        double g = V.dcontrol ? V.dcontrol[(long long)b * V.sdc + cu] : 0.0;
        if (V.dtraj) {
            const int j = cu / nu, bb = cu % nu;
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

// entry s of the x0 tangent of direction d (the identity's column d for the gain)
__device__ __forceinline__ double x0_tangent(const JvpParams& J, int b, int nx, int d, int s)
{
    if (J.gain) return s == d ? 1.0 : 0.0;
    return J.tx0 ? J.tx0[((long long)b * J.k + d) * nx + s] : 0.0;
}

__global__ void __launch_bounds__(kSensThreads) k9_tangent_kernel(const __grid_constant__ BuildParams P, const __grid_constant__ JvpParams J)
{
    const int lb = blockIdx.x, b = J.b0 + lb;
    const int n = J.n, nu = P.nu, nx = P.nx, nU = P.nU, mg = P.meq + P.mineq, nm = J.nm, k = J.k;
    const int off = P.initial_state ? nx : 0;
    double* slab = sens_gather(J, lb, b, mg, [&](int idx, int col) {
        return col < off ? initial_row_entry(P, b, idx, col) : general_row_entry(P, b, nu, idx, col - off);
    });
    if (J.status[b] != 0) return;
    const int na = J.nact[b];
    const int* iact = J.iact + (long long)b * n;
    const bool has_x0 = !off && (J.gain || J.tx0); // initial-state mode: x0 moves only the bounds that defaulted to it
    // -cdot_d: cdot[col] = sum_costs (sum_s E[s, col] x0dot[s] + fdot[col]),  fdot[(j, bb)] = -sum_{i >= j} sum_l
    // w[l] pdot_i[l] MGx[l, bb, i - j]  (the tangent of dev_ef's f through res_i = M xi_i - p_i); in initial-state mode
    // cdot[s < nx] = rdot[s] + sum_a (Rdot[s, a] + Rdot[a, s]) / 2 x0*[a]
    for (int t = threadIdx.x; t < n * k; t += blockDim.x) {
        const int cl = t % n, d = t / n;
        if (cl < off) {
            double c = J.tr ? J.tr[((long long)b * k + d) * nx + cl] : 0.0;
            if (J.tR) {
                const double* Rd = J.tR + ((long long)b * k + d) * nx * nx;
                const double* xs = J.x + (long long)b * n;
                double s = 0.0;
                for (int a = 0; a < nx; ++a) s += 0.5 * (Rd[cl + a * nx] + Rd[a + cl * nx]) * xs[a];
                c += s;
            }
            slab[cl + (long long)(nm + d) * J.lds] = -c;
            continue;
        }
        const int col = cl - off;
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
        slab[cl + (long long)(nm + d) * J.lds] = -c;
    }
    // bdot_act (nm x k): an Aeq / Aineq row's fdot at its (step, line) minus Y_row x0dot (LMPC mode); a bound row's lbdot /
    // ubdot, in initial-state mode x0lbdot / x0ubdot for the rows k < nx (x0dot where that bound defaulted to x0)
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
                const bool up = (idx - mg) < n; // upper rows first, then lower rows
                if (var < off) {
                    const double* src = up ? (P.x0ub.p ? J.tx0ub : J.tx0) : (P.x0lb.p ? J.tx0lb : J.tx0);
                    if (src) v = src[((long long)b * k + d) * nx + var];
                } else {
                    const int vu = var - off;
                    const double* src = up ? J.tupper : J.tlower;
                    if (src) v = src[((long long)b * k + d) * J.cblen + (J.cblen == nU ? vu : vu % nu)];
                }
            }
        }
        J.rhs[(long long)lb * nm * k + t] = v;
    }
}

// Gf: (nm+k) x (nm+k) Gram matrix of [Y1 | T] per instance -> Gq (nm x nm, padded diagonal 1) and rhs = Y1' T - bdot_act
__global__ void sens_gram_kernel(const __grid_constant__ SensChunk S)
{
    const int lb = blockIdx.x, b = S.b0 + lb, nm = S.nm, k = S.k, ld = nm + k;
    const int na = sens_nact(S, b);
    const double* Gf = S.Gf + (long long)lb * ld * ld;
    double* Gq = S.Gq + (long long)lb * nm * nm;
    for (int t = threadIdx.x; t < nm * nm; t += blockDim.x) {
        const int i = t % nm, j = t / nm;
        Gq[t] = (i < na && j < na) ? Gf[i + (long long)j * ld] : (i == j ? 1.0 : 0.0);
    }
    double* rhs = S.rhs + (long long)lb * nm * k;
    for (int t = threadIdx.x; t < nm * k; t += blockDim.x) {
        const int i = t % nm, d = t / nm;
        rhs[t] = i < na ? Gf[i + (long long)(nm + d) * ld] - rhs[t] : 0.0;
    }
}

// M = J_G J_G' rhs (J_G = R_G^-1) and W = T - Y1 M for every right-hand side, TILE per pass: k when k <= 2, so one or two
// right-hand sides do not pay for kDirTile predicated lanes, else kDirTile.  Each column's arithmetic is the same for every
// TILE.  With TILE <= 2 (the VJP) M goes back to rhs.  A Gram matrix that is not positive definite
// (linearly dependent active rows) or a Hessian factor that failed gives NaN rather than silently wrong results.
template <int TILE> __global__ void __launch_bounds__(kSensThreads) sens_solve_kernel(const __grid_constant__ SensChunk S)
{
    extern __shared__ double sens_sm[];
    const int lb = blockIdx.x, b = S.b0 + lb, nm = S.nm, n = S.n, k = S.k;
    const int na = sens_nact(S, b);
    double* rm = sens_sm;               // nm x min(k, TILE): rhs, then M
    double* s = rm + nm * min(k, TILE); // nm x min(k, TILE)
    const double* Y = S.Y + (long long)lb * S.ldy * (nm + k);
    const double* Jg = S.GJ + (long long)lb * S.ldg * nm;
    const bool ok = na == 0 || S.gpd[lb] != 0;
    const bool qok = S.qpd[(long long)b * S.qpd_stride] != 0;
    const bool live = S.status[b] == 0;
    double* rhs = S.rhs + (long long)lb * nm * k;
    double* W = S.W + (long long)lb * S.lds * k;
    for (int d0 = 0; d0 < k; d0 += TILE) {
        const int kt = min(TILE, k - d0);
        __syncthreads(); // the previous tile's M is no longer read
        if (na > 0) {
            for (int t = threadIdx.x; t < nm * kt; t += blockDim.x) rm[t] = rhs[(long long)d0 * nm + t];
            __syncthreads();
            for (int j = threadIdx.x; j < na; j += blockDim.x) {
                double acc[TILE];
#pragma unroll
                for (int dd = 0; dd < TILE; ++dd) acc[dd] = 0.0;
                for (int i = 0; i <= j; ++i) {
                    const double g = Jg[i + (long long)j * S.ldg];
#pragma unroll
                    for (int dd = 0; dd < TILE; ++dd)
                        if (dd < kt) acc[dd] += g * rm[i + dd * nm];
                }
#pragma unroll
                for (int dd = 0; dd < TILE; ++dd)
                    if (dd < kt) s[j + dd * nm] = acc[dd];
            }
            __syncthreads();
            for (int i = threadIdx.x; i < na; i += blockDim.x) {
                double acc[TILE];
#pragma unroll
                for (int dd = 0; dd < TILE; ++dd) acc[dd] = 0.0;
                for (int j = i; j < na; ++j) {
                    const double g = Jg[i + (long long)j * S.ldg];
#pragma unroll
                    for (int dd = 0; dd < TILE; ++dd)
                        if (dd < kt) acc[dd] += g * s[j + dd * nm];
                }
#pragma unroll
                for (int dd = 0; dd < TILE; ++dd)
                    if (dd < kt) {
                        const double m = (ok && qok) ? acc[dd] : CUDART_NAN;
                        rm[i + dd * nm] = m;
                        // the VJP's multipliers mu (and, k = 2, the forward lambda), for k8_adjoint / k8_model_grad;
                        // TILE <= 2 is launched with k = TILE, so d0 = 0
                        if (TILE <= 2) rhs[i + dd * nm] = m;
                    }
            }
            __syncthreads();
        }
        for (int r = threadIdx.x; r < S.lds; r += blockDim.x) {
            double acc[TILE];
#pragma unroll
            for (int dd = 0; dd < TILE; ++dd) acc[dd] = 0.0;
            if (r < n && live) {
#pragma unroll
                for (int dd = 0; dd < TILE; ++dd)
                    if (dd < kt) acc[dd] = Y[r + (long long)(nm + d0 + dd) * S.ldy];
                for (int a = 0; a < na; ++a) {
                    const double y = Y[r + (long long)a * S.ldy];
#pragma unroll
                    for (int dd = 0; dd < TILE; ++dd)
                        if (dd < kt) acc[dd] -= y * rm[a + dd * nm];
                }
            }
#pragma unroll
            for (int dd = 0; dd < TILE; ++dd)
                if (dd < kt) W[r + (long long)(d0 + dd) * S.lds] = (r < n && live && !qok) ? CUDART_NAN : acc[dd];
        }
    }
}

__global__ void __launch_bounds__(kSensThreads) k8_adjoint_kernel(const __grid_constant__ BuildParams P, const __grid_constant__ VjpParams V)
{
    extern __shared__ double sens_sm[];
    __shared__ double red[2 * kMaxWarps];
    const int lb = blockIdx.x, b = V.b0 + lb;
    if (V.status[b] != 0) return; // gradients stay at the zeros they were initialised to
    const int n = V.n, nx = P.nx, nu = P.nu, N = P.N, X = P.X, meq = P.meq, mineq = P.mineq, mg = meq + mineq, nm = V.nm;
    const int nU = P.nU, off = P.initial_state ? nx : 0;
    const int na = V.nact[b];
    const int tid = threadIdx.x, T = blockDim.x;
    double* ch = sens_sm;          // n    c^ = -v
    double* bh = ch + n;           // mg + 2n: b^eq | b^in | ub^ | lb^  (the solver's constraint index space)
    double* tmp = bh + mg + 2 * n; // per-step partials of one cost
    for (int t = tid; t < n; t += T) ch[t] = -V.V[(long long)lb * V.lds * V.k + t];
    for (int t = tid; t < mg + 2 * n; t += T) bh[t] = 0.0;
    __syncthreads();
    const int* iact = V.iact + (long long)b * n;
    for (int k = tid; k < na; k += T) bh[iact[k] - 1] = V.rhs[(long long)lb * nm * V.k + k]; // mu, from sens_solve
    __syncthreads();
    if (off) {
        // initial-state mode: c[0:nx] = r, Q_tl = R + E Qb^-1 E', the bound rows 0..nx-1 are [x0lb, x0ub] (x0 where not given)
        const double* ubh = bh + mg;
        const double* lbh = bh + mg + n;
        const double* xs = V.U + (long long)b * n; // x0* = the solution's first nx entries
        for (int s = tid; s < nx; s += T) {
            if (V.dr) V.dr[(long long)b * nx + s] = ch[s];
            if (V.dx0lb) V.dx0lb[(long long)b * nx + s] = lbh[s];
            if (V.dx0ub) V.dx0ub[(long long)b * nx + s] = ubh[s];
            if (V.dx0) V.dx0[(long long)b * nx + s] = (P.x0lb.p ? 0.0 : lbh[s]) + (P.x0ub.p ? 0.0 : ubh[s]);
        }
        if (V.dR)
            for (int q = tid; q < nx * nx; q += T) {
                const int s = q % nx, u = q / nx;
                // no contraction, so that dR is exactly symmetric
                V.dR[(long long)b * nx * nx + q] = 0.5 * __dadd_rn(__dmul_rn(ch[s], xs[u]), __dmul_rn(xs[s], ch[u]));
            }
    }
    // dx0 = sum_costs E c^ - Yeq' b^eq - Yin' b^in + Phi' dtraj (LMPC mode)
    if (V.dx0 && !off) {
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
    const double* cu = ch + off; // c^ of U
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
                for (int bb = 0; bb < nu; ++bb) acc += MG[l + r * (bb + nu * (i - j))] * cu[j * nu + bb];
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
    // control bounds: lb[off + k] = lower[cb_full ? k : k % nu] (dev_finalize)
    for (int side = 0; side < 2; ++side) {
        double* out = side == 0 ? V.dlower : V.dupper;
        if (!out) continue;
        const double* g = bh + mg + (side == 0 ? n : 0) + off;
        out += (long long)b * V.cblen;
        if (V.cblen == nU)
            for (int k = tid; k < nU; k += T) out[k] = g[k];
        else
            for (int e = tid; e < nu; e += T) {
                double acc = 0.0;
                for (int k = e; k < nU; k += nu) acc += g[k];
                out[e] = acc;
            }
    }
}

// dw, dM and dN of every requested cost (see the file comment), one CTA per instance of the chunk.  Shared memory: c^ and U
// (n each), x^ = Psi c^ and xd = Phi x0 + Psi U (X each; x_i = xd_i + xi_i), then e and t of one cost (rows x steps each).
// e_i = res_i + M xd_i + N u_i with the resident res_i = M xi_i - p_i.  Every sum runs in a fixed order; an instance whose
// status is not 0 keeps the zeros its outputs were initialised to, a failed factorisation reaches the outputs as NaN through v.
__global__ void __launch_bounds__(kSensThreads) k8_cost_grad_kernel(const __grid_constant__ BuildParams P, const __grid_constant__ VjpParams V)
{
    extern __shared__ double sens_sm[];
    const int lb = blockIdx.x, b = V.b0 + lb;
    if (V.status[b] != 0) return;
    const int n = V.n, nx = P.nx, nu = P.nu, N = P.N, X = P.X, NX = N * nx;
    const int tid = threadIdx.x, T = blockDim.x;
    double* ch = sens_sm;  // n  c^ = -v
    double* u = ch + n;    // n  U
    double* xh = u + n;    // X  Psi c^
    double* xd = xh + X;   // X  Phi x0 + Psi U
    double* et = xd + X;   // 2 x rows x steps: e, then t, of one cost
    for (int t = tid; t < n; t += T) {
        ch[t] = -V.V[(long long)lb * V.lds * V.k + t];
        u[t] = V.U[(long long)b * n + t];
    }
    __syncthreads();
    const double* Phi = P.Phi + (long long)b * X * nx;
    const double* Gs = P.Gs + (long long)b * NX * nu;
    const double* xi = P.xi + (long long)b * X;
    const double* x0 = P.x0.at(b);
    for (int row = tid; row < X; row += T) {
        const int i = row / nx, r = row % nx;
        double sh = 0.0, su = 0.0;
        int go = (i - 1) * nx + r; // G_{i-1-j}[r, :]
        for (int j = 0; j < i; ++j, go -= nx)
            for (int cc = 0; cc < nu; ++cc) {
                const double g = Gs[go + (long long)cc * NX];
                sh += g * ch[j * nu + cc];
                su += g * u[j * nu + cc];
            }
        double s0 = 0.0;
        for (int a = 0; a < nx; ++a) s0 += Phi[row + (long long)a * X] * x0[a];
        xh[row] = sh;
        xd[row] = s0 + su;
    }
    for (int ci = 0; ci < P.ncost; ++ci) {
        double *ow = V.dw[ci], *oM = V.dM[ci], *oN = V.dN[ci];
        if (!ow && !oM && !oN) continue;
        const CostFam& F = P.cost[ci];
        const int r = F.rows, ns = F.i1 - F.i0, len = r * ns;
        const double* M = F.hasM ? F.M.at(b) : nullptr; // r x nx
        const double* Nm = F.hasN ? F.N.at(b) : nullptr; // r x nu
        const double* w = F.w.at(b);
        const double* res = F.res + (long long)b * F.sres;
        __syncthreads(); // xh / xd complete; the previous cost's e / t are no longer read
        for (int t = tid; t < len; t += T) {
            const int l = t % r, i = F.i0 + t / r;
            double e = res[t], tt = 0.0;
            if (M)
                for (int a = 0; a < nx; ++a) {
                    const double m = M[l + r * a];
                    e += m * xd[i * nx + a];
                    tt += m * xh[i * nx + a];
                }
            if (Nm && i < N)
                for (int bb = 0; bb < nu; ++bb) {
                    const double m = Nm[l + r * bb];
                    e += m * u[i * nu + bb];
                    tt += m * ch[i * nu + bb];
                }
            et[t] = e;
            et[len + t] = tt;
        }
        __syncthreads();
        const double* e = et;
        const double* tv = et + len;
        if (ow)
            for (int l = tid; l < r; l += T) {
                double acc = 0.0;
                for (int s = 0; s < ns; ++s) acc += tv[s * r + l] * e[s * r + l];
                ow[(long long)b * r + l] = acc;
            }
        if (oM)
            for (int q = tid; q < r * nx; q += T) {
                const int l = q % r, a = q / r;
                double acc = 0.0;
                for (int s = 0; s < ns; ++s) {
                    const int k = (F.i0 + s) * nx + a;
                    acc += e[s * r + l] * xh[k] + tv[s * r + l] * (xd[k] + xi[k]);
                }
                oM[(long long)b * r * nx + q] = w[l] * acc;
            }
        if (oN)
            for (int q = tid; q < r * nu; q += T) {
                const int l = q % r, bb = q / r;
                double acc = 0.0;
                for (int s = 0; s < ns && F.i0 + s < N; ++s) {
                    const int k = (F.i0 + s) * nu + bb;
                    acc += e[s * r + l] * ch[k] + tv[s * r + l] * u[k];
                }
                oN[(long long)b * r * nu + q] = w[l] * acc;
            }
    }
}

// dA, dB, dd and the dE / dG of every requested row constraint (see the file comment), one CTA per instance of the chunk.
// Shared memory: c^ and U (n each); x^ = Psi c^ and x = Phi x0 + Psi U + xi (X each); gx, then rho, and gh, then rho^ (X
// each); mu and lambda spread over the general rows [eq | ineq] (mg each: the bound rows do not depend on the model).  A is
// Phi's block 1 and B is Gs's block 0.  Every sum runs in a fixed order; an instance whose status is not 0 keeps the zeros its
// outputs were initialised to, a failed factorisation reaches the outputs as NaN through v, mu and lambda.
__global__ void __launch_bounds__(kSensThreads) k8_model_grad_kernel(const __grid_constant__ BuildParams P, const __grid_constant__ VjpParams V)
{
    extern __shared__ double sens_sm[];
    const int lb = blockIdx.x, b = V.b0 + lb;
    if (V.status[b] != 0) return;
    const int n = V.n, nx = P.nx, nu = P.nu, N = P.N, X = P.X, NX = N * nx, meq = P.meq, mg = meq + P.mineq, nm = V.nm;
    const int na = V.nact[b];
    const int tid = threadIdx.x, T = blockDim.x;
    double* ch = sens_sm;    // n   c^ = -v
    double* u = ch + n;      // n   U
    double* xh = u + n;      // X   Psi c^
    double* x = xh + X;      // X   Phi x0 + Psi U + xi
    double* rho = x + X;     // X   gx, then rho
    double* rhoh = rho + X;  // X   gh, then rho^
    double* mu = rhoh + X;   // mg  the adjoint's multipliers
    double* lam = mu + mg;   // mg  the forward solve's multipliers
    const double* v = V.V + (long long)lb * V.lds * V.k;
    for (int t = tid; t < n; t += T) {
        ch[t] = -v[t];
        u[t] = V.U[(long long)b * n + t];
    }
    for (int t = tid; t < mg; t += T) mu[t] = lam[t] = 0.0;
    __syncthreads();
    const int* iact = V.iact + (long long)b * n;
    const double* rhs = V.rhs + (long long)lb * nm * V.k;
    for (int a = tid; a < na; a += T) {
        const int idx = iact[a] - 1;
        if (idx < mg) {
            mu[idx] = rhs[a];
            lam[idx] = rhs[nm + a];
        }
    }
    const double* Phi = P.Phi + (long long)b * X * nx;
    const double* Gs = P.Gs + (long long)b * NX * nu;
    const double* xi = P.xi + (long long)b * X;
    const double* x0 = P.x0.at(b);
    for (int row = tid; row < X; row += T) {
        const int i = row / nx, r = row % nx;
        double sh = 0.0, su = 0.0;
        int go = (i - 1) * nx + r; // G_{i-1-j}[r, :]
        for (int j = 0; j < i; ++j, go -= nx)
            for (int cc = 0; cc < nu; ++cc) {
                const double g = Gs[go + (long long)cc * NX];
                sh += g * ch[j * nu + cc];
                su += g * u[j * nu + cc];
            }
        double s0 = 0.0;
        for (int a = 0; a < nx; ++a) s0 += Phi[row + (long long)a * X] * x0[a];
        xh[row] = sh;
        x[row] = s0 + su + xi[row];
    }
    __syncthreads();
    // gx_i = dtraj_i + sum_costs M'W t_i - sum_rows mu E_l',  gh_i = sum_costs M'W e_i + sum_rows lambda E_l'
    const double* dt = V.dtraj ? V.dtraj + (long long)b * V.sdt : nullptr;
    for (int row = tid; row < X; row += T) {
        const int i = row / nx, r = row % nx;
        double gx = dt ? dt[row] : 0.0, gh = 0.0;
        for (int ci = 0; ci < P.ncost; ++ci) {
            const CostFam& F = P.cost[ci];
            if (!F.hasM || i < F.i0 || i >= F.i1) continue;
            const int rr = F.rows;
            const double* M = F.M.at(b);
            const double* Nm = F.hasN && i < N ? F.N.at(b) : nullptr;
            const double* w = F.w.at(b);
            const double* res = F.res + (long long)b * F.sres + (long long)(i - F.i0) * rr; // M xi_i - p_i
            for (int l = 0; l < rr; ++l) {
                double e = res[l], tt = 0.0;
                for (int a = 0; a < nx; ++a) {
                    const double m = M[l + rr * a];
                    e += m * (x[i * nx + a] - xi[i * nx + a]);
                    tt += m * xh[i * nx + a];
                }
                if (Nm)
                    for (int bb = 0; bb < nu; ++bb) {
                        const double m = Nm[l + rr * bb];
                        e += m * u[i * nu + bb];
                        tt += m * ch[i * nu + bb];
                    }
                const double mw = M[l + rr * r] * w[l];
                gx += mw * tt;
                gh += mw * e;
            }
        }
        for (int fi = 0; fi < P.nfam; ++fi) {
            const CstrFam& F = P.fam[fi];
            if (!F.hasE || i < F.i0 || i >= F.i1) continue;
            const double* E = F.E.at(b); // a trajectory bound's selector: quirk Q1 keeps its lower rows as x <= lower
            const int j0 = (F.is_eq ? 0 : meq) + F.row_off + (i - F.i0) * F.rows;
            for (int l = 0; l < F.rows; ++l) {
                const double ev = E[l + F.rows * r];
                gx -= ev * mu[j0 + l];
                gh += ev * lam[j0 + l];
            }
        }
        rho[row] = gx;
        rhoh[row] = gh;
    }
    // rho_N = gx_N, rho_i = gx_i + A' rho_{i+1} (and rho^ from gh) down to rho_1: the outputs need no rho_0 (= dx0)
    for (int i = N - 1; i >= 1; --i) {
        __syncthreads();
        for (int r = tid; r < nx; r += T) {
            double s = 0.0, sh = 0.0;
            for (int a = 0; a < nx; ++a) {
                const double A = Phi[nx + a + (long long)r * X]; // A[a, r]
                s += A * rho[(i + 1) * nx + a];
                sh += A * rhoh[(i + 1) * nx + a];
            }
            rho[i * nx + r] += s;
            rhoh[i * nx + r] += sh;
        }
    }
    __syncthreads();
    if (V.dA)
        for (int q = tid; q < nx * nx; q += T) {
            const int r = q % nx, a = q / nx;
            double acc = 0.0;
            for (int i = 0; i < N; ++i) acc += rho[(i + 1) * nx + r] * x[i * nx + a] + rhoh[(i + 1) * nx + r] * xh[i * nx + a];
            V.dA[(long long)b * nx * nx + q] = acc;
        }
    if (V.dB)
        for (int q = tid; q < nx * nu; q += T) {
            const int r = q % nx, cc = q / nx;
            double acc = 0.0;
            for (int i = 0; i < N; ++i) acc += rho[(i + 1) * nx + r] * u[i * nu + cc] + rhoh[(i + 1) * nx + r] * ch[i * nu + cc];
            V.dB[(long long)b * nx * nu + q] = acc;
        }
    if (V.dd)
        for (int r = tid; r < nx; r += T) {
            double acc = 0.0;
            for (int i = 0; i < N; ++i) acc += rho[(i + 1) * nx + r];
            V.dd[(long long)b * nx + r] = acc;
        }
    // dE_l = sum_i lambda_(i,l) x^_i' - mu_(i,l) x_i',  dG_l = sum_i lambda_(i,l) c^_i' - mu_(i,l) u_i'
    for (int fi = 0; fi < P.nfam; ++fi) {
        const CstrFam& F = P.fam[fi];
        const int rr = F.rows, j0 = (F.is_eq ? 0 : meq) + F.row_off;
        if (V.dE[fi])
            for (int q = tid; q < rr * nx; q += T) {
                const int l = q % rr, a = q / rr;
                double acc = 0.0;
                for (int i = F.i0; i < F.i1; ++i) {
                    const int j = j0 + (i - F.i0) * rr + l;
                    acc += lam[j] * xh[i * nx + a] - mu[j] * x[i * nx + a];
                }
                V.dE[fi][(long long)b * rr * nx + q] = acc;
            }
        if (V.dG[fi])
            for (int q = tid; q < rr * nu; q += T) {
                const int l = q % rr, cc = q / rr;
                double acc = 0.0;
                for (int i = F.i0; i < F.i1 && i < N; ++i) {
                    const int j = j0 + (i - F.i0) * rr + l;
                    acc += lam[j] * ch[i * nu + cc] - mu[j] * u[i * nu + cc];
                }
                V.dG[fi][(long long)b * rr * nu + q] = acc;
            }
    }
}

// The raw QP (copra_b200_qp_vjp): [A_act' | dx] into the zero-padded slab, A_act read from the caller's column-major Aeq /
// Aineq through iact; with row-matrix gradients (k = 2) also -c in slab column nm + 1 and beta of the active rows in rhs
// column 1, as k8_gather
__global__ void __launch_bounds__(kSensThreads) qp_gather_kernel(const __grid_constant__ QpVjpParams V)
{
    const int lb = blockIdx.x, b = V.b0 + lb;
    const int n = V.n, meq = V.meq, m = V.m, mg = meq + m, nm = V.nm;
    const double* Aeq = V.Aeq.at(b);
    const double* Aineq = V.Aineq.at(b);
    double* slab = sens_gather(V, lb, b, mg, [&](int idx, int col) {
        return idx < meq ? Aeq[idx + (long long)meq * col] : Aineq[idx - meq + (long long)m * col];
    });
    vjp_rhs(V, lb, b, [&](int idx) { return active_beta(idx, meq, mg, n, V.beq.at(b), V.bineq.at(b), V.ub.at(b), V.lb.at(b)); });
    if (V.status[b] != 0) return;
    const double* c = V.c.at(b);
    const double* dx = V.dx + (long long)b * n;
    for (int col = threadIdx.x; col < n; col += blockDim.x) {
        slab[col + (long long)nm * V.lds] = dx[col];
        if (V.k == 2) slab[col + (long long)(nm + 1) * V.lds] = -c[col];
    }
}

// The raw QP's gradients from v (S.V), mu (rhs column 0), lambda (rhs column 1, k = 2) and the solution x, one CTA per
// instance: dc = -v, dQ = -(v x' + x v') / 2, dbeta_j = mu_j at active row j's index (beq | bineq | ub | lb), and the row of
// dAeq / dAineq of an active general row j = -lambda_j v - mu_j x.  Shared memory: v and x (n each).  An instance whose status
// is not 0 keeps the zeros its outputs were initialised to; a failed factorisation reaches the outputs as NaN through v, mu
// and lambda.
__global__ void __launch_bounds__(kSensThreads) qp_grad_kernel(const __grid_constant__ QpVjpParams V)
{
    extern __shared__ double sens_sm[];
    const int lb = blockIdx.x, b = V.b0 + lb;
    if (V.status[b] != 0) return;
    const int n = V.n, meq = V.meq, m = V.m, mg = meq + m, nm = V.nm, na = V.nact[b];
    const int tid = threadIdx.x, T = blockDim.x;
    double* v = sens_sm; // n
    double* x = v + n;   // n
    const double* Vb = V.V + (long long)lb * V.lds * V.k;
    for (int t = tid; t < n; t += T) {
        v[t] = Vb[t];
        x[t] = V.x[(long long)b * n + t];
    }
    __syncthreads();
    if (V.dc)
        for (int t = tid; t < n; t += T) V.dc[(long long)b * n + t] = -v[t];
    if (V.dQ)
        for (int q = tid; q < n * n; q += T) {
            const int i = q % n, j = q / n;
            // no contraction, so that dQ is exactly symmetric
            V.dQ[(long long)b * n * n + q] = -0.5 * __dadd_rn(__dmul_rn(v[i], x[j]), __dmul_rn(x[i], v[j]));
        }
    const int* iact = V.iact + (long long)b * n;
    const double* rhs = V.rhs + (long long)lb * nm * V.k;
    for (int a = tid; a < na; a += T) {
        const int idx = iact[a] - 1;
        double* out = idx < meq ? (V.dbeq ? V.dbeq + (long long)b * meq + idx : nullptr)
                    : idx < mg ? (V.dbineq ? V.dbineq + (long long)b * m + idx - meq : nullptr)
                    : idx < mg + n ? (V.dub ? V.dub + (long long)b * n + idx - mg : nullptr)
                    : (V.dlb ? V.dlb + (long long)b * n + idx - mg - n : nullptr);
        if (out) *out = rhs[a];
    }
    if (V.k == 2)
        for (int t = tid; t < na * n; t += T) {
            const int a = t / n, j = t % n, idx = iact[a] - 1;
            if (idx >= mg) continue;
            const double g = -rhs[nm + a] * v[j] - rhs[a] * x[j];
            if (idx < meq) {
                if (V.dAeq) V.dAeq[(long long)b * meq * n + idx + (long long)meq * j] = g;
            } else if (V.dAineq) {
                V.dAineq[(long long)b * m * n + idx - meq + (long long)m * j] = g;
            }
        }
}

// The values of COPRA_B200_QP_WRT_*: the input whose identity columns qp_tangent writes (QpJvpParams::wrt)
constexpr int kWrtC = 0, kWrtBeq = 1, kWrtBineq = 2, kWrtLb = 3, kWrtUb = 4;

// entry `col` of general row idx (< meq + m) of a raw QP: the caller's column-major Aeq / Aineq of one instance
struct QpRows {
    const double* Aeq;
    const double* Aineq;
    int meq, m;
    __device__ double operator()(int idx, int col) const
    {
        return idx < meq ? Aeq[idx + (long long)meq * col] : Aineq[idx - meq + (long long)m * col];
    }
};

// direction d of a raw-QP tangent (len doubles per direction, column-major) of instance b, null when not given
__device__ __forceinline__ const double* qp_dir(const DArr& t, int b, long long len, int d)
{
    return t.p ? t.at(b) + len * d : nullptr;
}

// The raw QP's lambda pass (k = 1): [A_act' | -c] into the slab and beta of the active rows in rhs, so that sens_solve leaves
// the forward multipliers lambda in rhs
__global__ void __launch_bounds__(kSensThreads) qp_lambda_gather_kernel(const __grid_constant__ QpJvpParams J)
{
    const int lb = blockIdx.x, b = J.b0 + lb;
    const int n = J.n, meq = J.meq, m = J.m, mg = meq + m, nm = J.nm;
    double* slab = sens_gather(J, lb, b, mg, QpRows{ J.Aeq.at(b), J.Aineq.at(b), meq, m });
    const int na = sens_nact(J, b);
    const int* iact = J.iact + (long long)b * n;
    for (int a = threadIdx.x; a < nm; a += blockDim.x)
        J.rhs[(long long)lb * nm + a] = a < na ? active_beta(iact[a] - 1, meq, mg, n, J.beq.at(b), J.bineq.at(b), J.ub.at(b), J.lb.at(b)) : 0.0;
    if (J.status[b] != 0) return;
    const double* c = J.c.at(b);
    for (int col = threadIdx.x; col < n; col += blockDim.x) slab[col + (long long)nm * J.lds] = -c[col];
}

// lambda (rhs after sens_solve, k = 1) into the whole-batch workspace, by active position
__global__ void __launch_bounds__(kSensThreads) qp_lambda_store_kernel(const __grid_constant__ QpJvpParams J)
{
    const int lb = blockIdx.x, b = J.b0 + lb, na = sens_nact(J, b);
    for (int a = threadIdx.x; a < na; a += blockDim.x) J.lam[(long long)b * J.n + a] = J.rhs[(long long)lb * J.nm + a];
}

// The raw QP's tangent pass: [A_act' | -cdot_eff,1 .. -cdot_eff,k] into the slab and bdot_eff (nm x k) in rhs, with
//   cdot_eff = cdot + sym(Qdot) x + sum_active lambda_j adot_j,   bdot_eff,j = bdot_j - adot_j' x (general row), lbdot / ubdot
// (bound row); in identity mode (wrt >= 0) cdot or bdot of direction d is the unit vector e_d and every other tangent is zero.
// The symmetric-part product is formed without contraction, so that Qdot and Qdot' give the same bits.
__global__ void __launch_bounds__(kSensThreads) qp_tangent_kernel(const __grid_constant__ QpJvpParams J)
{
    const int lb = blockIdx.x, b = J.b0 + lb;
    const int n = J.n, meq = J.meq, m = J.m, mg = meq + m, nm = J.nm, k = J.k, wrt = J.wrt;
    double* slab = sens_gather(J, lb, b, mg, QpRows{ J.Aeq.at(b), J.Aineq.at(b), meq, m });
    if (J.status[b] != 0) return; // sens_gram zeroes the rhs of an instance without an active set
    const int na = J.nact[b];
    const int* iact = J.iact + (long long)b * n;
    const double* x = J.x + (long long)b * n;
    const double* lam = J.lam ? J.lam + (long long)b * n : nullptr;
    const long long nn = (long long)n * n;
    for (int t = threadIdx.x; t < n * k; t += blockDim.x) {
        const int i = t % n, d = t / n;
        const double* tc = qp_dir(J.tc, b, n, d);
        double c = wrt == kWrtC ? (i == d ? 1.0 : 0.0) : tc ? tc[i] : 0.0;
        if (const double* Qd = qp_dir(J.tQ, b, nn, d)) {
            double s = 0.0;
            for (int a = 0; a < n; ++a)
                s = __dadd_rn(s, __dmul_rn(__dmul_rn(0.5, __dadd_rn(Qd[i + (long long)a * n], Qd[a + (long long)i * n])), x[a]));
            c += s;
        }
        if (lam) {
            const double* Ae = qp_dir(J.tAeq, b, (long long)meq * n, d);
            const double* Ai = qp_dir(J.tAineq, b, (long long)m * n, d);
            for (int a = 0; a < na; ++a) {
                const int idx = iact[a] - 1;
                if (idx < meq) {
                    if (Ae) c += lam[a] * Ae[idx + (long long)meq * i];
                } else if (idx < mg && Ai) {
                    c += lam[a] * Ai[idx - meq + (long long)m * i];
                }
            }
        }
        slab[i + (long long)(nm + d) * J.lds] = -c;
    }
    for (int t = threadIdx.x; t < nm * k; t += blockDim.x) {
        const int a = t % nm, d = t / nm;
        double v = 0.0;
        if (a < na) {
            const int idx = iact[a] - 1;
            if (idx < mg) {
                const bool eq = idx < meq;
                const int r = eq ? idx : idx - meq, rows = eq ? meq : m;
                const double* tb = qp_dir(eq ? J.tbeq : J.tbineq, b, rows, d);
                const double* tA = qp_dir(eq ? J.tAeq : J.tAineq, b, (long long)rows * n, d);
                if (wrt == (eq ? kWrtBeq : kWrtBineq)) v = r == d ? 1.0 : 0.0;
                else if (tb) v = tb[r];
                if (tA) {
                    double s = 0.0;
                    for (int i = 0; i < n; ++i) s += tA[r + (long long)rows * i] * x[i];
                    v -= s;
                }
            } else {
                const int var = (idx - mg) % n;
                const bool up = idx - mg < n; // upper rows first, then lower rows
                const double* tv = qp_dir(up ? J.tub : J.tlb, b, n, d);
                if (wrt == (up ? kWrtUb : kWrtLb)) v = var == d ? 1.0 : 0.0;
                else if (tv) v = tv[var];
            }
        }
        J.rhs[(long long)lb * nm * k + t] = v;
    }
}

// xdot = V, n x k per instance (column-major); zeros for an instance whose status is not 0
__global__ void __launch_bounds__(kSensThreads) qp_output_kernel(const __grid_constant__ QpJvpParams J)
{
    const int lb = blockIdx.x, b = J.b0 + lb, n = J.n, k = J.k;
    const bool live = J.status[b] == 0;
    const double* V = J.V + (long long)lb * J.lds * k;
    double* out = J.dx + (long long)b * n * k;
    for (int t = threadIdx.x; t < n * k; t += blockDim.x) out[t] = live ? V[t % n + (long long)(t / n) * J.lds] : 0.0;
}

// dcontrol = the first ru rows of Udot; dtraj = the first rx rows of Phi x0dot + Psi Udot, Psi applied as the block-Toeplitz
// product over the compact Gs (K7 without xi).  In initial-state mode Udot = zdot[nx:] and x0dot = zdot[0:nx].  Zeros for an
// instance whose status is not 0.
__global__ void __launch_bounds__(kSensThreads) k9_output_kernel(const __grid_constant__ BuildParams P, const __grid_constant__ JvpParams J)
{
    const int lb = blockIdx.x, b = J.b0 + lb, k = J.k;
    const int nx = P.nx, nu = P.nu, X = P.X, NX = P.N * P.nx, off = P.initial_state ? nx : 0;
    const bool live = J.status[b] == 0;
    const double* Zd = J.V + (long long)lb * J.lds * k;
    const double* Ud = Zd + off;
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
            const double* z = Zd + (long long)d * J.lds;
            double s1 = 0.0;
            for (int a = 0; a < nx; ++a) s1 += Phi[row + (long long)a * X] * (off ? z[a] : x0_tangent(J, b, nx, d, a));
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

int k8_gather_launch(const BuildParams& P, const VjpParams& V, int nb, cudaStream_t st)
{
    k8_gather_kernel<<<nb, kSensThreads, 0, st>>>(P, V);
    return launched(cudaGetLastError());
}

int k9_tangent_launch(const BuildParams& P, const JvpParams& J, int nb, cudaStream_t st)
{
    k9_tangent_kernel<<<nb, kSensThreads, 0, st>>>(P, J);
    return launched(cudaGetLastError());
}

int sens_gram_launch(const SensChunk& S, int nb, cudaStream_t st)
{
    sens_gram_kernel<<<nb, kSensThreads, 0, st>>>(S);
    return launched(cudaGetLastError());
}

size_t sens_solve_smem(int k, int nm)
{
    const int tile = k <= 2 ? k : kDirTile;
    return sizeof(double) * 2 * std::min(k, tile) * size_t(std::max(nm, 1));
}

int sens_solve_launch(const SensChunk& S, int nb, cudaStream_t st)
{
    const auto kernel = S.k == 1 ? sens_solve_kernel<1> : S.k == 2 ? sens_solve_kernel<2> : sens_solve_kernel<kDirTile>;
    const size_t smem = sens_solve_smem(S.k, S.nm);
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return -int(e);
    kernel<<<nb, kSensThreads, smem, st>>>(S);
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
    k8_adjoint_kernel<<<nb, kSensThreads, smem, st>>>(P, V);
    return launched(cudaGetLastError());
}

size_t k8_cost_grad_smem(const BuildParams& P)
{
    int et = 1;
    for (int ci = 0; ci < P.ncost; ++ci) et = std::max(et, 2 * P.cost[ci].rows * (P.cost[ci].i1 - P.cost[ci].i0));
    return sizeof(double) * (2 * size_t(P.nvar) + 2 * size_t(P.X) + size_t(et));
}

int k8_cost_grad_launch(const BuildParams& P, const VjpParams& V, int nb, cudaStream_t st)
{
    const size_t smem = k8_cost_grad_smem(P);
    cudaError_t e = cudaFuncSetAttribute(k8_cost_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return -int(e);
    k8_cost_grad_kernel<<<nb, kSensThreads, smem, st>>>(P, V);
    return launched(cudaGetLastError());
}

size_t k8_model_grad_smem(const BuildParams& P)
{
    return sizeof(double) * (2 * size_t(P.nvar) + 4 * size_t(P.X) + 2 * size_t(P.meq + P.mineq));
}

int k8_model_grad_launch(const BuildParams& P, const VjpParams& V, int nb, cudaStream_t st)
{
    const size_t smem = k8_model_grad_smem(P);
    cudaError_t e = cudaFuncSetAttribute(k8_model_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return -int(e);
    k8_model_grad_kernel<<<nb, kSensThreads, smem, st>>>(P, V);
    return launched(cudaGetLastError());
}

int k9_output_launch(const BuildParams& P, const JvpParams& J, int nb, cudaStream_t st)
{
    k9_output_kernel<<<nb, kSensThreads, 0, st>>>(P, J);
    return launched(cudaGetLastError());
}

int qp_gather_launch(const QpVjpParams& V, int nb, cudaStream_t st)
{
    qp_gather_kernel<<<nb, kSensThreads, 0, st>>>(V);
    return launched(cudaGetLastError());
}

size_t qp_grad_smem(int n) { return sizeof(double) * 2 * size_t(n); }

int qp_grad_launch(const QpVjpParams& V, int nb, cudaStream_t st)
{
    const size_t smem = qp_grad_smem(V.n);
    cudaError_t e = cudaFuncSetAttribute(qp_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return -int(e);
    qp_grad_kernel<<<nb, kSensThreads, smem, st>>>(V);
    return launched(cudaGetLastError());
}

int qp_lambda_gather_launch(const QpJvpParams& J, int nb, cudaStream_t st)
{
    qp_lambda_gather_kernel<<<nb, kSensThreads, 0, st>>>(J);
    return launched(cudaGetLastError());
}

int qp_lambda_store_launch(const QpJvpParams& J, int nb, cudaStream_t st)
{
    qp_lambda_store_kernel<<<nb, kSensThreads, 0, st>>>(J);
    return launched(cudaGetLastError());
}

int qp_tangent_launch(const QpJvpParams& J, int nb, cudaStream_t st)
{
    qp_tangent_kernel<<<nb, kSensThreads, 0, st>>>(J);
    return launched(cudaGetLastError());
}

int qp_output_launch(const QpJvpParams& J, int nb, cudaStream_t st)
{
    qp_output_kernel<<<nb, kSensThreads, 0, st>>>(J);
    return launched(cudaGetLastError());
}

} // namespace cb
