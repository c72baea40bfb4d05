// k6_solver.cu -- batched Goldfarb-Idnani kernel (K5+K6): persistent CTAs pull instances off an
// atomic work queue (iteration counts diverge per instance, SURVEY.md 7).
#include "gi_solver.cuh"
#include "gi_small.cuh"
#include "gi_cluster.cuh"
#include "launch.h"

#include <algorithm>

namespace cb {

template <int MAXT, int MINB>
__global__ void __launch_bounds__(MAXT, MINB) gi_batch_kernel(const __grid_constant__ GiBatch B)
{
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ int s_next;
    const GiLayout L = gi_layout(B.n, B.meq, B.m, blockDim.x, B.j_smem, B.s_smem, B.a_smem);
    double* gJ = B.ws ? B.ws + (long long)blockIdx.x * B.ws_stride : nullptr;
    double* gS = gJ ? gJ + (B.j_smem ? 0 : size_t(L.ldj) * B.n) : nullptr;
    GiWork W = gi_carve(L, smem, gJ, gS);
    for (;;) {
        if (threadIdx.x == 0) s_next = atomicAdd(B.counter, 1);
        __syncthreads();
        const int b = s_next;
        __syncthreads();
        if (b >= B.batch) break;
        GiView P;
        P.n = B.n; P.meq = B.meq; P.m = B.m;
        P.Q = B.Q.at(b); P.c = B.c.at(b);
        P.Aeq = B.Aeq.p ? B.Aeq.at(b) : nullptr; P.beq = B.beq.p ? B.beq.at(b) : nullptr;
        P.Aineq = B.Aineq.p ? B.Aineq.at(b) : nullptr; P.bineq = B.bineq.p ? B.bineq.at(b) : nullptr;
        P.lb = B.lb.at(b); P.ub = B.ub.at(b);
        GiOut O;
        O.x = B.x ? B.x + (long long)b * B.n : nullptr;
        O.status = B.status ? B.status + b : nullptr;
        O.iters = B.iters ? B.iters + 2LL * b : nullptr;
        O.nact = B.nact ? B.nact + b : nullptr;
        O.iact = B.iact ? B.iact + (long long)b * B.n : nullptr;
        gi_solve(P, W, O, B.vsmall, B.max_iter);
        __syncthreads();
    }
}

// n <= 64: latency-optimised 128-thread variant (gi_small.cuh).  J always lives in shared memory; the variants
// differ in where S = R^-1 and the general constraint rows live (shared memory, or global/L2) and therefore in
// how many instances are resident per SM (kSmMinB = 4 CTAs per SM sets the register budget: 128).
template <bool AG, bool SG> __global__ void __launch_bounds__(kSmT, kSmMinB) gi_small_kernel(const __grid_constant__ GiBatch B)
{
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ int s_next;
    const GsLayout L = gs_layout(B.n, B.meq, B.m, !SG, !AG);
    GsWork W = gs_carve(L, smem);
    double* Sg = SG ? B.ws + (long long)blockIdx.x * B.ws_stride : nullptr;
    for (;;) {
        if (threadIdx.x == 0) s_next = atomicAdd(B.counter, 1);
        __syncthreads();
        const int b = s_next;
        __syncthreads();
        if (b >= B.batch) break;
        GiView P;
        P.n = B.n; P.meq = B.meq; P.m = B.m;
        P.Q = B.Q.at(b); P.c = B.c.at(b);
        P.Aeq = B.Aeq.p ? B.Aeq.at(b) : nullptr; P.beq = B.beq.p ? B.beq.at(b) : nullptr;
        P.Aineq = B.Aineq.p ? B.Aineq.at(b) : nullptr; P.bineq = B.bineq.p ? B.bineq.at(b) : nullptr;
        P.lb = B.lb.at(b); P.ub = B.ub.at(b);
        if (B.jmode) {
            double* jc = B.jcache + (long long)b * L.ld * L.n2;
            P.Jin = (B.jmode == 2 && B.jflag[b] == 1) ? jc : nullptr;
            P.Jout = P.Jin ? nullptr : jc;
            P.Jflag = B.jflag + b;
        }
        GiOut O;
        O.x = B.x ? B.x + (long long)b * B.n : nullptr;
        O.status = B.status ? B.status + b : nullptr;
        O.iters = B.iters ? B.iters + 2LL * b : nullptr;
        O.nact = B.nact ? B.nact + b : nullptr;
        O.iact = B.iact ? B.iact + (long long)b * B.n : nullptr;
        gs_solve<AG, SG>(P, L, W, Sg, O, B.vsmall, B.max_iter);
        __syncthreads();
    }
}

// ---- large n: one thread-block cluster per instance (gi_cluster.cuh) -----------------------------------
__global__ void __launch_bounds__(512, 1) gi_cluster_kernel(const __grid_constant__ GiBatch B, double* __restrict__ Sws, int C)
{
    extern __shared__ __align__(16) unsigned char smem[];
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = int(cluster.block_rank());
    const int cid = blockIdx.x / C; // cluster index
    const GcLayout L = gc_layout(B.n, B.meq, B.m, C, blockDim.x);
    GcWork W = gc_carve(L, smem);
    const int lds = odd_ld(B.n);
    double* S = Sws + (long long)cid * lds * B.n;
    for (;;) {
        cluster.sync(); // every CTA is done with the previous instance (DSMEM buffers are free)
        if (rank == 0 && threadIdx.x == 0) {
            const int nb = atomicAdd(B.counter, 1);
            for (int t = 0; t < C; ++t) cluster.map_shared_rank(W.ctl, t)[0] = nb;
        }
        cluster.sync();
        const int b = W.ctl[0];
        if (b >= B.batch) break;
        GiOut O;
        O.x = B.x ? B.x + (long long)b * B.n : nullptr;
        O.status = B.status ? B.status + b : nullptr;
        O.iters = B.iters ? B.iters + 2LL * b : nullptr;
        O.nact = B.nact ? B.nact + b : nullptr;
        O.iact = B.iact ? B.iact + (long long)b * B.n : nullptr;
        GiView P;
        P.n = B.n; P.meq = B.meq; P.m = B.m;
        P.Q = B.Q.at(b); P.c = B.c.at(b);
        P.Aeq = B.Aeq.p ? B.Aeq.at(b) : nullptr; P.beq = B.beq.p ? B.beq.at(b) : nullptr;
        P.Aineq = B.Aineq.p ? B.Aineq.at(b) : nullptr; P.bineq = B.bineq.p ? B.bineq.at(b) : nullptr;
        P.lb = B.lb.at(b); P.ub = B.ub.at(b);
        gc_solve(P, L, W, S, lds, O, B.vsmall, B.max_iter);
    }
}

double gi_vsmall()
{
    // Powell's ZQPCVX estimate as coded in qpgen2 (SURVEY.md 3.3 step 1)
    double vsmall = 1.0e-60;
    for (;;) {
        vsmall += vsmall;
        volatile double tmpa = 1.0 + 0.1 * vsmall;
        volatile double tmpb = 1.0 + 0.2 * vsmall;
        if (tmpa <= 1.0) continue;
        if (tmpb <= 1.0) continue;
        break;
    }
    return vsmall;
}

GiPlan gi_plan(int n, int meq, int m, int batch, int sms, size_t smem_optin, int small_variant)
{
    GiPlan p;
    p.small = 0;
    p.cluster = 0;
    if (n <= kSmMaxN) {
        // Residency variants, in order of preference: J,S,A in shared memory; S in global (L2); S and A in global.
        // Measured on C2/C4 (profiles/r01_summary.md): 4 resident CTAs per SM at <= 128 registers is the sweet spot --
        // fewer CTAs leave issue slots idle, more cost registers -- so take the first variant that reaches 4 per SM,
        // else the one with the most.
        int best = -1, best_per_sm = 0;
        size_t best_bytes = 0;
        for (int v = 0; v < 3; ++v) {
            const size_t b = gs_layout(n, meq, m, v < 1, v < 2).bytes;
            if (b + 2048 > smem_optin) continue;
            const int per_sm = int(std::min<size_t>(kSmMinB, (smem_optin + 1024) / (b + 1024)));
            if (per_sm > best_per_sm) { best = v; best_per_sm = per_sm; best_bytes = b; }
            if (per_sm >= kSmMinB) break;
        }
        if (small_variant >= 1 && small_variant <= 3) { // testing: force residency variant small_variant - 1 when it fits
            const int v = small_variant - 1;
            const size_t b = gs_layout(n, meq, m, v < 1, v < 2).bytes;
            if (b + 2048 <= smem_optin) { best = v; best_bytes = b; best_per_sm = int(std::min<size_t>(kSmMinB, (smem_optin + 1024) / (b + 1024))); }
        }
        if (best >= 0) {
            p.small = 1;
            p.threads = kSmT;
            p.j_smem = 1; p.s_smem = best < 1; p.a_smem = best < 2;
            p.smem_bytes = best_bytes;
            p.ws_stride = p.s_smem ? 0 : (long long)odd_ld(n) * n;
            p.grid = std::max(1, std::min(batch, sms * best_per_sm));
            return p;
        }
    }
    // n too large for one SM's shared memory: a cluster of C CTAs shares J through DSMEM
    if (size_t(odd_ld(n)) * n * sizeof(double) + 24 * 1024 > smem_optin) {
        for (int C = 2; C <= kClMaxC; C *= 2) {
            const size_t b = gc_layout(n, meq, m, C, 512).bytes;
            if (b + 2048 <= smem_optin) {
                p.cluster = C;
                p.threads = 512;
                p.smem_bytes = b;
                p.j_smem = 1; p.s_smem = 0; p.a_smem = 0;
                p.ws_stride = 0;
                p.grid = 0; // sized at launch from cudaOccupancyMaxActiveClusters
                return p;
            }
        }
    }
    // general path: many threads per instance (every phase is a CTA-wide GEMV / rank-1 / reduction)
    p.threads = n <= 32 ? 128 : (n <= 128 ? 256 : 512);
    const size_t budget = smem_optin > 1024 ? smem_optin - 1024 : 0; // headroom for static smem
    const size_t small = 76 * 1024;                                  // keep >= 3 CTAs/SM when the problem is small
    int cfg[4][3] = { { 1, 1, 1 }, { 1, 1, 0 }, { 1, 0, 0 }, { 0, 0, 0 } };
    int pick = 3;
    for (int k = 0; k < 4; ++k) {
        const size_t b = gi_layout(n, meq, m, p.threads, cfg[k][0], cfg[k][1], cfg[k][2]).bytes;
        if (k == 0 && b > small) continue;
        if (b <= budget) { pick = k; break; }
    }
    p.j_smem = cfg[pick][0]; p.s_smem = cfg[pick][1]; p.a_smem = cfg[pick][2];
    const GiLayout L = gi_layout(n, meq, m, p.threads, p.j_smem, p.s_smem, p.a_smem);
    p.smem_bytes = L.bytes;
    p.ws_stride = (p.j_smem ? 0 : (long long)L.ldj * n) + (p.s_smem ? 0 : (long long)L.lds * n);
    int per_sm = 1;
    if (p.smem_bytes > 0) per_sm = int(std::max<size_t>(1, std::min<size_t>(16, (smem_optin + 1024) / (p.smem_bytes + 1024))));
    per_sm = std::min(per_sm, 2048 / p.threads);
    p.grid = std::max(1, std::min(batch, sms * per_sm));
    return p;
}

template <int MAXT, int MINB> static cudaError_t gi_launch_t(const GiBatch& B, const GiPlan& plan, cudaStream_t st)
{
    cudaError_t e = cudaFuncSetAttribute(gi_batch_kernel<MAXT, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(plan.smem_bytes));
    if (e != cudaSuccess) return e;
    gi_batch_kernel<MAXT, MINB><<<plan.grid, plan.threads, plan.smem_bytes, st>>>(B);
    return cudaGetLastError();
}

template <bool AG, bool SG> static cudaError_t gi_small_launch_t(const GiBatch& B, const GiPlan& plan, cudaStream_t st)
{
    cudaError_t e = cudaFuncSetAttribute(gi_small_kernel<AG, SG>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(plan.smem_bytes));
    if (e != cudaSuccess) return e;
    gi_small_kernel<AG, SG><<<plan.grid, plan.threads, plan.smem_bytes, st>>>(B);
    return cudaGetLastError();
}

cudaError_t gi_cluster_launch(const GiBatch& B, const GiPlan& plan, double* Sws, int nclusters, cudaStream_t st)
{
    cudaError_t e;
    // cluster solve
    e = cudaFuncSetAttribute(gi_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(plan.smem_bytes));
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(unsigned(nclusters * plan.cluster));
    cfg.blockDim = dim3(unsigned(plan.threads));
    cfg.dynamicSmemBytes = plan.smem_bytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = unsigned(plan.cluster);
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int C = plan.cluster;
    return cudaLaunchKernelEx(&cfg, gi_cluster_kernel, B, Sws, C);
}

int gi_cluster_max_clusters(const GiPlan& plan)
{
    if (cudaFuncSetAttribute(gi_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(plan.smem_bytes)) != cudaSuccess) return 0;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(unsigned(plan.cluster * 64));
    cfg.blockDim = dim3(unsigned(plan.threads));
    cfg.dynamicSmemBytes = plan.smem_bytes;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = unsigned(plan.cluster);
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int nc = 0;
    if (cudaOccupancyMaxActiveClusters(&nc, gi_cluster_kernel, &cfg) != cudaSuccess) return 0;
    return nc;
}

cudaError_t gi_launch(const GiBatch& B, const GiPlan& plan, cudaStream_t st)
{
    if (plan.small) {
        if (plan.s_smem) return gi_small_launch_t<false, false>(B, plan, st);
        if (plan.a_smem) return gi_small_launch_t<false, true>(B, plan, st);
        return gi_small_launch_t<true, true>(B, plan, st);
    }
    // register budgets: 128 thr x 6 CTA/SM, 256 thr x 3 CTA/SM (<= 80 regs), 512 thr x 1 (<= 128 regs)
    if (plan.threads <= 128) return gi_launch_t<128, 6>(B, plan, st);
    if (plan.threads <= 256) return gi_launch_t<256, 3>(B, plan, st);
    return gi_launch_t<512, 1>(B, plan, st);
}

} // namespace cb
