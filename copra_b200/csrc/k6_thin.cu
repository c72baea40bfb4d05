// k6_thin.cu -- kernels of the throughput-oriented solver (gi_thin.cuh): the once-per-Hessian factorisation and the
// persistent one-CTA-per-instance active-set kernel.
#include "gi_thin.cuh"
#include "launch.h"

#include <cub/device/device_radix_sort.cuh>

#include <algorithm>

namespace cb {

// Jt = R^-1 (Q = R'R) for `count` Hessians, one CTA each (blocked DMMA Cholesky + inverse of gi_factor.cuh working in
// global memory / L2), plus the transposed copy the row-oriented mat-vec reads.  pd[h] = 0 when Q is not positive
// definite (QuadProg's fail code 2).
__global__ void __launch_bounds__(512, 1) gt_factor_kernel(DArr Q, int n, int ld, int count, double* __restrict__ Jt,
    double* __restrict__ JtT, int* __restrict__ pd)
{
    extern __shared__ __align__(16) unsigned char smem[];
    double* scratch = reinterpret_cast<double*>(smem);
    const int tid = threadIdx.x, T = blockDim.x;
    const size_t sz = size_t(ld) * n;
    for (int h = blockIdx.x; h < count; h += gridDim.x) {
        double* J = Jt + (long long)h * sz;
        double* JT = JtT + (long long)h * sz;
        const double* q = Q.at(h);
        __syncthreads();
        for (size_t idx = tid; idx < sz; idx += T) {
            const int i = int(idx % ld), j = int(idx / ld);
            J[idx] = (i < n) ? q[i + size_t(j) * n] : 0.0;
            JT[idx] = 0.0;
        }
        __syncthreads();
        const bool ok = gi_factor_blocked(J, ld, n, scratch);
        __syncthreads();
        if (tid == 0) pd[h] = ok ? 1 : 0;
        if (!ok) continue;
        // transpose through 32 x 32 tiles (scratch holds >= 33 * 32 doubles)
        double* tile = scratch;
        const int nt = (n + 31) >> 5;
        for (int t = 0; t < nt * nt; ++t) {
            const int ti = t % nt, tj = t / nt; // tile rows ti*32.., cols tj*32..
            if (ti > tj) continue;              // strictly lower tiles are zero
            __syncthreads();
            for (int e = tid; e < 1024; e += T) {
                const int i = ti * 32 + (e & 31), j = tj * 32 + (e >> 5);
                tile[(e >> 5) * 33 + (e & 31)] = (i < n && j < n) ? J[i + size_t(j) * ld] : 0.0;
            }
            __syncthreads();
            for (int e = tid; e < 1024; e += T) {
                const int j = tj * 32 + (e & 31), i = ti * 32 + (e >> 5);
                if (i < n && j < n) JT[j + size_t(i) * ld] = tile[(e & 31) * 33 + (e >> 5)];
            }
        }
    }
}

// Psi' (nU x X, column-major) of ONE system from its compact first block column Gs: Psi[s nx + a, j nu + b] = (A^(s-1-j) B)[a, b]
// for j < s, zero otherwise (src/PreviewSystem.cpp:63-71).  Right-hand operand of Dpsi = Jt' Psi'.
__global__ void gt_psit_fill_kernel(const double* __restrict__ Gs, double* __restrict__ PsiT, int nx, int nu, int N)
{
    const int nU = nu * N, X = nx * (N + 1);
    const long long total = (long long)nU * X;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int i = int(idx % nU), c = int(idx / nU);
        const int j = i / nu, bb = i - j * nu, st = c / nx, a = c - st * nx;
        PsiT[idx] = (j < st) ? Gs[size_t(st - 1 - j) * nx + a + size_t(bb) * N * nx] : 0.0;
    }
}

cudaError_t gt_psit_fill_launch(const double* Gs, double* PsiT, int nx, int nu, int N, cudaStream_t st)
{
    gt_psit_fill_kernel<<<296, 256, 0, st>>>(Gs, PsiT, nx, nu, N);
    return cudaGetLastError();
}

int gt_cluster_capacity(const GtPlan& plan, int csize); // k6_thin_cluster.cu

// Global workspace per CTA: Q1 (or P, ld x n) then S (n x n).  The kernels read Q1 with 128-bit loads, so every CTA's slice
// starts on a 16-byte boundary: for odd n, ld n + n n is odd and is rounded up.
static long long gt_ws_stride(const GtShape& sh)
{
    return ((long long)sh.ld * sh.n + (long long)sh.n * sh.n + 1) & ~1LL;
}

GtPlan gt_plan(const GtShape& sh, int batch, int sms, size_t smem_optin)
{
    GtPlan p{};
    // 512 threads per instance: 256 (47.7 k solves/s on C3) and 1024 x 1 CTA/SM (51.1 k) were measured against 512 x 2 (63.0 k) and
    // dropped -- every extra instantiation of the solver costs minutes of compile time
    p.threads = 512;
    const size_t base = gt_layout(sh.n, sh.meq, sh.m, sh.tab_doubles, p.threads, 0, sh.ss_doubles).bytes;
    p.ok = base + 2048 <= smem_optin;
    if (!p.ok) return p;
    if (sh.cluster > 1) {
        // one cluster per instance: one CTA per SM, Q1 entirely in the global workspace (every CTA of the cluster reads it)
        p.cluster = sh.cluster;
        p.q1s = 0;
        p.per_sm = 1;
        p.smem_bytes = base;
        p.ws_stride = gt_ws_stride(sh);
        const int cap = gt_cluster_capacity(p, sh.cluster);
        if (cap <= 0) { p.ok = 0; return p; }
        p.grid = std::max(1, std::min(batch, cap)) * sh.cluster;
        return p;
    }
    // one CTA per instance, two per SM when their shared memory fits; whatever shared memory the vectors and tables leave
    // holds the head columns of Q1
    const int per_sm = std::min<int>(2, int((smem_optin + 1024) / (base + 1024)));
    const size_t budget = (smem_optin + 1024) / per_sm - 1024 - 1024; // per CTA, minus static shared memory headroom
    int q1s = budget > base ? int((budget - base) / (size_t(sh.ld) * sizeof(double))) : 0;
    q1s = std::min(q1s, sh.n);
    if (sh.pform) q1s = 0; // the shared-factor kernels are compiled without the shared-memory head of P
    p.q1s = q1s;
    p.smem_bytes = gt_layout(sh.n, sh.meq, sh.m, sh.tab_doubles, p.threads, q1s, sh.ss_doubles).bytes;
    p.per_sm = per_sm;
    p.grid = std::max(1, std::min(batch, sms * per_sm));
    p.ws_stride = gt_ws_stride(sh);
    return p;
}

size_t gt_factor_smem(int n) { return std::max<size_t>(gi_factor_scratch(n), 33 * 32) * sizeof(double); }

cudaError_t gt_factor_launch(DArr Q, int n, int ld, int count, double* Jt, double* JtT, int* pd, int sms, cudaStream_t st)
{
    const size_t smem = gt_factor_smem(n);
    cudaError_t e = cudaFuncSetAttribute(gt_factor_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
    // (two CTAs per SM fit for n = 800 but cap the kernel at 64 registers: 165 ms instead of 145 ms for 1024 Hessians)
    gt_factor_kernel<<<std::max(1, std::min(count, sms)), 512, smem, st>>>(Q, n, ld, count, Jt, JtT, pd);
    return cudaGetLastError();
}

size_t gt_sort_temp_bytes(int count)
{
    size_t bytes = 0;
    cub::DeviceRadixSort::SortPairsDescending(nullptr, bytes, (const int*)nullptr, (int*)nullptr, (const int*)nullptr, (int*)nullptr, count);
    return bytes;
}

cudaError_t gt_sort_launch(const int* keys, int* keys_sorted, const int* idx, int* order, int count, void* temp, size_t temp_bytes, cudaStream_t st)
{
    return cub::DeviceRadixSort::SortPairsDescending(temp, temp_bytes, keys, keys_sorted, idx, order, count, 0, 32, st);
}

// one translation unit per form (k6_thin_f0/f1/f2.cu, k6_thin_cluster.cu): the solver is one large inlined function and the
// forms compile in parallel
cudaError_t gt_launch_form0(const GtBatch& B, const GtPlan& plan, cudaStream_t st);
cudaError_t gt_launch_form1(const GtBatch& B, const GtPlan& plan, cudaStream_t st);
cudaError_t gt_launch_form2(const GtBatch& B, const GtPlan& plan, cudaStream_t st);
cudaError_t gt_launch_cluster(const GtBatch& B, const GtPlan& plan, cudaStream_t st);

cudaError_t gt_launch(const GtBatch& B, const GtPlan& plan, cudaStream_t st)
{
    if (plan.cluster > 1) return gt_launch_cluster(B, plan, st);
    // shared-factor form (C3-like batches: 2 CTAs/SM whenever it applies) / general form
    if (B.Hpsi && B.ss && B.structured && !B.warm && !B.prekey) return gt_launch_form2(B, plan, st);
    if (B.Hpsi) return gt_launch_form1(B, plan, st);
    return gt_launch_form0(B, plan, st);
}

} // namespace cb
