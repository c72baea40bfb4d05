// dgemm_dmma.cu -- batched FP64 GEMM on the tensor cores: the dense contraction of QP assembly for
// FULL-SIZE (autoSpan'd) entries, where the cost / constraint matrices are dense R x X blocks:
//   T = M Psi (+ N)                        reference src/costFunctions.cpp:65,197   (NN)
//   Q += T' W T, E = (M Phi)' W T          src/costFunctions.cpp:66-69,199-202      (TN)
//   A = E Psi (+ G), Y = E Phi             src/constraints.cpp:68-72,199-203        (NN)
// sm_100a has no f64 kind in tcgen05; FP64 MMA is the warp-level mma.sync m8n8k4 (SASS DMMA.8x8x4).
//
//   C[b] = alpha * op(A[b]) * B[b] + beta * C[b],   op(A) = A (M x K) or A' (A stored K x M); column-major.
//
// CTA tile 64 x 64, K tile 16, 8 warps as 4 (M) x 2 (N), each warp 16 x 32 = 2 x 4 DMMA tiles.
// Shared-memory layouts are chosen so that every fragment load is conflict-free for 64-bit words (a
// half-warp must hit 16 distinct 8-byte banks): A as [k][m] with ld 68 (op N) or [m][k] with ld 20
// (op T), B as [n][k] with ld 20 -- 68 = 4 (mod 16) and 20 = 4 (mod 16).
// The A tile of the NN case is a set of contiguous 512-byte column segments: when the operand is
// 16-byte aligned they are fetched by the TMA engine (cp.async.bulk.shared.global + mbarrier
// complete_tx) and overlap with the B tile's register-staged loads.
//
// Two kernels.  dgemm_dmma_tma_kernel (the one that runs whenever the operands are 16-byte aligned with even leading
// dimensions) is a warp-specialised pipeline: ONE producer thread feeds a 4-stage ring of 128 x 16 (A) and 16 x 64 (B)
// tiles with 2-D/3-D tensor-map TMA (cp.async.bulk.tensor, SWIZZLE_128B -- SASS UTMALDG), full / empty mbarriers per stage,
// and 8 consumer warps (4 x 2, warp tile 32 x 32 = 4 x 4 DMMA tiles) read their fragments straight from the swizzled tiles;
// out-of-range rows / columns / k are zero-filled by the TMA unit, so the main loop has no bounds code.
// dgemm_dmma_kernel is the fallback for unaligned operands (single-buffered, register-staged loads).
#include "launch.h"

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace cb {

namespace {

constexpr int TM = 64, TN = 64, TK = 16;
constexpr int LDA_N = 68; // A stored [k][m]
constexpr int LDK = 20;   // [m][k] / [n][k]

__device__ __forceinline__ void dmma8x8x4(double& d0, double& d1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    }
}
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

struct GemmArgs {
    int transA, M, N, K, batch;
    double alpha, beta;
    const double* A; int lda; long long sA;
    const double* B; int ldb; long long sB;
    double* C; int ldc; long long sC;
};

template <bool TRANSA> __global__ void __launch_bounds__(256) dgemm_dmma_kernel(const GemmArgs g)
{
    __shared__ __align__(16) double As[TRANSA ? TM * LDK : TK * LDA_N];
    __shared__ __align__(16) double Bs[TN * LDK];
    __shared__ __align__(8) uint64_t bar;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp >> 1, wn = warp & 1; // 4 x 2 warps
    const int m0 = blockIdx.x * TM, n0 = blockIdx.y * TN;
    const long long b = blockIdx.z;
    const double* A = g.A + b * g.sA;
    const double* B = g.B + b * g.sB;
    double* C = g.C + b * g.sC;
    const int M = g.M, N = g.N, K = g.K;

    double acc[2][4][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    // TMA is usable for the NN A tile when every 64-double column segment is in range and 16-byte aligned
    const bool tma_ok = !TRANSA && (m0 + TM <= M) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0) && ((g.lda & 1) == 0);
    if (tid == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    }
    __syncthreads();
    uint32_t phase = 0;

    for (int k0 = 0; k0 < K; k0 += TK) {
        // ---- A tile ----
        if (TRANSA) {
            // As[m][k] = A[(k0+k) + (m0+m) * lda] : k contiguous in global
            for (int idx = tid; idx < TM * TK; idx += 256) {
                const int k = idx % TK, m = idx / TK;
                const int gm = m0 + m, gk = k0 + k;
                As[m * LDK + k] = (gm < M && gk < K) ? A[gk + (long long)gm * g.lda] : 0.0;
            }
        } else if (tma_ok) {
            if (tid == 0) {
                const int kk = min(TK, K - k0);
                mbar_expect_tx(&bar, uint32_t(kk) * TM * sizeof(double));
                for (int k = 0; k < kk; ++k) tma_load_1d(&As[k * LDA_N], A + m0 + (long long)(k0 + k) * g.lda, TM * sizeof(double), &bar);
            }
            if (k0 + TK > K)
                for (int idx = tid; idx < TM * TK; idx += 256) {
                    const int m = idx % TM, k = idx / TM;
                    if (k0 + k >= K) As[k * LDA_N + m] = 0.0;
                }
        } else {
            // As[k][m] = A[(m0+m) + (k0+k) * lda] : m contiguous in global
            for (int idx = tid; idx < TM * TK; idx += 256) {
                const int m = idx % TM, k = idx / TM;
                const int gm = m0 + m, gk = k0 + k;
                As[k * LDA_N + m] = (gm < M && gk < K) ? A[gm + (long long)gk * g.lda] : 0.0;
            }
        }
        // ---- B tile: Bs[n][k] = B[(k0+k) + (n0+n) * ldb] ----
        for (int idx = tid; idx < TN * TK; idx += 256) {
            const int k = idx % TK, n = idx / TK;
            const int gn = n0 + n, gk = k0 + k;
            Bs[n * LDK + k] = (gn < N && gk < K) ? B[gk + (long long)gn * g.ldb] : 0.0;
        }
        if (!TRANSA && tma_ok) { mbar_wait(&bar, phase); phase ^= 1; }
        __syncthreads();
        // ---- 4 k-steps of DMMA ----
#pragma unroll
        for (int ks = 0; ks < TK; ks += 4) {
            double af[2], bf[4];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int m = wm * 16 + i * 8 + (lane >> 2), k = ks + (lane & 3);
                af[i] = TRANSA ? As[m * LDK + k] : As[k * LDA_N + m];
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int n = wn * 32 + j * 8 + (lane >> 2), k = ks + (lane & 3);
                bf[j] = Bs[n * LDK + k];
            }
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) dmma8x8x4(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
        }
        __syncthreads();
    }
    // ---- epilogue ----
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int m = m0 + wm * 16 + i * 8 + (lane >> 2);
                const int n = n0 + wn * 32 + j * 8 + 2 * (lane & 3) + e;
                if (m < M && n < N) {
                    double* cp = C + m + (long long)n * g.ldc;
                    const double v = g.alpha * acc[i][j][e];
                    *cp = (g.beta == 0.0) ? v : v + g.beta * (*cp);
                }
            }
}


// ---- the TMA pipeline ----------------------------------------------------------------------------------------------------
constexpr int PM = 128, PN = 64, PK = 16, STAGES = 4;
constexpr int A_BYTES = PM * PK * 8, B_BYTES = PN * PK * 8, STAGE_BYTES = A_BYTES + B_BYTES;

__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst_smem, const CUtensorMap* tm, int c0, int c1, int c2, uint64_t* bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];\n" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
                 : "memory");
}
// byte offset of element (row r, inner index i in [0,16)) of a tile whose rows are 128 bytes, SWIZZLE_128B
__device__ __forceinline__ uint32_t swz(int r, int i) { return uint32_t(r) * 128u + (uint32_t(((i >> 1) ^ (r & 7))) << 4) + (uint32_t(i & 1) << 3); }

template <bool TRANSA>
__global__ void __launch_bounds__(288, 2) dgemm_dmma_tma_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
    const GemmArgs g, const int zA, const int zB)
{
    extern __shared__ __align__(1024) unsigned char dsm_raw[];
    __shared__ __align__(8) uint64_t full[STAGES], empty[STAGES];
    unsigned char* dsm = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(dsm_raw) + 1023) & ~uintptr_t(1023));
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int m0 = blockIdx.x * PM, n0 = blockIdx.y * PN;
    const int b = blockIdx.z;
    const int M = g.M, N = g.N, K = g.K;
    const int nk = (K + PK - 1) / PK;
    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 8); }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    }
    __syncthreads();
    if (warp == 8) {
        if (lane == 0) {
            for (int kt = 0; kt < nk; ++kt) {
                const int s = kt % STAGES, ph = (kt / STAGES) & 1, k0 = kt * PK;
                if (kt >= STAGES) mbar_wait(&empty[s], uint32_t(ph ^ 1));
                unsigned char* as = dsm + size_t(s) * STAGE_BYTES;
                mbar_expect_tx(&full[s], STAGE_BYTES);
                if (TRANSA) tma_load_3d(as, &tmA, k0, m0, zA ? b : 0, &full[s]);                // box {16 k, 128 m}
                else
                    for (int j = 0; j < PM / 16; ++j) tma_load_3d(as + j * 2048, &tmA, m0 + 16 * j, k0, zA ? b : 0, &full[s]); // box {16 m, 16 k}
                tma_load_3d(as + A_BYTES, &tmB, k0, n0, zB ? b : 0, &full[s]);                  // box {16 k, 64 n}
            }
        }
        return;
    }
    const int wm = warp >> 1, wn = warp & 1; // 4 x 2 consumer warps, warp tile 32 x 32
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    const int fr = lane >> 2, fk = lane & 3;
    // per-lane fragment offsets inside a stage, hoisted out of the loop: everything else is an immediate
    //   k-inner tiles (B, A of the TN case): row r = base + 8 j + fr -> swz(r, ks + fk) = r 128 + (((ks + fk) >> 1) ^ fr) 16 + (fk & 1) 8
    //   m-inner boxes (A of the NN case):    m = wm 32 + 8 i + fr   -> (m >> 4) 2048 + (ks + fk) 128 + chunk 16 + (fr & 1) 8,
    //                                        chunk = ((fr >> 1) ^ fk) + 4 ((i & 1) ^ ((ks >> 2) & 1))
    uint32_t offB[4], offA[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int ks = 4 * q;
        offB[q] = A_BYTES + swz(wn * 32 + fr, ks + fk);
        offA[q] = TRANSA ? swz(wm * 32 + fr, ks + fk) : uint32_t(wm * 4096 + (ks + fk) * 128 + (((fr >> 1) ^ fk) << 4) + ((fr & 1) << 3));
    }
    for (int kt = 0; kt < nk; ++kt) {
        const int s = kt % STAGES, ph = (kt / STAGES) & 1;
        mbar_wait(&full[s], uint32_t(ph));
        const unsigned char* st = dsm + size_t(s) * STAGE_BYTES;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            double af[4], bf[4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
                af[i] = TRANSA ? *reinterpret_cast<const double*>(st + offA[q] + i * 1024)
                               : *reinterpret_cast<const double*>(st + offA[q] + (i >> 1) * 2048 + (((i & 1) ^ (q & 1)) << 6));
#pragma unroll
            for (int j = 0; j < 4; ++j) bf[j] = *reinterpret_cast<const double*>(st + offB[q] + j * 1024);
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) dmma8x8x4(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
    }
    double* C = g.C + (long long)b * g.sC;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int m = m0 + wm * 32 + i * 8 + fr;
                const int n = n0 + wn * 32 + j * 8 + 2 * fk + e;
                if (m < M && n < N) {
                    double* cp = C + m + (long long)n * g.ldc;
                    const double v = g.alpha * acc[i][j][e];
                    *cp = (g.beta == 0.0) ? v : v + g.beta * (*cp);
                }
            }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn()
{
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// column-major `inner x outer` matrices, `count` of them `stride` doubles apart (0: one shared matrix)
bool make_map(CUtensorMap* tm, const double* base, int inner, int outer, int ld, long long stride, int count, int box_inner, int box_outer)
{
    EncodeTiledFn fn = encode_fn();
    if (!fn) return false;
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (ld & 1) || (stride & 1) || ld < inner) return false;
    const bool z = stride != 0 && count > 1;
    cuuint64_t dims[3] = { cuuint64_t(inner), cuuint64_t(outer), cuuint64_t(z ? count : 1) };
    cuuint64_t strides[2] = { cuuint64_t(ld) * 8, z ? cuuint64_t(stride) * 8 : cuuint64_t(ld) * 8 * cuuint64_t(outer) };
    cuuint32_t box[3] = { cuuint32_t(box_inner), cuuint32_t(box_outer), 1 };
    cuuint32_t estr[3] = { 1, 1, 1 };
    return fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, const_cast<double*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <bool TRANSA> cudaError_t launch_tma(const GemmArgs& g, const CUtensorMap& ta, const CUtensorMap& tb, cudaStream_t st)
{
    const int smem = STAGES * STAGE_BYTES + 1024;
    cudaError_t e = cudaFuncSetAttribute(dgemm_dmma_tma_kernel<TRANSA>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); // per device
    if (e != cudaSuccess) return e;
    dim3 grid((g.M + PM - 1) / PM, (g.N + PN - 1) / PN, g.batch);
    dgemm_dmma_tma_kernel<TRANSA><<<grid, 288, smem, st>>>(ta, tb, g, g.sA != 0, g.sB != 0);
    return cudaGetLastError();
}

} // namespace

int dgemm_dmma_launch(int transA, int M, int N, int K, double alpha, const double* A, int lda, long long sA, const double* B, int ldb,
    long long sB, double beta, double* C, int ldc, long long sC, int batch, cudaStream_t st)
{
    if (M <= 0 || N <= 0 || batch <= 0) return 0;
    int launches = 0;
    for (int b0 = 0; b0 < batch; b0 += 65535) {
        const int nb = batch - b0 < 65535 ? batch - b0 : 65535;
        GemmArgs g;
        g.transA = transA; g.M = M; g.N = N; g.K = K; g.batch = nb; g.alpha = alpha; g.beta = beta;
        g.A = A + (long long)b0 * sA; g.lda = lda; g.sA = sA;
        g.B = B + (long long)b0 * sB; g.ldb = ldb; g.sB = sB;
        g.C = C + (long long)b0 * sC; g.ldc = ldc; g.sC = sC;
        // tensor-map TMA pipeline when the operands qualify (16-byte aligned, even leading dimensions / batch strides)
        CUtensorMap ta, tb;
        const bool tma = K >= 1 &&
            (transA ? make_map(&ta, g.A, K, M, lda, sA, nb, PK, PM) : make_map(&ta, g.A, M, K, lda, sA, nb, 16, PK)) &&
            make_map(&tb, g.B, K, N, ldb, sB, nb, PK, PN);
        cudaError_t e;
        if (tma) {
            e = transA ? launch_tma<true>(g, ta, tb, st) : launch_tma<false>(g, ta, tb, st);
        } else {
            dim3 grid((M + TM - 1) / TM, (N + TN - 1) / TN, nb);
            if (transA) dgemm_dmma_kernel<true><<<grid, 256, 0, st>>>(g);
            else dgemm_dmma_kernel<false><<<grid, 256, 0, st>>>(g);
            e = cudaGetLastError();
        }
        if (e != cudaSuccess) return -int(e);
        ++launches;
    }
    return launches;
}

} // namespace cb
