// K2 (exact-fp32 engine) -- shared-memory tiled FFMA GEMM with fused epilogues.
// Serves CODAE_F32 mode (the reference's own precision: parity at fp32 rounding) and every shape the
// tcgen05 engine cannot tile (abalone's 11x11 layers, odd pitches).  One kernel template covers the three
// contractions of nn.Linear:  C[m,n] = sum_k A(m,k) * B(k,n)
//   fwd   : A = X  (k contiguous)   B(k,n) = W[n,k]  (k contiguous)   epilogue bias + ReLU
//   dgrad : A = dY (k contiguous)   B(k,n) = W[k,n]  (n contiguous)   epilogue ReLU mask of the layer input
//   wgrad : A(m,k) = dY[k,m] (m contiguous)   B(k,n) = X[k,n] (n contiguous)
#include <stdio.h>
#include <stdlib.h>

#include "common.cuh"
#include "gemm.h"

namespace {

enum { EPI_NONE = 0, EPI_BIAS_ACT = 1, EPI_RELU_MASK = 2 };

template <int BM, int BN, int BK, bool A_KC, bool B_KC, int EPI>
__global__ void __launch_bounds__((BM / 4) * (BN / 4)) simt_gemm_kernel(const float* __restrict__ A, int64_t lda,
                                                                        const float* __restrict__ B, int64_t ldb,
                                                                        float* __restrict__ C, int64_t ldc, int M, int N,
                                                                        int K, const float* __restrict__ bias, int act,
                                                                        const float* __restrict__ mask_src, int64_t ldm) {
    constexpr int NT = (BM / 4) * (BN / 4);
    __shared__ __align__(16) float As[BK][BM + 4];
    __shared__ __align__(16) float Bs[BK][BN + 4];
    const int tid = threadIdx.x;
    const int tx = tid % (BN / 4), ty = tid / (BN / 4);
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int k0 = 0; k0 < K; k0 += BK) {
        for (int e = tid; e < BM * BK; e += NT) {
            int m, k;
            if (A_KC) { m = e / BK; k = e % BK; } else { k = e / BM; m = e % BM; }
            const int gm = m0 + m, gk = k0 + k;
            float val = 0.f;
            if (gm < M && gk < K) val = A_KC ? A[(int64_t)gm * lda + gk] : A[(int64_t)gk * lda + gm];
            As[k][m] = val;
        }
        for (int e = tid; e < BN * BK; e += NT) {
            int n, k;
            if (B_KC) { n = e / BK; k = e % BK; } else { k = e / BN; n = e % BN; }
            const int gn = n0 + n, gk = k0 + k;
            float val = 0.f;
            if (gn < N && gk < K) val = B_KC ? B[(int64_t)gn * ldb + gk] : B[(int64_t)gk * ldb + gn];
            Bs[k][n] = val;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int gm = m0 + ty * 4 + i;
        if (gm >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int gn = n0 + tx * 4 + j;
            if (gn >= N) continue;
            float r = acc[i][j];
            if (EPI == EPI_BIAS_ACT) {
                if (bias) r += bias[gn];
                if (act == CODAE_ACT_RELU) r = fmaxf(r, 0.f);
            } else if (EPI == EPI_RELU_MASK) {
                if (mask_src) r = mask_src[(int64_t)gm * ldm + gn] > 0.f ? r : 0.f;
            }
            C[(int64_t)gm * ldc + gn] = r;
        }
    }
}

// Split-K variant for small batches (few 64x64 tiles, long K): the K range is spread over a thread-block cluster along
// grid z; every CTA parks its 64x64 fp32 partial in shared memory and, after a cluster barrier, CTA r reduces rows
// [64 r / S, 64 (r+1) / S) of all S partials through distributed shared memory in rank order (deterministic), applies
// the epilogue and stores.  Same scheme as the tensor-core engine's split-K.
template <bool A_KC, bool B_KC, int EPI>
__global__ void __launch_bounds__(256) simt_gemm_splitk_kernel(const float* __restrict__ A, int64_t lda,
                                                               const float* __restrict__ B, int64_t ldb,
                                                               float* __restrict__ C, int64_t ldc, int M, int N, int K,
                                                               const float* __restrict__ bias, int act,
                                                               const float* __restrict__ mask_src, int64_t ldm) {
    constexpr int BM = 64, BN = 64, BK = 16, NT = 256, kPitch = BN + 4;
    __shared__ __align__(16) float As[BK][BM + 4];
    __shared__ __align__(16) float Bs[BK][BN + 4];
    __shared__ __align__(16) float part[BM * kPitch];
    const int tid = threadIdx.x;
    const int tx = tid % (BN / 4), ty = tid / (BN / 4);
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const int nsplit = gridDim.z, rank = blockIdx.z;
    const int k_per = ((K + nsplit - 1) / nsplit + BK - 1) / BK * BK;
    const int k_begin = rank * k_per, k_end = min(K, k_begin + k_per);
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int k0 = k_begin; k0 < k_end; k0 += BK) {
        for (int e = tid; e < BM * BK; e += NT) {
            int m, k;
            if (A_KC) { m = e / BK; k = e % BK; } else { k = e / BM; m = e % BM; }
            const int gm = m0 + m, gk = k0 + k;
            float val = 0.f;
            if (gm < M && gk < k_end) val = A_KC ? A[(int64_t)gm * lda + gk] : A[(int64_t)gk * lda + gm];
            As[k][m] = val;
        }
        for (int e = tid; e < BN * BK; e += NT) {
            int n, k;
            if (B_KC) { n = e / BK; k = e % BK; } else { k = e / BN; n = e % BN; }
            const int gn = n0 + n, gk = k0 + k;
            float val = 0.f;
            if (gn < N && gk < k_end) val = B_KC ? B[(int64_t)gn * ldb + gk] : B[(int64_t)gk * ldb + gn];
            Bs[k][n] = val;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
        *reinterpret_cast<float4*>(&part[(ty * 4 + i) * kPitch + tx * 4]) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    const int r_begin = (rank * BM) / nsplit, r_end = ((rank + 1) * BM) / nsplit;
    const uint32_t base = (uint32_t)__cvta_generic_to_shared(part);
    for (int it = tid; it < (r_end - r_begin) * (BN / 4); it += NT) {
        const int rl = r_begin + it / (BN / 4), c4 = it % (BN / 4);
        const uint32_t off = (uint32_t)(rl * kPitch + 4 * c4) * 4u;
        float4 p[8];
#pragma unroll
        for (int sp = 0; sp < 8; ++sp) {
            if (sp < nsplit) {
                uint32_t remote;
                asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(base + off), "r"(sp));
                asm volatile("ld.shared::cluster.v4.f32 {%0,%1,%2,%3}, [%4];"
                             : "=f"(p[sp].x), "=f"(p[sp].y), "=f"(p[sp].z), "=f"(p[sp].w) : "r"(remote) : "memory");
            }
        }
        float r[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int sp = 0; sp < 8; ++sp)
            if (sp < nsplit) { r[0] += p[sp].x; r[1] += p[sp].y; r[2] += p[sp].z; r[3] += p[sp].w; }
        const int gm = m0 + rl;
        if (gm >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int gn = n0 + 4 * c4 + j;
            if (gn >= N) continue;
            float o = r[j];
            if (EPI == EPI_BIAS_ACT) {
                if (bias) o += bias[gn];
                if (act == CODAE_ACT_RELU) o = fmaxf(o, 0.f);
            } else if (EPI == EPI_RELU_MASK) {
                if (mask_src) o = mask_src[(int64_t)gm * ldm + gn] > 0.f ? o : 0.f;
            }
            C[(int64_t)gm * ldc + gn] = o;
        }
    }
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// db[n] = sum_m dY[m, n]: block (32 columns x 32 row groups), fixed-order reduction through smem.
template <bool kBf16>
__global__ void __launch_bounds__(1024) colsum_kernel(const void* __restrict__ dY, int64_t ld, int M, int N,
                                                      float* __restrict__ db) {
    __shared__ float part[32][33];
    const int n = blockIdx.x * 32 + threadIdx.x;
    float s = 0.f;
    if (n < N) {
        for (int m = threadIdx.y; m < M; m += 32) {
            s += kBf16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(dY)[(int64_t)m * ld + n])
                       : reinterpret_cast<const float*>(dY)[(int64_t)m * ld + n];
        }
    }
    part[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y == 0 && n < N) {
        float t = 0.f;
#pragma unroll
        for (int r = 0; r < 32; ++r) t += part[r][threadIdx.x];
        db[n] = t;
    }
}

template <bool A_KC, bool B_KC, int EPI>
int launch(codae_ctx* ctx, const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int M, int N,
           int K, const float* bias, int act, const float* mask_src, int64_t ldm, cudaStream_t s) {
    const long ctas64 = (long)((M + 63) / 64) * ((N + 63) / 64);
    static const bool debug_plan = getenv("CODAE_DEBUG_PLAN") != nullptr;
    if (ctas64 >= 2L * ctx->sm_count) {
        if (debug_plan) fprintf(stderr, "codae plan: simt M=%d N=%d K=%d EPI=%d tile 64 split 1\n", M, N, K, EPI);
        dim3 grid((N + 63) / 64, (M + 63) / 64);
        simt_gemm_kernel<64, 64, 16, A_KC, B_KC, EPI><<<grid, 256, 0, s>>>(A, lda, B, ldb, C, ldc, M, N, K, bias, act, mask_src, ldm);
    } else if (ctx->splitk && K >= 256 && M * (long)N >= 64 * 64) {
        // small batch, long contraction: cluster split-K so that ~one CTA per SM streams the weights
        int nsplit = (int)(ctx->sm_count / ctas64);
        if (nsplit > 8) nsplit = 8;
        if (nsplit > K / 128) nsplit = K / 128;
        if (nsplit < 1) nsplit = 1;
        if (debug_plan) fprintf(stderr, "codae plan: simt M=%d N=%d K=%d EPI=%d tile 64 split %d\n", M, N, K, EPI, nsplit);
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((N + 63) / 64, (M + 63) / 64, nsplit);
        cfg.blockDim = dim3(256);
        cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 1;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = nsplit;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        cudaError_t le = cudaLaunchKernelEx(&cfg, simt_gemm_splitk_kernel<A_KC, B_KC, EPI>, A, lda, B, ldb, C, ldc, M, N, K, bias, act,
                                            mask_src, ldm);
        if (le != cudaSuccess) {
            cudaGetLastError();
            return codae_fail(ctx, CODAE_ECUDA, "simt_gemm_splitk_kernel launch (split %d): %s", nsplit, cudaGetErrorString(le));
        }
    } else {
        if (debug_plan) fprintf(stderr, "codae plan: simt M=%d N=%d K=%d EPI=%d tile 32 split 1\n", M, N, K, EPI);
        dim3 grid((N + 31) / 32, (M + 31) / 32);
        simt_gemm_kernel<32, 32, 32, A_KC, B_KC, EPI><<<grid, 64, 0, s>>>(A, lda, B, ldb, C, ldc, M, N, K, bias, act, mask_src, ldm);
    }
    return codae_check_launch(ctx, "simt_gemm_kernel");
}

}  // namespace

int codae_simt_linear_fwd(codae_ctx* ctx, const float* X, int64_t ldx, const float* W, int64_t ldw, const float* bias,
                          float* Y, int64_t ldy, int M, int N, int K, int act, cudaStream_t s) {
    return launch<true, true, EPI_BIAS_ACT>(ctx, X, ldx, W, ldw, Y, ldy, M, N, K, bias, act, nullptr, 0, s);
}

int codae_simt_linear_dgrad(codae_ctx* ctx, const float* dY, int64_t lddy, const float* W, int64_t ldw, const float* A_prev,
                            int64_t lda, float* dX, int64_t lddx, int M, int N, int K, cudaStream_t s) {
    // dX[M,K] = dY[M,N] . W[N,K]: contraction over N; output columns = K
    return launch<true, false, EPI_RELU_MASK>(ctx, dY, lddy, W, ldw, dX, lddx, M, K, N, nullptr, 0, A_prev, lda, s);
}

int codae_simt_linear_wgrad(codae_ctx* ctx, const float* dY, int64_t lddy, const float* X, int64_t ldx, float* dW,
                            int64_t lddw, int M, int N, int K, cudaStream_t s) {
    // dW[N,K] = dY[M,N]^T . X[M,K]: contraction over M
    return launch<false, false, EPI_NONE>(ctx, dY, lddy, X, ldx, dW, lddw, N, K, M, nullptr, 0, nullptr, 0, s);
}

int codae_colsum(codae_ctx* ctx, const void* dY, int dtype, int64_t ld, int M, int N, float* db, cudaStream_t s) {
    dim3 block(32, 32), grid((N + 31) / 32);
    if (dtype == CODAE_BF16) colsum_kernel<true><<<grid, block, 0, s>>>(dY, ld, M, N, db);
    else colsum_kernel<false><<<grid, block, 0, s>>>(dY, ld, M, N, db);
    return codae_check_launch(ctx, "colsum_kernel");
}
