// Internal (non-ABI) entry points of the two GEMM engines; linear.cu dispatches between them.
#pragma once
#include <cuda.h>

#include "common.cuh"

int codae_simt_linear_fwd(codae_ctx* ctx, const float* X, int64_t ldx, const float* W, int64_t ldw, const float* bias,
                          float* Y, int64_t ldy, int M, int N, int K, int act, cudaStream_t s);
int codae_simt_linear_dgrad(codae_ctx* ctx, const float* dY, int64_t lddy, const float* W, int64_t ldw, const float* A_prev,
                            int64_t lda, float* dX, int64_t lddx, int M, int N, int K, cudaStream_t s);
int codae_simt_linear_wgrad(codae_ctx* ctx, const float* dY, int64_t lddy, const float* X, int64_t ldx, float* dW,
                            int64_t lddw, int M, int N, int K, cudaStream_t s);
int codae_colsum(codae_ctx* ctx, const void* dY, int dtype, int64_t ld, int M, int N, float* db, cudaStream_t s);

// tcgen05 engine (gemm_tcgen05.cu).  All operands bf16, fp32 accumulation in TMEM.
//   a_kmajor / b_kmajor: whether the contraction index is the contiguous one of that operand.
//   C[M,N] (f32 or bf16, pitch ldc) = epilogue(sum_k A(m,k) B(n,k))
struct Tc05Gemm {
    const void* A; int64_t lda; bool a_kmajor;   // A(m,k): kmajor -> A[m*lda+k], else A[k*lda+m]
    const void* B; int64_t ldb; bool b_kmajor;   // B(n,k): kmajor -> B[n*ldb+k], else B[k*ldb+n]
    void* C; int64_t ldc; int c_dtype;
    int M, N, K;
    const float* bias; int act;                  // bias[n] + activation (fwd)
    const void* mask_src; int64_t ldm;           // bf16 [M, ldm]: C *= (mask_src > 0) (dgrad)
    bool b_is_weight = false;                    // B holds layer weights: its tiles may be fetched ahead of the stream dependency
    double* sq_partial = nullptr;                // f32 outputs: every CTA writes the sum of squares of what it stored into its slot
    int sq_slots = 0;                            // must equal codae_tc05_gemm_ctas(ctx, g)
    // fp32-parity mode (CODAE_F32X3): A and B are THREE bf16 planes each (hi, mid, lo: x = hi + mid + lo to 2^-24), plane p at
    // base + p * plane_stride elements; six MMAs per k-step (hh | hm, mh | mm, hl, lh) into three TMEM accumulators by
    // magnitude class, summed in the epilogue.  C is f32 (c_dtype CODAE_F32) or three bf16 planes (c_dtype CODAE_F32X3).
    int planes = 1;
    int64_t a_plane_stride = 0, b_plane_stride = 0, c_plane_stride = 0;
};
bool codae_tc05_supported(const codae_ctx* ctx, const Tc05Gemm& g);
int codae_tc05_gemm(codae_ctx* ctx, const Tc05Gemm& g, cudaStream_t s);
// CTAs codae_tc05_gemm launches for this shape under the context's current options (0: shape not supported).
int codae_tc05_gemm_ctas(const codae_ctx* ctx, const Tc05Gemm& g);
// bf16 tensor map over a row-major [rows, cols] matrix with pitch ld (elements), box {box_cols, box_rows}, 128-byte swizzle,
// out-of-range elements read as zero; planes > 1: a 3-D map {cols, rows, plane} over matrices plane_stride elements apart.
int codae_tc05_make_map(codae_ctx* ctx, CUtensorMap* map, const void* base, long long rows, long long cols, long long ld,
                        int box_cols, int box_rows, int planes, long long plane_stride);

// Candidate pass of the batched top-k (score_tc.cu): one launch = one catalog chunk against query blocks qb0 .. qb0 + G - 1,
// W CTAs per query block.  Every (CTA worker w, query q) keeps a sorted list of kp (bound key, global index) pairs in
// ls / li [W][Q][kp] that persists across launches.  See the header comment of score_tc.cu for the keys.
struct ScoreTcPass {
    int metric;
    const void* cat; int cat_planes;          // 1: the bf16 catalog rows in place; 2: hi / mid bf16 planes of an fp32 chunk
    int64_t cat_ld, cat_plane_stride;
    int64_t n_rows, row0;                     // rows of this chunk, global index of its row 0
    const __nv_bfloat16* q_planes;            // hi / mid planes of the queries [2][Q][q_ld]
    int64_t q_ld, q_plane_stride;
    int Q, E, qb0, G, W, kp;
    const float* cc;                          // [n_rows] row norms of the chunk
    const float* qq;                          // [Q] query norms
    float inv_scale, c_rel;                   // c_rel: relative error bound (score_tc.cu)
    float* ls; int64_t* li;
    const uint8_t* allow;                     // [n_rows] eligibility of the chunk's rows, or NULL (every row)
    const int64_t* exclude; int n_exclude;    // [Q][n_exclude] excluded global indices per query (entries < 0: padding)
};
int codae_score_tc_pass(codae_ctx* ctx, const ScoreTcPass& p, cudaStream_t s);
