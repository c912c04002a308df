// K3 -- complementarity inference: sweep a catalog shard against query vectors staged in shared
// memory, reduce each candidate's score with warp shuffles and keep the best k per query in-kernel.
// HBM-bound: E*sizeof(dtype) bytes per candidate, nothing written per candidate.
// Ordering is the total order (score, index) -> the selected set and its order do not depend on the
// sweep schedule, so results are bit-reproducible and shard-invariant.
#include <float.h>

#include "common.cuh"
#include "gemm.h"

namespace {

constexpr int kWarps = 8;                 // warps per CTA
constexpr int kThreads = kWarps * 32;
constexpr int kMaxK = 128;
constexpr int64_t kEmptyIdx = 0x7fffffffffffffffLL;

// "a is strictly better than b" under the total order; sqerr: smaller score first, cosine: larger first.
template <int METRIC>
__device__ __forceinline__ bool better(float sa, int64_t ia, float sb, int64_t ib) {
    if (METRIC == CODAE_METRIC_SQERR) return sa < sb || (sa == sb && ia < ib);
    return sa > sb || (sa == sb && ia < ib);
}
template <int METRIC>
__device__ __forceinline__ float worst_score() { return METRIC == CODAE_METRIC_SQERR ? INFINITY : -INFINITY; }

// Warp-cooperative sorted insertion into a k-entry list held in shared memory (best first).
// Returns true if the entry made it into the list.  All lanes must call with identical (s, i).
template <int METRIC>
__device__ __forceinline__ bool list_insert(float* ls, int64_t* li, int k, float s, int64_t i, int lane) {
    if (!better<METRIC>(s, i, ls[k - 1], li[k - 1])) return false;
    // position = number of entries strictly better than the new one
    int pos = 0;
    for (int b = 0; b < k; b += 32) {
        const int e = b + lane;
        const bool bt = e < k && better<METRIC>(ls[e], li[e], s, i);
        pos += __popc(__ballot_sync(0xffffffffu, bt));
    }
    // shift [pos, k-1) one slot towards the tail, highest chunk first
    for (int b = ((k - 1) / 32) * 32; b >= 0; b -= 32) {
        const int e = b + lane;
        float ts = 0.f; int64_t ti = 0;
        const bool mv = e > pos && e < k;
        if (mv) { ts = ls[e - 1]; ti = li[e - 1]; }
        __syncwarp();
        if (mv) { ls[e] = ts; li[e] = ti; }
        __syncwarp();
    }
    if (lane == 0) { ls[pos] = s; li[pos] = i; }
    __syncwarp();
    return true;
}

// Filtered instantiations (kFilter): may local row r, global index gi, enter the list of a query with exclusion list
// ex[n_ex]?  Asked only after the candidate has beaten the list's worst entry -- the rare path -- so the mask byte and the
// exclusion list are read from global memory there.  Warp-cooperative: all lanes must call with identical arguments.
__device__ __forceinline__ bool eligible(const uint8_t* __restrict__ allow, int64_t r, const int64_t* __restrict__ ex, int n_ex,
                                         int64_t gi, int lane) {
    if (allow && !allow[r]) return false;
    bool hit = false;
    for (int e = lane; e < n_ex; e += 32) hit |= ex[e] == gi;      // padding (< 0) never equals gi >= 0
    return !__any_sync(0xffffffffu, hit);
}

// The filtered instantiations' insertion: list_insert of an eligible row.  Kept out of line so that the sweep loop around it is
// allocated as in the unfiltered kernels (inlined, the rare path raised the loop's register count and cost up to 1.6x).
template <int METRIC>
__device__ __noinline__ void filtered_insert(float* ls, int64_t* li, int k, float s, int64_t gi, const uint8_t* __restrict__ allow,
                                             int64_t r, const int64_t* __restrict__ ex, int n_ex, int lane) {
    if (eligible(allow, r, ex, n_ex, gi, lane)) list_insert<METRIC>(ls, li, k, s, gi, lane);
}

// R candidate rows against QC queries (smem), partial sums per lane.  All loads of a 256-element (bf16) / 128-element (f32)
// column block of the R rows are issued before the first use: R x 16 bytes (bf16) or R x 16 bytes x 1 (f32, four column blocks
// per unrolled pass) in flight per lane -- a 1 KB bf16 row alone leaves a warp with 2 loads in flight and the sweep at half of
// the HBM rate (measured 0.52 of the copy bandwidth; fp32 rows are twice as long and reached 0.94).
// The per-row arithmetic (order of the FMAs inside a lane, then the shuffle tree) does not depend on R: scores are bit-identical
// to the one-row-at-a-time sweep.
//   SQERR : acc[q] = sum (q_d - c_d*inv_scale)^2 ; COSINE: acc[q] = sum c_d q_d, cc = sum c_d^2
template <int METRIC, int QC, bool kBf16, int R>
__device__ __forceinline__ void rows_partial(const unsigned char* const (&row)[R], int E, const float* __restrict__ qs,
                                             float inv_scale, int lane, float (&acc)[R][QC], float (&cc)[R]) {
#pragma unroll
    for (int j = 0; j < R; ++j) {
        cc[j] = 0.f;
#pragma unroll
        for (int q = 0; q < QC; ++q) acc[j][q] = 0.f;
    }
    if (kBf16) {
        for (int c = lane * 8; c < E; c += 256) {
            uint4 p[R];
#pragma unroll
            for (int j = 0; j < R; ++j) p[j] = ldg_stream_u4(reinterpret_cast<const __nv_bfloat16*>(row[j]) + c);
#pragma unroll
            for (int j = 0; j < R; ++j) {
                const float v[8] = {bf16_lo(p[j].x), bf16_hi(p[j].x), bf16_lo(p[j].y), bf16_hi(p[j].y),
                                    bf16_lo(p[j].z), bf16_hi(p[j].z), bf16_lo(p[j].w), bf16_hi(p[j].w)};
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    if (METRIC == CODAE_METRIC_COSINE) cc[j] = fmaf(v[e], v[e], cc[j]);
#pragma unroll
                    for (int q = 0; q < QC; ++q) {
                        const float qv = qs[q * E + c + e];
                        if (METRIC == CODAE_METRIC_SQERR) { const float d = qv - v[e] * inv_scale; acc[j][q] = fmaf(d, d, acc[j][q]); }
                        else acc[j][q] = fmaf(v[e], qv, acc[j][q]);
                    }
                }
            }
        }
    } else {
        for (int c = lane * 4; c < E; c += 128) {
            float4 p[R];
#pragma unroll
            for (int j = 0; j < R; ++j) p[j] = ldg_stream_f4(reinterpret_cast<const float*>(row[j]) + c);
#pragma unroll
            for (int j = 0; j < R; ++j) {
                const float v[4] = {p[j].x, p[j].y, p[j].z, p[j].w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    if (METRIC == CODAE_METRIC_COSINE) cc[j] = fmaf(v[e], v[e], cc[j]);
#pragma unroll
                    for (int q = 0; q < QC; ++q) {
                        const float qv = qs[q * E + c + e];
                        if (METRIC == CODAE_METRIC_SQERR) { const float d = qv - v[e] * inv_scale; acc[j][q] = fmaf(d, d, acc[j][q]); }
                        else acc[j][q] = fmaf(v[e], qv, acc[j][q]);
                    }
                }
            }
        }
    }
}

// One row (rank mode).
template <int METRIC, int QC, bool kBf16>
__device__ __forceinline__ void row_partial(const void* __restrict__ row, int E, const float* __restrict__ qs, float inv_scale,
                                            int lane, float (&acc)[QC], float& cc) {
    const unsigned char* const rows[1] = {reinterpret_cast<const unsigned char*>(row)};
    float a[1][QC], c1[1];
    rows_partial<METRIC, QC, kBf16, 1>(rows, E, qs, inv_scale, lane, a, c1);
#pragma unroll
    for (int q = 0; q < QC; ++q) acc[q] = a[0][q];
    cc = c1[0];
}

template <int METRIC>
__device__ __forceinline__ float finish_score(float acc, float cc, float qq) {
    if (METRIC == CODAE_METRIC_SQERR) return acc;
    return acc / fmaxf(sqrtf(cc * qq), 1e-8f);
}

// Workspace layout: [grid][QC][k] entries per launch (scores then indices).
// kFilter: allow [n_rows] (NULL: every row) and exclude [QC][n_exclude] global indices of the CTA's queries; a row that fails
// them is treated as absent.  The unfiltered instantiation ignores both.
template <int METRIC, int QC, bool kBf16, bool kFilter>
__global__ void __launch_bounds__(kThreads) score_topk_kernel(const void* __restrict__ catalog, int64_t n_rows, int64_t ld,
                                                              int E, int64_t row_offset, const float* __restrict__ query,
                                                              float inv_scale, int k, float* __restrict__ ws_score,
                                                              int64_t* __restrict__ ws_idx, const uint8_t* __restrict__ allow,
                                                              const int64_t* __restrict__ exclude, int n_exclude) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* qs = reinterpret_cast<float*>(smem_raw);                        // [QC][E]
    float* qq = qs + QC * E;                                               // [QC] |q|^2
    int64_t* li = reinterpret_cast<int64_t*>(qq + ((QC + 3) & ~3));         // [kWarps][QC][k]
    float* ls = reinterpret_cast<float*>(li + kWarps * QC * k);            // [kWarps][QC][k]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int e = threadIdx.x; e < QC * E; e += kThreads) qs[e] = query[e];
    for (int e = threadIdx.x; e < kWarps * QC * k; e += kThreads) { ls[e] = worst_score<METRIC>(); li[e] = kEmptyIdx; }
    __syncthreads();
    if (warp < QC) {
        float s = 0.f;
        for (int c = lane; c < E; c += 32) s = fmaf(qs[warp * E + c], qs[warp * E + c], s);
        s = warp_sum(s);
        if (lane == 0) qq[warp] = s;
    }
    __syncthreads();
    float* my_s = ls + warp * QC * k;
    int64_t* my_i = li + warp * QC * k;
    const size_t esz = kBf16 ? 2 : 4;
    const int64_t wstride = (int64_t)gridDim.x * kWarps;
    // rows per warp pass = independent 16-byte loads per lane and column block (fewer with four queries: register budget)
    constexpr int R = (kBf16 ? 8 : 4) / (QC == 1 ? 1 : 2);
    for (int64_t r = (int64_t)blockIdx.x * kWarps + warp; r < n_rows; r += R * wstride) {
        const unsigned char* row[R];
#pragma unroll
        for (int j = 0; j < R; ++j) {
            const int64_t rj = r + j * wstride;
            row[j] = reinterpret_cast<const unsigned char*>(catalog) + (size_t)(rj < n_rows ? rj : r) * ld * esz;   // tail: re-read row r, result unused
        }
        float acc[R][QC], cc[R];
        rows_partial<METRIC, QC, kBf16, R>(row, E, qs, inv_scale, lane, acc, cc);
        // R x QC independent shuffle trees: the compiler interleaves them
#pragma unroll
        for (int j = 0; j < R; ++j) {
            if (METRIC == CODAE_METRIC_COSINE) cc[j] = warp_sum(cc[j]);
#pragma unroll
            for (int q = 0; q < QC; ++q) acc[j][q] = warp_sum(acc[j][q]);
        }
#pragma unroll
        for (int j = 0; j < R; ++j) {
            const int64_t rj = r + j * wstride;
            if (rj >= n_rows) break;
#pragma unroll
            for (int q = 0; q < QC; ++q) {
                const float s = finish_score<METRIC>(acc[j][q], cc[j], qq[q]);
                if constexpr (!kFilter) {
                    if (s == s) list_insert<METRIC>(my_s + q * k, my_i + q * k, k, s, row_offset + rj, lane);  // NaN never ranks
                } else if (s == s && better<METRIC>(s, row_offset + rj, my_s[q * k + k - 1], my_i[q * k + k - 1])) {
                    filtered_insert<METRIC>(my_s + q * k, my_i + q * k, k, s, row_offset + rj, allow, rj,
                                            exclude + (int64_t)q * n_exclude, n_exclude, lane);
                }
            }
        }
    }
    __syncthreads();
    // CTA merge: warp w (< QC) folds the lists of query w from all warps; sorted inputs -> stop at first reject
    for (int q = warp; q < QC; q += kWarps) {
        float* dst_s = ls + q * k;            // warp 0's list of query q
        int64_t* dst_i = li + q * k;
        for (int w = 1; w < kWarps; ++w) {
            const float* src_s = ls + (w * QC + q) * k;
            const int64_t* src_i = li + (w * QC + q) * k;
            for (int e = 0; e < k; ++e) {
                if (src_i[e] == kEmptyIdx) break;
                if (!list_insert<METRIC>(dst_s, dst_i, k, src_s[e], src_i[e], lane)) break;
            }
        }
        for (int e = lane; e < k; e += 32) {
            ws_score[((int64_t)blockIdx.x * QC + q) * k + e] = dst_s[e];
            ws_idx[((int64_t)blockIdx.x * QC + q) * k + e] = dst_i[e];
        }
    }
}

// Merge `n_lists` sorted k-lists per query (layout [n_lists][Q][k]) into out [Q][k].  One CTA per query;
// every warp folds a strided subset of the lists, then warp 0 folds the per-warp results.
// A warp first copies its lists into shared memory with all lanes loading (hundreds of independent loads in flight), then
// folds them from there: folding straight from global memory is a chain of dependent ~0.6 us loads per list (measured 48.9 us
// for the 592 lists of one sweep).
constexpr int kMergeStage = 1024;          // entries per warp staged per pass (12 KB)
inline size_t merge_smem() { return (size_t)kWarps * kMergeStage * 12; }
template <int METRIC>
__global__ void __launch_bounds__(kThreads) topk_merge_kernel(const float* __restrict__ in_s, const int64_t* __restrict__ in_i,
                                                              int n_lists, int Q, int k, float* __restrict__ out_s,
                                                              int64_t* __restrict__ out_i, int q_out_offset, int q_out_stride) {
    __shared__ float ls[kWarps][kMaxK];
    __shared__ int64_t li[kWarps][kMaxK];
    extern __shared__ __align__(16) unsigned char merge_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, q = blockIdx.x;
    int64_t* st_i = reinterpret_cast<int64_t*>(merge_raw) + warp * kMergeStage;
    float* st_s = reinterpret_cast<float*>(merge_raw + (size_t)kWarps * kMergeStage * 8) + warp * kMergeStage;
    for (int e = lane; e < k; e += 32) { ls[warp][e] = worst_score<METRIC>(); li[warp][e] = kEmptyIdx; }
    __syncwarp();
    const int per_pass = kMergeStage / k;                              // lists per pass (k <= 128 -> at least 8)
    const int mine = n_lists > warp ? (n_lists - warp + kWarps - 1) / kWarps : 0;    // lists warp, warp + kWarps, ...
    for (int j0 = 0; j0 < mine; j0 += per_pass) {
        const int nl = min(per_pass, mine - j0);
        for (int t = lane; t < nl * k; t += 32) {
            const int j = t / k, e = t - j * k;
            const int64_t src = ((int64_t)(warp + (j0 + j) * kWarps) * Q + q) * k + e;
            st_s[t] = in_s[src];
            st_i[t] = in_i[src];
        }
        __syncwarp();
        for (int j = 0; j < nl; ++j)
            for (int e = 0; e < k; ++e) {
                const int64_t ii = st_i[j * k + e];
                if (ii == kEmptyIdx || ii < 0) break;
                if (!list_insert<METRIC>(ls[warp], li[warp], k, st_s[j * k + e], ii, lane)) break;
            }
        __syncwarp();
    }
    __syncthreads();
    if (warp == 0) {
        for (int w = 1; w < kWarps; ++w)
            for (int e = 0; e < k; ++e) {
                if (li[w][e] == kEmptyIdx) break;
                if (!list_insert<METRIC>(ls[0], li[0], k, ls[w][e], li[w][e], lane)) break;
            }
        const int qo = q_out_offset + q * q_out_stride;
        for (int e = lane; e < k; e += 32) {
            const bool empty = li[0][e] == kEmptyIdx;
            out_s[(int64_t)qo * k + e] = ls[0][e];
            out_i[(int64_t)qo * k + e] = empty ? -1 : li[0][e];
        }
    }
}

inline void merge_attrs() {      // the staging buffers need the opt-in shared-memory size (once per process)
    static const bool done = (cudaFuncSetAttribute(topk_merge_kernel<CODAE_METRIC_SQERR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)merge_smem()),
                              cudaFuncSetAttribute(topk_merge_kernel<CODAE_METRIC_COSINE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)merge_smem()), true);
    (void)done;
}

// Rank mode: s_true[q] = score(query q, row true_idx[q]); out_rank[q] = #{j in subset : s_true[q] better-than s_q[j]}.
template <int METRIC, bool kBf16>
__global__ void __launch_bounds__(kThreads) score_rank_kernel(const void* __restrict__ catalog, int64_t n_rows, int64_t ld,
                                                              int E, const float* __restrict__ query, int Q, float inv_scale,
                                                              const int64_t* __restrict__ true_idx,
                                                              const int64_t* __restrict__ subset, int64_t n_subset,
                                                              unsigned long long* __restrict__ out_rank) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* s_true = reinterpret_cast<float*>(smem_raw);     // [Q]
    float* qq = s_true + Q;                                 // [Q]
    int* cnt = reinterpret_cast<int*>(qq + Q);              // [Q]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t esz = kBf16 ? 2 : 4;
    for (int q = threadIdx.x; q < Q; q += kThreads) cnt[q] = 0;
    for (int q = warp; q < Q; q += kWarps) {
        float s = 0.f;
        for (int c = lane; c < E; c += 32) { const float v = query[(int64_t)q * E + c]; s = fmaf(v, v, s); }
        s = warp_sum(s);
        float acc[1], cc;
        row_partial<METRIC, 1, kBf16>(reinterpret_cast<const unsigned char*>(catalog) + (size_t)true_idx[q] * ld * esz, E,
                                      query + (int64_t)q * E, inv_scale, lane, acc, cc);
        if (METRIC == CODAE_METRIC_COSINE) cc = warp_sum(cc);
        const float st = finish_score<METRIC>(warp_sum(acc[0]), cc, s);
        if (lane == 0) { qq[q] = s; s_true[q] = st; }
    }
    __syncthreads();
    const int64_t wstride = (int64_t)gridDim.x * kWarps;
    for (int64_t t = (int64_t)blockIdx.x * kWarps + warp; t < n_subset; t += wstride) {
        const int64_t r = subset ? subset[t] : t;
        const unsigned char* row = reinterpret_cast<const unsigned char*>(catalog) + (size_t)r * ld * esz;
        for (int q = 0; q < Q; ++q) {
            float acc[1], cc;
            row_partial<METRIC, 1, kBf16>(row, E, query + (int64_t)q * E, inv_scale, lane, acc, cc);
            if (METRIC == CODAE_METRIC_COSINE) cc = warp_sum(cc);
            const float s = finish_score<METRIC>(warp_sum(acc[0]), cc, qq[q]);
            const bool b = METRIC == CODAE_METRIC_SQERR ? (s_true[q] < s) : (s_true[q] > s);
            if (lane == 0 && b) atomicAdd(&cnt[q], 1);
        }
    }
    __syncthreads();
    for (int q = threadIdx.x; q < Q; q += kThreads)
        if (cnt[q]) atomicAdd(&out_rank[q], (unsigned long long)cnt[q]);
}

// ---- rank mode for large query batches: the Q x n dot products come from the fp32-parity tensor-core GEMM ---------------------
// RankingLoss.get runs for every validation batch (train_dae_on_embedding.py:241-261; metering.py:46-79).  For Q >= 64 queries of
// one category the dot products q . c_j are one [Q, E] x [E, n] contraction (codae_linear_fwd_x3: fp32 fidelity on tensor cores);
// these two kernels supply the norms and turn the score matrix into ranks.
//   row_sqnorm_kernel  out[r] = sum_d X[r, d]^2                  (warp per row, fixed shuffle tree)
//   rank_count_kernel  out_rank[q] = #{ j < n : cos(q, true_q) > cos(q, c_j) } with cos = dot / max(sqrt(|c|^2 |q|^2), 1e-8),
//                      dot(q, true_q) = scores[q, n + q] (the true rows are appended to the catalog operand so that a true item
//                      that is itself in the subset gets bit-identical scores on both sides of the strict comparison)
//                      (T = __nv_bfloat16: the row norms of a bf16 catalog for the batched top-k)
template <typename T>
__global__ void __launch_bounds__(kThreads) row_sqnorm_kernel(const T* __restrict__ X, int64_t ld, int64_t rows, int E,
                                                              float* __restrict__ out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t r = (int64_t)blockIdx.x * kWarps + warp; r < rows; r += (int64_t)gridDim.x * kWarps) {
        const T* row = X + r * ld;
        float s = 0.f;
        for (int c = lane; c < E; c += 32) { const float v = (float)row[c]; s = fmaf(v, v, s); }
        s = warp_sum(s);
        if (lane == 0) out[r] = s;
    }
}

__global__ void __launch_bounds__(kThreads) rank_count_kernel(const float* __restrict__ scores, int64_t ld, int Q, int64_t n,
                                                              const float* __restrict__ cc, const float* __restrict__ qq,
                                                              unsigned long long* __restrict__ out_rank) {
    __shared__ unsigned int part[kWarps];
    const int q = blockIdx.y;
    const float* row = scores + (int64_t)q * ld;
    const float nq = qq[q];
    const float s_true = row[n + q] / fmaxf(sqrtf(cc[n + q] * nq), 1e-8f);
    unsigned int cnt = 0;
    for (int64_t j = (int64_t)blockIdx.x * kThreads + threadIdx.x; j < n; j += (int64_t)gridDim.x * kThreads) {
        const float s = row[j] / fmaxf(sqrtf(cc[j] * nq), 1e-8f);
        cnt += (s_true > s) ? 1u : 0u;
    }
    cnt = warp_sum(cnt);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int t = 0;
        for (int w = 0; w < kWarps; ++w) t += part[w];
        if (t) atomicAdd(&out_rank[q], (unsigned long long)t);      // integer counts: order-independent
    }
}

// ---- batched top-k: tensor-core proposals (score_tc.cu), certified here with the sweep's own arithmetic -------------------
// hi / mid bf16 planes of fp32 rows (pitch `pitch`, columns E .. pitch - 1 zero): the A operand (queries) and, chunk by chunk, the
// B operand of an fp32 catalog.  A padded pitch (multiple of 8 elements) keeps every plane row a whole number of 16-byte units,
// which the tensor maps need; codae_split_x3 writes unpadded rows.
__global__ void __launch_bounds__(kThreads) split_hm_kernel(const float* __restrict__ src, int64_t ld, int64_t rows, int E,
                                                            __nv_bfloat16* __restrict__ dst, int64_t pitch, int64_t plane) {
    const int64_t total = rows * pitch;
    for (int64_t e = (int64_t)blockIdx.x * kThreads + threadIdx.x; e < total; e += (int64_t)gridDim.x * kThreads) {
        const int64_t r = e / pitch;
        const int c = (int)(e - r * pitch);
        float h = 0.f, m = 0.f, l;
        if (c < E) split3(src[r * ld + c], h, m, l);
        dst[e] = __float2bfloat16_rn(h);
        dst[plane + e] = __float2bfloat16_rn(m);
    }
}

template <int METRIC>
__global__ void __launch_bounds__(kThreads) list_init_kernel(float* __restrict__ ls, int64_t* __restrict__ li, int64_t n) {
    for (int64_t e = (int64_t)blockIdx.x * kThreads + threadIdx.x; e < n; e += (int64_t)gridDim.x * kThreads) {
        ls[e] = worst_score<METRIC>();
        li[e] = kEmptyIdx;
    }
}

// One CTA per query.  The merged proposal list of query q holds the kp best (bound key, index) pairs of the whole shard; every
// row outside it has key >= the worst key b_w (SQERR; <= for COSINE) and, by the bound, an exact score no better than its key.
// Re-score the kp rows exactly as score_topk_kernel does (query in shared memory, rows_partial, warp_sum tree, the same qq,
// finish_score, NaN never ranks), keep the best k under (score, index), and CERTIFY the query when the exact k-th score is
// strictly better than b_w -- then no outside row can enter -- or when the list holds every row of the shard.  Uncertified
// queries are appended to uncert[] (count in *n_uncert); their outputs are written but unspecified.
// Filtered calls need nothing here: the candidate pass proposes eligible rows only, so every proposal is eligible.  A row outside
// the merged list is either ineligible, or had a key no better than its worker's threshold when it was seen -- and thresholds
// only improve -- so the b_w test still bounds every eligible row left out.  A list with an empty slot (iw < 0) or a shard of at
// most kp rows still means that every eligible row was proposed.
template <int METRIC, bool kBf16>
__global__ void __launch_bounds__(kThreads) score_certify_kernel(const void* __restrict__ catalog, int64_t n_rows, int64_t ld, int E,
                                                                 int64_t row_offset, const float* __restrict__ query, float inv_scale,
                                                                 int k, int kp, const float* __restrict__ m_key,
                                                                 const int64_t* __restrict__ m_idx, float* __restrict__ out_score,
                                                                 int64_t* __restrict__ out_idx, int* __restrict__ n_uncert,
                                                                 int* __restrict__ uncert) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int64_t* ex_i = reinterpret_cast<int64_t*>(smem_raw);          // [kp] exact scores of the proposals
    int64_t* li = ex_i + kp;                                        // [k]  best k
    float* qs = reinterpret_cast<float*>(li + k);                   // [E]
    float* ex_s = qs + E;                                           // [kp]
    float* ls = ex_s + kp;                                          // [k]
    float* qq = ls + k;                                             // [1]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, q = blockIdx.x;
    for (int e = threadIdx.x; e < E; e += kThreads) qs[e] = query[(int64_t)q * E + e];
    for (int e = threadIdx.x; e < k; e += kThreads) { ls[e] = worst_score<METRIC>(); li[e] = kEmptyIdx; }
    __syncthreads();
    if (warp == 0) {
        float s = 0.f;
        for (int c = lane; c < E; c += 32) s = fmaf(qs[c], qs[c], s);
        s = warp_sum(s);
        if (lane == 0) qq[0] = s;
    }
    __syncthreads();
    const size_t esz = kBf16 ? 2 : 4;
    for (int e = warp; e < kp; e += kWarps) {
        const int64_t gi = m_idx[(int64_t)q * kp + e];
        float s = 0.f;
        if (gi >= 0) {
            float acc[1], cc;
            row_partial<METRIC, 1, kBf16>(reinterpret_cast<const unsigned char*>(catalog) + (size_t)(gi - row_offset) * ld * esz, E, qs,
                                          inv_scale, lane, acc, cc);
            if (METRIC == CODAE_METRIC_COSINE) cc = warp_sum(cc);
            s = finish_score<METRIC>(warp_sum(acc[0]), cc, qq[0]);
        }
        if (lane == 0) { ex_s[e] = s; ex_i[e] = (gi >= 0 && s == s) ? gi : kEmptyIdx; }    // NaN never ranks
    }
    __syncthreads();
    if (warp != 0) return;
    for (int e = 0; e < kp; ++e)
        if (ex_i[e] != kEmptyIdx) list_insert<METRIC>(ls, li, k, ex_s[e], ex_i[e], lane);
    const float bw = m_key[(int64_t)q * kp + kp - 1];
    const int64_t iw = m_idx[(int64_t)q * kp + kp - 1];
    bool cert = n_rows <= kp || iw < 0;             // the list holds every row of the shard
    if (!cert) cert = li[k - 1] != kEmptyIdx && (METRIC == CODAE_METRIC_SQERR ? ls[k - 1] < bw : ls[k - 1] > bw);
    for (int e = lane; e < k; e += 32) {
        out_score[(int64_t)q * k + e] = ls[e];
        out_idx[(int64_t)q * k + e] = li[e] == kEmptyIdx ? -1 : li[e];
    }
    if (!cert && lane == 0) uncert[atomicAdd(n_uncert, 1)] = q;
}

// Proposal list length k' (> k, <= the merge's 128) and relative error bound (derivation: score_tc.cu).
inline int batched_kp(int k) { return 2 * k + 32 < kMaxK ? 2 * k + 32 : kMaxK; }
inline float batched_c_rel(int E, bool bf16_catalog) {
    const double P = bf16_catalog ? 2 : 3;
    const double c = ldexp(1.0, -14) + (P * ((E + 15) / 16) + 8) * ldexp(1.0, -21) + (E / 32.0 + 16) * ldexp(1.0, -21);
    return (float)(c * (1 + ldexp(1.0, -10)));
}
constexpr int kTcTileM = 128;              // queries per tensor-core tile
// Rows of one catalog chunk: bf16 catalogs are read in place (the chunk only bounds the row-norm buffer), fp32 chunks are split
// into two bf16 planes of 2 * rows * pitch elements -- at most 512 MB of scratch.
inline int64_t batched_chunk_rows(bool bf16_catalog, int64_t pitch) {
    if (bf16_catalog) return (int64_t)1 << 24;
    const int64_t r = (((int64_t)1 << 27) / pitch) & ~(int64_t)255;
    return r < 256 ? 256 : r;
}
struct BatchedLayout {         // workspace of codae_score_topk_batched, in this order, each part 256-byte aligned
    int kp, W, G0, QB;
    int64_t pitch, chunk, crow;   // crow: rows of the largest chunk (the row-norm and plane buffers hold that many)
    size_t m_key, m_idx, ls, li, cc, qq, qplanes, cplanes, total;
};
inline size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }
inline BatchedLayout batched_layout(const codae_ctx* ctx, bool bf, int64_t n_rows, int E, int Q, int k) {
    BatchedLayout L;
    L.kp = batched_kp(k);
    L.QB = (Q + kTcTileM - 1) / kTcTileM;
    L.G0 = L.QB < ctx->sm_count ? L.QB : ctx->sm_count;
    L.W = ctx->sm_count / L.G0;
    L.pitch = (E + 7) & ~7;
    L.chunk = batched_chunk_rows(bf, L.pitch);
    const int64_t crow = L.crow = n_rows < L.chunk ? (n_rows > 0 ? n_rows : 1) : L.chunk;
    const size_t lists = (size_t)L.W * Q * L.kp;
    size_t o = 0;
    L.m_key = o; o = al256(o + (size_t)Q * L.kp * 4);
    L.m_idx = o; o = al256(o + (size_t)Q * L.kp * 8);
    L.ls = o;    o = al256(o + lists * 4);
    L.li = o;    o = al256(o + lists * 8);
    L.cc = o;    o = al256(o + (size_t)crow * 4);
    L.qq = o;    o = al256(o + (size_t)Q * 4);
    L.qplanes = o; o = al256(o + (size_t)2 * Q * L.pitch * 2);
    L.cplanes = o; if (!bf) o = al256(o + (size_t)2 * crow * L.pitch * 2);
    L.total = o + 256;
    return L;
}

// ---- candidate SWAPS scored by full reconstruction error --------------------------------------------------------
// Second reading of "scores candidate item swaps by reconstruction error": put candidate j into slot c of the outfit, run
// the DAE on the swapped outfit (the tensor-core GEMMs, batched over candidates) and score the swap by
// || DAE(outfit_j) - outfit_j ||^2 over all io dimensions.  Two small kernels bracket the forward pass:
//   swap_build_kernel      x'[b, :] = outfit with columns [slot*E, (slot+1)*E) replaced by catalog[first_row + b] * inv_scale
//   swap_error_topk_kernel err_b = sum_d (y[b, d] - x'[b, d])^2 (x' recomputed in fp32), best k per CTA, then topk_merge_kernel
template <bool kBf16Cat, bool kBf16Out>
__global__ void __launch_bounds__(256) swap_build_kernel(const float* __restrict__ outfit, const void* __restrict__ catalog,
                                                         int64_t ld_cat, int64_t first_row, int B, int E, int slot, int io,
                                                         float inv_scale, void* __restrict__ out, int64_t ld_out) {
    const int64_t total = (int64_t)B * io;
    const int lo = slot * E, hi = lo + E;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int b = (int)(e / io), d = (int)(e - (int64_t)b * io);
        float v;
        if (d >= lo && d < hi) {
            const int64_t off = (first_row + b) * ld_cat + (d - lo);
            v = (kBf16Cat ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(catalog)[off])
                          : reinterpret_cast<const float*>(catalog)[off]) * inv_scale;
        } else {
            v = outfit[d];
        }
        if (kBf16Out) reinterpret_cast<__nv_bfloat16*>(out)[(int64_t)b * ld_out + d] = __float2bfloat16_rn(v);
        else reinterpret_cast<float*>(out)[(int64_t)b * ld_out + d] = v;
    }
}

// Swap error of built row b: sum_d (y[b, d] - x'_d)^2 with x' recomputed in fp32 from the outfit and catalog row first_row + b
// (lane-strided fmaf over io, then the warp_sum tree).  The one definition of a swap's error: codae_swap_error_topk and
// codae_swap_error_pairs both call it, so a pair's error equals the row sweep's bit for bit whenever the GEMM chain computed the
// same y row.  The row is passed as (first_row, b) because that is how swap_error_topk_kernel indexed it before this helper existed:
// written so, the kernel keeps its SASS opcode sequence (profiles/r05_sass_swap_error.jsonl).
template <bool kBf16Cat>
__device__ __forceinline__ float swap_row_error(const float* __restrict__ outfit, const void* __restrict__ catalog, int64_t ld_cat,
                                                int64_t first_row, int lo, int hi, int io, float inv_scale, const float* __restrict__ y,
                                                int64_t ld_y, int b, int lane) {
    float acc = 0.f;
    for (int d = lane; d < io; d += 32) {
        float t;
        if (d >= lo && d < hi) {
            const int64_t off = (first_row + b) * ld_cat + (d - lo);
            t = (kBf16Cat ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(catalog)[off])
                          : reinterpret_cast<const float*>(catalog)[off]) * inv_scale;
        } else {
            t = outfit[d];
        }
        const float df = y[(int64_t)b * ld_y + d] - t;
        acc = fmaf(df, df, acc);
    }
    return warp_sum(acc);
}

// kFilter: allow indexed by catalog row (first_row + b), exclude [n_exclude] global indices, as in score_topk_kernel.
template <bool kBf16Cat, bool kFilter>
__global__ void __launch_bounds__(kThreads) swap_error_topk_kernel(const float* __restrict__ outfit, const void* __restrict__ catalog,
                                                                   int64_t ld_cat, int64_t first_row, int B, int E, int slot, int io,
                                                                   float inv_scale, const float* __restrict__ y, int64_t ld_y,
                                                                   int64_t row_offset, int k, float* __restrict__ ws_score,
                                                                   int64_t* __restrict__ ws_idx, const uint8_t* __restrict__ allow,
                                                                   const int64_t* __restrict__ exclude, int n_exclude) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int64_t* li = reinterpret_cast<int64_t*>(smem_raw);                    // [kWarps][k]
    float* ls = reinterpret_cast<float*>(li + kWarps * k);                 // [kWarps][k]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int e = threadIdx.x; e < kWarps * k; e += kThreads) { ls[e] = INFINITY; li[e] = kEmptyIdx; }
    __syncthreads();
    const int lo = slot * E, hi = lo + E;
    for (int b = blockIdx.x * kWarps + warp; b < B; b += gridDim.x * kWarps) {
        const float acc = swap_row_error<kBf16Cat>(outfit, catalog, ld_cat, first_row, lo, hi, io, inv_scale, y, ld_y, b, lane);
        if constexpr (!kFilter) {
            if (acc == acc) list_insert<CODAE_METRIC_SQERR>(ls + warp * k, li + warp * k, k, acc, row_offset + first_row + b, lane);
        } else {
            const int64_t gi = row_offset + first_row + b;
            if (acc == acc && better<CODAE_METRIC_SQERR>(acc, gi, ls[warp * k + k - 1], li[warp * k + k - 1]))
                filtered_insert<CODAE_METRIC_SQERR>(ls + warp * k, li + warp * k, k, acc, gi, allow, first_row + b, exclude, n_exclude,
                                                    lane);
        }
    }
    __syncthreads();
    if (warp == 0) {
        for (int w = 1; w < kWarps; ++w)
            for (int e = 0; e < k; ++e) {
                if (li[w * k + e] == kEmptyIdx) break;
                if (!list_insert<CODAE_METRIC_SQERR>(ls, li, k, ls[w * k + e], li[w * k + e], lane)) break;
            }
        for (int e = lane; e < k; e += 32) {
            ws_score[(int64_t)blockIdx.x * k + e] = ls[e];
            ws_idx[(int64_t)blockIdx.x * k + e] = li[e];
        }
    }
}

// ---- swaps over per-outfit candidate lists (re-ranking) -------------------------------------------------------------------
// The list is candidates [Q][m] (global row ids, < 0 padding), flattened to pairs p = q * m + j.  A chunk of B built rows takes
// its pairs from pos [B] (indices into the flattened list).  Row b is valid when 0 <= pos[b] < Q m and its local catalog row
// candidates[pos[b]] - row_offset lies in [0, n_rows); an invalid row is built as zeros and gets no error, so device-side ids and
// positions are never dereferenced out of range.
__device__ __forceinline__ bool pair_row(const int64_t* __restrict__ pos, const int64_t* __restrict__ candidates, int64_t n_pairs,
                                         int m, int64_t n_rows, int64_t row_offset, int b, int64_t& p, int64_t& q, int64_t& r) {
    p = pos[b];
    if (p < 0 || p >= n_pairs) return false;
    q = p / m;
    r = candidates[p] - row_offset;
    return r >= 0 && r < n_rows;
}

//   swap_build_pairs_kernel   x'[b, :] = outfit q with columns [slot*E, (slot+1)*E) replaced by catalog row r * inv_scale --
//                             swap_build_kernel's values, gathered per pair.  V = 4: four columns per thread, the outfit read with
//                             one 16-byte load (io, E, ld_outfit multiples of 4 and a 16-byte aligned outfit base).
template <bool kBf16Cat, bool kBf16Out, int V>
__global__ void __launch_bounds__(256) swap_build_pairs_kernel(const float* __restrict__ outfits, int64_t ld_outfit, int64_t n_pairs,
                                                               const void* __restrict__ catalog, int64_t ld_cat, int64_t n_rows,
                                                               int64_t row_offset, const int64_t* __restrict__ candidates, int m,
                                                               const int64_t* __restrict__ pos, int B, int E, int slot, int io,
                                                               float inv_scale, void* __restrict__ out, int64_t ld_out) {
    const int per_row = io / V;
    const int64_t total = (int64_t)B * per_row;
    const int lo = slot * E, hi = lo + E;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int b = (int)(e / per_row), d0 = (int)(e - (int64_t)b * per_row) * V;
        int64_t p, q, r;
        float v[V];
        if (!pair_row(pos, candidates, n_pairs, m, n_rows, row_offset, b, p, q, r)) {
#pragma unroll
            for (int j = 0; j < V; ++j) v[j] = 0.f;
        } else if (d0 >= lo && d0 < hi) {           // V divides E: the V columns are all inside the slot or all outside
            const int64_t off = r * ld_cat + (d0 - lo);
#pragma unroll
            for (int j = 0; j < V; ++j)
                v[j] = (kBf16Cat ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(catalog)[off + j])
                                 : reinterpret_cast<const float*>(catalog)[off + j]) * inv_scale;
        } else if constexpr (V == 4) {
            const float4 o = *reinterpret_cast<const float4*>(outfits + q * ld_outfit + d0);
            v[0] = o.x; v[1] = o.y; v[2] = o.z; v[3] = o.w;
        } else {
            v[0] = outfits[q * ld_outfit + d0];
        }
#pragma unroll
        for (int j = 0; j < V; ++j) {
            if (kBf16Out) reinterpret_cast<__nv_bfloat16*>(out)[(int64_t)b * ld_out + d0 + j] = __float2bfloat16_rn(v[j]);
            else reinterpret_cast<float*>(out)[(int64_t)b * ld_out + d0 + j] = v[j];
        }
    }
}

//   swap_error_pairs_kernel   err[p] = swap_row_error of built row b (one warp per row, as swap_error_topk_kernel)
template <bool kBf16Cat>
__global__ void __launch_bounds__(kThreads) swap_error_pairs_kernel(const float* __restrict__ outfits, int64_t ld_outfit,
                                                                    int64_t n_pairs, const void* __restrict__ catalog, int64_t ld_cat,
                                                                    int64_t n_rows, int64_t row_offset,
                                                                    const int64_t* __restrict__ candidates, int m,
                                                                    const int64_t* __restrict__ pos, int B, int E, int slot, int io,
                                                                    float inv_scale, const float* __restrict__ y, int64_t ld_y,
                                                                    float* __restrict__ err) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int lo = slot * E, hi = lo + E;
    for (int b = blockIdx.x * kWarps + warp; b < B; b += gridDim.x * kWarps) {
        int64_t p, q, r;
        if (!pair_row(pos, candidates, n_pairs, m, n_rows, row_offset, b, p, q, r)) continue;
        const float acc = swap_row_error<kBf16Cat>(outfits + q * ld_outfit, catalog, ld_cat, r - b /* row r */, lo, hi, io, inv_scale,
                                                   y, ld_y, b, lane);
        if (lane == 0) err[p] = acc;
    }
}

//   swap_pairs_topk_kernel    one warp per outfit: the best k of err[q][0..m) by (error, candidate id) in a shared-memory list
//                             (list_insert of the sweep: the same ties; NaN -- unscored -- entries and ids < 0 never rank)
__global__ void __launch_bounds__(kThreads) swap_pairs_topk_kernel(const float* __restrict__ err, const int64_t* __restrict__ candidates,
                                                                   int Q, int m, int k, float* __restrict__ out_score,
                                                                   int64_t* __restrict__ out_idx) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int64_t* li = reinterpret_cast<int64_t*>(smem_raw) + warp * k;                       // [kWarps][k]
    float* ls = reinterpret_cast<float*>(reinterpret_cast<int64_t*>(smem_raw) + kWarps * k) + warp * k;
    const int q = blockIdx.x * kWarps + warp;
    if (q >= Q) return;
    for (int e = lane; e < k; e += 32) { ls[e] = INFINITY; li[e] = kEmptyIdx; }
    __syncwarp();
    const float* es = err + (int64_t)q * m;
    const int64_t* ci = candidates + (int64_t)q * m;
    for (int j0 = 0; j0 < m; j0 += 32) {
        const int n = m - j0 < 32 ? m - j0 : 32;
        float s_l = NAN;
        int64_t i_l = -1;
        if (lane < n) { s_l = es[j0 + lane]; i_l = ci[j0 + lane]; }
        for (int j = 0; j < n; ++j) {
            const float s = __shfl_sync(0xffffffffu, s_l, j);
            const int64_t i = __shfl_sync(0xffffffffu, i_l, j);
            if (s == s && i >= 0) list_insert<CODAE_METRIC_SQERR>(ls, li, k, s, i, lane);
        }
    }
    for (int e = lane; e < k; e += 32) {
        out_score[(int64_t)q * k + e] = ls[e];
        out_idx[(int64_t)q * k + e] = li[e] == kEmptyIdx ? -1 : li[e];
    }
}

// ---- outfit compatibility: leave-one-slot-out reconstruction errors ------------------------------------------------------
// The reconstructions y come slot-major: row s * Q + i is outfit i with slot s multiplied by 0 (codae_corrupt_fwd, run s).
//   outfit_loo_error_kernel  one warp per outfit: err[i, s] = sum_{d < E} (y[s Q + i, s E + d] - outfits[i, s E + d])^2 (lane-strided
//                            fmaf, then the warp_sum tree), score[i] = err[i, 0] + err[i, 1] + ... in slot order, odd[i] = the first
//                            slot of largest error; a NaN error makes score NaN and odd -1.  An outfit holding a NaN or inf gets NaN
//                            errors throughout: the GEMM epilogue's ReLU (fmaxf) turns NaN into 0, so its reconstructions can be finite
//                            and meaningless.
__global__ void __launch_bounds__(kThreads) outfit_loo_error_kernel(const float* __restrict__ outfits, int64_t ld_outfit, int Q, int S,
                                                                    int E, const float* __restrict__ y, int64_t ld_y,
                                                                    float* __restrict__ err, float* __restrict__ score,
                                                                    int64_t* __restrict__ odd) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = blockIdx.x * kWarps + warp; i < Q; i += gridDim.x * kWarps) {
        const float* x = outfits + (int64_t)i * ld_outfit;
        float sum = 0.f, best = -INFINITY;
        int arg = 0;
        bool nan = false, nonfinite = false;
        for (int s = 0; s < S; ++s) {
            const float* yr = y + ((int64_t)s * Q + i) * ld_y + (int64_t)s * E;
            const float* xr = x + (int64_t)s * E;
            float acc = 0.f;
            for (int d = lane; d < E; d += 32) {
                const float xv = xr[d];
                nonfinite |= !isfinite(xv);
                const float df = yr[d] - xv;
                acc = fmaf(df, df, acc);
            }
            acc = warp_sum(acc);
            if (lane == 0) err[(int64_t)i * S + s] = acc;
            sum += acc;
            if (acc != acc) nan = true;
            else if (acc > best) { best = acc; arg = s; }
        }
        nonfinite = __any_sync(0xffffffffu, nonfinite);
        if (lane == 0) {
            if (nonfinite)
                for (int s = 0; s < S; ++s) err[(int64_t)i * S + s] = NAN;
            score[i] = nan || nonfinite ? NAN : sum;
            odd[i] = nan || nonfinite ? -1 : arg;
        }
    }
}

// ---- outfit completion: every missing slot filled together, each combination scored by swap error -------------------------
// Combination p of the flattened [Q, C] grid (include/codae_b200.h: outfit completion) -- the one decode and validity rule of both
// completion kernels.  Returns whether p is valid and sets q and, in row, the pool row that slot `want` takes (-1 for a given slot).
// The j-th missing slot of outfit q (ascending slot order) takes digit (c / depth^j) % depth; c < depth^m_q exactly when nothing of
// c is left after m_q digits.  Every pool row the combination takes is checked before any of it is read.
__device__ __forceinline__ bool complete_row(const int64_t* __restrict__ pos, const int64_t* __restrict__ slot_base,
                                             const int64_t* __restrict__ pool_id, int64_t n_pool, int Q, int S, int depth, int C,
                                             int b, int want, int64_t& p, int64_t& q, int64_t& row) {
    p = pos[b];
    row = -1;
    if (p < 0 || p >= (int64_t)Q * C) return false;
    q = p / C;
    int c = (int)(p - q * C);
    const int64_t* sb = slot_base + q * S;
    for (int s = 0; s < S; ++s) {
        const int64_t base = sb[s];
        if (base < 0) continue;
        const int digit = c % depth;
        c /= depth;
        if (base >= n_pool || digit >= n_pool - base) return false;
        if (pool_id[base + digit] < 0) return false;
        if (s == want) row = base + digit;
    }
    return c == 0;
}

//   complete_build_kernel   x'[b, :] = outfit q with each missing slot replaced by its pool row * inv_scale (swap_build_pairs_kernel's
//                           values for one missing slot).  V = 4: four columns per thread, the outfit read with one 16-byte load (E,
//                           ld_outfit multiples of 4 and a 16-byte aligned outfit base).
template <bool kBf16Out, int V>
__global__ void __launch_bounds__(256) complete_build_kernel(const float* __restrict__ outfits, int64_t ld_outfit, int Q, int S, int E,
                                                             const int64_t* __restrict__ slot_base, const float* __restrict__ pool,
                                                             int64_t ld_pool, int64_t n_pool, const int64_t* __restrict__ pool_id,
                                                             int depth, int C, const int64_t* __restrict__ pos, int B, float inv_scale,
                                                             void* __restrict__ out, int64_t ld_out) {
    const int per_row = S * E / V;
    const int64_t total = (int64_t)B * per_row;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int b = (int)(e / per_row), d0 = (int)(e - (int64_t)b * per_row) * V;
        const int s = d0 / E;                        // V divides E: the V columns lie in one slot
        int64_t p, q, r;
        float v[V];
        if (!complete_row(pos, slot_base, pool_id, n_pool, Q, S, depth, C, b, s, p, q, r)) {
#pragma unroll
            for (int j = 0; j < V; ++j) v[j] = 0.f;
        } else if (r >= 0) {
            const float* src = pool + r * ld_pool + (d0 - s * E);
#pragma unroll
            for (int j = 0; j < V; ++j) v[j] = src[j] * inv_scale;
        } else if constexpr (V == 4) {
            const float4 o = *reinterpret_cast<const float4*>(outfits + q * ld_outfit + d0);
            v[0] = o.x; v[1] = o.y; v[2] = o.z; v[3] = o.w;
        } else {
            v[0] = outfits[q * ld_outfit + d0];
        }
#pragma unroll
        for (int j = 0; j < V; ++j) {
            if (kBf16Out) reinterpret_cast<__nv_bfloat16*>(out)[(int64_t)b * ld_out + d0 + j] = __float2bfloat16_rn(v[j]);
            else reinterpret_cast<float*>(out)[(int64_t)b * ld_out + d0 + j] = v[j];
        }
    }
}

//   complete_error_kernel   err[p] = sum_d (y[b, d] - x'_d)^2 over io, one warp per row: swap_row_error's loop (lane-strided fmaf over
//                           io, then the warp_sum tree), x'_d recomputed in fp32; a lane looks up its slot's pool row when it enters it.
__global__ void __launch_bounds__(kThreads) complete_error_kernel(const float* __restrict__ outfits, int64_t ld_outfit, int Q, int S,
                                                                  int E, const int64_t* __restrict__ slot_base,
                                                                  const float* __restrict__ pool, int64_t ld_pool, int64_t n_pool,
                                                                  const int64_t* __restrict__ pool_id, int depth, int C,
                                                                  const int64_t* __restrict__ pos, int B, float inv_scale,
                                                                  const float* __restrict__ y, int64_t ld_y, float* __restrict__ err) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int io = S * E;
    for (int b = blockIdx.x * kWarps + warp; b < B; b += gridDim.x * kWarps) {
        int64_t p, q, r;
        if (!complete_row(pos, slot_base, pool_id, n_pool, Q, S, depth, C, b, 0, p, q, r)) continue;
        const float* x = outfits + q * ld_outfit;
        float acc = 0.f;
        int lo = 0;
        for (int d = lane; d < io; d += 32) {
            if (d >= lo + E) {
                const int s = d / E;
                lo = s * E;
                complete_row(pos, slot_base, pool_id, n_pool, Q, S, depth, C, b, s, p, q, r);
            }
            const float t = r >= 0 ? pool[r * ld_pool + (d - lo)] * inv_scale : x[d];
            const float df = y[(int64_t)b * ld_y + d] - t;
            acc = fmaf(df, df, acc);
        }
        acc = warp_sum(acc);
        if (lane == 0) err[p] = acc;
    }
}

// ---- beam completion: the missing slots filled one level at a time, the slots not yet filled hidden -------------------------
constexpr int64_t kHiddenSlot = -2;
// v /= d, returning v % d, for 0 <= v and 1 <= d <= 128 in 32-bit divisions (a 64-bit division is a call, which spills here):
// the high word, then the low word in two 16-bit steps, each dividend below 2^23.
__device__ __forceinline__ int divmod_small(int64_t& v, int d) {
    const uint32_t ud = (uint32_t)d, hi = (uint32_t)((uint64_t)v >> 32), lo = (uint32_t)v;
    const uint32_t a = ((hi % ud) << 16) | (lo >> 16), b = ((a % ud) << 16) | (lo & 0xffffu);
    v = (int64_t)(((uint64_t)(hi / ud) << 32) | ((a / ud) << 16) | (b / ud));
    return (int)(b % ud);
}
// Child p of the flattened [Q, W depth] grid at `level` (include/codae_b200.h: beam completion) -- the one decode and validity rule of
// both beam kernels.  Child (q, t, b) extends parent beam_c[q, t] by candidate b of the level-th missing slot of outfit q.  Returns
// whether it is valid and sets q and, in row, what slot `want` holds: its pool row, -1 for a given slot, kHiddenSlot for a missing
// slot past the level.  The parent's digits (complete_row's convention) fill missing slots 0 .. level-1; the parent is < depth^level
// exactly when nothing of it is left after them, and the level is < m_q exactly when more than `level` missing slots were seen.  Every
// pool row the child takes is checked before any of it is read.
__device__ __forceinline__ bool beam_row(const int64_t* __restrict__ pos, const int64_t* __restrict__ beam_c, int W,
                                         const int64_t* __restrict__ slot_base, const int64_t* __restrict__ pool_id, int64_t n_pool,
                                         int Q, int S, int depth, int level, int b, int want, int64_t& p, int64_t& q, int64_t& row) {
    p = pos[b];
    row = -1;
    const int wd = W * depth;
    if (p < 0 || p >= (int64_t)Q * wd) return false;
    const int pc = (int)p;                             // Q W depth <= INT32_MAX: 32-bit divisions from here on
    q = pc / wd;
    const int t = (pc - (int)q * wd) / depth;
    const int cand = pc - (int)q * wd - t * depth;
    int64_t parent = beam_c[q * W + t];
    if (parent < 0) return false;
    const int64_t* sb = slot_base + q * S;
    int j = 0;
    for (int s = 0; s < S; ++s) {
        const int64_t base = sb[s];
        if (base < 0) continue;
        const int jj = j++;
        if (jj > level) {
            if (s == want) row = kHiddenSlot;
            continue;
        }
        int digit = cand;
        if (jj < level) digit = divmod_small(parent, depth);
        if (base >= n_pool || digit >= n_pool - base) return false;
        if (pool_id[base + digit] < 0) return false;
        if (s == want) row = base + digit;
    }
    return j > level && parent == 0;
}

//   beam_build_kernel   x'[b, :] = outfit q with missing slots 0 .. level filled (pool row * inv_scale, complete_build_kernel's
//                       values) and the later missing slots +0.0; V = 4 as in complete_build_kernel.
template <bool kBf16Out, int V>
__global__ void __launch_bounds__(256) beam_build_kernel(const float* __restrict__ outfits, int64_t ld_outfit, int Q, int S, int E,
                                                         const int64_t* __restrict__ slot_base, const float* __restrict__ pool,
                                                         int64_t ld_pool, int64_t n_pool, const int64_t* __restrict__ pool_id,
                                                         int depth, const int64_t* __restrict__ beam_c, int W, int level,
                                                         const int64_t* __restrict__ pos, int B, float inv_scale,
                                                         void* __restrict__ out, int64_t ld_out) {
    const int per_row = S * E / V;
    const int64_t total = (int64_t)B * per_row;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int b = (int)(e / per_row), d0 = (int)(e - (int64_t)b * per_row) * V;
        const int s = d0 / E;                        // V divides E: the V columns lie in one slot
        int64_t p, q, r;
        float v[V];
        if (!beam_row(pos, beam_c, W, slot_base, pool_id, n_pool, Q, S, depth, level, b, s, p, q, r) || r == kHiddenSlot) {
#pragma unroll
            for (int j = 0; j < V; ++j) v[j] = 0.f;
        } else if (r >= 0) {
            const float* src = pool + r * ld_pool + (d0 - s * E);
#pragma unroll
            for (int j = 0; j < V; ++j) v[j] = src[j] * inv_scale;
        } else if constexpr (V == 4) {
            const float4 o = *reinterpret_cast<const float4*>(outfits + q * ld_outfit + d0);
            v[0] = o.x; v[1] = o.y; v[2] = o.z; v[3] = o.w;
        } else {
            v[0] = outfits[q * ld_outfit + d0];
        }
#pragma unroll
        for (int j = 0; j < V; ++j) {
            if (kBf16Out) reinterpret_cast<__nv_bfloat16*>(out)[(int64_t)b * ld_out + d0 + j] = __float2bfloat16_rn(v[j]);
            else reinterpret_cast<float*>(out)[(int64_t)b * ld_out + d0 + j] = v[j];
        }
    }
}

//   beam_error_kernel   err[p] = sum_d (y[b, d] - x'_d)^2 over the columns of the given slots and of missing slots 0 .. level: the loop
//                       of complete_error_kernel with the hidden columns skipped, so at a child's last level it is complete_error's
//                       value bit for bit.  The minimum of one CTA per SM in the launch bounds lets ptxas use the 40 registers the
//                       decode needs; without it ptxas held the kernel to 32 and spilled.
__global__ void __launch_bounds__(kThreads, 1) beam_error_kernel(const float* __restrict__ outfits, int64_t ld_outfit, int Q, int S, int E,
                                                              const int64_t* __restrict__ slot_base, const float* __restrict__ pool,
                                                              int64_t ld_pool, int64_t n_pool, const int64_t* __restrict__ pool_id,
                                                              int depth, const int64_t* __restrict__ beam_c, int W, int level,
                                                              const int64_t* __restrict__ pos, int B, float inv_scale,
                                                              const float* __restrict__ y, int64_t ld_y, float* __restrict__ err) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int io = S * E;
    for (int b = blockIdx.x * kWarps + warp; b < B; b += gridDim.x * kWarps) {
        int64_t p, q, r;
        if (!beam_row(pos, beam_c, W, slot_base, pool_id, n_pool, Q, S, depth, level, b, 0, p, q, r)) continue;
        const float* x = outfits + q * ld_outfit;
        float acc = 0.f;
        int lo = 0;
        for (int d = lane; d < io; d += 32) {
            if (d >= lo + E) {
                const int s = d / E;
                lo = s * E;
                beam_row(pos, beam_c, W, slot_base, pool_id, n_pool, Q, S, depth, level, b, s, p, q, r);
            }
            if (r == kHiddenSlot) continue;
            const float t = r >= 0 ? pool[r * ld_pool + (d - lo)] * inv_scale : x[d];
            const float df = y[(int64_t)b * ld_y + d] - t;
            acc = fmaf(df, df, acc);
        }
        acc = warp_sum(acc);
        if (lane == 0) err[p] = acc;
    }
}

// ---- outfit revision: the outfit as given and every single-item replacement of it, each scored by swap error --------------
// Row p of the flattened [Q, 1 + S depth] grid (include/codae_b200.h: outfit revision) -- the one decode and validity rule of both
// revision kernels.  Column 0 of outfit q is the outfit as given (slot = -1); column 1 + s depth + c replaces slot s by its candidate
// c, pool row slot_base[q, s] + c.  Returns whether p is valid and sets q, slot and row (-1 for column 0).  The pool row is checked
// before it is read; Q (1 + S depth) <= INT32_MAX, so the decode uses 32-bit divisions.
__device__ __forceinline__ bool revise_row(const int64_t* __restrict__ pos, const int64_t* __restrict__ slot_base,
                                           const int64_t* __restrict__ pool_id, int64_t n_pool, int Q, int S, int depth, int b,
                                           int64_t& p, int64_t& q, int& slot, int64_t& row) {
    p = pos[b];
    slot = -1;
    row = -1;
    const int g = 1 + S * depth;
    if (p < 0 || p >= (int64_t)Q * g) return false;
    const int pc = (int)p;
    q = pc / g;
    const int col = pc - (int)q * g;
    if (col == 0) return true;
    slot = (col - 1) / depth;
    const int cand = col - 1 - slot * depth;
    const int64_t base = slot_base[q * S + slot];
    if (base < 0 || base >= n_pool || cand >= n_pool - base) return false;
    row = base + cand;
    return pool_id[row] >= 0;
}

//   revise_build_kernel   x'[b, :] = outfit q with slot `slot` replaced by its pool row * inv_scale (complete_build_kernel's values),
//                         the outfit itself for column 0.  V = 4 as in complete_build_kernel.
template <bool kBf16Out, int V>
__global__ void __launch_bounds__(256) revise_build_kernel(const float* __restrict__ outfits, int64_t ld_outfit, int Q, int S, int E,
                                                           const int64_t* __restrict__ slot_base, const float* __restrict__ pool,
                                                           int64_t ld_pool, int64_t n_pool, const int64_t* __restrict__ pool_id,
                                                           int depth, const int64_t* __restrict__ pos, int B, float inv_scale,
                                                           void* __restrict__ out, int64_t ld_out) {
    const int per_row = S * E / V;
    const int64_t total = (int64_t)B * per_row;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int b = (int)(e / per_row), d0 = (int)(e - (int64_t)b * per_row) * V;
        const int s = d0 / E;                        // V divides E: the V columns lie in one slot
        int64_t p, q, r;
        int slot;
        float v[V];
        if (!revise_row(pos, slot_base, pool_id, n_pool, Q, S, depth, b, p, q, slot, r)) {
#pragma unroll
            for (int j = 0; j < V; ++j) v[j] = 0.f;
        } else if (s == slot) {
            const float* src = pool + r * ld_pool + (d0 - s * E);
#pragma unroll
            for (int j = 0; j < V; ++j) v[j] = src[j] * inv_scale;
        } else if constexpr (V == 4) {
            const float4 o = *reinterpret_cast<const float4*>(outfits + q * ld_outfit + d0);
            v[0] = o.x; v[1] = o.y; v[2] = o.z; v[3] = o.w;
        } else {
            v[0] = outfits[q * ld_outfit + d0];
        }
#pragma unroll
        for (int j = 0; j < V; ++j) {
            if (kBf16Out) reinterpret_cast<__nv_bfloat16*>(out)[(int64_t)b * ld_out + d0 + j] = __float2bfloat16_rn(v[j]);
            else reinterpret_cast<float*>(out)[(int64_t)b * ld_out + d0 + j] = v[j];
        }
    }
}

//   revise_error_kernel   err[p] = sum_d (y[b, d] - x'_d)^2 over io, one warp per row: complete_error_kernel's loop (lane-strided fmaf
//                         over io, then the warp_sum tree), x'_d recomputed in fp32, the pool read only in the swapped slot.  A swap
//                         whose x' equals the outfit value for value (the held item proposed again) gets no error: it is not a change.
__global__ void __launch_bounds__(kThreads) revise_error_kernel(const float* __restrict__ outfits, int64_t ld_outfit, int Q, int S,
                                                                int E, const int64_t* __restrict__ slot_base,
                                                                const float* __restrict__ pool, int64_t ld_pool, int64_t n_pool,
                                                                const int64_t* __restrict__ pool_id, int depth,
                                                                const int64_t* __restrict__ pos, int B, float inv_scale,
                                                                const float* __restrict__ y, int64_t ld_y, float* __restrict__ err) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int io = S * E;
    for (int b = blockIdx.x * kWarps + warp; b < B; b += gridDim.x * kWarps) {
        int64_t p, q, r;
        int slot;
        if (!revise_row(pos, slot_base, pool_id, n_pool, Q, S, depth, b, p, q, slot, r)) continue;
        const float* x = outfits + q * ld_outfit;
        const int lo = slot < 0 ? io : slot * E, hi = lo + E;
        float acc = 0.f;
        bool same = true;
        for (int d = lane; d < io; d += 32) {
            const bool in = d >= lo && d < hi;
            const float t = in ? pool[r * ld_pool + (d - lo)] * inv_scale : x[d];
            same &= !in || t == x[d];
            const float df = y[(int64_t)b * ld_y + d] - t;
            acc = fmaf(df, df, acc);
        }
        acc = warp_sum(acc);
        if (slot >= 0 && __all_sync(0xffffffffu, same)) continue;
        if (lane == 0) err[p] = acc;
    }
}

inline int sweep_grid(const codae_ctx* ctx, int64_t n_rows) {
    int64_t g = (n_rows + kWarps - 1) / kWarps;
    const int64_t cap = (int64_t)ctx->sm_count * 4;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

inline size_t topk_smem(int QC, int E, int k) {
    return (size_t)QC * E * 4 + (size_t)((QC + 3) & ~3) * 4 + (size_t)kWarps * QC * k * 12;
}

// Arguments of the *_filtered entry points (include/codae_b200.h).  Global indices must be >= 0 so that padding never matches.
inline int check_filter(codae_ctx* ctx, const char* fn, int64_t row_offset, const int64_t* exclude, int n_exclude) {
    CODAE_REQUIRE(ctx, n_exclude >= 0 && n_exclude <= CODAE_TOPK_MAX_EXCLUDE, "%s: n_exclude %d outside [0, %d]", fn, n_exclude,
                  CODAE_TOPK_MAX_EXCLUDE);
    CODAE_REQUIRE(ctx, (exclude != nullptr) == (n_exclude > 0), "%s: exclude must be non-NULL exactly when n_exclude > 0", fn);
    CODAE_REQUIRE(ctx, row_offset >= 0, "%s: row_offset %lld < 0", fn, (long long)row_offset);
    return CODAE_OK;
}

}  // namespace

extern "C" {

size_t codae_score_topk_workspace_bytes(const codae_ctx* ctx, int Q, int k) {
    if (!ctx || Q < 1 || k < 1) return 0;
    return (size_t)ctx->sm_count * 4 * 4 /*QC max*/ * (size_t)k * 12 + 256;
}

// codae_score_topk and codae_score_topk_filtered; no filter (allow NULL, n_exclude 0) runs the unfiltered instantiations.
static int score_topk(codae_ctx* ctx, const void* catalog, int cat_dtype, int64_t n_rows, int64_t ld, int E, int64_t row_offset,
                      const float* query, int Q, float inv_scale, int metric, int k, const uint8_t* allow, const int64_t* exclude,
                      int n_exclude, float* out_score, int64_t* out_idx, void* workspace, size_t ws_bytes, void* stream) {
    CODAE_REQUIRE(ctx, ctx && catalog && query && out_score && out_idx && workspace, "codae_score_topk: NULL argument");
    CODAE_REQUIRE(ctx, k >= 1 && k <= kMaxK, "codae_score_topk: k %d outside [1, %d]", k, kMaxK);
    CODAE_REQUIRE(ctx, Q >= 1 && n_rows >= 0, "codae_score_topk: bad Q / n_rows");
    CODAE_REQUIRE(ctx, metric == CODAE_METRIC_SQERR || metric == CODAE_METRIC_COSINE, "codae_score_topk: bad metric %d", metric);
    const bool bf = cat_dtype == CODAE_BF16;
    CODAE_REQUIRE(ctx, cat_dtype == CODAE_F32 || bf, "codae_score_topk: bad cat_dtype %d", cat_dtype);
    const int vec = bf ? 8 : 4;
    CODAE_REQUIRE(ctx, E >= vec && E <= 4096 && E % vec == 0 && ld >= E && ld % vec == 0 &&
                           (reinterpret_cast<uintptr_t>(catalog) & 15) == 0,
                  "codae_score_topk: E=%d ld=%lld must be multiples of %d (16-byte rows), E <= 4096", E, (long long)ld, vec);
    if (ws_bytes < codae_score_topk_workspace_bytes(ctx, Q, k))
        return codae_fail(ctx, CODAE_ENOMEM, "codae_score_topk: workspace %zu < %zu bytes", ws_bytes,
                          codae_score_topk_workspace_bytes(ctx, Q, k));
    cudaStream_t s = as_stream(stream);
    merge_attrs();
    const bool filtered = allow || n_exclude > 0;
    const int grid0 = sweep_grid(ctx, n_rows);
    int64_t* ws_idx = reinterpret_cast<int64_t*>(workspace);
    float* ws_score = reinterpret_cast<float*>(ws_idx + (size_t)grid0 * 4 * k);
    for (int q0 = 0; q0 < Q; q0 += 4) {
        int grid = grid0;
        const int qc = (Q - q0 >= 4) ? 4 : 1;
        const int reps = (Q - q0 >= 4) ? 1 : (Q - q0);  // leftover queries one at a time
        for (int rpt = 0; rpt < reps; ++rpt) {
            const float* qptr = query + (int64_t)(q0 + rpt) * E;
            const int64_t* xptr = exclude ? exclude + (int64_t)(q0 + rpt) * n_exclude : nullptr;
            const size_t smem = topk_smem(qc, E, k);
#define LAUNCH_F(MET, QC, BF, F)                                                                                     \
    do {                                                                                                             \
        cudaFuncSetAttribute(score_topk_kernel<MET, QC, BF, F>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        /* one resident wave: the grid-stride sweep balances itself only if every CTA runs from the start */             \
        const int occ = resident_ctas_per_sm(score_topk_kernel<MET, QC, BF, F>, kThreads, smem);                          \
        if (grid > ctx->sm_count * occ) grid = ctx->sm_count * occ;                                                     \
        score_topk_kernel<MET, QC, BF, F><<<grid, kThreads, smem, s>>>(catalog, n_rows, ld, E, row_offset, qptr, inv_scale, k, \
                                                                       ws_score, ws_idx, allow, xptr, n_exclude);   \
    } while (0)
#define LAUNCH(MET, QC, BF) do { if (filtered) LAUNCH_F(MET, QC, BF, true); else LAUNCH_F(MET, QC, BF, false); } while (0)
            if (metric == CODAE_METRIC_SQERR) {
                if (qc == 4) { if (bf) LAUNCH(CODAE_METRIC_SQERR, 4, true); else LAUNCH(CODAE_METRIC_SQERR, 4, false); }
                else { if (bf) LAUNCH(CODAE_METRIC_SQERR, 1, true); else LAUNCH(CODAE_METRIC_SQERR, 1, false); }
            } else {
                if (qc == 4) { if (bf) LAUNCH(CODAE_METRIC_COSINE, 4, true); else LAUNCH(CODAE_METRIC_COSINE, 4, false); }
                else { if (bf) LAUNCH(CODAE_METRIC_COSINE, 1, true); else LAUNCH(CODAE_METRIC_COSINE, 1, false); }
            }
#undef LAUNCH
#undef LAUNCH_F
            int rc = codae_check_launch(ctx, "score_topk_kernel");
            if (rc) return rc;
            if (metric == CODAE_METRIC_SQERR)
                topk_merge_kernel<CODAE_METRIC_SQERR><<<qc, kThreads, merge_smem(), s>>>(ws_score, ws_idx, grid, qc, k, out_score, out_idx, q0 + rpt, 1);
            else
                topk_merge_kernel<CODAE_METRIC_COSINE><<<qc, kThreads, merge_smem(), s>>>(ws_score, ws_idx, grid, qc, k, out_score, out_idx, q0 + rpt, 1);
            rc = codae_check_launch(ctx, "topk_merge_kernel");
            if (rc) return rc;
        }
    }
    return CODAE_OK;
}

int codae_score_topk(codae_ctx* ctx, const void* catalog, int cat_dtype, int64_t n_rows, int64_t ld, int E,
                     int64_t row_offset, const float* query, int Q, float inv_scale, int metric, int k, float* out_score,
                     int64_t* out_idx, void* workspace, size_t ws_bytes, void* stream) {
    return score_topk(ctx, catalog, cat_dtype, n_rows, ld, E, row_offset, query, Q, inv_scale, metric, k, nullptr, nullptr, 0,
                      out_score, out_idx, workspace, ws_bytes, stream);
}

int codae_score_topk_filtered(codae_ctx* ctx, const void* catalog, int cat_dtype, int64_t n_rows, int64_t ld, int E,
                              int64_t row_offset, const float* query, int Q, float inv_scale, int metric, int k,
                              const uint8_t* allow, const int64_t* exclude, int n_exclude, float* out_score, int64_t* out_idx,
                              void* workspace, size_t ws_bytes, void* stream) {
    const int rc = check_filter(ctx, "codae_score_topk_filtered", row_offset, exclude, n_exclude);
    if (rc) return rc;
    return score_topk(ctx, catalog, cat_dtype, n_rows, ld, E, row_offset, query, Q, inv_scale, metric, k, allow, exclude,
                      n_exclude, out_score, out_idx, workspace, ws_bytes, stream);
}

int codae_topk_merge(codae_ctx* ctx, const float* scores, const int64_t* idx, int G, int Q, int k, int metric,
                     float* out_score, int64_t* out_idx, void* stream) {
    CODAE_REQUIRE(ctx, ctx && scores && idx && out_score && out_idx, "codae_topk_merge: NULL argument");
    CODAE_REQUIRE(ctx, G >= 1 && Q >= 1 && k >= 1 && k <= kMaxK, "codae_topk_merge: bad shape");
    merge_attrs();
    if (metric == CODAE_METRIC_SQERR)
        topk_merge_kernel<CODAE_METRIC_SQERR><<<Q, kThreads, merge_smem(), as_stream(stream)>>>(scores, idx, G, Q, k, out_score, out_idx, 0, 1);
    else if (metric == CODAE_METRIC_COSINE)
        topk_merge_kernel<CODAE_METRIC_COSINE><<<Q, kThreads, merge_smem(), as_stream(stream)>>>(scores, idx, G, Q, k, out_score, out_idx, 0, 1);
    else
        return codae_fail(ctx, CODAE_EINVAL, "codae_topk_merge: bad metric %d", metric);
    return codae_check_launch(ctx, "topk_merge_kernel");
}

int codae_swap_build(codae_ctx* ctx, const float* outfit, const void* catalog, int cat_dtype, int64_t ld_cat, int64_t first_row,
                     int B, int E, int slot, int io, float inv_scale, void* out_x, int x_dtype, int64_t ld_x, void* stream) {
    CODAE_REQUIRE(ctx, ctx && outfit && catalog && out_x, "codae_swap_build: NULL argument");
    CODAE_REQUIRE(ctx, B >= 1 && E >= 1 && slot >= 0 && (slot + 1) * E <= io && ld_x >= io && ld_cat >= E && first_row >= 0,
                  "codae_swap_build: bad shape (B=%d E=%d slot=%d io=%d)", B, E, slot, io);
    const bool bc = cat_dtype == CODAE_BF16, bo = x_dtype == CODAE_BF16;
    int64_t blocks = ((int64_t)B * io + 256 * 4 - 1) / (256 * 4);
    if (blocks > (int64_t)ctx->sm_count * 8) blocks = (int64_t)ctx->sm_count * 8;
    cudaStream_t s = as_stream(stream);
#define LAUNCH(BC, BO) swap_build_kernel<BC, BO><<<(unsigned)blocks, 256, 0, s>>>(outfit, catalog, ld_cat, first_row, B, E, slot, io, inv_scale, out_x, ld_x)
    if (bc && bo) LAUNCH(true, true); else if (bc) LAUNCH(true, false); else if (bo) LAUNCH(false, true); else LAUNCH(false, false);
#undef LAUNCH
    return codae_check_launch(ctx, "swap_build_kernel");
}

static int swap_error_topk(codae_ctx* ctx, const float* outfit, const void* catalog, int cat_dtype, int64_t ld_cat,
                           int64_t first_row, int B, int E, int slot, int io, float inv_scale, const float* y, int64_t ld_y,
                           int64_t row_offset, int k, const uint8_t* allow, const int64_t* exclude, int n_exclude,
                           float* out_score, int64_t* out_idx, void* workspace, size_t ws_bytes, void* stream) {
    CODAE_REQUIRE(ctx, ctx && outfit && catalog && y && out_score && out_idx && workspace, "codae_swap_error_topk: NULL argument");
    CODAE_REQUIRE(ctx, B >= 1 && E >= 1 && slot >= 0 && (slot + 1) * E <= io && ld_y >= io && ld_cat >= E && k >= 1 && k <= kMaxK,
                  "codae_swap_error_topk: bad shape");
    if (ws_bytes < codae_score_topk_workspace_bytes(ctx, 1, k))
        return codae_fail(ctx, CODAE_ENOMEM, "codae_swap_error_topk: workspace %zu < %zu bytes", ws_bytes,
                          codae_score_topk_workspace_bytes(ctx, 1, k));
    cudaStream_t s = as_stream(stream);
    const int grid = sweep_grid(ctx, B);
    int64_t* ws_idx = reinterpret_cast<int64_t*>(workspace);
    float* ws_score = reinterpret_cast<float*>(ws_idx + (size_t)grid * k);
    const size_t smem = (size_t)kWarps * k * 12;
    const bool bc = cat_dtype == CODAE_BF16, filtered = allow || n_exclude > 0;
#define LAUNCH(BC, F) swap_error_topk_kernel<BC, F><<<grid, kThreads, smem, s>>>(outfit, catalog, ld_cat, first_row, B, E, slot, io, inv_scale, y, ld_y, row_offset, k, ws_score, ws_idx, allow, exclude, n_exclude)
    if (bc && filtered) LAUNCH(true, true); else if (bc) LAUNCH(true, false); else if (filtered) LAUNCH(false, true); else LAUNCH(false, false);
#undef LAUNCH
    int rc = codae_check_launch(ctx, "swap_error_topk_kernel");
    if (rc) return rc;
    merge_attrs();
    topk_merge_kernel<CODAE_METRIC_SQERR><<<1, kThreads, merge_smem(), s>>>(ws_score, ws_idx, grid, 1, k, out_score, out_idx, 0, 1);
    return codae_check_launch(ctx, "topk_merge_kernel");
}

int codae_swap_error_topk(codae_ctx* ctx, const float* outfit, const void* catalog, int cat_dtype, int64_t ld_cat,
                          int64_t first_row, int B, int E, int slot, int io, float inv_scale, const float* y, int64_t ld_y,
                          int64_t row_offset, int k, float* out_score, int64_t* out_idx, void* workspace, size_t ws_bytes,
                          void* stream) {
    return swap_error_topk(ctx, outfit, catalog, cat_dtype, ld_cat, first_row, B, E, slot, io, inv_scale, y, ld_y, row_offset, k,
                           nullptr, nullptr, 0, out_score, out_idx, workspace, ws_bytes, stream);
}

int codae_swap_error_topk_filtered(codae_ctx* ctx, const float* outfit, const void* catalog, int cat_dtype, int64_t ld_cat,
                                   int64_t first_row, int B, int E, int slot, int io, float inv_scale, const float* y,
                                   int64_t ld_y, int64_t row_offset, int k, const uint8_t* allow, const int64_t* exclude,
                                   int n_exclude, float* out_score, int64_t* out_idx, void* workspace, size_t ws_bytes,
                                   void* stream) {
    const int rc = check_filter(ctx, "codae_swap_error_topk_filtered", row_offset, exclude, n_exclude);
    if (rc) return rc;
    return swap_error_topk(ctx, outfit, catalog, cat_dtype, ld_cat, first_row, B, E, slot, io, inv_scale, y, ld_y, row_offset, k,
                           allow, exclude, n_exclude, out_score, out_idx, workspace, ws_bytes, stream);
}

// Arguments shared by codae_swap_build_pairs and codae_swap_error_pairs.
static int check_pairs(codae_ctx* ctx, const char* fn, const float* outfits, int64_t ld_outfit, int Q, const void* catalog,
                       int cat_dtype, int64_t ld_cat, int64_t n_rows, int64_t row_offset, const int64_t* candidates, int m,
                       const int64_t* pos, int B, int E, int slot, int io) {
    CODAE_REQUIRE(ctx, ctx && outfits && catalog && candidates && pos, "%s: NULL argument", fn);
    CODAE_REQUIRE(ctx, Q >= 1 && m >= 1 && (int64_t)Q * m <= INT32_MAX, "%s: bad list shape Q=%d m=%d", fn, Q, m);
    CODAE_REQUIRE(ctx, B >= 1 && E >= 1 && slot >= 0 && (int64_t)(slot + 1) * E <= io && ld_outfit >= io && ld_cat >= E &&
                           n_rows >= 0 && row_offset >= 0,
                  "%s: bad shape (B=%d E=%d slot=%d io=%d)", fn, B, E, slot, io);
    CODAE_REQUIRE(ctx, cat_dtype == CODAE_F32 || cat_dtype == CODAE_BF16, "%s: bad cat_dtype %d", fn, cat_dtype);
    return CODAE_OK;
}

int codae_swap_build_pairs(codae_ctx* ctx, const float* outfits, int64_t ld_outfit, int Q, const void* catalog, int cat_dtype,
                           int64_t ld_cat, int64_t n_rows, int64_t row_offset, const int64_t* candidates, int m, const int64_t* pos,
                           int B, int E, int slot, int io, float inv_scale, void* out_x, int x_dtype, int64_t ld_x, void* stream) {
    int rc = check_pairs(ctx, "codae_swap_build_pairs", outfits, ld_outfit, Q, catalog, cat_dtype, ld_cat, n_rows, row_offset,
                         candidates, m, pos, B, E, slot, io);
    if (rc) return rc;
    CODAE_REQUIRE(ctx, out_x && ld_x >= io && (x_dtype == CODAE_F32 || x_dtype == CODAE_BF16),
                  "codae_swap_build_pairs: bad output (ld_x=%lld x_dtype=%d)", (long long)ld_x, x_dtype);
    const bool bc = cat_dtype == CODAE_BF16, bo = x_dtype == CODAE_BF16;
    const bool v4 = io % 4 == 0 && E % 4 == 0 && ld_outfit % 4 == 0 && (reinterpret_cast<uintptr_t>(outfits) & 15) == 0;
    const int V = v4 ? 4 : 1;
    int64_t blocks = ((int64_t)B * (io / V) + 256 * 4 - 1) / (256 * 4);
    if (blocks > (int64_t)ctx->sm_count * 8) blocks = (int64_t)ctx->sm_count * 8;
    const int64_t n_pairs = (int64_t)Q * m;
    cudaStream_t s = as_stream(stream);
#define LAUNCH(BC, BO, VV) swap_build_pairs_kernel<BC, BO, VV><<<(unsigned)blocks, 256, 0, s>>>(outfits, ld_outfit, n_pairs, catalog, ld_cat, n_rows, row_offset, candidates, m, pos, B, E, slot, io, inv_scale, out_x, ld_x)
#define LAUNCH_V(BC, BO) do { if (v4) LAUNCH(BC, BO, 4); else LAUNCH(BC, BO, 1); } while (0)
    if (bc && bo) LAUNCH_V(true, true); else if (bc) LAUNCH_V(true, false); else if (bo) LAUNCH_V(false, true); else LAUNCH_V(false, false);
#undef LAUNCH_V
#undef LAUNCH
    return codae_check_launch(ctx, "swap_build_pairs_kernel");
}

int codae_swap_error_pairs(codae_ctx* ctx, const float* outfits, int64_t ld_outfit, int Q, const void* catalog, int cat_dtype,
                           int64_t ld_cat, int64_t n_rows, int64_t row_offset, const int64_t* candidates, int m, const int64_t* pos,
                           int B, int E, int slot, int io, float inv_scale, const float* y, int64_t ld_y, float* err, void* stream) {
    int rc = check_pairs(ctx, "codae_swap_error_pairs", outfits, ld_outfit, Q, catalog, cat_dtype, ld_cat, n_rows, row_offset,
                         candidates, m, pos, B, E, slot, io);
    if (rc) return rc;
    CODAE_REQUIRE(ctx, y && err && ld_y >= io, "codae_swap_error_pairs: bad output (ld_y=%lld)", (long long)ld_y);
    const int64_t n_pairs = (int64_t)Q * m;
    cudaStream_t s = as_stream(stream);
    if (cat_dtype == CODAE_BF16)
        swap_error_pairs_kernel<true><<<sweep_grid(ctx, B), kThreads, 0, s>>>(outfits, ld_outfit, n_pairs, catalog, ld_cat, n_rows, row_offset, candidates, m, pos, B, E, slot, io, inv_scale, y, ld_y, err);
    else
        swap_error_pairs_kernel<false><<<sweep_grid(ctx, B), kThreads, 0, s>>>(outfits, ld_outfit, n_pairs, catalog, ld_cat, n_rows, row_offset, candidates, m, pos, B, E, slot, io, inv_scale, y, ld_y, err);
    return codae_check_launch(ctx, "swap_error_pairs_kernel");
}

int codae_swap_pairs_topk(codae_ctx* ctx, const float* err, const int64_t* candidates, int Q, int m, int k, float* out_score,
                          int64_t* out_idx, void* stream) {
    CODAE_REQUIRE(ctx, ctx && err && candidates && out_score && out_idx, "codae_swap_pairs_topk: NULL argument");
    CODAE_REQUIRE(ctx, Q >= 1 && m >= 1 && (int64_t)Q * m <= INT32_MAX, "codae_swap_pairs_topk: bad list shape Q=%d m=%d", Q, m);
    CODAE_REQUIRE(ctx, k >= 1 && k <= kMaxK, "codae_swap_pairs_topk: k %d outside [1, %d]", k, kMaxK);
    const int grid = (Q + kWarps - 1) / kWarps;
    swap_pairs_topk_kernel<<<grid, kThreads, (size_t)kWarps * k * 12, as_stream(stream)>>>(err, candidates, Q, m, k, out_score, out_idx);
    return codae_check_launch(ctx, "swap_pairs_topk_kernel");
}

int codae_outfit_loo_error(codae_ctx* ctx, const float* outfits, int64_t ld_outfit, int Q, int S, int E, const float* y, int64_t ld_y,
                           float* err, float* score, int64_t* odd, void* stream) {
    CODAE_REQUIRE(ctx, ctx && outfits && y && err && score && odd, "codae_outfit_loo_error: NULL argument");
    CODAE_REQUIRE(ctx, Q >= 1 && S >= 1 && S <= 64 && E >= 4 && E % 4 == 0,
                  "codae_outfit_loo_error: bad shape Q=%d S=%d E=%d (Q >= 1, 1 <= S <= 64, E a positive multiple of 4)", Q, S, E);
    CODAE_REQUIRE(ctx, ld_outfit >= (int64_t)S * E && ld_y >= (int64_t)S * E,
                  "codae_outfit_loo_error: pitches ld_outfit=%lld ld_y=%lld shorter than S E = %lld", (long long)ld_outfit,
                  (long long)ld_y, (long long)S * E);
    const auto al = [](const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; };
    CODAE_REQUIRE(ctx, al(outfits, 4) && al(y, 4) && al(err, 4) && al(score, 4) && al(odd, 8),
                  "codae_outfit_loo_error: misaligned buffer");
    outfit_loo_error_kernel<<<sweep_grid(ctx, Q), kThreads, 0, as_stream(stream)>>>(outfits, ld_outfit, Q, S, E, y, ld_y, err, score,
                                                                                     odd);
    return codae_check_launch(ctx, "outfit_loo_error_kernel");
}

// Arguments shared by codae_complete_build and codae_complete_error.
static int check_complete(codae_ctx* ctx, const char* fn, const float* outfits, int64_t ld_outfit, int Q, int S, int E,
                          const int64_t* slot_base, const float* pool, int64_t ld_pool, int64_t n_pool, const int64_t* pool_id,
                          int depth, int C, const int64_t* pos, int B) {
    CODAE_REQUIRE(ctx, ctx && outfits && slot_base && pool && pool_id && pos, "%s: NULL argument", fn);
    CODAE_REQUIRE(ctx, Q >= 1 && S >= 1 && S <= 64 && E >= 1 && (int64_t)S * E <= INT32_MAX && B >= 1,
                  "%s: bad shape Q=%d S=%d E=%d B=%d (Q, B >= 1, 1 <= S <= 64)", fn, Q, S, E, B);
    CODAE_REQUIRE(ctx, depth >= 1 && depth <= kMaxK && C >= 1 && C <= CODAE_COMPLETE_MAX_COMBOS && (int64_t)Q * C <= INT32_MAX,
                  "%s: bad combinations depth=%d C=%d (1 <= depth <= %d, 1 <= C <= %d, Q C <= INT32_MAX)", fn, depth, C, kMaxK,
                  CODAE_COMPLETE_MAX_COMBOS);
    CODAE_REQUIRE(ctx, n_pool >= 1 && ld_pool >= E && ld_outfit >= (int64_t)S * E,
                  "%s: bad pool or pitch (n_pool=%lld ld_pool=%lld ld_outfit=%lld)", fn, (long long)n_pool, (long long)ld_pool,
                  (long long)ld_outfit);
    const auto al = [](const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; };
    CODAE_REQUIRE(ctx, al(outfits, 4) && al(pool, 4) && al(slot_base, 8) && al(pool_id, 8) && al(pos, 8), "%s: misaligned buffer", fn);
    return CODAE_OK;
}

int codae_complete_build(codae_ctx* ctx, const float* outfits, int64_t ld_outfit, int Q, int S, int E, const int64_t* slot_base,
                         const float* pool, int64_t ld_pool, int64_t n_pool, const int64_t* pool_id, int depth, int C,
                         const int64_t* pos, int B, float inv_scale, void* out_x, int x_dtype, int64_t ld_x, void* stream) {
    int rc = check_complete(ctx, "codae_complete_build", outfits, ld_outfit, Q, S, E, slot_base, pool, ld_pool, n_pool, pool_id,
                            depth, C, pos, B);
    if (rc) return rc;
    const int io = S * E;
    const bool bo = x_dtype == CODAE_BF16;
    CODAE_REQUIRE(ctx, out_x && ld_x >= io && (x_dtype == CODAE_F32 || bo) &&
                           (reinterpret_cast<uintptr_t>(out_x) & (bo ? 1 : 3)) == 0,
                  "codae_complete_build: bad output (ld_x=%lld x_dtype=%d)", (long long)ld_x, x_dtype);
    const bool v4 = E % 4 == 0 && ld_outfit % 4 == 0 && (reinterpret_cast<uintptr_t>(outfits) & 15) == 0;
    const int V = v4 ? 4 : 1;
    int64_t blocks = ((int64_t)B * (io / V) + 256 * 4 - 1) / (256 * 4);
    if (blocks > (int64_t)ctx->sm_count * 8) blocks = (int64_t)ctx->sm_count * 8;
    cudaStream_t s = as_stream(stream);
#define LAUNCH(BO, VV) complete_build_kernel<BO, VV><<<(unsigned)blocks, 256, 0, s>>>(outfits, ld_outfit, Q, S, E, slot_base, pool, ld_pool, n_pool, pool_id, depth, C, pos, B, inv_scale, out_x, ld_x)
    if (bo) { if (v4) LAUNCH(true, 4); else LAUNCH(true, 1); } else { if (v4) LAUNCH(false, 4); else LAUNCH(false, 1); }
#undef LAUNCH
    return codae_check_launch(ctx, "complete_build_kernel");
}

int codae_complete_error(codae_ctx* ctx, const float* outfits, int64_t ld_outfit, int Q, int S, int E, const int64_t* slot_base,
                         const float* pool, int64_t ld_pool, int64_t n_pool, const int64_t* pool_id, int depth, int C,
                         const int64_t* pos, int B, float inv_scale, const float* y, int64_t ld_y, float* err, void* stream) {
    int rc = check_complete(ctx, "codae_complete_error", outfits, ld_outfit, Q, S, E, slot_base, pool, ld_pool, n_pool, pool_id,
                            depth, C, pos, B);
    if (rc) return rc;
    CODAE_REQUIRE(ctx, y && err && ld_y >= (int64_t)S * E && (reinterpret_cast<uintptr_t>(y) & 3) == 0 &&
                           (reinterpret_cast<uintptr_t>(err) & 3) == 0,
                  "codae_complete_error: bad output (ld_y=%lld)", (long long)ld_y);
    complete_error_kernel<<<sweep_grid(ctx, B), kThreads, 0, as_stream(stream)>>>(outfits, ld_outfit, Q, S, E, slot_base, pool, ld_pool,
                                                                                   n_pool, pool_id, depth, C, pos, B, inv_scale, y, ld_y,
                                                                                   err);
    return codae_check_launch(ctx, "complete_error_kernel");
}

// Arguments shared by codae_complete_beam_build and codae_complete_beam_error.
static int check_beam(codae_ctx* ctx, const char* fn, const float* outfits, int64_t ld_outfit, int Q, int S, int E,
                      const int64_t* slot_base, const float* pool, int64_t ld_pool, int64_t n_pool, const int64_t* pool_id, int depth,
                      const int64_t* beam_c, int W, int level, const int64_t* pos, int B) {
    CODAE_REQUIRE(ctx, ctx && outfits && slot_base && pool && pool_id && beam_c && pos, "%s: NULL argument", fn);
    CODAE_REQUIRE(ctx, Q >= 1 && S >= 1 && S <= 64 && E >= 1 && (int64_t)S * E <= INT32_MAX && B >= 1,
                  "%s: bad shape Q=%d S=%d E=%d B=%d (Q, B >= 1, 1 <= S <= 64)", fn, Q, S, E, B);
    CODAE_REQUIRE(ctx, depth >= 1 && depth <= kMaxK && W >= 1 && W <= kMaxK && (int64_t)Q * W * depth <= INT32_MAX,
                  "%s: bad beam depth=%d W=%d (1 <= depth, W <= %d, Q W depth <= INT32_MAX)", fn, depth, W, kMaxK);
    bool fits = level >= 0 && level < S;                 // the keys of level `level` are < depth^(level+1) <= 2^62
    for (int64_t pw = 1, i = 0; fits && i <= level; ++i) {
        fits = pw <= ((int64_t)1 << 62) / depth;
        pw *= depth;
    }
    CODAE_REQUIRE(ctx, fits, "%s: bad level %d (0 <= level < S, depth^(level+1) <= 2^62)", fn, level);
    CODAE_REQUIRE(ctx, n_pool >= 1 && ld_pool >= E && ld_outfit >= (int64_t)S * E,
                  "%s: bad pool or pitch (n_pool=%lld ld_pool=%lld ld_outfit=%lld)", fn, (long long)n_pool, (long long)ld_pool,
                  (long long)ld_outfit);
    const auto al = [](const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; };
    CODAE_REQUIRE(ctx, al(outfits, 4) && al(pool, 4) && al(slot_base, 8) && al(pool_id, 8) && al(beam_c, 8) && al(pos, 8),
                  "%s: misaligned buffer", fn);
    return CODAE_OK;
}

int codae_complete_beam_build(codae_ctx* ctx, const float* outfits, int64_t ld_outfit, int Q, int S, int E, const int64_t* slot_base,
                              const float* pool, int64_t ld_pool, int64_t n_pool, const int64_t* pool_id, int depth,
                              const int64_t* beam_c, int W, int level, const int64_t* pos, int B, float inv_scale, void* out_x,
                              int x_dtype, int64_t ld_x, void* stream) {
    int rc = check_beam(ctx, "codae_complete_beam_build", outfits, ld_outfit, Q, S, E, slot_base, pool, ld_pool, n_pool, pool_id,
                        depth, beam_c, W, level, pos, B);
    if (rc) return rc;
    const int io = S * E;
    const bool bo = x_dtype == CODAE_BF16;
    CODAE_REQUIRE(ctx, out_x && ld_x >= io && (x_dtype == CODAE_F32 || bo) &&
                           (reinterpret_cast<uintptr_t>(out_x) & (bo ? 1 : 3)) == 0,
                  "codae_complete_beam_build: bad output (ld_x=%lld x_dtype=%d)", (long long)ld_x, x_dtype);
    const bool v4 = E % 4 == 0 && ld_outfit % 4 == 0 && (reinterpret_cast<uintptr_t>(outfits) & 15) == 0;
    const int V = v4 ? 4 : 1;
    int64_t blocks = ((int64_t)B * (io / V) + 256 * 4 - 1) / (256 * 4);
    if (blocks > (int64_t)ctx->sm_count * 8) blocks = (int64_t)ctx->sm_count * 8;
    cudaStream_t s = as_stream(stream);
#define LAUNCH(BO, VV) beam_build_kernel<BO, VV><<<(unsigned)blocks, 256, 0, s>>>(outfits, ld_outfit, Q, S, E, slot_base, pool, ld_pool, n_pool, pool_id, depth, beam_c, W, level, pos, B, inv_scale, out_x, ld_x)
    if (bo) { if (v4) LAUNCH(true, 4); else LAUNCH(true, 1); } else { if (v4) LAUNCH(false, 4); else LAUNCH(false, 1); }
#undef LAUNCH
    return codae_check_launch(ctx, "beam_build_kernel");
}

int codae_complete_beam_error(codae_ctx* ctx, const float* outfits, int64_t ld_outfit, int Q, int S, int E, const int64_t* slot_base,
                              const float* pool, int64_t ld_pool, int64_t n_pool, const int64_t* pool_id, int depth,
                              const int64_t* beam_c, int W, int level, const int64_t* pos, int B, float inv_scale, const float* y,
                              int64_t ld_y, float* err, void* stream) {
    int rc = check_beam(ctx, "codae_complete_beam_error", outfits, ld_outfit, Q, S, E, slot_base, pool, ld_pool, n_pool, pool_id,
                        depth, beam_c, W, level, pos, B);
    if (rc) return rc;
    CODAE_REQUIRE(ctx, y && err && ld_y >= (int64_t)S * E && (reinterpret_cast<uintptr_t>(y) & 3) == 0 &&
                           (reinterpret_cast<uintptr_t>(err) & 3) == 0,
                  "codae_complete_beam_error: bad output (ld_y=%lld)", (long long)ld_y);
    beam_error_kernel<<<sweep_grid(ctx, B), kThreads, 0, as_stream(stream)>>>(outfits, ld_outfit, Q, S, E, slot_base, pool, ld_pool,
                                                                               n_pool, pool_id, depth, beam_c, W, level, pos, B,
                                                                               inv_scale, y, ld_y, err);
    return codae_check_launch(ctx, "beam_error_kernel");
}

// Arguments shared by codae_revise_build and codae_revise_error.
static int check_revise(codae_ctx* ctx, const char* fn, const float* outfits, int64_t ld_outfit, int Q, int S, int E,
                        const int64_t* slot_base, const float* pool, int64_t ld_pool, int64_t n_pool, const int64_t* pool_id, int depth,
                        const int64_t* pos, int B) {
    CODAE_REQUIRE(ctx, ctx && outfits && slot_base && pool && pool_id && pos, "%s: NULL argument", fn);
    CODAE_REQUIRE(ctx, Q >= 1 && S >= 1 && S <= 64 && E >= 1 && (int64_t)S * E <= INT32_MAX && B >= 1,
                  "%s: bad shape Q=%d S=%d E=%d B=%d (Q, B >= 1, 1 <= S <= 64)", fn, Q, S, E, B);
    CODAE_REQUIRE(ctx, depth >= 1 && depth <= kMaxK && (int64_t)Q * (1 + (int64_t)S * depth) <= INT32_MAX,
                  "%s: bad grid depth=%d (1 <= depth <= %d, Q (1 + S depth) <= INT32_MAX)", fn, depth, kMaxK);
    CODAE_REQUIRE(ctx, n_pool >= 1 && ld_pool >= E && ld_outfit >= (int64_t)S * E,
                  "%s: bad pool or pitch (n_pool=%lld ld_pool=%lld ld_outfit=%lld)", fn, (long long)n_pool, (long long)ld_pool,
                  (long long)ld_outfit);
    const auto al = [](const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; };
    CODAE_REQUIRE(ctx, al(outfits, 4) && al(pool, 4) && al(slot_base, 8) && al(pool_id, 8) && al(pos, 8), "%s: misaligned buffer", fn);
    return CODAE_OK;
}

int codae_revise_build(codae_ctx* ctx, const float* outfits, int64_t ld_outfit, int Q, int S, int E, const int64_t* slot_base,
                       const float* pool, int64_t ld_pool, int64_t n_pool, const int64_t* pool_id, int depth, const int64_t* pos, int B,
                       float inv_scale, void* out_x, int x_dtype, int64_t ld_x, void* stream) {
    int rc = check_revise(ctx, "codae_revise_build", outfits, ld_outfit, Q, S, E, slot_base, pool, ld_pool, n_pool, pool_id, depth,
                          pos, B);
    if (rc) return rc;
    const int io = S * E;
    const bool bo = x_dtype == CODAE_BF16;
    CODAE_REQUIRE(ctx, out_x && ld_x >= io && (x_dtype == CODAE_F32 || bo) &&
                           (reinterpret_cast<uintptr_t>(out_x) & (bo ? 1 : 3)) == 0,
                  "codae_revise_build: bad output (ld_x=%lld x_dtype=%d)", (long long)ld_x, x_dtype);
    const bool v4 = E % 4 == 0 && ld_outfit % 4 == 0 && (reinterpret_cast<uintptr_t>(outfits) & 15) == 0;
    const int V = v4 ? 4 : 1;
    int64_t blocks = ((int64_t)B * (io / V) + 256 * 4 - 1) / (256 * 4);
    if (blocks > (int64_t)ctx->sm_count * 8) blocks = (int64_t)ctx->sm_count * 8;
    cudaStream_t s = as_stream(stream);
#define LAUNCH(BO, VV) revise_build_kernel<BO, VV><<<(unsigned)blocks, 256, 0, s>>>(outfits, ld_outfit, Q, S, E, slot_base, pool, ld_pool, n_pool, pool_id, depth, pos, B, inv_scale, out_x, ld_x)
    if (bo) { if (v4) LAUNCH(true, 4); else LAUNCH(true, 1); } else { if (v4) LAUNCH(false, 4); else LAUNCH(false, 1); }
#undef LAUNCH
    return codae_check_launch(ctx, "revise_build_kernel");
}

int codae_revise_error(codae_ctx* ctx, const float* outfits, int64_t ld_outfit, int Q, int S, int E, const int64_t* slot_base,
                       const float* pool, int64_t ld_pool, int64_t n_pool, const int64_t* pool_id, int depth, const int64_t* pos, int B,
                       float inv_scale, const float* y, int64_t ld_y, float* err, void* stream) {
    int rc = check_revise(ctx, "codae_revise_error", outfits, ld_outfit, Q, S, E, slot_base, pool, ld_pool, n_pool, pool_id, depth,
                          pos, B);
    if (rc) return rc;
    CODAE_REQUIRE(ctx, y && err && ld_y >= (int64_t)S * E && (reinterpret_cast<uintptr_t>(y) & 3) == 0 &&
                           (reinterpret_cast<uintptr_t>(err) & 3) == 0,
                  "codae_revise_error: bad output (ld_y=%lld)", (long long)ld_y);
    revise_error_kernel<<<sweep_grid(ctx, B), kThreads, 0, as_stream(stream)>>>(outfits, ld_outfit, Q, S, E, slot_base, pool, ld_pool,
                                                                                 n_pool, pool_id, depth, pos, B, inv_scale, y, ld_y, err);
    return codae_check_launch(ctx, "revise_error_kernel");
}

int codae_score_rank(codae_ctx* ctx, const void* catalog, int cat_dtype, int64_t n_rows, int64_t ld, int E,
                     const float* query, int Q, float inv_scale, int metric, const int64_t* true_idx,
                     const int64_t* subset_idx, int64_t n_subset, int64_t* out_rank, void* stream) {
    CODAE_REQUIRE(ctx, ctx && catalog && query && true_idx && out_rank, "codae_score_rank: NULL argument");
    CODAE_REQUIRE(ctx, Q >= 1 && Q <= 1024, "codae_score_rank: Q %d outside [1, 1024]", Q);
    const bool bf = cat_dtype == CODAE_BF16;
    const int vec = bf ? 8 : 4;
    CODAE_REQUIRE(ctx, E >= vec && E <= 4096 && E % vec == 0 && ld >= E && ld % vec == 0 &&
                           (reinterpret_cast<uintptr_t>(catalog) & 15) == 0 && (reinterpret_cast<uintptr_t>(query) & 15) == 0,
                  "codae_score_rank: E=%d ld=%lld must be multiples of %d", E, (long long)ld, vec);
    cudaStream_t s = as_stream(stream);
    if (!subset_idx) n_subset = n_rows;
    cudaError_t e = cudaMemsetAsync(out_rank, 0, sizeof(int64_t) * Q, s);
    if (e != cudaSuccess) return codae_fail(ctx, CODAE_ECUDA, "cudaMemsetAsync: %s", cudaGetErrorString(e));
    const int grid = sweep_grid(ctx, n_subset);
    const size_t smem = (size_t)Q * 12;
    unsigned long long* out = reinterpret_cast<unsigned long long*>(out_rank);
#define LAUNCH(MET, BF) score_rank_kernel<MET, BF><<<grid, kThreads, smem, s>>>(catalog, n_rows, ld, E, query, Q, inv_scale, true_idx, subset_idx, n_subset, out)
    if (metric == CODAE_METRIC_SQERR) { if (bf) LAUNCH(CODAE_METRIC_SQERR, true); else LAUNCH(CODAE_METRIC_SQERR, false); }
    else if (metric == CODAE_METRIC_COSINE) { if (bf) LAUNCH(CODAE_METRIC_COSINE, true); else LAUNCH(CODAE_METRIC_COSINE, false); }
    else return codae_fail(ctx, CODAE_EINVAL, "codae_score_rank: bad metric %d", metric);
#undef LAUNCH
    return codae_check_launch(ctx, "score_rank_kernel");
}

int codae_row_sqnorm(codae_ctx* ctx, const float* X, int64_t ld, int64_t rows, int E, float* out, void* stream) {
    CODAE_REQUIRE(ctx, ctx && X && out && rows >= 0 && E >= 1 && ld >= E, "codae_row_sqnorm: bad argument");
    if (rows == 0) return CODAE_OK;
    row_sqnorm_kernel<float><<<sweep_grid(ctx, rows), kThreads, 0, as_stream(stream)>>>(X, ld, rows, E, out);
    return codae_check_launch(ctx, "row_sqnorm_kernel");
}

int codae_rank_count(codae_ctx* ctx, const float* scores, int64_t ld, int Q, int64_t n, const float* cc, const float* qq,
                     int64_t* out_rank, void* stream) {
    CODAE_REQUIRE(ctx, ctx && scores && cc && qq && out_rank, "codae_rank_count: NULL argument");
    CODAE_REQUIRE(ctx, Q >= 1 && Q <= 65535 && n >= 0 && ld >= n + Q, "codae_rank_count: bad shape Q=%d n=%lld ld=%lld", Q, (long long)n, (long long)ld);
    cudaStream_t s = as_stream(stream);
    cudaError_t e = cudaMemsetAsync(out_rank, 0, sizeof(int64_t) * Q, s);
    if (e != cudaSuccess) return codae_fail(ctx, CODAE_ECUDA, "cudaMemsetAsync: %s", cudaGetErrorString(e));
    int gx = (int)((n + kThreads * 8 - 1) / (kThreads * 8));
    if (gx < 1) gx = 1;
    if (gx > ctx->sm_count) gx = ctx->sm_count;
    rank_count_kernel<<<dim3(gx, Q), kThreads, 0, s>>>(scores, ld, Q, n, cc, qq, reinterpret_cast<unsigned long long*>(out_rank));
    return codae_check_launch(ctx, "rank_count_kernel");
}

size_t codae_score_topk_batched_workspace_bytes(const codae_ctx* ctx, int cat_dtype, int64_t n_rows, int E, int Q, int k) {
    if (!ctx || Q < 1 || k < 1 || E < 1 || n_rows < 0 || (cat_dtype != CODAE_F32 && cat_dtype != CODAE_BF16)) return 0;
    return batched_layout(ctx, cat_dtype == CODAE_BF16, n_rows, E, Q, k).total;
}

static int score_topk_batched(codae_ctx* ctx, const void* catalog, int cat_dtype, int64_t n_rows, int64_t ld, int E,
                              int64_t row_offset, const float* query, int Q, float inv_scale, int metric, int k,
                              const uint8_t* allow, const int64_t* exclude, int n_exclude, float* out_score, int64_t* out_idx,
                              int* n_uncertified, int* uncertified, void* workspace, size_t ws_bytes, void* stream) {
    CODAE_REQUIRE(ctx, ctx && catalog && query && out_score && out_idx && n_uncertified && uncertified && workspace,
                  "codae_score_topk_batched: NULL argument");
    CODAE_REQUIRE(ctx, k >= 1 && k <= CODAE_TOPK_BATCHED_MAX_K, "codae_score_topk_batched: k %d outside [1, %d]", k,
                  CODAE_TOPK_BATCHED_MAX_K);
    CODAE_REQUIRE(ctx, Q >= 1 && n_rows >= 0, "codae_score_topk_batched: bad Q / n_rows");
    CODAE_REQUIRE(ctx, metric == CODAE_METRIC_SQERR || metric == CODAE_METRIC_COSINE, "codae_score_topk_batched: bad metric %d", metric);
    const bool bf = cat_dtype == CODAE_BF16;
    CODAE_REQUIRE(ctx, cat_dtype == CODAE_F32 || bf, "codae_score_topk_batched: bad cat_dtype %d", cat_dtype);
    const int vec = bf ? 8 : 4;
    CODAE_REQUIRE(ctx, E >= vec && E <= 4096 && E % vec == 0 && ld >= E && ld % vec == 0 &&
                           (reinterpret_cast<uintptr_t>(catalog) & 15) == 0,
                  "codae_score_topk_batched: E=%d ld=%lld must be multiples of %d (16-byte rows), E <= 4096", E, (long long)ld, vec);
    const BatchedLayout L = batched_layout(ctx, bf, n_rows, E, Q, k);
    if (ws_bytes < L.total)
        return codae_fail(ctx, CODAE_ENOMEM, "codae_score_topk_batched: workspace %zu < %zu bytes", ws_bytes, L.total);
    cudaStream_t s = as_stream(stream);
    unsigned char* ws = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
    float* m_key = reinterpret_cast<float*>(ws + L.m_key);
    int64_t* m_idx = reinterpret_cast<int64_t*>(ws + L.m_idx);
    float* ls = reinterpret_cast<float*>(ws + L.ls);
    int64_t* li = reinterpret_cast<int64_t*>(ws + L.li);
    float* cc = reinterpret_cast<float*>(ws + L.cc);
    float* qq = reinterpret_cast<float*>(ws + L.qq);
    __nv_bfloat16* qplanes = reinterpret_cast<__nv_bfloat16*>(ws + L.qplanes);
    __nv_bfloat16* cplanes = reinterpret_cast<__nv_bfloat16*>(ws + L.cplanes);
    const int64_t q_plane = (int64_t)Q * L.pitch;
    const int64_t c_plane = L.crow * L.pitch;

    cudaError_t e = cudaMemsetAsync(n_uncertified, 0, sizeof(int), s);
    if (e != cudaSuccess) return codae_fail(ctx, CODAE_ECUDA, "cudaMemsetAsync: %s", cudaGetErrorString(e));
    split_hm_kernel<<<sweep_grid(ctx, (int64_t)Q * L.pitch / 8), kThreads, 0, s>>>(query, E, Q, E, qplanes, L.pitch, q_plane);
    row_sqnorm_kernel<float><<<sweep_grid(ctx, Q), kThreads, 0, s>>>(query, E, Q, E, qq);
    const int64_t nl = (int64_t)L.W * Q * L.kp;
    if (metric == CODAE_METRIC_SQERR) list_init_kernel<CODAE_METRIC_SQERR><<<sweep_grid(ctx, nl / 8), kThreads, 0, s>>>(ls, li, nl);
    else list_init_kernel<CODAE_METRIC_COSINE><<<sweep_grid(ctx, nl / 8), kThreads, 0, s>>>(ls, li, nl);
    int rc = codae_check_launch(ctx, "codae_score_topk_batched prologue");
    if (rc) return rc;

    ScoreTcPass p;
    p.metric = metric;
    p.q_planes = qplanes; p.q_ld = L.pitch; p.q_plane_stride = q_plane;
    p.Q = Q; p.E = E; p.W = L.W; p.kp = L.kp;
    p.cc = cc; p.qq = qq;
    p.inv_scale = inv_scale; p.c_rel = batched_c_rel(E, bf);
    p.ls = ls; p.li = li;
    p.exclude = exclude; p.n_exclude = n_exclude;
    for (int64_t c0 = 0; c0 < n_rows; c0 += L.chunk) {
        const int64_t rows = n_rows - c0 < L.chunk ? n_rows - c0 : L.chunk;
        if (bf) {
            const __nv_bfloat16* src = reinterpret_cast<const __nv_bfloat16*>(catalog) + c0 * ld;
            row_sqnorm_kernel<__nv_bfloat16><<<sweep_grid(ctx, rows), kThreads, 0, s>>>(src, ld, rows, E, cc);
            p.cat = src; p.cat_planes = 1; p.cat_ld = ld; p.cat_plane_stride = 0;
        } else {
            const float* src = reinterpret_cast<const float*>(catalog) + c0 * ld;
            row_sqnorm_kernel<float><<<sweep_grid(ctx, rows), kThreads, 0, s>>>(src, ld, rows, E, cc);
            split_hm_kernel<<<sweep_grid(ctx, rows * L.pitch / 8), kThreads, 0, s>>>(src, ld, rows, E, cplanes, L.pitch, c_plane);
            p.cat = cplanes; p.cat_planes = 2; p.cat_ld = L.pitch; p.cat_plane_stride = c_plane;
        }
        rc = codae_check_launch(ctx, "codae_score_topk_batched chunk");
        if (rc) return rc;
        p.n_rows = rows; p.row0 = row_offset + c0;
        p.allow = allow ? allow + c0 : nullptr;
        for (int qb0 = 0; qb0 < L.QB; qb0 += L.G0) {
            p.qb0 = qb0;
            p.G = L.QB - qb0 < L.G0 ? L.QB - qb0 : L.G0;
            rc = codae_score_tc_pass(ctx, p, s);
            if (rc) return rc;
        }
    }
    merge_attrs();
    const size_t csmem = (size_t)(L.kp + k) * 12 + (size_t)E * 4 + 16;
    if (metric == CODAE_METRIC_SQERR) {
        topk_merge_kernel<CODAE_METRIC_SQERR><<<Q, kThreads, merge_smem(), s>>>(ls, li, L.W, Q, L.kp, m_key, m_idx, 0, 1);
        if (bf) score_certify_kernel<CODAE_METRIC_SQERR, true><<<Q, kThreads, csmem, s>>>(catalog, n_rows, ld, E, row_offset, query, inv_scale, k, L.kp, m_key, m_idx, out_score, out_idx, n_uncertified, uncertified);
        else score_certify_kernel<CODAE_METRIC_SQERR, false><<<Q, kThreads, csmem, s>>>(catalog, n_rows, ld, E, row_offset, query, inv_scale, k, L.kp, m_key, m_idx, out_score, out_idx, n_uncertified, uncertified);
    } else {
        topk_merge_kernel<CODAE_METRIC_COSINE><<<Q, kThreads, merge_smem(), s>>>(ls, li, L.W, Q, L.kp, m_key, m_idx, 0, 1);
        if (bf) score_certify_kernel<CODAE_METRIC_COSINE, true><<<Q, kThreads, csmem, s>>>(catalog, n_rows, ld, E, row_offset, query, inv_scale, k, L.kp, m_key, m_idx, out_score, out_idx, n_uncertified, uncertified);
        else score_certify_kernel<CODAE_METRIC_COSINE, false><<<Q, kThreads, csmem, s>>>(catalog, n_rows, ld, E, row_offset, query, inv_scale, k, L.kp, m_key, m_idx, out_score, out_idx, n_uncertified, uncertified);
    }
    return codae_check_launch(ctx, "score_certify_kernel");
}

int codae_score_topk_batched(codae_ctx* ctx, const void* catalog, int cat_dtype, int64_t n_rows, int64_t ld, int E,
                             int64_t row_offset, const float* query, int Q, float inv_scale, int metric, int k, float* out_score,
                             int64_t* out_idx, int* n_uncertified, int* uncertified, void* workspace, size_t ws_bytes,
                             void* stream) {
    return score_topk_batched(ctx, catalog, cat_dtype, n_rows, ld, E, row_offset, query, Q, inv_scale, metric, k, nullptr,
                              nullptr, 0, out_score, out_idx, n_uncertified, uncertified, workspace, ws_bytes, stream);
}

int codae_score_topk_batched_filtered(codae_ctx* ctx, const void* catalog, int cat_dtype, int64_t n_rows, int64_t ld, int E,
                                      int64_t row_offset, const float* query, int Q, float inv_scale, int metric, int k,
                                      const uint8_t* allow, const int64_t* exclude, int n_exclude, float* out_score,
                                      int64_t* out_idx, int* n_uncertified, int* uncertified, void* workspace, size_t ws_bytes,
                                      void* stream) {
    const int rc = check_filter(ctx, "codae_score_topk_batched_filtered", row_offset, exclude, n_exclude);
    if (rc) return rc;
    return score_topk_batched(ctx, catalog, cat_dtype, n_rows, ld, E, row_offset, query, Q, inv_scale, metric, k, allow, exclude,
                              n_exclude, out_score, out_idx, n_uncertified, uncertified, workspace, ws_bytes, stream);
}

}  // extern "C"
