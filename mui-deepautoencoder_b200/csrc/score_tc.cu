// K3b -- candidate pass of the batched complementarity top-k (codae_score_topk_batched, score.cu): Q queries against a
// catalog shard as ONE [Q, E] x [E, n] contraction on 5th-generation tensor cores.  The tensor cores only PROPOSE
// candidates: scores never leave TMEM, no [Q, n] matrix is written, and every thread keeps a short list of the rows whose
// approximate score could still beat its list.  score_certify_kernel (score.cu) re-scores the proposals with the sweep's own
// arithmetic and proves (or refutes) that nothing outside them can enter the top-k.
//
// Tile = 128 queries (M: TMEM lane t = query t of the block) x 256 catalog rows (N: TMEM column j = row j of the tile).
//   A: hi / mid bf16 planes of the fp32 queries (3-D tensor map, rows past Q read as zero -> padded lanes are ignored)
//   B: bf16 catalog rows in place (products c.q_hi + c.q_mid), or the hi / mid planes of an fp32 catalog chunk
//      (c_hi.q_hi + c_mid.q_hi + c_hi.q_mid); all products of a tile accumulate into one fp32 TMEM accumulator.
// CTA = 6 warps: warp 0 TMA producer, warp 1 TMEM allocator + MMA issuer, warps 2..5 epilogue.  The accumulator is
// double-buffered (2 x 256 columns = all of TMEM) and the shared-memory ring runs on across tiles, as in the persistent GEMM.
// Grid = G query blocks x W workers: CTA (w, qb) walks catalog tiles w, w + W, ... -- the CTAs of all query blocks read the same
// catalog tile at about the same time, so the catalog comes from HBM about once per launch and the other G - 1 reads hit L2.
//
// ---- Epilogue and the error bound ------------------------------------------------------------------------------------------
// Thread t turns column j into the approximate score a_j and a BOUND KEY that no exact score can beat:
//   SQERR  : a_j = qq - 2 s dot_j + s^2 cc_j,               key_j = a_j - delta_j,  delta_j = c_rel (qq + s^2 cc_j)
//   COSINE : a_j = dot_j / max(sqrt(cc_j qq), 1e-8),        key_j = a_j + delta_j,  delta_j = c_rel (1 + |a_j|)
// with s = inv_scale, dot_j the tensor-core sum, cc_j / qq the fp32 row / query norms, and s_j the fp32 score the sweep computes.
// Claim: |a_j - s_j| <= delta_j (so key_j is never better than s_j).  Let u = 2^-24, P = products per k-step (2 or 3), and
// D = sum_d |c_d| |q_d| <= sqrt(cc qq) (Cauchy-Schwarz; 2|s| sqrt(cc qq) <= qq + s^2 cc).
//   (1) dropped plane products: x = hi + mid + r with |r| <= 2^-16 |x| (two round-to-nearest bf16 splits, 2^-8 each).  bf16
//       catalog: c.q - c.(q_hi + q_mid) = c.r_q -> <= 2^-16 D.  fp32 catalog: c_hi r_q + c_mid q_mid + c_mid r_q + r_c q
//       -> <= 3.1 * 2^-16 D.  Both <= 2^-14 D.
//   (2) TMEM accumulation rounds toward zero (DESIGN 5): the P ceil(E/16) MMAs of a tile each round the running sum once
//       (error < 2^-23 of a partial sum <= (1 + 2^-8) D; the bf16 x bf16 products themselves are exact in fp32).  Taken with
//       a factor 4 of headroom for the adder's internal alignment: <= (P ceil(E/16) + 8) 2^-21 D.
//   (3) fp32 rounding of qq, cc and the epilogue: qq and cc are lane chains of E/32 fmas plus a 5-level shuffle tree
//       (relative error <= (E/32 + 6) u each); the epilogue's 3-4 roundings add <= 8 u (qq + 2|s| D + s^2 cc).
//   (4) the sweep's own rounding: the same chain / tree shape over E terms ((E/32 + 7) u of a sum of non-negative terms for
//       SQERR, of D for COSINE) plus the rounding of d = q - c s (<= 12 u (qq + s^2 cc) over the row).
//   SQERR: (1) + (2) scale with 2|s| D <= qq + s^2 cc; (3) + (4) sum to <= (3 E/32 + 47) u (qq + s^2 cc) <= (E/32 + 16) 2^-21
//   (qq + s^2 cc).  COSINE: the dot error over the (clamped) norm is <= ((1) + (2)) / sqrt(cc qq) <= 2^-14 + (2), the norm
//   roundings are relative errors of a_j, all <= (E/32 + 16) 2^-21 (1 + |a|).  Hence, with a factor (1 + 2^-10) for computing
//   delta itself in fp32:
//       c_rel = (2^-14 + (P ceil(E/16) + 8) 2^-21 + (E/32 + 16) 2^-21) (1 + 2^-10)            (batched_c_rel, score.cu)
//   (Operand values are assumed to lie in the normal fp32 range; a non-finite a_j or key_j becomes the BEST key, so such rows
//   always reach the re-scoring, which applies the sweep's NaN / inf rules exactly.)
// A key is compared with the thread's threshold -- the worst entry of its list, in registers -- and inserted into the sorted list
// (global memory, [W][Q][kp]) only when it beats it: after the first few tiles almost every column is one compare.
// Filtered calls (kFilter) test the row's mask byte and the query's exclusion list only behind that compare, and an ineligible
// row is skipped as if it were absent: the lists hold eligible rows only (the certification argument: score.cu).
#include <float.h>

#include "common.cuh"
#include "gemm.h"
#include "tc05_ptx.cuh"

namespace {

constexpr int kThreads = 192;
constexpr int kTileN = 256;                       // catalog rows per tile
constexpr int64_t kEmptyIdx = 0x7fffffffffffffffLL;

template <int NPB>     // catalog planes per stage
struct SCfg {
    static constexpr uint32_t kBTileBytes = kTileN * BK * 2;                      // 32 KB
    static constexpr uint32_t kStageBytes = 2 * kATileBytes + NPB * kBTileBytes;  // [A_hi | A_mid | B_hi (| B_mid)]
    static constexpr int kStages = NPB == 1 ? 3 : 2;
    static constexpr uint32_t kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;
};

template <int METRIC>
__device__ __forceinline__ bool key_better(float sa, int64_t ia, float sb, int64_t ib) {
    if (METRIC == CODAE_METRIC_SQERR) return sa < sb || (sa == sb && ia < ib);
    return sa > sb || (sa == sb && ia < ib);
}

template <int METRIC, int NPB, bool kFilter>
__global__ void __launch_bounds__(kThreads, 1) score_tc_kernel(const __grid_constant__ CUtensorMap tma_q,
                                                               const __grid_constant__ CUtensorMap tma_c, const ScoreTcPass p) {
    using C = SCfg<NPB>;
    constexpr int kS = C::kStages;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kS * C::kStageBytes);
    uint64_t* empty_bar = full_bar + kS;
    uint64_t* tmem_full_bar = empty_bar + kS;      // [2]
    uint64_t* tmem_empty_bar = tmem_full_bar + 2;  // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int qb = p.qb0 + (int)blockIdx.x % p.G, worker = (int)blockIdx.x / p.G;
    const int tiles = (int)((p.n_rows + kTileN - 1) / kTileN);
    const int num_kb = (p.E + BK - 1) / BK;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_q)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_c)) : "memory");
        for (int s = 0; s < kS; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full_bar[a], 1); mbar_init(&tmem_empty_bar[a], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, 2 * kTileN);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===== TMA producer: the ring index and phase run on across tiles =====
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            for (int t = worker; t < tiles; t += p.W) {
                for (int kb = 0; kb < num_kb; ++kb, s = (s + 1 == kS ? 0 : s + 1), ph ^= (s == 0)) {
                    mbar_wait(&empty_bar[s], ph ^ 1);
                    uint8_t* a_dst = smem + s * C::kStageBytes;
                    uint8_t* b_dst = a_dst + 2 * kATileBytes;
                    mbar_expect_tx(&full_bar[s], C::kStageBytes);
                    const int k0 = kb * BK;
                    tma_load_3d(&tma_q, &full_bar[s], a_dst, k0, qb * BM, 0);
                    tma_load_3d(&tma_q, &full_bar[s], a_dst + kATileBytes, k0, qb * BM, 1);
                    if constexpr (NPB == 1) {
                        tma_load_2d(&tma_c, &full_bar[s], b_dst, k0, t * kTileN);
                    } else {
                        tma_load_3d(&tma_c, &full_bar[s], b_dst, k0, t * kTileN, 0);
                        tma_load_3d(&tma_c, &full_bar[s], b_dst + C::kBTileBytes, k0, t * kTileN, 1);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: tile i accumulates into TMEM buffer i & 1 =====
        if (lane == 0) {
            const uint32_t idesc = make_idesc(kTileN, true, true);
            int s = 0, it = 0;
            uint32_t ph = 0;
            for (int t = worker; t < tiles; t += p.W, ++it) {
                const int acc = it & 1;
                mbar_wait(&tmem_empty_bar[acc], ((it >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * kTileN);
                for (int kb = 0; kb < num_kb; ++kb, s = (s + 1 == kS ? 0 : s + 1), ph ^= (s == 0)) {
                    mbar_wait(&full_bar[s], ph);
                    tc_fence_after();
                    const uint32_t a_addr = smem_u32(smem + s * C::kStageBytes);
                    const uint32_t b_addr = a_addr + 2 * kATileBytes;
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        const uint64_t ah = make_desc(a_addr + k * UMMA_K * 2, true), am = make_desc(a_addr + kATileBytes + k * UMMA_K * 2, true);
                        const uint64_t bh = make_desc(b_addr + k * UMMA_K * 2, true);
                        umma_bf16(d_tmem, ah, bh, idesc, (kb | k) != 0);
                        umma_bf16(d_tmem, am, bh, idesc, 1);
                        if constexpr (NPB == 2) umma_bf16(d_tmem, ah, make_desc(b_addr + C::kBTileBytes + k * UMMA_K * 2, true), idesc, 1);
                    }
                    umma_commit(&empty_bar[s]);
                }
                umma_commit(&tmem_full_bar[acc]);
            }
        }
    } else {
        // ===== epilogue: thread = query, column = catalog row; compare with the threshold, rarely insert =====
        const int qd = warp & 3;                      // TMEM lane quarter this warp may read
        const int qrow = qb * BM + qd * 32 + lane;
        const bool live = qrow < p.Q;
        const size_t list = ((size_t)worker * p.Q + (live ? qrow : 0)) * p.kp;
        float* Ls = p.ls + list;
        int64_t* Li = p.li + list;
        float thr_s = live ? Ls[p.kp - 1] : 0.f;
        int64_t thr_i = live ? Li[p.kp - 1] : 0;
        const float qq = live ? p.qq[qrow] : 0.f;
        const int64_t* ex = kFilter && live ? p.exclude + (size_t)qrow * p.n_exclude : nullptr;
        const float sc = p.inv_scale, s2 = sc * sc, m2s = -2.f * sc, c_rel = p.c_rel;
        int it = 0;
        for (int t = worker; t < tiles; t += p.W, ++it) {
            const int acc = it & 1;
            mbar_wait(&tmem_full_bar[acc], (it >> 1) & 1);
            tc_fence_after();
            const int64_t r0 = (int64_t)t * kTileN;
#pragma unroll 1
            for (int c = 0; c < kTileN / 32; ++c) {
                uint32_t v[32];
                tmem_ld32(tmem_base + ((uint32_t)(qd * 32) << 16) + (uint32_t)(acc * kTileN + c * 32), v);
                if (c == kTileN / 32 - 1) {
                    // every column of this buffer is in registers: hand it back to the MMA warp
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
                }
                const int64_t rc = r0 + c * 32;
                if (rc >= p.n_rows) continue;                                   // warp-uniform
                const float my_cc = rc + lane < p.n_rows ? __ldg(p.cc + rc + lane) : 0.f;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float ccj = __shfl_sync(0xffffffffu, my_cc, j);
                    if (!live || rc + j >= p.n_rows) continue;
                    const float dot = __uint_as_float(v[j]);
                    float key;
                    if (METRIC == CODAE_METRIC_SQERR) {
                        const float base = fmaf(s2, ccj, qq);
                        key = fmaf(m2s, dot, base) - c_rel * base;
                        if (!(fabsf(key) <= FLT_MAX)) key = -INFINITY;
                    } else {
                        const float a = dot / fmaxf(sqrtf(ccj * qq), 1e-8f);
                        key = a + c_rel * (1.f + fabsf(a));
                        if (!(fabsf(key) <= FLT_MAX)) key = INFINITY;
                    }
                    const int64_t gi = p.row0 + rc + j;
                    if (key_better<METRIC>(key, gi, thr_s, thr_i)) {
                        if constexpr (kFilter) {
                            if (p.allow && !p.allow[rc + j]) continue;
                            int e = 0;
                            while (e < p.n_exclude && ex[e] != gi) ++e;
                            if (e < p.n_exclude) continue;
                        }
                        int pos = p.kp - 1;
                        while (pos > 0) {
                            const float ps = Ls[pos - 1];
                            const int64_t pi = Li[pos - 1];
                            if (!key_better<METRIC>(key, gi, ps, pi)) break;
                            Ls[pos] = ps;
                            Li[pos] = pi;
                            --pos;
                        }
                        Ls[pos] = key;
                        Li[pos] = gi;
                        thr_s = Ls[p.kp - 1];
                        thr_i = Li[p.kp - 1];
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 2 * kTileN);
    }
}

template <int METRIC, int NPB, bool kFilter>
int launch_pass(codae_ctx* ctx, const ScoreTcPass& p, cudaStream_t s) {
    using C = SCfg<NPB>;
    static const cudaError_t attr =
        cudaFuncSetAttribute(score_tc_kernel<METRIC, NPB, kFilter>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::kSmemBytes);
    if (attr != cudaSuccess) return codae_fail(ctx, CODAE_ECUDA, "score_tc_kernel: cudaFuncSetAttribute: %s", cudaGetErrorString(attr));
    CUtensorMap mq, mc;
    int rc = codae_tc05_make_map(ctx, &mq, p.q_planes, p.Q, p.E, p.q_ld, BK, BM, 2, p.q_plane_stride);
    if (rc) return rc;
    rc = codae_tc05_make_map(ctx, &mc, p.cat, p.n_rows, p.E, p.cat_ld, BK, kTileN, NPB, p.cat_plane_stride);
    if (rc) return rc;
    score_tc_kernel<METRIC, NPB, kFilter><<<p.G * p.W, kThreads, C::kSmemBytes, s>>>(mq, mc, p);
    return codae_check_launch(ctx, "score_tc_kernel");
}

}  // namespace

int codae_score_tc_pass(codae_ctx* ctx, const ScoreTcPass& p, cudaStream_t s) {
    if (!ctx->encode_tiled) return codae_fail(ctx, CODAE_EARCH, "score_tc_kernel: no tensor-map encoder (driver too old)");
    if (p.n_rows < 1) return CODAE_OK;
    const bool two = p.cat_planes == 2;
    if (p.allow || p.n_exclude > 0) {
        if (p.metric == CODAE_METRIC_SQERR) return two ? launch_pass<CODAE_METRIC_SQERR, 2, true>(ctx, p, s) : launch_pass<CODAE_METRIC_SQERR, 1, true>(ctx, p, s);
        return two ? launch_pass<CODAE_METRIC_COSINE, 2, true>(ctx, p, s) : launch_pass<CODAE_METRIC_COSINE, 1, true>(ctx, p, s);
    }
    if (p.metric == CODAE_METRIC_SQERR) return two ? launch_pass<CODAE_METRIC_SQERR, 2, false>(ctx, p, s) : launch_pass<CODAE_METRIC_SQERR, 1, false>(ctx, p, s);
    return two ? launch_pass<CODAE_METRIC_COSINE, 2, false>(ctx, p, s) : launch_pass<CODAE_METRIC_COSINE, 1, false>(ctx, p, s);
}
