// K2 (tensor-core engine) -- bf16 GEMM on 5th-generation tensor cores: tcgen05.mma with the fp32
// accumulator in TMEM, operands staged in shared memory by TMA (128-byte swizzle), fused epilogues.
//
//   C[M,N] = epilogue( sum_k A(m,k) * B(n,k) )        A: M x K, B: N x K (each K-major or MN-major in HBM)
//
// One kernel covers nn.Linear's three contractions (see linear.cu):
//   fwd   Y  = X . W^T      A = X  K-major, B = W  K-major,  epilogue bias + ReLU
//   dgrad dX = dY . W       A = dY K-major, B = W  MN-major, epilogue ReLU mask of the layer input
//   wgrad dW = dY^T . X     A = dY MN-major, B = X MN-major, fp32 output into the flat gradient buffer
//
// CTA = 6 warps, one 128 x BN output tile: warp 0 = TMA producer (one elected lane), warp 1 = TMEM
// allocator + MMA issuer (one elected lane), warps 2..5 = epilogue (tcgen05.ld 32 lanes x 32 columns each).
// Pipeline: kStages smem slots guarded by full/empty mbarriers; tcgen05.commit releases a slot when the
// MMAs that read it have drained, and signals the epilogue after the last k-block.
//
// Two epilogues:
//   direct : TMEM -> registers -> fused epilogue -> HBM (bf16 activations of the large-batch layers)
//   staged : TMEM -> registers -> fp32 tile in shared memory (over the drained pipeline slots) -> coalesced
//            epilogue + store.  Used for fp32 outputs (weight gradients) and for split-K.
// Split-K (small batches: too few output tiles to keep 148 SMs streaming the weights): the k-blocks of one tile are
// spread over a thread-block CLUSTER along grid z; every CTA stages its partial tile in its own shared memory and,
// after a cluster barrier, CTA r reduces rows [128 r / S, 128 (r+1) / S) of all S partials through distributed
// shared memory (ld.shared::cluster) in rank order -- deterministic, no HBM round trip, no atomics.
// (A push variant -- st.shared::cluster into the owner, one barrier -- was measured slower: 8.1 vs 6.8 us per
// dependent launch; remote stores cost more than the second barrier saves.)
//
// Large problems (more than 2 output tiles per SM) use tc05_gemm_persistent_kernel further down: one CTA per SM walks
// tiles in L2-friendly groups, the accumulator is double-buffered in TMEM so that the epilogue of tile i overlaps the
// MMAs of tile i+1, and the shared-memory ring keeps running across tile boundaries.  Its 256-wide form runs as CTA PAIRS
// (tcgen05.mma.cta_group::2 on 256 x 256 tiles, see the comment above PCfg).
#include <cuda.h>
#include <stdlib.h>

#include "common.cuh"
#include "gemm.h"
#include "tc05_ptx.cuh"

namespace {

constexpr int kThreads = 192;
constexpr int kMaxSplit = 8;     // portable cluster size limit
// fp32-parity engine: k-blocks (of 64) accumulated in TMEM before the partial sum is folded into registers (x3_chunk_kb():
// tuning knob CODAE_X3_CHUNK_KB, read once)
inline int x3_chunk_kb() {
    static const int v = [] {
        const char* e = getenv("CODAE_X3_CHUNK_KB");
        const int x = e ? atoi(e) : 0;
        return x >= 1 && x <= 64 ? x : 8;
    }();
    return v;
}
constexpr uint32_t kPersistentStageBytes = 4 * 2 * 4096;   // persistent kernel, bulk-store epilogue: 4 warps x 2 boxes of 32 rows x 128 B

struct Params {
    int M, N, K;
    int a_kmajor, b_kmajor;
    void* C;
    long long ldc;
    int c_bf16;
    const float* bias;
    int act;
    const __nv_bfloat16* mask_src;
    long long ldm;
    int stages;                  // pipeline depth actually used (<= Cfg::kStages)
    int staged;                  // 1: epilogue through the shared-memory tile (required when gridDim.z > 1)
    int prefetch_b;              // 1: B holds weights no running predecessor writes: fetch its first tiles before the PDL wait
    int group_m;                 // persistent kernel: row-tiles per raster group
    int tma_store;               // 1: staged f32 tile leaves through cp.async.bulk.tensor stores (nsplit == 1, plain epilogue)
    double* sq_partial;          // f32 outputs only: slot [linear CTA id] receives the sum of squares of what this CTA stored (or NULL)
    unsigned long long* trace;   // debugging: CTA (0,0,0) writes %globaltimer stamps of its phases here (or NULL)
    int c_planes;                // NP == 3 only: 1 -> C is three bf16 planes (hi, mid, lo) c_plane_stride elements apart
    long long c_plane_stride;
    int chunk_kb;                // NP == 3, CH: k-blocks per TMEM accumulation chunk
    int trace_cta;               // debugging: linear (y * gridDim.x + x) id of the CTA that writes the trace stamps
    int tmem_cols;               // TMEM columns this CTA allocates (NP == 3: 2 BN while one chunk covers the k-range, else 4 BN)
};

// NP = operand planes: 1 (bf16 engine) or 3 (fp32-parity engine, CODAE_F32X3: every operand is the bf16 triple hi + mid + lo of
// an fp32 value; a stage holds [A_hi | A_mid | A_lo | B_hi | B_mid | B_lo]).  Six MMAs per k-step instead of one:
//     hi.hi                                  -> one of NB accumulators "big" (round-robin over the k-steps, see x3_load_sum)
//     hi.mid, mid.hi, mid.mid, hi.lo, lo.hi  -> accumulator "small", everything <= 2^-8 of the big terms
// and the epilogue adds them.  Dropped terms (mid.lo, lo.mid, lo.lo) are <= 2^-24 of a product, the representation error of
// the triple is 2^-24: measured against fp64 products of the same fp32 operands the contraction is as accurate as the FFMA engine
// and torch's fp32 GEMM (1.6e-7 vs 6e-7 vs 1.3e-6 of max |result| at 128 x 1536 x 1536, tools/probes/x3_chunk_accuracy.py).
template <int BN, int NP = 1>
struct Cfg {
    static_assert(NP == 1 || (NP == 3 && BN <= 128), "three-plane stages of a 256-wide tile do not fit in shared memory");
    static constexpr uint32_t kBTileBytes = BN * BK * 2;
    static constexpr uint32_t kStageBytes = NP * (kATileBytes + kBTileBytes);
    static constexpr int kStages = NP == 3 ? (BN == 128 ? 2 : 3) : ((BN == 256) ? 4 : (BN == 128 ? 6 : 8));
    static constexpr uint32_t kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;
    static constexpr uint32_t kTmemCols = NP == 3 ? 512 : BN;        // NP == 3: all columns -- one or two sets of NB + 1 accumulators
};

// fp32-parity engine: 32 columns of one TMEM accumulator set -> registers: ((big_0 + big_1) + ...) + small, round-to-nearest adds.
// The "big" products (hi.hi) are dealt round-robin over nbig accumulators (k-step j -> accumulator j % nbig): TMEM accumulation
// rounds TOWARD ZERO, a systematic error that grows with the number of MMA steps one accumulator takes and -- unlike
// round-to-nearest noise -- adds up coherently from layer to layer (measured: forward error 3.7e-7 after layer 1 growing to
// 1.2e-6 after layer 6 with one accumulator, where the FFMA engine stays at 4e-7).  nbig accumulators see 1/nbig of the steps each.
// NB "big" accumulators per set (compile time): x3_nbig<BN, CH>() fills the 512 TMEM columns with one set (k-range within one
// chunk) or two sets (chunked).
template <int BN, bool CH>
__host__ __device__ constexpr int x3_nbig() { return 512 / ((CH ? 2 : 1) * BN) - 1 > 4 ? 4 : 512 / ((CH ? 2 : 1) * BN) - 1; }
template <int NB, bool kBatched>
__device__ __forceinline__ void x3_load_sum(uint32_t taddr_set_chunk, int bn, uint32_t (&v)[32]) {
    if constexpr (kBatched) {
        // all NB + 1 loads in flight before the single tcgen05.wait::ld: one TMEM round trip per 32-column chunk
        uint32_t u[NB][32];
        tmem_ld32_nowait(taddr_set_chunk, v);
#pragma unroll
        for (int i = 1; i <= NB; ++i) tmem_ld32_nowait(taddr_set_chunk + (uint32_t)(i * bn), u[i - 1]);
        tmem_ld_wait();
#pragma unroll
        for (int i = 1; i <= NB; ++i) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(u[i - 1][j]));
        }
    } else {
        tmem_ld32(taddr_set_chunk, v);
        uint32_t u[32];
#pragma unroll
        for (int i = 1; i <= NB; ++i) {                           // i == NB: the "small" accumulator
            tmem_ld32(taddr_set_chunk + (uint32_t)(i * bn), u);
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(u[j]));
        }
    }
}

// One operand tile per plane: plane pl lands plane_bytes after plane pl - 1.
template <int NP>
__device__ __forceinline__ void tma_load_op(const CUtensorMap* map, uint64_t* bar, uint8_t* dst, int c0, int c1, uint32_t plane_bytes) {
    if constexpr (NP == 1) {
        tma_load_2d(map, bar, dst, c0, c1);
    } else {
#pragma unroll
        for (int pl = 0; pl < NP; ++pl) tma_load_3d(map, bar, dst + pl * plane_bytes, c0, c1, pl);
    }
}

__device__ __forceinline__ void trace_stamp(const Params& p, int slot) {
    if (p.trace && (int)(blockIdx.y * gridDim.x + blockIdx.x) == p.trace_cta && blockIdx.z == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        p.trace[slot] = t;
    }
}

// Sum of squares of the stored outputs (the weight-gradient norm of clip_grad_norm_, taken while the gradient tile is
// still in registers): the four epilogue warps combine their per-thread sums with a fixed tree and thread 64 writes the
// CTA's slot.  Called by all 128 epilogue threads (warps 2..5); named barrier 1.
__device__ __forceinline__ void sq_partial_store(double* slot, double sq, double* red) {
    const int lane = threadIdx.x & 31, w = (threadIdx.x >> 5) - 2;
    sq = warp_sum(sq);
    if (lane == 0) red[w] = sq;
    asm volatile("bar.sync 1, 128;" ::: "memory");
    if (threadIdx.x == 64) *slot = (red[0] + red[1]) + (red[2] + red[3]);
}
template <int W>
__device__ __forceinline__ float chunk_sq(const float (&f)[W], int col0, int n) {
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < W; ++j) if (col0 + j < n) s = fmaf(f[j], f[j], s);
    return s;
}

// Fused epilogue of one W-column chunk (W = 16 or 32) of one output row: bias + activation / ReLU mask of the
// layer input, cast, 128-bit stores.
template <int W>
__device__ __forceinline__ void epilogue_chunk(const Params& p, int row, int col0, float (&f)[W]) {
    const bool full = col0 + W <= p.N;
    if (p.bias) {
#pragma unroll
        for (int j = 0; j < W; ++j) if (full || col0 + j < p.N) f[j] += __ldg(p.bias + col0 + j);
    }
    if (p.act == CODAE_ACT_RELU) {
#pragma unroll
        for (int j = 0; j < W; ++j) f[j] = fmaxf(f[j], 0.f);
    }
    if (p.mask_src) {
        const __nv_bfloat16* mrow = p.mask_src + (long long)row * p.ldm + col0;
        if (full) {
#pragma unroll
            for (int j = 0; j < W / 8; ++j) {
                const uint4 mv = *reinterpret_cast<const uint4*>(mrow + 8 * j);
                const uint32_t w[4] = {mv.x, mv.y, mv.z, mv.w};
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    if (!(bf16_lo(w[t]) > 0.f)) f[8 * j + 2 * t] = 0.f;
                    if (!(bf16_hi(w[t]) > 0.f)) f[8 * j + 2 * t + 1] = 0.f;
                }
            }
        } else {
#pragma unroll
            for (int j = 0; j < W; ++j)
                if (col0 + j < p.N && !(__bfloat162float(mrow[j]) > 0.f)) f[j] = 0.f;
        }
    }
}
template <int W>
__device__ __forceinline__ void store_chunk(const Params& p, int row, int col0, float (&f)[W]) {
    const bool full = col0 + W <= p.N;
    epilogue_chunk<W>(p, row, col0, f);
    if (p.c_planes) {
        // fp32-parity engine: the value leaves as its bf16 triple, one 8-byte store per plane and four columns
        __nv_bfloat16* crow = reinterpret_cast<__nv_bfloat16*>(p.C) + (long long)row * p.ldc + col0;
        if (full) {
#pragma unroll
            for (int j = 0; j < W / 4; ++j)
                store_planes4(crow + 4 * j, p.c_plane_stride, make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]));
        } else {
#pragma unroll
            for (int j = 0; j < W; ++j) if (col0 + j < p.N) store_planes1(crow + j, p.c_plane_stride, f[j]);
        }
    } else if (p.c_bf16) {
        __nv_bfloat16* crow = reinterpret_cast<__nv_bfloat16*>(p.C) + (long long)row * p.ldc + col0;
        if (full) {
#pragma unroll
            for (int j = 0; j < W / 8; ++j) {
                uint4 o;
                o.x = pack_bf16x2(f[8 * j + 0], f[8 * j + 1]);
                o.y = pack_bf16x2(f[8 * j + 2], f[8 * j + 3]);
                o.z = pack_bf16x2(f[8 * j + 4], f[8 * j + 5]);
                o.w = pack_bf16x2(f[8 * j + 6], f[8 * j + 7]);
                *reinterpret_cast<uint4*>(crow + 8 * j) = o;
            }
        } else {
#pragma unroll
            for (int j = 0; j < W; ++j) if (col0 + j < p.N) crow[j] = __float2bfloat16_rn(f[j]);
        }
    } else {
        float* crow = reinterpret_cast<float*>(p.C) + (long long)row * p.ldc + col0;
        if (full) {
#pragma unroll
            for (int j = 0; j < W / 4; ++j)
                *reinterpret_cast<float4*>(crow + 4 * j) = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
        } else {
#pragma unroll
            for (int j = 0; j < W; ++j) if (col0 + j < p.N) crow[j] = f[j];
        }
    }
}

// CH (NP == 3 only): the k-range of a CTA is longer than one chunk -> chunked accumulation with the running sum in registers
// (BN more registers per epilogue thread; the short-k-range variant stays light enough for 2 CTAs per SM).
template <int BN, int NP, bool CH = false>
__global__ void __launch_bounds__(kThreads, 1) tc05_gemm_kernel(const __grid_constant__ CUtensorMap tma_a,
                                                                const __grid_constant__ CUtensorMap tma_b,
                                                                const __grid_constant__ CUtensorMap tma_c, const Params p) {
    using C = Cfg<BN, NP>;
    constexpr uint32_t kBOff = NP * kATileBytes;      // B planes follow the A planes of a stage
    constexpr int NB = NP == 3 ? x3_nbig<BN, CH>() : 1;   // "big" accumulators per TMEM set (fp32-parity engine)
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int nstages = p.stages;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + nstages * C::kStageBytes);
    uint64_t* empty_bar = full_bar + nstages;
    uint64_t* tmem_full_bar = empty_bar + nstages;     // [2] (NP == 1 uses slot 0 only)
    uint64_t* tmem_empty_bar = tmem_full_bar + 2;      // [2] NP == 3: chunked accumulation, see Params::chunk_kb
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
    constexpr int kStagePitch = BN + 4;               // floats per row of the staged fp32 tile
    __shared__ double sq_red[4];
    double sq_acc = 0.0;                              // epilogue threads: sum of squares of the values this thread stored

    pdl_launch_dependents();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nsplit = gridDim.z;
    // Single-pass launches walk the tiles column-tile-major: the CTAs of the LAST column tile get the highest linear ids.  tcgen05
    // kernels run one CTA per SM, so a grid of more than 148 CTAs has a second wave; the weight gradients of an augmented layer
    // (K = 128 k + 1: the last column tile holds only the bias column) then leave the cheap one-column tiles for it instead of full
    // ones (156 tiles: second wave = 8 ragged tiles, which also start as soon as the first-wave ragged tiles have exited).
    int m_idx = blockIdx.y, n_idx = blockIdx.x;
    if (nsplit == 1) {
        const int lin = blockIdx.y * gridDim.x + blockIdx.x;
        n_idx = lin / (int)gridDim.y;
        m_idx = lin - n_idx * (int)gridDim.y;
    }
    const int m0 = m_idx * BM, n0 = n_idx * BN;
    if (threadIdx.x == 0) trace_stamp(p, 0);                       // kernel entry
    const int total_kb = (p.K + BK - 1) / BK;
    const int kb_per = (total_kb + nsplit - 1) / nsplit;
    const int kb_begin = blockIdx.z * kb_per;
    const int num_kb = min(total_kb, kb_begin + kb_per) - kb_begin;      // >= 1 by construction (host)

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_a)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_b)) : "memory");
        if (p.tma_store) asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_c)) : "memory");
        for (int s = 0; s < nstages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full_bar[a], 1); mbar_init(&tmem_empty_bar[a], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0) trace_stamp(p, 1);                       // prologue done (barriers, TMEM)
    // Weight tiles of the first ring pass are requested NOW, while the stream predecessor (which produces A) is still
    // finishing: the full barrier of a slot is armed for both operands, B arrives early, A is requested after the wait.
    const int npre = p.prefetch_b ? min(num_kb, nstages) : 0;
    if (warp == 0 && lane == 0) {
        for (int kb = 0; kb < npre; ++kb) {
            uint8_t* b_dst = smem + kb * C::kStageBytes + kBOff;
            mbar_expect_tx(&full_bar[kb], C::kStageBytes);
            const int k0 = (kb_begin + kb) * BK;
            if (p.b_kmajor) {
                tma_load_op<NP>(&tma_b, &full_bar[kb], b_dst, k0, n0, C::kBTileBytes);
            } else {
#pragma unroll
                for (int j = 0; j < BN / 64; ++j) tma_load_op<NP>(&tma_b, &full_bar[kb], b_dst + j * 8192, n0 + 64 * j, k0, C::kBTileBytes);
            }
        }
    }
    pdl_wait();
    if (threadIdx.x == 0) trace_stamp(p, 2);                       // predecessor complete     // everything above overlapped the previous kernel's tail; operands and outputs are global memory

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            for (int kb = 0; kb < num_kb; ++kb, s = (s + 1 == nstages ? 0 : s + 1), ph ^= (s == 0)) {
                const bool b_requested = kb < npre;                                          // first ring pass, before the wait
                if (!b_requested) mbar_wait(&empty_bar[s], ph ^ 1);
                uint8_t* a_dst = smem + s * C::kStageBytes;
                uint8_t* b_dst = a_dst + kBOff;
                if (!b_requested) mbar_expect_tx(&full_bar[s], C::kStageBytes);
                const int k0 = (kb_begin + kb) * BK;
                if (p.a_kmajor) {
                    tma_load_op<NP>(&tma_a, &full_bar[s], a_dst, k0, m0, kATileBytes);              // box {64 k, 128 m}
                } else {
                    tma_load_op<NP>(&tma_a, &full_bar[s], a_dst, m0, k0, kATileBytes);              // box {64 m, 64 k} x 2
                    tma_load_op<NP>(&tma_a, &full_bar[s], a_dst + 8192, m0 + 64, k0, kATileBytes);
                }
                if (b_requested) continue;
                if (p.b_kmajor) {
                    tma_load_op<NP>(&tma_b, &full_bar[s], b_dst, k0, n0, C::kBTileBytes);           // box {64 k, BN n}
                } else {
#pragma unroll
                    for (int j = 0; j < BN / 64; ++j) tma_load_op<NP>(&tma_b, &full_bar[s], b_dst + j * 8192, n0 + 64 * j, k0, C::kBTileBytes);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            // a ragged last column tile only pays for the MMA width it needs (multiples of 16)
            const int n_eff = min(BN, ((p.N - n0) + 15) & ~15);
            const uint32_t idesc = make_idesc(n_eff, p.a_kmajor != 0, p.b_kmajor != 0);
            const uint32_t a_adv = p.a_kmajor ? (UMMA_K * 2) : (UMMA_K * 128);   // bytes per UMMA_K step
            const uint32_t b_adv = p.b_kmajor ? (UMMA_K * 2) : (UMMA_K * 128);
            int s = 0;
            uint32_t ph = 0;
            for (int kb = 0; kb < num_kb; ++kb, s = (s + 1 == nstages ? 0 : s + 1), ph ^= (s == 0)) {
                mbar_wait(&full_bar[s], ph);
                if (kb == 0) trace_stamp(p, 3);                    // first operands landed
                tc_fence_after();
                const uint32_t a_addr = smem_u32(smem + s * C::kStageBytes);
                const uint32_t b_addr = a_addr + kBOff;
#pragma unroll
                for (int k = 0; k < BK / UMMA_K; ++k) {
                    if constexpr (NP == 1) {
                        umma_bf16(tmem_base, make_desc(a_addr + k * a_adv, p.a_kmajor != 0),
                                  make_desc(b_addr + k * b_adv, p.b_kmajor != 0), idesc, (kb | k) != 0);
                    } else {
                        // chunked accumulation: k-blocks [ci chunk_kb, (ci + 1) chunk_kb) accumulate into TMEM set ci & 1 from
                        // zero; the epilogue warps fold finished chunks into fp32 registers with round-to-nearest adds
                        const int ci = CH ? kb / p.chunk_kb : 0, within = kb - ci * p.chunk_kb;
                        const int step = within * (BK / UMMA_K) + k;                     // k-step inside the chunk
                        const uint32_t set_base = tmem_base + (uint32_t)((ci & 1) * (NB + 1) * BN);
                        const uint32_t d_big = set_base + (uint32_t)((step % NB) * BN), d_small = set_base + (uint32_t)(NB * BN);
                        if (CH && within == 0 && k == 0) {
                            mbar_wait(&tmem_empty_bar[ci & 1], (((uint32_t)ci >> 1) & 1) ^ 1);     // set drained (first use: free)
                            tc_fence_after();
                        }
                        const bool ak = p.a_kmajor != 0, bk = p.b_kmajor != 0;
                        const uint64_t ah = make_desc(a_addr + k * a_adv, ak), am = make_desc(a_addr + kATileBytes + k * a_adv, ak),
                                       al = make_desc(a_addr + 2 * kATileBytes + k * a_adv, ak);
                        const uint64_t bh = make_desc(b_addr + k * b_adv, bk), bm = make_desc(b_addr + C::kBTileBytes + k * b_adv, bk),
                                       bl = make_desc(b_addr + 2 * C::kBTileBytes + k * b_adv, bk);
                        umma_bf16(d_big, ah, bh, idesc, step >= NB);              // big: the first use of an accumulator overwrites
                        umma_bf16(d_small, ah, bm, idesc, step != 0);               // small: five terms <= 2^-8 of the big one
                        umma_bf16(d_small, am, bh, idesc, 1);
                        umma_bf16(d_small, am, bm, idesc, 1);
                        umma_bf16(d_small, ah, bl, idesc, 1);
                        umma_bf16(d_small, al, bh, idesc, 1);
                    }
                }
                umma_commit(&empty_bar[s]);          // slot reusable once these MMAs have read it
                if constexpr (NP == 3 && CH) {
                    if ((kb + 1) % p.chunk_kb == 0 && kb + 1 < num_kb) umma_commit(&tmem_full_bar[(kb / p.chunk_kb) & 1]);   // chunk complete
                }
            }
            umma_commit(&tmem_full_bar[(NP == 3 && CH) ? ((num_kb - 1) / p.chunk_kb) & 1 : 0]);      // accumulator complete
            trace_stamp(p, 4);                       // all MMAs issued
        }
    } else {
        // ===== epilogue, part 1: TMEM -> registers -> HBM (direct) or -> shared-memory tile (staged) =====
        const int q = warp & 3;                      // TMEM lane quarter this warp may read
        uint32_t tmem_acc = tmem_base;               // accumulator set the last (or only) chunk lands in
        [[maybe_unused]] float racc[(NP == 3 && CH) ? BN : 1];   // running fp32 sum of the finished chunks (this thread's row)
        if constexpr (NP == 3 && CH) {
#pragma unroll
            for (int j = 0; j < BN; ++j) racc[j] = 0.f;
            const int nchunks = (num_kb + p.chunk_kb - 1) / p.chunk_kb;
            for (int ci = 0; ci + 1 < nchunks; ++ci) {
                const int set = ci & 1;
                mbar_wait(&tmem_full_bar[set], ((uint32_t)ci >> 1) & 1);
                tc_fence_after();
#pragma unroll
                for (int c = 0; c < BN / 32; ++c) {
                    uint32_t v[32];
                    x3_load_sum<NB, false>(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(set * (NB + 1) * BN + c * 32), BN, v);
#pragma unroll
                    for (int j = 0; j < 32; ++j) racc[c * 32 + j] += __uint_as_float(v[j]);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tmem_empty_bar[set]);
            }
            const int last = nchunks - 1;
            mbar_wait(&tmem_full_bar[last & 1], ((uint32_t)last >> 1) & 1);
            tmem_acc = tmem_base + (uint32_t)((last & 1) * (NB + 1) * BN);
        } else {
            mbar_wait(tmem_full_bar, 0);
        }
        if (threadIdx.x == 64) trace_stamp(p, 5);                  // accumulator complete
        tc_fence_after();
        const int row = m0 + q * 32 + lane;
        const bool row_ok = row < p.M;
        float* stage_row = reinterpret_cast<float*>(smem) + (size_t)(q * 32 + lane) * kStagePitch;
        auto emit = [&](const int c, uint32_t (&v)[32]) {
            const int col0 = n0 + c * 32;
            if (!p.staged) {
                if (!row_ok || col0 >= p.N) return;
                float f[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
                store_chunk<32>(p, row, col0, f);
                if (p.sq_partial) sq_acc += (double)chunk_sq<32>(f, col0, p.N);
            } else if (p.tma_store) {
                // box c = [128 rows][32 floats] at smem + c * 16 KB in the 128-byte-swizzle layout the store's tensor map
                // names: 16-byte chunk j of row r sits at chunk j ^ (r & 7), so the 8 lanes of a store phase (8 consecutive
                // rows) hit 8 distinct bank groups
                uint8_t* brow = smem + c * 16384 + (q * 32 + lane) * 128;
                const int sw = lane & 7;
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    *reinterpret_cast<float4*>(brow + ((j ^ sw) << 4)) =
                        make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                                    __uint_as_float(v[4 * j + 3]));
                if (p.sq_partial && row_ok && col0 < p.N) {
                    float f[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
                    sq_acc += (double)chunk_sq<32>(f, col0, p.N);
                }
            } else {
                // row pitch BN+4 floats: the 8 lanes of a 128-bit store phase hit 8 distinct 16-byte bank groups
                float4* dst = reinterpret_cast<float4*>(stage_row + c * 32);
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    dst[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                         __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
            }
        };
        if constexpr (NP == 3) {
            // last chunk: (big + small) + the running sum; fully unrolled, racc stays in registers
#pragma unroll
            for (int c = 0; c < BN / 32; ++c) {
                uint32_t v[32];
                x3_load_sum<NB, !CH>(tmem_acc + ((uint32_t)(q * 32) << 16) + (uint32_t)(c * 32), BN, v);
                if constexpr (CH) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + racc[c * 32 + j]);
                }
                emit(c, v);
            }
        } else {
#pragma unroll 1
            for (int c = 0; c < BN / 32; ++c) {
                uint32_t v[32];
                tmem_ld32(tmem_acc + ((uint32_t)(q * 32) << 16) + (uint32_t)(c * 32), v);
                emit(c, v);
            }
        }
    }

    if (p.staged && p.tma_store) {
        // ===== epilogue, part 2 (bulk store): the tile leaves through the TMA unit, BN/32 boxes of 128 x 32 floats =====
        // The store's tensor map ends at the last whole 16-byte unit of a row (n4 columns): TMA clips a ragged row end at
        // 16-byte granularity (measured: it zero-fills up to 3 floats past the last valid column), so the N & 3 tail
        // columns -- the bias-gradient column of an augmented layer -- are stored by the threads and padding stays untouched.
        if (warp >= 2) {
            const int n4 = p.N & ~3;
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic-proxy smem writes -> async proxy
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (threadIdx.x == 64) {
                trace_stamp(p, 6);
#pragma unroll 1
                for (int c = 0; c < BN / 32; ++c)
                    if (n0 + c * 32 < n4) tma_store_2d(&tma_c, smem + c * 16384, n0 + c * 32, m0);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            if (n4 < p.N && n4 >= n0 && n4 < n0 + BN) {
                const int rl = threadIdx.x - 64, row = m0 + rl;
                if (row < p.M) {
                    const int c = (n4 - n0) >> 5, j = ((n4 - n0) & 31) >> 2;
                    const float* src = reinterpret_cast<const float*>(smem + c * 16384 + rl * 128 + ((j ^ (rl & 7)) << 4));
                    float* crow = reinterpret_cast<float*>(p.C) + (long long)row * p.ldc + n4;
                    for (int e = 0; e < p.N - n4; ++e) crow[e] = src[e];
                }
            }
            if (threadIdx.x == 64) {
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // smem is released at the barrier below
                trace_stamp(p, 8);
            }
        }
    } else if (p.staged) {
        // ===== epilogue, part 2 (staged): [cluster reduce +] fused epilogue + coalesced stores =====
        __syncwarp();
        if (threadIdx.x == 64) trace_stamp(p, 6);                  // tile staged in shared memory
        if (nsplit > 1) cluster_sync();                      // every thread of every CTA of the cluster
        else if (warp >= 2) asm volatile("bar.sync 1, 128;" ::: "memory");
        if (threadIdx.x == 64) trace_stamp(p, 7);                  // cluster barrier 1 passed
        if (warp >= 2) {
            const int t = threadIdx.x - 64;                  // 0..127
            const int rank = blockIdx.z;                     // == %cluster_ctarank (cluster spans grid z only)
            const int r_begin = (rank * BM) / nsplit, r_end = ((rank + 1) * BM) / nsplit;
            constexpr int kVecPerRow = BN / 4;
            const int items = (r_end - r_begin) * kVecPerRow;
            const uint32_t stage_base = smem_u32(smem);
            for (int it = t; it < items; it += 128) {
                const int rl = r_begin + it / kVecPerRow;    // row within the tile
                const int c4 = it % kVecPerRow;
                const uint32_t off = (uint32_t)(rl * kStagePitch + 4 * c4) * 4u;
                float4 acc;
                if (nsplit == 1) {
                    acc = *reinterpret_cast<const float4*>(smem + off);
                } else {
                    // all remote loads in flight before the first add (a rolled loop serialises one DSMEM round trip
                    // of ~110 ns per split: measured 2.5 us for this phase), then summed in rank order
                    float4 part[kMaxSplit];
#pragma unroll
                    for (int sp = 0; sp < kMaxSplit; ++sp)
                        if (sp < nsplit) part[sp] = ld_dsmem_f4(stage_base + off, (uint32_t)sp);
                    acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int sp = 0; sp < kMaxSplit; ++sp)
                        if (sp < nsplit) { acc.x += part[sp].x; acc.y += part[sp].y; acc.z += part[sp].z; acc.w += part[sp].w; }
                }
                const int row = m0 + rl, col = n0 + 4 * c4;
                if (row >= p.M || col >= p.N) continue;
                float f[4] = {acc.x, acc.y, acc.z, acc.w};
                const bool full = col + 4 <= p.N;
                if (p.bias) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) if (full || col + j < p.N) f[j] += __ldg(p.bias + col + j);
                }
                if (p.act == CODAE_ACT_RELU) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) f[j] = fmaxf(f[j], 0.f);
                }
                if (p.mask_src) {
                    const __nv_bfloat16* mrow = p.mask_src + (long long)row * p.ldm + col;
                    if (full) {
                        const uint2 mv = *reinterpret_cast<const uint2*>(mrow);
                        if (!(bf16_lo(mv.x) > 0.f)) f[0] = 0.f;
                        if (!(bf16_hi(mv.x) > 0.f)) f[1] = 0.f;
                        if (!(bf16_lo(mv.y) > 0.f)) f[2] = 0.f;
                        if (!(bf16_hi(mv.y) > 0.f)) f[3] = 0.f;
                    } else {
#pragma unroll
                        for (int j = 0; j < 4; ++j) if (col + j < p.N && !(__bfloat162float(mrow[j]) > 0.f)) f[j] = 0.f;
                    }
                }
                if (p.sq_partial) sq_acc += (double)chunk_sq<4>(f, col, p.N);
                if (p.c_planes) {
                    __nv_bfloat16* crow = reinterpret_cast<__nv_bfloat16*>(p.C) + (long long)row * p.ldc + col;
                    if (full) {
                        store_planes4(crow, p.c_plane_stride, make_float4(f[0], f[1], f[2], f[3]));
                    } else {
#pragma unroll
                        for (int j = 0; j < 4; ++j) if (col + j < p.N) store_planes1(crow + j, p.c_plane_stride, f[j]);
                    }
                } else if (p.c_bf16) {
                    __nv_bfloat16* crow = reinterpret_cast<__nv_bfloat16*>(p.C) + (long long)row * p.ldc + col;
                    if (full) {
                        uint2 o;
                        o.x = pack_bf16x2(f[0], f[1]);
                        o.y = pack_bf16x2(f[2], f[3]);
                        *reinterpret_cast<uint2*>(crow) = o;
                    } else {
#pragma unroll
                        for (int j = 0; j < 4; ++j) if (col + j < p.N) crow[j] = __float2bfloat16_rn(f[j]);
                    }
                } else {
                    float* crow = reinterpret_cast<float*>(p.C) + (long long)row * p.ldc + col;
                    if (full) {
                        *reinterpret_cast<float4*>(crow) = make_float4(f[0], f[1], f[2], f[3]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 4; ++j) if (col + j < p.N) crow[j] = f[j];
                    }
                }
            }
        }
        if (threadIdx.x == 64) trace_stamp(p, 8);                  // reduced + stored
        if (nsplit > 1) cluster_sync();                      // peers may still be reading this CTA's tile
        if (threadIdx.x == 64) trace_stamp(p, 9);                  // cluster barrier 2 passed
    }
    if (p.sq_partial && warp >= 2)
        sq_partial_store(p.sq_partial + ((size_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x, sq_acc, sq_red);
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
    }
    if (p.trace && threadIdx.x == 0) {          // debugging: slot 10 = exit of CTA (0,0,0), slot 11 = last CTA exit, slot 12 = first entry
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        if ((int)(blockIdx.y * gridDim.x + blockIdx.x) == p.trace_cta && blockIdx.z == 0) p.trace[10] = t;
        atomicMax(&p.trace[11], t);
    }
}

// ---- persistent variant for large problems (tiles > 2 x SMs): one CTA per SM walks output tiles t, t + grid, ... -----------
// The accumulator is double-buffered in TMEM (2 x BN columns): while the epilogue warps drain tile i (tcgen05.ld, fused
// epilogue, stores), the MMA warp already accumulates tile i+1 and the producer keeps the shared-memory ring full across
// tile boundaries.  Tiles are walked m-fastest so that concurrently running CTAs share the same weight tile in L2.
// Tile order of the persistent kernel: groups of group_m (16) row-tiles; inside a group all column-tiles of one row-tile
// column are adjacent (m fastest).  The ~148 tiles in flight then span group_m x ~9 tiles: every operand tile is shared by
// many concurrent CTAs and the working set (tens of MB) stays in L2.  (Plain m-fastest order re-streamed the whole 67 MB
// activation matrix for every pair of column tiles: ncu showed 350-530 MB of DRAM reads for 100-135 MB of operands.)
__device__ __forceinline__ void tile_coords(int t, int tiles_m, int tiles_n, int group_m, int& m_idx, int& n_idx) {
    const int per_group = group_m * tiles_n;
    const int g = t / per_group, r = t - g * per_group;
    const int gm = min(group_m, tiles_m - g * group_m);
    m_idx = g * group_m + r % gm;
    n_idx = r / gm;
}

//
// kPair (BN = 256, launched as clusters of 2 along x): a CTA PAIR works on one 256 x 256 tile with cta_group::2 MMAs.  CTA r of
// the pair stages its own 128 rows of A and its own HALF (128 columns) of B -- 32 KB per k-block instead of 48 KB, six ring
// slots instead of four --, the leader (cluster rank 0) issues one 256 x 256 x 16 MMA per k-step that reads both CTAs' shared
// memory and leaves rows 0..127 of the accumulator in the leader's TMEM and rows 128..255 in the peer's; every CTA drains its
// own 128 x 256 half exactly like the single-CTA kernel.  Barriers: the full barriers live in the leader and count both CTAs'
// TMA bytes (the peer's loads name the leader's barrier, cp.async.bulk.tensor.cta_group::2); empty and accumulator-full
// barriers are per CTA and signalled by multicast tcgen05.commit; the leader's accumulator-empty barriers take the arrivals of
// all eight epilogue warps of the pair.  Same k order per output element as the single-CTA kernel.
template <int BN, bool kPair = false>
struct PCfg {
    static_assert(!kPair || BN == 256, "CTA pairs work on 256 x 256 tiles");
    static constexpr uint32_t kBTileBytes = (kPair ? BN / 2 : BN) * BK * 2;      // this CTA's share of B
    static constexpr uint32_t kStageBytes = kATileBytes + kBTileBytes;
    static constexpr int kStages = kPair ? 6 : Cfg<BN>::kStages;
    static constexpr uint32_t kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;
};

template <int BN, bool kPair>
__global__ void __launch_bounds__(kThreads, 1) tc05_gemm_persistent_kernel(const __grid_constant__ CUtensorMap tma_a,
                                                                           const __grid_constant__ CUtensorMap tma_b,
                                                                           const __grid_constant__ CUtensorMap tma_c,
                                                                           const Params p) {
    using C = PCfg<BN, kPair>;
    constexpr int kRowsPerTile = kPair ? 2 * BM : BM;         // rows of the tile a CTA (pair) works on
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    constexpr int kS = C::kStages;
    // bulk-store epilogue: 2 x 4 KB staging boxes per epilogue warp between the ring and the barriers (only allocated then)
    uint8_t* stage_base = smem + kS * C::kStageBytes;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(stage_base + (p.tma_store ? kPersistentStageBytes : 0));
    uint64_t* empty_bar = full_bar + kS;
    uint64_t* tmem_full_bar = empty_bar + kS;          // [2]
    uint64_t* tmem_empty_bar = tmem_full_bar + 2;      // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
    __shared__ double sq_red[4];

    pdl_launch_dependents();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles_m = (p.M + kRowsPerTile - 1) / kRowsPerTile, tiles_n = (p.N + BN - 1) / BN;
    const int total_tiles = tiles_m * tiles_n;
    const int num_kb = (p.K + BK - 1) / BK;
    // work items: a CTA (kPair: a pair) walks tiles worker, worker + num_workers, ...
    const int rank = kPair ? (int)cluster_ctarank() : 0;
    const int worker = kPair ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int num_workers = kPair ? (int)(gridDim.x >> 1) : (int)gridDim.x;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_a)) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_b)) : "memory");
        if (p.tma_store) asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tma_c)) : "memory");
        for (int s = 0; s < kS; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full_bar[a], 1); mbar_init(&tmem_empty_bar[a], kPair ? 8 : 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) {
        if constexpr (kPair) tmem_alloc_pair(tmem_slot, 2 * BN);
        else tmem_alloc(tmem_slot, 2 * BN);
    }
    tc_fence_before();
    if constexpr (kPair) cluster_sync();      // the peer's barriers are initialised before anything is signalled across the pair
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();

    if (warp == 0) {
        // ===== TMA producer: the ring index and phase run on across tiles =====
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            for (int t = worker; t < total_tiles; t += num_workers) {
                int m_idx, n_idx;
                tile_coords(t, tiles_m, tiles_n, p.group_m, m_idx, n_idx);
                const int m0 = m_idx * kRowsPerTile + rank * BM, n0 = n_idx * BN;
                if constexpr (kPair) {
                    // this CTA's half of B: columns [n0 + rank n_half, + n_half) of the n_eff columns the pair's MMA covers
                    const int n_half = min(BN, ((p.N - n0) + 31) & ~31) >> 1;
                    const int nb0 = n0 + rank * n_half;
                    for (int kb = 0; kb < num_kb; ++kb, s = (s + 1 == kS ? 0 : s + 1), ph ^= (s == 0)) {
                        mbar_wait(&empty_bar[s], ph ^ 1);                       // own slot drained (multicast commit of the leader)
                        uint8_t* a_dst = smem + s * C::kStageBytes;
                        uint8_t* b_dst = a_dst + kATileBytes;
                        if (rank == 0) mbar_expect_tx(&full_bar[s], 2 * C::kStageBytes);   // the leader's barrier counts both CTAs' bytes
                        const uint32_t bar = mapa_u32(smem_u32(&full_bar[s]), 0);
                        const int k0 = kb * BK;
                        if (p.a_kmajor) {
                            tma_load_2d_pair(&tma_a, bar, a_dst, k0, m0);
                        } else {
                            tma_load_2d_pair(&tma_a, bar, a_dst, m0, k0);
                            tma_load_2d_pair(&tma_a, bar, a_dst + 8192, m0 + 64, k0);
                        }
                        if (p.b_kmajor) {
                            tma_load_2d_pair(&tma_b, bar, b_dst, k0, nb0);                  // box {64 k, 128 n}
                        } else {
                            tma_load_2d_pair(&tma_b, bar, b_dst, nb0, k0);                  // box {64 n, 64 k} x 2
                            tma_load_2d_pair(&tma_b, bar, b_dst + 8192, nb0 + 64, k0);
                        }
                    }
                } else {
                    for (int kb = 0; kb < num_kb; ++kb, s = (s + 1 == kS ? 0 : s + 1), ph ^= (s == 0)) {
                        mbar_wait(&empty_bar[s], ph ^ 1);
                        uint8_t* a_dst = smem + s * C::kStageBytes;
                        uint8_t* b_dst = a_dst + kATileBytes;
                        mbar_expect_tx(&full_bar[s], C::kStageBytes);
                        const int k0 = kb * BK;
                        if (p.a_kmajor) {
                            tma_load_2d(&tma_a, &full_bar[s], a_dst, k0, m0);
                        } else {
                            tma_load_2d(&tma_a, &full_bar[s], a_dst, m0, k0);
                            tma_load_2d(&tma_a, &full_bar[s], a_dst + 8192, m0 + 64, k0);
                        }
                        if (p.b_kmajor) {
                            tma_load_2d(&tma_b, &full_bar[s], b_dst, k0, n0);
                        } else {
#pragma unroll
                            for (int j = 0; j < BN / 64; ++j) tma_load_2d(&tma_b, &full_bar[s], b_dst + j * 8192, n0 + 64 * j, k0);
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: tile i accumulates into TMEM buffer i & 1 =====
        if (lane == 0 && rank == 0) {                 // kPair: the leader issues the pair's MMAs
            const uint32_t a_adv = p.a_kmajor ? (UMMA_K * 2) : (UMMA_K * 128);
            const uint32_t b_adv = p.b_kmajor ? (UMMA_K * 2) : (UMMA_K * 128);
            int s = 0;
            uint32_t ph = 0;
            int it = 0;
            for (int t = worker; t < total_tiles; t += num_workers, ++it) {
                int m_idx, n_idx;
                tile_coords(t, tiles_m, tiles_n, p.group_m, m_idx, n_idx);
                // a ragged last column tile (the bias column of the augmented weight gradient: 1 of 256 columns) only
                // pays for the MMA width it needs (multiples of 16; a pair: multiples of 32, half from each CTA)
                const int n_eff = kPair ? min(BN, ((p.N - n_idx * BN) + 31) & ~31) : min(BN, ((p.N - n_idx * BN) + 15) & ~15);
                const uint32_t idesc = make_idesc(n_eff, p.a_kmajor != 0, p.b_kmajor != 0, kRowsPerTile);
                const int acc = it & 1;
                const uint32_t acc_ph = (it >> 1) & 1;
                // epilogue has drained this buffer (first use: free); kPair: the warps of both CTAs
                if constexpr (kPair) mbar_wait_cluster(&tmem_empty_bar[acc], acc_ph ^ 1);
                else mbar_wait(&tmem_empty_bar[acc], acc_ph ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                for (int kb = 0; kb < num_kb; ++kb, s = (s + 1 == kS ? 0 : s + 1), ph ^= (s == 0)) {
                    mbar_wait(&full_bar[s], ph);
                    tc_fence_after();
                    const uint32_t a_addr = smem_u32(smem + s * C::kStageBytes);
                    const uint32_t b_addr = a_addr + kATileBytes;
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        const uint64_t ad = make_desc(a_addr + k * a_adv, p.a_kmajor != 0), bd = make_desc(b_addr + k * b_adv, p.b_kmajor != 0);
                        if constexpr (kPair) umma_bf16_pair(d_tmem, ad, bd, idesc, (kb | k) != 0);
                        else umma_bf16(d_tmem, ad, bd, idesc, (kb | k) != 0);
                    }
                    if constexpr (kPair) umma_commit_pair(&empty_bar[s]);
                    else umma_commit(&empty_bar[s]);
                }
                if constexpr (kPair) umma_commit_pair(&tmem_full_bar[acc]);
                else umma_commit(&tmem_full_bar[acc]);
            }
        }
    } else {
        // ===== epilogue warps: drain buffer i & 1 while the MMA warp fills the other one =====
        const int q = warp & 3;
        int it = 0;
        double sq_acc = 0.0;
        // bulk-store epilogue (p.tma_store): every warp stages 32 rows x 128 B (32 floats, or 2 x 32 bf16) in one of its two
        // 4 KB boxes (128-byte swizzle) and lane 0 issues a cp.async.bulk.tensor store; a box is rewritten after the store
        // issued two units earlier has read it.  The store's tensor map ends at the last whole 16-byte unit of a row (TMA
        // clips ragged row ends at that granularity); the tail columns are stored by the threads.
        const bool tma_st = p.tma_store != 0;
        const int tail_mask = p.c_bf16 ? 7 : 3;
        const int n4 = p.N & ~tail_mask;
        uint8_t* wbuf = stage_base + q * 8192;
        int unit = 0;
        for (int t = worker; t < total_tiles; t += num_workers, ++it) {
            const int acc = it & 1;
            const uint32_t acc_ph = (it >> 1) & 1;
            int m_idx, n_idx;
            tile_coords(t, tiles_m, tiles_n, p.group_m, m_idx, n_idx);
            const int m0 = m_idx * kRowsPerTile + rank * BM, n0 = n_idx * BN;
            mbar_wait(&tmem_full_bar[acc], acc_ph);
            tc_fence_after();
            const int row = m0 + q * 32 + lane;
            const bool row_ok = row < p.M;
            const int n_chunks = min(BN / 32, (p.N - n0 + 31) / 32);        // >= 1
#pragma unroll 1
            for (int c = 0; c < n_chunks; ++c) {
                uint32_t v[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN + c * 32), v);
                if (c == n_chunks - 1) {
                    // every column of this buffer is in registers: hand it back to the MMA warp before the last stores
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        if constexpr (kPair) mbar_arrive_cluster(mapa_u32(smem_u32(&tmem_empty_bar[acc]), 0));   // the leader's barrier
                        else mbar_arrive(&tmem_empty_bar[acc]);
                    }
                }
                const int col0 = n0 + c * 32;
                if (!tma_st) {
                    if (!row_ok || col0 >= p.N) continue;
                    float f[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
                    store_chunk<32>(p, row, col0, f);
                    if (p.sq_partial) sq_acc += (double)chunk_sq<32>(f, col0, p.N);
                    continue;
                }
                float f[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
                if (row_ok) {
                    epilogue_chunk<32>(p, row, col0, f);
                    if (p.sq_partial) sq_acc += (double)chunk_sq<32>(f, col0, p.N);
                }
                const bool opens = !p.c_bf16 || (c & 1) == 0;                        // first (or only) half of a box
                const bool closes = !p.c_bf16 || (c & 1) == 1 || c == n_chunks - 1;
                uint8_t* box = wbuf + (unit & 1) * 4096;
                if (opens) {
                    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                    __syncwarp();
                }
                uint8_t* brow = box + lane * 128;
                const int sw = lane & 7;
                if (p.c_bf16) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        uint4 o;
                        o.x = pack_bf16x2(f[8 * j + 0], f[8 * j + 1]);
                        o.y = pack_bf16x2(f[8 * j + 2], f[8 * j + 3]);
                        o.z = pack_bf16x2(f[8 * j + 4], f[8 * j + 5]);
                        o.w = pack_bf16x2(f[8 * j + 6], f[8 * j + 7]);
                        *reinterpret_cast<uint4*>(brow + ((((c & 1) * 4 + j) ^ sw) << 4)) = o;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        *reinterpret_cast<float4*>(brow + ((j ^ sw) << 4)) = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
                }
                if (row_ok && n4 < p.N && n4 >= col0 && n4 < col0 + 32) {               // ragged tail of the row
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        if (col0 + j >= n4 && col0 + j < p.N) {
                            if (p.c_bf16) reinterpret_cast<__nv_bfloat16*>(p.C)[(long long)row * p.ldc + col0 + j] = __float2bfloat16_rn(f[j]);
                            else reinterpret_cast<float*>(p.C)[(long long)row * p.ldc + col0 + j] = f[j];
                        }
                    }
                }
                if (closes) {
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) {
                        const int cbase = p.c_bf16 ? (n0 + (c & ~1) * 32) : col0;
                        if (cbase < n4 && m0 + q * 32 < p.M) tma_store_2d(&tma_c, box, cbase, m0 + q * 32);
                        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                    }
                    ++unit;
                }
            }
        }
        if (tma_st) {
            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // boxes are read before the CTA exits
            __syncwarp();
        }
        if (p.sq_partial) sq_partial_store(p.sq_partial + blockIdx.x, sq_acc, sq_red);
    }
    tc_fence_before();
    if constexpr (kPair) cluster_sync();      // neither CTA leaves (or frees TMEM) while the other may still signal or write into it
    else __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        if constexpr (kPair) tmem_dealloc_pair(tmem_base, 2 * BN);
        else tmem_dealloc(tmem_base, 2 * BN);
    }
}


int g_trace_cta = 0;
unsigned long long* g_trace_buf = nullptr;   // set through codae_debug_set_trace (debugging hook, not part of the ABI)

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 2-D bf16 tensor map over a row-major [rows, cols] matrix with pitch ld (elements); box {box_cols, box_rows}.
// planes == 3: a 3-D map {cols, rows, plane} over three such matrices plane_stride elements apart, box depth 1.
int make_map(codae_ctx* ctx, CUtensorMap* map, const void* base, long long rows, long long cols, long long ld, int box_cols,
             int box_rows, int planes = 1, long long plane_stride = 0) {
    const cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)planes};
    const cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)plane_stride * 2};
    const cuuint32_t box[3] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = reinterpret_cast<EncodeTiledFn>(ctx->encode_tiled)(
        map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, planes == 1 ? 2 : 3, const_cast<void*>(base), dims, strides, box, estr,
        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return codae_fail(ctx, CODAE_ECUDA, "cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
    return CODAE_OK;
}

// Launch shape of one contraction, decided up front (also reported by codae_tc05_gemm_ctas).
struct Plan {
    int nsplit;        // cluster split-K factor (grid z)
    bool staged;       // epilogue through the shared-memory tile
    bool persistent;   // one CTA per SM walking tiles
    bool pair = false; // persistent kernel as CTA pairs (cta_group::2, 256 x 256 tiles)
    int gx, gy;        // output tiles along N and M
    int ctas;          // CTAs the launch will have (= sum-of-squares slots it writes)
    int stages = 0;    // NP == 3: pipeline depth chosen by x3_geometry (0: the launch code's default)
    int tmem_cols = 0; // NP == 3: TMEM columns per CTA
};
// 2-D tensor map over the row-major OUTPUT [rows, cols] with pitch ld (elements) for cp.async.bulk.tensor stores:
// boxes of 128 bytes x box_rows rows, 128-byte swizzle (f32: 32 columns, bf16: 64 columns).
int make_store_map(codae_ctx* ctx, CUtensorMap* map, void* base, int c_dtype, long long rows, long long cols, long long ld,
                   int box_rows) {
    const bool bf = c_dtype == CODAE_BF16;
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * (bf ? 2 : 4)};
    const cuuint32_t box[2] = {(cuuint32_t)(bf ? 64 : 32), (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = reinterpret_cast<EncodeTiledFn>(ctx->encode_tiled)(
        map, bf ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr,
        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return codae_fail(ctx, CODAE_ECUDA, "cuTensorMapEncodeTiled (store map) failed (CUresult %d)", (int)r);
    return CODAE_OK;
}

// ---- fp32-parity engine: launch geometry ---------------------------------------------------------------------------------
// Measured on a B200 (tools/probes/occ_probe.cu): a kernel that contains tcgen05.alloc is scheduled ONE CTA per SM whatever its
// shared memory and registers are (cudaOccupancyMaxActiveBlocksPerMultiprocessor returns 1 even at 1 KB).  The bf16 split-K
// launches (24 clusters of 6) happen to fit the GPCs; with 72 KB three-plane stages the same geometry was measured as a second
// wave that doubled the launch (21 vs 12 us per dgrad): the cluster size is therefore the largest one for which
// cudaOccupancyMaxActiveClusters says every cluster of the launch is resident at once.
template <int BN, bool CH>
bool x3_set_smem_attr() {
    static bool ok = cudaFuncSetAttribute(tc05_gemm_kernel<BN, 3, CH>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)Cfg<BN, 3>::kSmemBytes) == cudaSuccess;
    return ok;
}
template <int BN, bool CH>
int x3_max_clusters(int nsplit, size_t smem) {
    static std::mutex mu;
    static int cache[kMaxSplit + 1][Cfg<BN, 3>::kStages + 1];
    const int st = (int)(smem / Cfg<BN, 3>::kStageBytes);
    std::lock_guard<std::mutex> lk(mu);
    int& slot = cache[nsplit][st];
    if (slot == 0) {
        x3_set_smem_attr<BN, CH>();
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(1, 1, nsplit);
        cfg.blockDim = dim3(kThreads);
        cfg.dynamicSmemBytes = smem;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 1;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = nsplit;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, tc05_gemm_kernel<BN, 3, CH>, &cfg) != cudaSuccess || n < 1) {
            cudaGetLastError();
            n = 1 << 20;      // no answer: do not constrain
        }
        slot = n;
    }
    return slot;
}
template <int BN, int NP = 1>
Plan make_plan(const codae_ctx* ctx, const Tc05Gemm& g) {
    Plan pl;
    pl.gx = (g.N + BN - 1) / BN;
    pl.gy = (g.M + BM - 1) / BM;
    // split-K over a thread-block cluster (see the header comment): only when the tiles alone would leave most SMs
    // idle and every split still gets at least 2 k-blocks.
    const int tiles = pl.gx * pl.gy;
    const int total_kb = (g.K + BK - 1) / BK;
    int nsplit = 1;
    if (ctx->splitk && 2 * tiles <= ctx->sm_count && total_kb >= 8) {
        int want = ctx->sm_count / tiles;
        if (want > total_kb / 2) want = total_kb / 2;
        if (want > kMaxSplit) want = kMaxSplit;
        static const int dgrad_maxsplit = getenv("CODAE_DGRAD_MAXSPLIT") ? atoi(getenv("CODAE_DGRAD_MAXSPLIT")) : 0;
        if (dgrad_maxsplit > 0 && g.a_kmajor && !g.b_kmajor && want > dgrad_maxsplit) want = dgrad_maxsplit;
        if (want > 1) {
            const int kb_per = (total_kb + want - 1) / want;
            nsplit = (total_kb + kb_per - 1) / kb_per;               // no empty split
        }
    }
    if constexpr (NP == 3) {
        using C3 = Cfg<BN, 3>;
        auto smem_for = [](int stages) { return (size_t)stages * C3::kStageBytes + 1024 + 256; };
        // split-K: shrink the cluster until every cluster of the launch is resident at once
        while (nsplit > 1) {
            const int kb_per = (total_kb + nsplit - 1) / nsplit;
            const int st = kb_per < C3::kStages ? kb_per : C3::kStages;
            const int fit = kb_per > x3_chunk_kb() ? x3_max_clusters<BN, true>(nsplit, smem_for(st)) : x3_max_clusters<BN, false>(nsplit, smem_for(st));
            if (fit >= tiles) break;
            int want = nsplit - 1;
            const int kb2 = (total_kb + want - 1) / want;
            nsplit = (total_kb + kb2 - 1) / kb2;
        }
        const int kb_per = (total_kb + nsplit - 1) / nsplit;
        pl.tmem_cols = 512;       // one set of NB + 1 accumulators, or two sets when the k-range is chunked (x3_nbig)
        const int st = kb_per < C3::kStages ? kb_per : C3::kStages;
        pl.stages = st;
    }
    pl.nsplit = nsplit;
    // staged (coalesced) epilogue: always for split-K; for fp32 outputs only while the grid is at most ~2 waves
    // (measured: the direct epilogue is faster for the 4096-wide weight gradients, 247 vs 261 us)
    pl.staged = nsplit > 1 || (g.c_dtype == CODAE_F32 && tiles <= 2 * ctx->sm_count);
    pl.persistent = NP == 1 && nsplit == 1 && !pl.staged && ctx->persistent && tiles > 2 * ctx->sm_count;
    pl.pair = pl.persistent && BN == 256 && ctx->cta_pair && ctx->sm_count >= 2;
    pl.ctas = pl.persistent ? (pl.pair ? (ctx->sm_count & ~1) : ctx->sm_count) : tiles * nsplit;
    return pl;
}

template <int BN, int NP = 1>
int launch(codae_ctx* ctx, const Tc05Gemm& g, cudaStream_t s) {
    using C = Cfg<BN, NP>;
    const Plan pl = make_plan<BN, NP>(ctx, g);
    if (g.sq_partial && (g.c_dtype != CODAE_F32 || g.sq_slots != pl.ctas))
        return codae_fail(ctx, CODAE_EINVAL, "codae_tc05_gemm: %d sum-of-squares slots passed, this launch writes %d (f32 outputs only)",
                          g.sq_slots, pl.ctas);
    CUtensorMap ma, mb;
    int rc;
    // A(m,k): K-major storage [M rows, K cols]; MN-major storage [K rows, M cols]
    if (g.a_kmajor) rc = make_map(ctx, &ma, g.A, g.M, g.K, g.lda, BK, BM, NP, g.a_plane_stride);
    else rc = make_map(ctx, &ma, g.A, g.K, g.M, g.lda, 64, BK, NP, g.a_plane_stride);
    if (rc) return rc;
    if (g.b_kmajor) rc = make_map(ctx, &mb, g.B, g.N, g.K, g.ldb, BK, BN, NP, g.b_plane_stride);
    else rc = make_map(ctx, &mb, g.B, g.K, g.N, g.ldb, 64, BK, NP, g.b_plane_stride);
    if (rc) return rc;
    Params p;
    p.c_planes = g.c_dtype == CODAE_F32X3 ? 1 : 0;
    p.c_plane_stride = g.c_plane_stride;
    p.M = g.M; p.N = g.N; p.K = g.K;
    p.a_kmajor = g.a_kmajor; p.b_kmajor = g.b_kmajor;
    p.C = g.C; p.ldc = g.ldc; p.c_bf16 = g.c_dtype == CODAE_BF16;
    p.bias = g.bias; p.act = g.act;
    p.mask_src = reinterpret_cast<const __nv_bfloat16*>(g.mask_src); p.ldm = g.ldm;
    p.sq_partial = g.sq_partial;
    const int total_kb = (g.K + BK - 1) / BK;
    const int nsplit = pl.nsplit;
    p.trace = g_trace_buf;
    p.trace_cta = g_trace_cta;
    p.staged = pl.staged ? 1 : 0;
    // bulk-store epilogue: plain f32 tiles of a single-pass launch (the weight gradients of the small-batch step)
    p.tma_store = (ctx->tma_store && pl.staged && nsplit == 1 && g.c_dtype == CODAE_F32 && !g.bias && g.act == CODAE_ACT_NONE &&
                   !g.mask_src && (g.ldc % 4) == 0) ? 1 : 0;
    CUtensorMap mc;
    memset(&mc, 0, sizeof(mc));
    if (p.tma_store) {
        rc = make_store_map(ctx, &mc, g.C, CODAE_F32, g.M, g.N & ~3, g.ldc, BM);     // whole 16-byte units only; the kernel stores the tail
        if (rc) return rc;
    }
    p.prefetch_b = (g.b_is_weight && ctx->pdl && ctx->weight_prefetch) ? 1 : 0;
    p.group_m = 16;
    if constexpr (NP == 1) if (pl.persistent) {
        static bool pattr_set = false;
        if (!pattr_set) {
            cudaError_t e = cudaFuncSetAttribute(tc05_gemm_persistent_kernel<BN, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)(C::kSmemBytes + kPersistentStageBytes));
            if constexpr (BN == 256) {
                if (e == cudaSuccess)
                    e = cudaFuncSetAttribute(tc05_gemm_persistent_kernel<BN, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)(PCfg<BN, true>::kSmemBytes + kPersistentStageBytes));
            }
            if (e != cudaSuccess) return codae_fail(ctx, CODAE_ECUDA, "cudaFuncSetAttribute(smem=%u): %s", C::kSmemBytes + kPersistentStageBytes, cudaGetErrorString(e));
            pattr_set = true;
        }
        // bulk-store epilogue of the persistent kernel (opt-in): needs a row of at least one whole 16-byte unit
        const int unit = g.c_dtype == CODAE_BF16 ? 8 : 4;
        p.tma_store = (ctx->tma_store_persistent && (g.N & ~(unit - 1)) > 0 && (g.ldc % unit) == 0) ? 1 : 0;
        if (p.tma_store) {
            rc = make_store_map(ctx, &mc, g.C, g.c_dtype, g.M, g.N & ~(unit - 1), g.ldc, 32);
            if (rc) return rc;
        }
        // raster group: 16 row-tiles measured best on the 4096-wide step (8: 7.48, 16: 7.14, 32: 7.33, 64: 7.43 ms/step);
        // CODAE_GROUP_M overrides it for tuning runs (read once)
        static int env_group_m = -1;
        if (env_group_m < 0) {
            const char* e = getenv("CODAE_GROUP_M");
            env_group_m = (e && atoi(e) > 0) ? atoi(e) : 16;
        }
        p.group_m = env_group_m;
        p.stages = C::kStages;
        static const bool debug_persistent = getenv("CODAE_DEBUG_PLAN") != nullptr;
        if (debug_persistent)
            fprintf(stderr, "codae plan: M=%d N=%d K=%d BN=%d persistent pair %d tma_store %d ctas %d\n", g.M, g.N, g.K, BN, (int)pl.pair,
                    p.tma_store, pl.ctas);
        if constexpr (BN == 256) if (pl.pair) {
            // CTA pairs: 256-row tiles (raster groups of group_m / 2 of them), this CTA's B box is 128 columns wide
            using PC = PCfg<BN, true>;
            p.group_m = env_group_m > 1 ? env_group_m / 2 : 1;
            p.stages = PC::kStages;
            if (g.b_kmajor) {
                rc = make_map(ctx, &mb, g.B, g.N, g.K, g.ldb, BK, BN / 2);
                if (rc) return rc;
            }
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(pl.ctas);
            cfg.blockDim = dim3(kThreads);
            cfg.dynamicSmemBytes = PC::kSmemBytes + (p.tma_store ? kPersistentStageBytes : 0);
            cfg.stream = s;
            cudaLaunchAttribute attr[2];
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = 2;
            attr[0].val.clusterDim.y = 1;
            attr[0].val.clusterDim.z = 1;
            int na = 1;
            if (codae_pdl_allowed(ctx, s)) {
                attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
                attr[na].val.programmaticStreamSerializationAllowed = 1;
                ++na;
            }
            cfg.attrs = attr;
            cfg.numAttrs = na;
            cudaError_t le = cudaLaunchKernelEx(&cfg, tc05_gemm_persistent_kernel<BN, true>, ma, mb, mc, p);
            if (le != cudaSuccess) {
                cudaGetLastError();
                return codae_fail(ctx, CODAE_ECUDA, "tc05_gemm_persistent_kernel<%d, pair> launch: %s", BN, cudaGetErrorString(le));
            }
            return codae_check_launch(ctx, "tc05_gemm_persistent_kernel<pair>");
        }
        cudaError_t le = launch_pdl(ctx, tc05_gemm_persistent_kernel<BN, false>, dim3(ctx->sm_count), dim3(kThreads),
                                    C::kSmemBytes + (p.tma_store ? kPersistentStageBytes : 0), s, ma, mb, mc, p);
        if (le != cudaSuccess) {
            cudaGetLastError();
            return codae_fail(ctx, CODAE_ECUDA, "tc05_gemm_persistent_kernel<%d> launch: %s", BN, cudaGetErrorString(le));
        }
        return codae_check_launch(ctx, "tc05_gemm_persistent_kernel");
    }
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(tc05_gemm_kernel<BN, NP, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::kSmemBytes);
        if (e == cudaSuccess && NP == 3)
            e = cudaFuncSetAttribute(tc05_gemm_kernel<BN, NP, NP == 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::kSmemBytes);
        if (e != cudaSuccess) return codae_fail(ctx, CODAE_ECUDA, "cudaFuncSetAttribute(smem=%u): %s", C::kSmemBytes, cudaGetErrorString(e));
        attr_set = true;
    }
    const int kb_per_cta = ((total_kb + nsplit - 1) / nsplit);
    p.stages = kb_per_cta < C::kStages ? (kb_per_cta < 2 ? 2 : kb_per_cta) : C::kStages;
    p.tmem_cols = BN;
    if constexpr (NP == 3) {
        p.stages = pl.stages;
        p.tmem_cols = pl.tmem_cols;
    }
    size_t pipe_bytes = (size_t)p.stages * C::kStageBytes;
    const size_t stage_tile = (size_t)BM * (BN + 4) * sizeof(float);          // staged epilogue overlays the pipeline
    if (p.staged && pipe_bytes < stage_tile) {
        p.stages = (int)((stage_tile + C::kStageBytes - 1) / C::kStageBytes);  // barriers sit after the last slot
        pipe_bytes = (size_t)p.stages * C::kStageBytes;
    }
    const size_t smem_bytes = pipe_bytes + 1024 + 256;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(pl.gx, pl.gy, nsplit);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem_bytes;
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    int na = 0;
    if (nsplit > 1) {
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = 1;
        attr[na].val.clusterDim.y = 1;
        attr[na].val.clusterDim.z = nsplit;
        ++na;
    }
    if (codae_pdl_allowed(ctx, s)) {
        attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[na].val.programmaticStreamSerializationAllowed = 1;
        ++na;
    }
    cfg.attrs = attr;
    cfg.numAttrs = na;
    const bool chunked = NP == 3 && kb_per_cta > x3_chunk_kb();
    p.chunk_kb = x3_chunk_kb();
    static const bool debug_plan = getenv("CODAE_DEBUG_PLAN") != nullptr;
    if (debug_plan) {
        int occ = -1;
        if (chunked) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, tc05_gemm_kernel<BN, NP, NP == 3>, kThreads, smem_bytes);
        else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, tc05_gemm_kernel<BN, NP, false>, kThreads, smem_bytes);
        fprintf(stderr, "codae plan: M=%d N=%d K=%d BN=%d NP=%d grid %d x %d x %d stages %d smem %zu tmem %d staged %d tma_store %d chunked %d occupancy %d\n",
                g.M, g.N, g.K, BN, NP, pl.gx, pl.gy, nsplit, p.stages, smem_bytes, p.tmem_cols, p.staged, p.tma_store, (int)chunked, occ);
    }
    cudaError_t le = chunked ? cudaLaunchKernelEx(&cfg, tc05_gemm_kernel<BN, NP, NP == 3>, ma, mb, mc, p)
                             : cudaLaunchKernelEx(&cfg, tc05_gemm_kernel<BN, NP, false>, ma, mb, mc, p);
    if (le != cudaSuccess) {
        cudaGetLastError();
        return codae_fail(ctx, CODAE_ECUDA, "tc05_gemm_kernel<%d, %d> launch (grid %u x %u x %d, smem %zu): %s", BN, NP, cfg.gridDim.x,
                          cfg.gridDim.y, nsplit, smem_bytes, cudaGetErrorString(le));
    }
    return codae_check_launch(ctx, "tc05_gemm_kernel");
}

inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

// Debugging hook (exported, deliberately absent from include/codae_b200.h): device buffer of >= 16 u64 that CTA (0,0,0) of
// every subsequent tcgen05 GEMM fills with %globaltimer stamps of its phases; NULL switches it off.
extern "C" int codae_debug_set_trace(void* device_buf) {
    g_trace_buf = reinterpret_cast<unsigned long long*>(device_buf);
    return 0;
}
extern "C" int codae_debug_set_trace_cta(int linear_cta) {
    g_trace_cta = linear_cta;
    return 0;
}

int codae_tc05_make_map(codae_ctx* ctx, CUtensorMap* map, const void* base, long long rows, long long cols, long long ld,
                        int box_cols, int box_rows, int planes, long long plane_stride) {
    return make_map(ctx, map, base, rows, cols, ld, box_cols, box_rows, planes, plane_stride);
}

bool codae_tc05_supported(const codae_ctx* ctx, const Tc05Gemm& g) {
    if (!ctx || !ctx->encode_tiled) return false;
    if (g.M < 1 || g.N < 1 || g.K < 1) return false;
    if (g.planes != 1 && g.planes != 3) return false;
    // TMA: 16-byte aligned bases and pitches (bf16 -> multiples of 8 elements)
    if (!al16(g.A) || !al16(g.B) || !al16(g.C) || (g.lda % 8) || (g.ldb % 8)) return false;
    if (g.c_dtype == CODAE_F32 ? (g.ldc % 4) : (g.ldc % 8)) return false;
    if (g.mask_src && (!al16(g.mask_src) || (g.ldm % 8))) return false;
    if (g.planes == 3) {
        if ((g.a_plane_stride % 8) || (g.b_plane_stride % 8) || g.a_plane_stride < 1 || g.b_plane_stride < 1) return false;
        if (g.c_dtype == CODAE_BF16) return false;                                  // f32 or its bf16 triple
        if (g.c_dtype == CODAE_F32X3 && ((g.c_plane_stride % 4) || g.c_plane_stride < 1)) return false;
    } else if (g.c_dtype == CODAE_F32X3) {
        return false;
    }
    // tiny problems (abalone 11x11) are not worth a 128-row tensor-core tile
    if (g.N < 32) return false;
    return true;
}

// Tile width: the widest tile that still yields at least one CTA per SM (small batches want many CTAs streaming the
// weights), 256-wide for large problems (bf16 engine only: three-plane stages of a 256-wide tile do not fit).
static int pick_bn(const codae_ctx* ctx, const Tc05Gemm& g) {
    const long tiles_m = (g.M + BM - 1) / BM;
    const long t256 = tiles_m * ((g.N + 255) / 256), t128 = tiles_m * ((g.N + 127) / 128);
    // tuning knobs (read once): CODAE_X3_BN / CODAE_DGRAD_BN = 64 | 128 force the tile width of the fp32-parity engine / of the
    // input-gradient contraction (K-major A, MN-major B)
    static const int x3_bn = getenv("CODAE_X3_BN") ? atoi(getenv("CODAE_X3_BN")) : 0;
    static const int dgrad_bn = getenv("CODAE_DGRAD_BN") ? atoi(getenv("CODAE_DGRAD_BN")) : 0;
    static const int wgrad_bn = getenv("CODAE_WGRAD_BN") ? atoi(getenv("CODAE_WGRAD_BN")) : 0;
    const bool is_dgrad = g.a_kmajor && !g.b_kmajor, is_wgrad = !g.a_kmajor && !g.b_kmajor;
    if (is_dgrad && (dgrad_bn == 64 || dgrad_bn == 128) && g.N >= dgrad_bn) return dgrad_bn;
    if (is_wgrad && (wgrad_bn == 64 || wgrad_bn == 128 || (wgrad_bn == 256 && g.planes == 1)) && g.N >= wgrad_bn) return wgrad_bn;
    if (g.planes == 3 && (x3_bn == 64 || x3_bn == 128) && g.N >= x3_bn) return x3_bn;
    if (g.planes == 1 && t256 >= ctx->sm_count && g.N >= 256) return 256;
    if (t128 >= ctx->sm_count && g.N >= 128) return 128;
    // Small-batch input gradients: 128-wide tiles (12 clusters of 8 = 96 CTAs at 1536 wide) although the launch alone is slower
    // than 24 x 6 CTAs of 64-wide tiles (86 vs 69 us for nine launches): tcgen05 kernels own their SM, and only this geometry
    // lets the weight gradient of the same layer (side stream) run beside it.  Measured per step on a B200
    // (tools/r02_ab_dgrad_bn.sh, r02_ab_bwd_split.sh): embedding.yaml bf16 0.3414 -> 0.3214 ms, fp32 0.5125 -> 0.4901,
    // modanet 0.2704 -> 0.2558; 72-CTA and 64-wide 96-CTA variants were slower than the default (0.356 - 0.367).
    if (is_dgrad && dgrad_bn == 0 && g.N >= 128 && tiles_m == 1) return 128;
    return 64;
}

int codae_tc05_gemm(codae_ctx* ctx, const Tc05Gemm& g, cudaStream_t s) {
    if (!codae_tc05_supported(ctx, g)) return codae_fail(ctx, CODAE_EINVAL, "codae_tc05_gemm: unsupported shape/alignment");
    if (g.planes == 3) return pick_bn(ctx, g) == 128 ? launch<128, 3>(ctx, g, s) : launch<64, 3>(ctx, g, s);
    switch (pick_bn(ctx, g)) {
        case 256: return launch<256>(ctx, g, s);
        case 128: return launch<128>(ctx, g, s);
        default: return launch<64>(ctx, g, s);
    }
}

int codae_tc05_gemm_ctas(const codae_ctx* ctx, const Tc05Gemm& g) {
    if (!ctx || !ctx->encode_tiled || g.M < 1 || g.N < 32 || g.K < 1) return 0;
    if (g.planes == 3) return pick_bn(ctx, g) == 128 ? make_plan<128, 3>(ctx, g).ctas : make_plan<64, 3>(ctx, g).ctas;
    switch (pick_bn(ctx, g)) {
        case 256: return make_plan<256>(ctx, g).ctas;
        case 128: return make_plan<128>(ctx, g).ctas;
        default: return make_plan<64>(ctx, g).ctas;
    }
}
