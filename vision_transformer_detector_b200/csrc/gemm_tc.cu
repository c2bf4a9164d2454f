// Dense layer on the 5th-gen tensor cores:  out = epilogue( A[M,K] * W[N,K]^T )
//
// Replaces every keras.layers.Dense / EinsumDense of the reference's forward pass in bf16 mode:
// linear_projection (det.py:297-301), the q/k/v and attention_output projections inside
// MultiHeadAttention (det.py:364-369), MLP_i_j (det.py:388-398) and the mlp_head Dense chain
// (det.py:468-480), together with the element-wise ops that follow them in the reference graph
// (bias add, MishActivation det.py:119-129 / tfa GELU det.py:402, keras.layers.add det.py:305,
// 371, 408-412), which run here as the epilogue of the same kernel.
//
// Structure (one persistent CTA per SM, 576 threads):
//   warp 0      TMA producer: cp.async.bulk.tensor 2-D boxes of A (128 x 64 bf16) and W (BN x 64
//               bf16) into a ring of 128B-swizzled shared-memory stages, completion on mbarriers.
//   warp 1      allocates 512 TMEM columns; one elected lane issues tcgen05.mma (M=128, N=BN, K=16,
//               bf16 x bf16 -> f32 in TMEM) and tcgen05.commit to free stages / publish accumulators.
//   warps 2..17 epilogue: tcgen05.ld the f32 accumulator (thread = one row of the tile, the four warps
//               of a TMEM lane quadrant split the 32-column chunks), bias / position scalar /
//               activation / residual, 16-byte global stores.  Sixteen warps because the Mish epilogue
//               of the wide layers is issue-bound: with four it capped the 28 -> 3584 layer at 5x its
//               HBM time (profiles/r01a_ncu_gemm.md).
// Two TMEM accumulator stages (2 x 256 columns) let the MMA of tile i+1 overlap the epilogue of
// tile i.  BN and the ring depth are run-time values (N lives in the instruction descriptor), so one
// binary serves every layer width of the model.
//
// CTA-pair form (PAIR, cta_group::2) for the large layers (the 3584 -> 1792 MLP layer is 37 % of the forward):
// two CTAs on the two SMs of a TPC form a cluster and compute one 256 x BN tile.  Each CTA stages ITS 128 rows
// of A and HALF of the BN rows of W per k-block; the producers' loads complete on the LEADER's full barrier, the
// leader's MMA warp issues tcgen05.mma.cta_group::2 (M = 256) and commits with multicast so that both CTAs'
// "stage empty" / "accumulator full" barriers fire, each CTA's TMEM receives the accumulator of its own 128 rows,
// and both CTAs' epilogue warps arrive on the leader's "accumulator drained" barrier.  Per SM and per MMA the
// tensor core then reads 4 KB (A) + 4 KB (half of B) of shared memory instead of 4 + 8 KB, and TMA fills 32 KB
// per k-block instead of 48 KB: the single-CTA kernel sat at 81 % tensor-pipe activity with the shared-memory
// operand pipe at 75 % of its rate (profiles/r01b_ncu_gemm.md).
#include <type_traits>

#include "common.cuh"
#include "kernels.h"
#include "launch.h"

namespace vitdet {

namespace {

template <int ACT, bool F32ACC>
__device__ __forceinline__ float act_out(float x) { return F32ACC ? apply_act_f32acc<ACT>(x) : apply_act<ACT, false>(x); }

// The cta_group::1 / cta_group::2 forms of the TMA load, the MMA and its commit
template <bool PAIR>
__device__ __forceinline__ void tma_load(uint32_t smem_dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    if constexpr (PAIR) tma_load_2d_2sm(smem_dst, map, bar, c0, c1); else tma_load_2d(smem_dst, map, bar, c0, c1);
}
template <bool PAIR>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    if constexpr (PAIR) umma_bf16_ss_2sm(tmem_d, desc_a, desc_b, idesc, accumulate); else umma_bf16_ss(tmem_d, desc_a, desc_b, idesc, accumulate);
}
template <bool PAIR>
__device__ __forceinline__ void commit(uint32_t bar) {
    if constexpr (PAIR) umma_commit_2sm(bar, 3); else umma_commit(bar);      // pair: the barrier at `bar` in both CTAs
}

constexpr int kBM = 128;              // rows of A per CTA (UMMA M of cta_group::1; the pair's M is 256)
constexpr int kBK = 64;               // one 128-byte swizzle row of bf16
constexpr int kUK = 16;               // UMMA K for 16-bit inputs
constexpr int kMaxBN = 256;
constexpr int kMaxStages = 8;
constexpr int kStageBytesA = kBM * kBK * 2;   // 16 KiB
constexpr int kEpiWarps = 16;          // 4 per TMEM lane quadrant; the quadrant's warps split the 32-column chunks
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kThreads = 64 + kEpiThreads;
// Role -> warp id.  The epilogue warps come first (warp & 3 is their TMEM lane quadrant); the TMA producer and the
// MMA issuer are the two HIGHEST warp ids because the warp arbiter favours high ids: the single thread that feeds
// the tensor pipe must never queue behind the ALU/SFU-heavy epilogue warps of its sub-partition.
constexpr int kProducerWarp = kEpiWarps, kMmaWarp = kEpiWarps + 1;
constexpr int kTmemCols = 512;
constexpr int kRingBytes = 192 * 1024;            // budget of the A/B stage ring (4 stages at BN = 256)
constexpr int kStoreTileBytes = 32 * 32 * 2;      // one epilogue warp's 32 x 32 bf16 sub-tile, 64B-swizzled
constexpr int kStoreBytes = kEpiWarps * kStoreTileBytes;
// Dynamic smem = ring + store staging = 224 KB; the static part (barriers, bias, ~2.2 KB) is padded to
// 3 KB by the 1024-byte alignment of the dynamic part, which makes exactly 227 KB.
constexpr int kMaxDynSmem = kRingBytes + kStoreBytes;

struct TcGemmArgs {
    int M, N, K;
    int block_n;
    int num_stages;
    int n_tiles;
    int num_tiles;
    int num_kb;
    const float* bias;
    const float* pos;
    int pos_period;
    const float* resid;
    int ldr;
    void* out;
    int ldc;
    int n_store;   // round_up(N, store vector): columns [N, n_store) are written as zero
    int split;     // 1: A and W are (hi, lo) bf16 planes; three passes over K (hi*hi, hi*lo, lo*hi)
};
// The single-CTA form's arguments add the fused LayerNorm of the output row (f32 output, N <= 32).  The pair form has none, so
// its kernel parameters end with TcGemmArgs: a parameter block of more than 128 bytes changes how the compiler loads the
// fields, and with it the machine code of the pair instances.
struct TcGemmLnArgs : TcGemmArgs {
    const float* ln_gamma;      // or nullptr
    const float* ln_beta;
    float ln_eps;
    __nv_bfloat16* ln_out;
    int ln_ld;
};

// OUT: 0 bf16 (TMA store), 1 float32 rows of <= 32 columns (direct stores, residual, fused LayerNorm), 2 split bf16 planes (hi, lo),
//      3 float32 rows wider than 32 columns (coalesced stores through the staging tile, residual prefetched)
// PRECISE: exact activations (the fp32-accumulate mode)
// PAIR: CTA-pair form, launched as clusters of two CTAs (no fused LayerNorm)
template <int ACT, int OUT, bool PRECISE, bool PAIR>
__global__ void __launch_bounds__(kThreads, 1)   // 96 registers is the most 576 threads can be granted (104 and 112 fail to launch)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmA_lo,
               const __grid_constant__ CUtensorMap tmB_lo, const __grid_constant__ CUtensorMap tmC_lo,
               const std::conditional_t<PAIR, TcGemmArgs, TcGemmLnArgs> p) {
    constexpr bool OUT_F32 = OUT == 1 || OUT == 3;
    constexpr bool WIDE_F32 = OUT == 3;      // float32 rows wider than one 32-column chunk: coalesced stores through the staging tile
    constexpr int kCtas = PAIR ? 2 : 1;      // CTAs per tile
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * kMaxStages + 4];
    __shared__ uint32_t tmem_base_s;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    pdl_launch_dependents();

    const uint32_t smem_base = smem_u32(smem_raw);
    if ((smem_base & 1023u) != 0u) __trap();          // 128B-swizzled stages need 1024-byte alignment
    // epilogue store staging after the ring: one 2 KB tile per warp, two (hi, lo) in the split-output mode
    constexpr uint32_t kStoreStride = OUT == 2 ? 2 * kStoreTileBytes : kStoreTileBytes;
    const uint32_t s_store0 = smem_base + (OUT == 2 ? kRingBytes - kStoreBytes : kRingBytes);
    const uint32_t stage_bytes_b = static_cast<uint32_t>(p.block_n / kCtas) * (kBK * 2);      // this CTA's part of the W tile
    const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0u;
    const bool leader = cta_rank == 0;
    const uint32_t sA0 = smem_base;
    const uint32_t sB0 = smem_base + static_cast<uint32_t>(p.num_stages) * kStageBytesA;

    const uint32_t bar_full = smem_u32(&bars[0]);
    const uint32_t bar_empty = smem_u32(&bars[kMaxStages]);
    const uint32_t bar_tfull = smem_u32(&bars[2 * kMaxStages]);
    const uint32_t bar_tempty = smem_u32(&bars[2 * kMaxStages + 2]);

    if (threadIdx.x == 0) {
        for (int s = 0; s < p.num_stages; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(bar_tfull + 8 * a, 1);
            mbar_init(bar_tempty + 8 * a, kCtas * kEpiWarps);     // pair: the leader's copy collects both CTAs' epilogue warps
        }
        fence_mbar_init();
    }
    if (warp == kProducerWarp && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        if (!OUT_F32) tma_prefetch_desc(&tmC);
        if (PRECISE && p.split) { tma_prefetch_desc(&tmA_lo); tma_prefetch_desc(&tmB_lo); }
        if (OUT == 2) tma_prefetch_desc(&tmC_lo);
    }
    if (warp == kMmaWarp) {
        if constexpr (PAIR) { tmem_alloc_2sm(smem_u32(&tmem_base_s), kTmemCols); tmem_relinquish_2sm(); }
        else { tmem_alloc(smem_u32(&tmem_base_s), kTmemCols); tmem_relinquish(); }
    }
    tc_fence_before();
    if constexpr (PAIR) cluster_sync_all();      // barriers of BOTH CTAs are initialised before any remote arrive / multicast commit
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    pdl_wait();       // set-up above overlapped the previous kernel; its outputs are read from here on

    if (warp == kProducerWarp) {
        // ------------------------------ TMA producer ------------------------------
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            // pair: this CTA's loads complete on the LEADER's full barrier (same offset, CTA rank 0)
            const uint32_t bar_full_leader = PAIR ? mapa_shared(bar_full, 0) : bar_full;
            const uint32_t tx_bytes = kCtas * (kStageBytesA + stage_bytes_b);       // pair: both CTAs' boxes
            for (int tile = blockIdx.x / kCtas; tile < p.num_tiles; tile += gridDim.x / kCtas) {
                const int m0 = (tile / p.n_tiles) * (kCtas * kBM) + static_cast<int>(cta_rank) * kBM;
                const int n0 = (tile % p.n_tiles) * p.block_n + static_cast<int>(cta_rank) * (p.block_n / 2);
                for (int kb = 0; kb < p.num_kb; ++kb) {
                    // split mode: the k-block is visited three times, with (A, W) = (hi, hi), (hi, lo), (lo, hi)
                    for (int t = 0; t < ((PRECISE && p.split) ? 3 : 1); ++t) {
                        mbar_wait(bar_empty + 8 * stage, phase ^ 1u);
                        if (leader) mbar_arrive_expect_tx(bar_full + 8 * stage, tx_bytes);
                        tma_load<PAIR>(sA0 + stage * kStageBytesA, t == 2 ? &tmA_lo : &tmA, bar_full_leader + 8 * stage, kb * kBK, m0);
                        tma_load<PAIR>(sB0 + stage * stage_bytes_b, t == 1 ? &tmB_lo : &tmB, bar_full_leader + 8 * stage, kb * kBK, n0);
                        if (++stage == p.num_stages) { stage = 0; phase ^= 1u; }
                    }
                }
            }
        }
    } else if (warp == kMmaWarp) {
        // ------------------------------ MMA issuer (pair: leader CTA only) --------
        // The WHOLE warp runs this loop (warp-uniform control flow keeps the loop state in uniform registers);
        // only the tcgen05 instructions are issued by one elected lane.
        if (leader) {
            const uint32_t idesc = umma_idesc_bf16_f32(kCtas * kBM, p.block_n);
            const uint64_t da0 = umma_desc_sw128_kmajor(sA0), db0 = umma_desc_sw128_kmajor(sB0);
            const uint32_t a_step = kStageBytesA >> 4, b_step = stage_bytes_b >> 4;      // descriptor address units (16 B)
            const int last_steps = (p.K - (p.num_kb - 1) * kBK + kUK - 1) / kUK;         // k-steps of the last k-block (1..4)
            int stage = 0;
            uint32_t phase = 0;
            int it = 0;
            for (int tile = blockIdx.x / kCtas; tile < p.num_tiles; tile += gridDim.x / kCtas, ++it) {
                const int acc = it & 1;
                const uint32_t acc_phase = (it >> 1) & 1;
                mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1u);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * kMaxBN);
                const int passes = (PRECISE && p.split) ? 3 : 1;      // split planes only exist in the fp32-accumulate mode
                for (int kb = 0; kb < p.num_kb; ++kb) {
                    const int ksteps = (kb == p.num_kb - 1) ? last_steps : kBK / kUK;
                    for (int t = 0; t < passes; ++t) {
                        mbar_wait(bar_full + 8 * stage, phase);
                        tc_fence_after();
                        if (elect_one()) {
                            const uint64_t da = da0 + static_cast<uint64_t>(stage * a_step), db = db0 + static_cast<uint64_t>(stage * b_step);
                            umma<PAIR>(d_tmem, da, db, idesc, (kb | t) != 0);
                            if (ksteps > 1) umma<PAIR>(d_tmem, da + 2u, db + 2u, idesc, 1u);
                            if (ksteps > 2) umma<PAIR>(d_tmem, da + 4u, db + 4u, idesc, 1u);
                            if (ksteps > 3) umma<PAIR>(d_tmem, da + 6u, db + 6u, idesc, 1u);
                            commit<PAIR>(bar_empty + 8 * stage);
                            if (kb == p.num_kb - 1 && t == passes - 1) commit<PAIR>(bar_tfull + 8 * acc);
                        }
                        __syncwarp();
                        if (++stage == p.num_stages) { stage = 0; phase ^= 1u; }
                    }
                }
            }
        }
    } else {
        // ------------------------------ epilogue ----------------------------------
        // Warp w may only read TMEM lanes [32*(w%4), +32).  The four warps of a quadrant take the
        // 32-column chunks round-robin (sub = 0..3), so a 256-wide tile is two chunks per warp.
        const int quad = warp & 3;                    // TMEM lane quadrant this warp may access
        const int sub = warp >> 2;                    // which chunks of the tile (c0 = 32*sub, +128, ...)
        int it = 0;
        const uint32_t bar_tempty_leader = PAIR ? mapa_shared(bar_tempty, 0) : bar_tempty;
        for (int tile = blockIdx.x / kCtas; tile < p.num_tiles; tile += gridDim.x / kCtas, ++it) {
            const int acc = it & 1;
            const uint32_t acc_phase = (it >> 1) & 1;
            const int m0 = (tile / p.n_tiles) * (kCtas * kBM) + static_cast<int>(cta_rank) * kBM;   // this CTA's 128 rows
            const int n0 = (tile % p.n_tiles) * p.block_n;

            // Bias is read straight from global memory below (a warp-wide broadcast that stays in L1): no staging
            // barrier per tile, so the sixteen epilogue warps drift apart and their SFU phases interleave.
            const float* bs = p.bias + n0;      // valid for columns < N only; the tail path guards its reads
            // The thread's row: the single-CTA form computes it before the wait for the accumulator (the residual prefetch
            // below needs it), the pair form after the wait, where its instances compile to 16 fewer instructions.
            int row = 0;
            bool row_ok = false;
            if constexpr (!PAIR) { row = m0 + quad * 32 + lane; row_ok = row < p.M; }
            // Narrow float32 rows (the 28-wide residual stream: output projection): the thread's residual row is fetched
            // BEFORE the wait for the accumulator, so that the global-load latency hides behind the tile's MMAs.
            float4 rpre[8];
            bool rpre_ok = false;
            if constexpr (OUT == 1) {
                if (p.resid != nullptr && p.block_n <= 32 && sub == 0 && row_ok) {
                    const float* rr = p.resid + static_cast<size_t>(row) * p.ldr + n0;
#pragma unroll
                    for (int g = 0; g < 8; ++g) rpre[g] = (n0 + 4 * g < p.n_store) ? *reinterpret_cast<const float4*>(rr + 4 * g) : make_float4(0.f, 0.f, 0.f, 0.f);
                    rpre_ok = true;
                }
            }
            mbar_wait(bar_tfull + 8 * acc, acc_phase);
            tc_fence_after();
            if constexpr (PAIR) { row = m0 + quad * 32 + lane; row_ok = row < p.M; }
            float pos_v = 0.f;
            if (p.pos != nullptr && row_ok) pos_v = __ldg(p.pos + (row % p.pos_period));
            const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) +
                                   static_cast<uint32_t>(acc * kMaxBN);

            for (int c0 = sub * 32; c0 < p.block_n; c0 += 128) {
                uint32_t v[32];
                tmem_ld_32x32(t_row + c0, v);
                const bool full = n0 + c0 + 32 <= p.N;
                float4 rres[2][4];      // residual values of this chunk, fetched under the TMEM load (dead code for bf16 outputs)
                const bool wide_f32 = WIDE_F32 && full;
                if constexpr (WIDE_F32) { if (wide_f32) prefetch_resid_chunk(rres, p.resid, p.ldr, lane, m0 + quad * 32, p.M, n0 + c0); }
                tmem_ld_wait();      // block_n is a multiple of 32: chunks are never partial in the tile
                if (OUT_F32) {
                    if (wide_f32) {
                        // wide float32 output (embedding_dim > 32): finished values of the lane's row, 16 columns at a
                        // time, through the staging tile to coalesced stores (common.cuh); residual added on that side
                        const uint32_t s_tile = s_store0 + static_cast<uint32_t>(warp) * kStoreStride;
#pragma unroll
                        for (int hh = 0; hh < 2; ++hh) {
                            float y16[16];
#pragma unroll
                            for (int g = 0; g < 4; ++g) {
                                const int c = c0 + 16 * hh + 4 * g;
                                const float4 b4 = p.bias ? __ldg(reinterpret_cast<const float4*>(bs + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
                                y16[4 * g + 0] = act_out<ACT, PRECISE>(__uint_as_float(v[16 * hh + 4 * g + 0]) + b4.x + pos_v);
                                y16[4 * g + 1] = act_out<ACT, PRECISE>(__uint_as_float(v[16 * hh + 4 * g + 1]) + b4.y + pos_v);
                                y16[4 * g + 2] = act_out<ACT, PRECISE>(__uint_as_float(v[16 * hh + 4 * g + 2]) + b4.z + pos_v);
                                y16[4 * g + 3] = act_out<ACT, PRECISE>(__uint_as_float(v[16 * hh + 4 * g + 3]) + b4.w + pos_v);
                            }
                            store_f32_half_chunk_coalesced(s_tile, y16, lane, m0 + quad * 32, p.M, reinterpret_cast<float*>(p.out), p.ldc,
                                                           rres[hh], n0 + c0 + 16 * hh);
                        }
                        continue;
                    }
                    if (!row_ok) continue;
                    float* orow = reinterpret_cast<float*>(p.out) + static_cast<size_t>(row) * p.ldc;
                    const float* rrow = p.resid ? p.resid + static_cast<size_t>(row) * p.ldr : nullptr;
                    float xr[32];        // the finished values of this chunk (kept for the fused LayerNorm)
#pragma unroll
                    for (int g = 0; g < 8; ++g) {
                        const int c = c0 + 4 * g;
                        const int n = n0 + c;
                        float x[4] = {0.f, 0.f, 0.f, 0.f};
                        if (full || n < p.n_store) {
                            float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (p.bias != nullptr) {
                                if (full) b4 = __ldg(reinterpret_cast<const float4*>(bs + c));
                                else {
                                    b4.x = (n + 0 < p.N) ? __ldg(bs + c + 0) : 0.f; b4.y = (n + 1 < p.N) ? __ldg(bs + c + 1) : 0.f;
                                    b4.z = (n + 2 < p.N) ? __ldg(bs + c + 2) : 0.f; b4.w = (n + 3 < p.N) ? __ldg(bs + c + 3) : 0.f;
                                }
                            }
                            x[0] = __uint_as_float(v[4 * g + 0]) + b4.x; x[1] = __uint_as_float(v[4 * g + 1]) + b4.y;
                            x[2] = __uint_as_float(v[4 * g + 2]) + b4.z; x[3] = __uint_as_float(v[4 * g + 3]) + b4.w;
                            float4 r4 = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (OUT == 1 && rpre_ok) r4 = rpre[g];
                            else if (rrow) r4 = *reinterpret_cast<const float4*>(rrow + n);
                            const float r[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float y = act_out<ACT, PRECISE>(x[j] + pos_v) + r[j];
                                x[j] = (full || n + j < p.N) ? y : 0.f;
                            }
                            *reinterpret_cast<float4*>(orow + n) = make_float4(x[0], x[1], x[2], x[3]);
                        }
#pragma unroll
                        for (int j = 0; j < 4; ++j) xr[4 * g + j] = x[j];
                    }
                    if constexpr (!PAIR) if (p.ln_out != nullptr) {
                        // keras LayerNormalization(axis=-1) of the row just produced (the host only sets ln_out when
                        // the whole row is this one chunk): biased variance, eps inside the rsqrt, f32 statistics
                        const float inv_n = 1.f / static_cast<float>(p.N);
                        float sum = 0.f;
#pragma unroll
                        for (int i = 0; i < 32; ++i) sum += xr[i];                 // columns >= N are zero
                        const float mean = sum * inv_n;
                        float sq = 0.f;
#pragma unroll
                        for (int i = 0; i < 32; ++i) { const float dv = (i < p.N) ? xr[i] - mean : 0.f; sq = fmaf(dv, dv, sq); }
                        const float rstd = rsqrtf(sq * inv_n + p.ln_eps);
                        __nv_bfloat16* yrow = p.ln_out + static_cast<size_t>(row) * p.ln_ld;
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            if (8 * g < p.ln_ld) {
                                float o8[8];
#pragma unroll
                                for (int j = 0; j < 8; ++j) {
                                    const int i = 8 * g + j;
                                    o8[j] = (i < p.N) ? (xr[i] - mean) * rstd * __ldg(p.ln_gamma + i) + __ldg(p.ln_beta + i) : 0.f;
                                }
                                uint4 w;
                                w.x = pack_bf16x2(o8[0], o8[1]); w.y = pack_bf16x2(o8[2], o8[3]);
                                w.z = pack_bf16x2(o8[4], o8[5]); w.w = pack_bf16x2(o8[6], o8[7]);
                                *reinterpret_cast<uint4*>(yrow + 8 * g) = w;
                            }
                        }
                    }
                } else {
                    // bf16 output: this warp's 32 x 32 sub-tile goes to its 64B-swizzled staging tile
                    // (row = lane, 64 B per row; 16-byte chunk c of row r sits at chunk c ^ ((r >> 1) & 3),
                    // which is both what CU_TENSOR_MAP_SWIZZLE_64B expects and bank-conflict free), then
                    // one TMA store writes it with full 64-byte row segments.  Rows >= M and columns past
                    // the tensor width are clipped by the TMA unit.
                    const uint32_t s_tile = s_store0 + static_cast<uint32_t>(warp) * kStoreStride;
                    uint32_t o[16];
                    uint32_t olo[OUT == 2 ? 16 : 1];
                    if (OUT == 2) {
                        // split output: y in float32 with the exact activation, hi = bf16(y), lo = bf16(y - hi)
#pragma unroll
                        for (int g = 0; g < 16; ++g) {
                            const int n = n0 + c0 + 2 * g;
                            const float bb0 = (p.bias && n < p.N) ? __ldg(bs + c0 + 2 * g) : 0.f;
                            const float bb1 = (p.bias && n + 1 < p.N) ? __ldg(bs + c0 + 2 * g + 1) : 0.f;
                            float y0 = apply_act_f32acc<ACT>(__uint_as_float(v[2 * g + 0]) + bb0);
                            float y1 = apply_act_f32acc<ACT>(__uint_as_float(v[2 * g + 1]) + bb1);
                            if (n >= p.N) y0 = 0.f;
                            if (n + 1 >= p.N) y1 = 0.f;
                            const __nv_bfloat162 hi = __floats2bfloat162_rn(y0, y1);
                            o[g] = *reinterpret_cast<const uint32_t*>(&hi);
                            olo[g] = pack_bf16x2(y0 - __low2float(hi), y1 - __high2float(hi));
                        }
                    } else if (full) {
#pragma unroll
                        for (int g = 0; g < 8; ++g) {
                            const float4 b4 = p.bias ? __ldg(reinterpret_cast<const float4*>(bs + c0 + 4 * g)) : make_float4(0.f, 0.f, 0.f, 0.f);
                            o[2 * g] = bias_act_bf16x2<ACT>(__uint_as_float(v[4 * g + 0]), __uint_as_float(v[4 * g + 1]), b4.x, b4.y);
                            o[2 * g + 1] = bias_act_bf16x2<ACT>(__uint_as_float(v[4 * g + 2]), __uint_as_float(v[4 * g + 3]), b4.z, b4.w);
                        }
                    } else {      // last N tile: columns >= N are written as zero
#pragma unroll
                        for (int g = 0; g < 16; ++g) {
                            const int n = n0 + c0 + 2 * g;
                            const float bb0 = (p.bias && n < p.N) ? __ldg(bs + c0 + 2 * g) : 0.f;
                            const float bb1 = (p.bias && n + 1 < p.N) ? __ldg(bs + c0 + 2 * g + 1) : 0.f;
                            const float y0 = apply_act<ACT, false>(__uint_as_float(v[2 * g + 0]) + bb0);
                            const float y1 = apply_act<ACT, false>(__uint_as_float(v[2 * g + 1]) + bb1);
                            o[g] = pack_bf16x2(n < p.N ? y0 : 0.f, n + 1 < p.N ? y1 : 0.f);
                        }
                    }
                    // only now wait for the previous TMA store of this warp to have left the staging
                    // tile: its read latency is hidden behind the arithmetic above
                    if (lane == 0) tma_store_wait_read();
                    __syncwarp();
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        const uint32_t dst = s_tile + static_cast<uint32_t>(lane * 64 + ((g ^ ((lane >> 1) & 3)) << 4));
                        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(o[4 * g]), "r"(o[4 * g + 1]),
                                     "r"(o[4 * g + 2]), "r"(o[4 * g + 3]) : "memory");
                        if (OUT == 2)
                            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst + kStoreTileBytes), "r"(olo[(4 * g) % (OUT == 2 ? 16 : 1)]),
                                         "r"(olo[(4 * g + 1) % (OUT == 2 ? 16 : 1)]), "r"(olo[(4 * g + 2) % (OUT == 2 ? 16 : 1)]),
                                         "r"(olo[(4 * g + 3) % (OUT == 2 ? 16 : 1)]) : "memory");
                    }
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        tma_store_2d(&tmC, s_tile, n0 + c0, m0 + quad * 32);
                        if (OUT == 2) tma_store_2d(&tmC_lo, s_tile + kStoreTileBytes, n0 + c0, m0 + quad * 32);
                        tma_store_commit();
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if constexpr (PAIR) mbar_arrive_cluster(bar_tempty_leader + 8 * acc);
                else mbar_arrive(bar_tempty + 8 * acc);
            }
        }
        if (!OUT_F32 && lane == 0) tma_store_wait_all();
    }

    tc_fence_before();
    if constexpr (PAIR) cluster_sync_all();      // the leader's MMAs touch the peer's smem and TMEM: nobody leaves early
    else __syncthreads();
    if (warp == kMmaWarp) {
        tc_fence_after();
        if constexpr (PAIR) tmem_dealloc_2sm(tmem_base, kTmemCols);
        else tmem_dealloc(tmem_base, kTmemCols);
    }
}

// ------------------------------------------------------------------------------------------------
// Host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn) return fn;
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess || sym == nullptr) {
        return nullptr;
    }
    fn = reinterpret_cast<EncodeTiledFn>(sym);
    return fn;
}

template <int ACT, int OUT, bool PRECISE, bool PAIR>
cudaError_t launch_variant(const TcGemmPlan& plan, const TcGemmLnArgs& a, cudaStream_t stream) {
    auto kern = gemm_tc_kernel<ACT, OUT, PRECISE, PAIR>;
    {
        cudaError_t e = ensure_max_dynamic_smem(reinterpret_cast<const void*>(kern), kMaxDynSmem);
        if (e != cudaSuccess) return e;
    }
    return launch_kernel(kern, dim3(plan.grid), dim3(kThreads), plan.smem_bytes, stream, PAIR ? 2 : 1, plan.tmA, plan.tmB, plan.tmC,
                         plan.tmA_lo, plan.tmB_lo, plan.tmC_lo, a);
}

template <int ACT, bool PAIR>
cudaError_t launch_act(const TcGemmPlan& plan, const TcGemmLnArgs& a, cudaStream_t stream) {
    const GemmDesc& d = plan.desc;
    // Wide float32 rows: separate instantiation, so that the narrow (28-wide) epilogue keeps its registers.  The pair form has
    // no narrow instantiation: its float32 layers are wide (N >= 128), and OUT = 3 handles a partial chunk as OUT = 1 does.
    if (d.out_f32 && (PAIR || (d.N > 32 && !d.ln_out)))
        return d.precise ? launch_variant<ACT, 3, true, PAIR>(plan, a, stream) : launch_variant<ACT, 3, false, PAIR>(plan, a, stream);
    if constexpr (!PAIR) {
        if (d.out_f32) return d.precise ? launch_variant<ACT, 1, true, PAIR>(plan, a, stream) : launch_variant<ACT, 1, false, PAIR>(plan, a, stream);
    }
    if (d.out_split) return launch_variant<ACT, 2, true, PAIR>(plan, a, stream);      // split planes only exist in the fp32-accumulate mode
    return launch_variant<ACT, 0, false, PAIR>(plan, a, stream);
}

}  // namespace

int choose_block_n(int N) {
    // Multiples of 32: the epilogue works on 32-column chunks (one tcgen05.ld, one TMA store box).
    if (N <= kMaxBN) return (N + 31) / 32 * 32;
    // Largest multiple of 32 whose padded width wastes <= 3 %; otherwise the least wasteful >= 64.
    int best = kMaxBN;
    double best_waste = 1e9;
    for (int bn = kMaxBN; bn >= 64; bn -= 32) {
        const int tiles = (N + bn - 1) / bn;
        const double waste = static_cast<double>(tiles) * bn / N - 1.0;
        if (waste <= 0.03) return bn;
        if (waste < best_waste - 1e-9) { best_waste = waste; best = bn; }
    }
    return best;
}

// 2-D bf16 tensor map, row-major [rows, cols] with `ld` elements between rows, box = 64 x box_rows,
// 128B swizzle, out-of-bounds elements read as zero (this is what pads K, M and N tails).
int make_tmap_bf16_2d_ex(CUtensorMap* map, const void* base, int rows, int cols, int ld, int box_cols, int box_rows,
                         int swizzle_bytes) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return -1;
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
    cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld) * 2};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows)};
    cuuint32_t estr[2] = {1, 1};
    const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -static_cast<int>(r) - 1000;
}

int make_tmap_bf16_2d(CUtensorMap* map, const void* base, int rows, int cols, int ld, int box_rows) {
    return make_tmap_bf16_2d_ex(map, base, rows, cols, ld, kBK, box_rows, 128);
}

// pair: tile = 256 rows x BN columns per cluster of two CTAs, W box = BN/2 rows per CTA.
int tc_gemm_make_plan(TcGemmPlan* plan, const GemmDesc& d, int num_sms, int pair) {
    if (d.M <= 0 || d.N <= 0 || d.K <= 0) return -2;
    if ((d.lda % 8) || (d.ldw % 8)) return -3;                        // 16-byte row pitch for TMA
    if ((reinterpret_cast<uintptr_t>(d.A) & 15) || (reinterpret_cast<uintptr_t>(d.W) & 15) ||
        (reinterpret_cast<uintptr_t>(d.out) & 15))
        return -4;
    const int vec = d.out_f32 ? 4 : 8;
    if ((d.ldc % vec) || d.ldc < (d.N + vec - 1) / vec * vec) return -5;
    if (d.resid && (!d.out_f32 || (d.ldr % 4) || d.ldr < (d.N + 3) / 4 * 4)) return -6;
    if (d.pos && !d.out_f32) return -8;      // the position scalar is only fused into f32-output layers
    if (d.split && !d.precise) return -12;      // split planes belong to the fp32-accumulate (precise) instantiations
    if (d.split && (!d.A_lo || !d.W_lo || (reinterpret_cast<uintptr_t>(d.A_lo) & 15) || (reinterpret_cast<uintptr_t>(d.W_lo) & 15))) return -10;
    if (d.out_split && (d.out_f32 || !d.out_lo || (reinterpret_cast<uintptr_t>(d.out_lo) & 15))) return -11;
    if (d.ln_out && (pair || !d.out_f32 || d.N > 32 || !d.ln_gamma || !d.ln_beta || (d.ln_ld % 8) || d.ln_ld < (d.N + 7) / 8 * 8 ||
                     d.ln_ld > 32 || (reinterpret_cast<uintptr_t>(d.ln_out) & 15)))
        return -9;                            // fused LayerNorm: single-CTA form only, the whole row in one 32-column chunk
    int bn = d.block_n > 0 ? d.block_n : choose_block_n(d.N);
    if (bn % 32 || bn < 32 || bn > kMaxBN) return -7;

    const int ctas = pair ? 2 : 1;
    const int box_n = bn / ctas;      // rows of W each CTA stages
    plan->desc = d;
    plan->pair = pair ? 1 : 0;
    plan->block_n = bn;
    const int stage = kStageBytesA + box_n * kBK * 2;
    const int ring = d.out_split ? kRingBytes - kStoreBytes : kRingBytes;       // split output: two staging tiles per epilogue warp
    int stages = ring / stage;
    if (stages > kMaxStages) stages = kMaxStages;
    plan->num_stages = stages;
    plan->smem_bytes = kMaxDynSmem;    // ring (up to 192 KB) + store staging, fixed layout
    const int m_tiles = (d.M + ctas * kBM - 1) / (ctas * kBM);
    const int n_tiles = (d.N + bn - 1) / bn;
    plan->n_tiles = n_tiles;
    plan->num_tiles = m_tiles * n_tiles;
    const int slots = num_sms / ctas;     // tiles in flight: one per CTA, or per cluster of two
    plan->grid = ctas * (plan->num_tiles < slots ? plan->num_tiles : slots);
    // Inner tensor dimension rounded up to the 16-byte granule (columns [K, K8) are zero in A and in the packed weights by the
    // contract above): with K = 28 the 56-byte rows put the out-of-bounds edge in the middle of a 16-byte chunk and the TMA
    // unit takes a slow path — the 28 -> 960 layer ran 44.5 instead of 35.6 us (experiments/microbench/gemm_sweep.cu).
    const int Kt = ((d.K + 7) / 8 * 8 <= d.lda && (d.K + 7) / 8 * 8 <= d.ldw) ? (d.K + 7) / 8 * 8 : d.K;
    int r = make_tmap_bf16_2d(&plan->tmA, d.A, d.M, Kt, d.lda, kBM);
    if (r) return r;
    r = make_tmap_bf16_2d(&plan->tmB, d.W, d.N, Kt, d.ldw, box_n);
    if (r) return r;
    if (!d.out_f32) {
        // store map: columns [N, round_up(N, 8)) are part of the tensor and receive zeros
        r = make_tmap_bf16_2d_ex(&plan->tmC, d.out, d.M, (d.N + 7) / 8 * 8, d.ldc, 32, 32, 64);
    } else {
        plan->tmC = plan->tmA;     // unused by the f32-output instantiations
    }
    if (r) return r;
    plan->tmA_lo = plan->tmA; plan->tmB_lo = plan->tmB; plan->tmC_lo = plan->tmC;      // placeholders when unused
    if (d.split) {
        r = make_tmap_bf16_2d(&plan->tmA_lo, d.A_lo, d.M, Kt, d.lda, kBM);
        if (r) return r;
        r = make_tmap_bf16_2d(&plan->tmB_lo, d.W_lo, d.N, Kt, d.ldw, box_n);
        if (r) return r;
    }
    if (d.out_split) r = make_tmap_bf16_2d_ex(&plan->tmC_lo, d.out_lo, d.M, (d.N + 7) / 8 * 8, d.ldc, 32, 32, 64);
    return r;
}

cudaError_t tc_gemm_launch(const TcGemmPlan& plan, cudaStream_t stream) {
    const GemmDesc& d = plan.desc;
    TcGemmLnArgs a;
    a.M = d.M; a.N = d.N; a.K = d.K;
    a.block_n = plan.block_n;
    a.num_stages = plan.num_stages;
    a.n_tiles = plan.n_tiles;
    a.num_tiles = plan.num_tiles;
    a.num_kb = (d.K + kBK - 1) / kBK;
    a.bias = d.bias;
    a.pos = d.pos;
    a.pos_period = d.pos_period > 0 ? d.pos_period : 1;
    a.resid = d.resid;
    a.ldr = d.ldr;
    a.out = d.out;
    a.ldc = d.ldc;
    a.n_store = d.out_f32 ? (d.N + 3) / 4 * 4 : (d.N + 7) / 8 * 8;
    a.ln_gamma = d.ln_gamma; a.ln_beta = d.ln_beta; a.ln_eps = d.ln_eps;
    a.ln_out = static_cast<__nv_bfloat16*>(d.ln_out); a.ln_ld = d.ln_ld;
    a.split = d.split;
    switch (d.act) {
        case ACT_NONE: return plan.pair ? launch_act<ACT_NONE, true>(plan, a, stream) : launch_act<ACT_NONE, false>(plan, a, stream);
        case ACT_MISH: return plan.pair ? launch_act<ACT_MISH, true>(plan, a, stream) : launch_act<ACT_MISH, false>(plan, a, stream);
        case ACT_GELU: return plan.pair ? launch_act<ACT_GELU, true>(plan, a, stream) : launch_act<ACT_GELU, false>(plan, a, stream);
    }
    return cudaErrorInvalidValue;
}

}  // namespace vitdet
