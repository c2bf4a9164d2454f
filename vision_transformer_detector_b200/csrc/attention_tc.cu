// Multi-head self-attention core on the 5th-gen tensor cores: softmax(q k^T / sqrt(d)) v per
// (image, head) without materialising the (B, H, T, T) score tensor of keras.layers.MultiHeadAttention
// (reference det.py:364-369).
//
// The product form (NB = 1, bf16, key_dim <= 64): one CTA = 128 queries of one (image, head); two CTAs are resident
// per SM so that the softmax of one overlaps the softmax latencies of the other.  192 threads:
//   warp 4      TMA producer: Q once, then 128-key K and V tiles (cp.async.bulk.tensor, 128B swizzle)
//               through a 3-stage mbarrier ring.
//   warp 5      allocates 256 TMEM columns; one lane issues
//                 S = Q K(j)^T        tcgen05.mma  M128 x N128 x K(16*ceil(d/16)), A and B K-major from smem
//                 O += P V(j)         tcgen05.mma  M128 x N64 x K128, A = P from TENSOR MEMORY, B = V MN-major
//               QK^T(j+1) is issued as soon as the softmax warps have S(j) in registers.
//   warps 0..3  softmax: thread = query row (TMEM lane).  One tcgen05.ld pass brings the 128 scores of
//               the row into registers (S is released to the MMA warp immediately), row maximum without
//               shuffles, p = ex2(s*c - m), row sum, P written back to TMEM as packed bf16 (tcgen05.st) —
//               never through shared memory.  The running maximum is only advanced (and O rescaled in
//               TMEM) when it grew by more than 2^8, so most tiles skip the correction.
// TMEM columns: S [0,128) f32 | P [128,192) bf16x2 | O [192,256) f32.
//
// Heads wider than 64 (64 < key_dim <= 128; the reference accepts any key_dim) run the same kernel with NB = 2: every Q / K /
// V tile is two 64-column boxes, QK^T walks up to eight k-steps across them, PV is issued once per box of V into O
// [192, 320), the CTA allocates 512 TMEM columns and the SM holds one CTA with two K/V stages.
//
// The fp32-accumulate mode runs the same kernel with SPLIT = true (key_dim <= 64): every operand is carried as two bf16
// planes (hi = bf16(x), lo = bf16(x - hi), |x - hi - lo| <= 2^-18 |x|) and every product is three passes with float32
// accumulation in TMEM:
//     S  = q_hi k_hi^T + q_hi k_lo^T + q_lo k_hi^T
//     O += p_hi v_hi   + p_hi v_lo   + p_lo v_hi          (p = 2^(s c - m) in float32, split like the other operands)
// with hi and lo tiles of Q, K, V in shared memory (160 KB, one CTA per SM, two K/V stages) and TMEM columns
// S [0,128) | P_hi [128,192) | P_lo [192,256) | O [256,320).  The float32 scores, their maximum, the exponentials and the
// row sums never leave float32; the context rows are written as (hi, lo) planes for the output projection.
//
// The binding unit is the SFU, not the tensor pipe: per 128 x 128 score tile the CTA needs 16 384 ex2 at
// 16/clk/SM = 1024 clk, against ~450 clk of MMA at head_dim 40 (DESIGN.md §4).  Tiles of 128 keys (not 64)
// because the per-tile fixed costs (barrier round trips, TMEM load/store latency) are what keeps the
// SFU idle (profiles/r01c_*).
#include "common.cuh"
#include "kernels.h"
#include "launch.h"

namespace vitdet {

namespace {

constexpr int kQ = 128;            // queries per CTA (UMMA M)
constexpr int kKV = 128;           // keys per tile (UMMA N of QK^T, K of PV)
constexpr int kHP = 64;            // head pitch in elements (one 128-byte swizzle row of bf16)
constexpr int kThreads = 192;
// softmax warps 0..3 (warp = TMEM lane quadrant); the TMA producer and the MMA issuer take the highest warp ids,
// which the warp arbiter favours: the MMA issuer's wake-up latency is on the critical path of every tile
constexpr int kProducerWarp = 4, kMmaWarp = 5;
// Shared memory: Q slot 0 | slot 1, then per stage the K slots | the V slots.  A slot is one 64-column box of a head tile,
// or in the split form one (hi, lo) plane of it.  Q and K / V slots are both 16 KiB.
constexpr int kQBytes = kQ * kHP * 2;         // 16 KiB per slot of Q
constexpr int kTileBytes = kKV * kHP * 2;     // 16 KiB: one slot of a K tile or a V tile = two TMA boxes of 64 rows
constexpr int kBoxBytes = 64 * kHP * 2;
static_assert(kQBytes == kTileBytes, "the MMA issuer steps over Q's and K's slots with one descriptor offset");
// NB = 64-column boxes per head tile: 1 for key_dim <= 64 (the product configuration: two CTAs per SM, three K/V stages),
// 2 for 64 < key_dim <= 128 (one CTA per SM: O needs 128 TMEM columns and the tiles twice the shared memory).
// SPLIT: the fp32-accumulate form (NB = 1), two planes per tile: one CTA per SM, like NB = 2.
template <int NB, bool SPLIT> struct AttnCfg {
    static_assert(NB == 1 || !SPLIT, "the split form holds one 64-column box per plane");
    static constexpr int kSlots = SPLIT ? 2 : NB;
    static constexpr int kStages = kSlots == 1 ? 3 : 2;
    static constexpr int kTmemCols = kSlots == 1 ? 256 : 512;
    static constexpr int kStageBytes = 2 * kSlots * kTileBytes;      // K slots, then V slots
    static constexpr int kMinBlocks = kSlots == 1 ? 2 : 1;
    static constexpr uint32_t kColPlo = 192;                         // P_lo [192,256) bf16x2 (split form only)
    static constexpr uint32_t kColO = SPLIT ? 256 : 192;             // O [kColO, kColO + 64 NB) f32
};
constexpr uint32_t kColS = 0, kColP = 128;    // S [0,128) f32 | P (P_hi) [128,192) bf16x2
constexpr float kRescaleThreshold = 8.f;      // log2 units: P stays <= 2^8 between rescales

// Tensor maps of qkv: one for the bf16 forms; the split form adds the lo plane (same shape and pitch).
template <bool SPLIT> struct AttnMaps { CUtensorMap qkv; };
template <> struct AttnMaps<true> { CUtensorMap qkv, lo; };

struct AttnTcArgs {
    __nv_bfloat16* ctx;      // context rows (the hi plane in the split form)
    int ldo;
    int T, H;
    int hp;              // elements per head in qkv / ctx (key_dim rounded up to 8)
    int k16;             // ceil(d / 16): K steps of the QK^T product
    float scale_log2;    // log2(e) / sqrt(key_dim)
    __nv_bfloat16* ctx_lo;   // split form: lo plane of the context rows (last, so that the bf16 forms' offsets stay put)
};

__device__ __forceinline__ float ex2f(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// One key tile of the online softmax for the calling thread's query row: NCH = number of 32-key chunks that
// hold at least one existing key (4 for a full tile), MASK = the last of them is partial.  Static loops only,
// so that the 128 scores stay in registers.
template <int NCH, bool MASK, int NB, bool SPLIT>
__device__ __forceinline__ void softmax_tile(uint32_t tS, uint32_t tP, uint32_t tPlo, uint32_t tO, uint32_t bar_s_free,
                                             uint32_t bar_pv_done, uint32_t bar_p_full, int lane, int j, int valid,
                                             float scale_log2, float& m_used, float& l) {
    // the row slice into registers (all loads in flight, one wait), then S belongs to the MMA warp again and
    // QK^T(j+1) overlaps this tile's softmax
    uint32_t v[NCH][32];
#pragma unroll
    for (int c = 0; c < NCH; ++c) tmem_ld_32x32(tS + 32u * c, v[c]);
    tmem_ld_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar_s_free);

    if (MASK) {
#pragma unroll
        for (int i = 0; i < 32; ++i)
            if (32 * (NCH - 1) + i >= valid) v[NCH - 1][i] = 0xff800000u;     // -inf: keys past the end of the image
    }
    // (three-input FMNMX3 maxima, 64 instead of 128 instructions, changed nothing: 2.776 vs 2.778 ms per step, r03b_ab.log)
    float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
    for (int c = 0; c < NCH; ++c)
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
            mx[0] = fmaxf(mx[0], __uint_as_float(v[c][i]));     mx[1] = fmaxf(mx[1], __uint_as_float(v[c][i + 1]));
            mx[2] = fmaxf(mx[2], __uint_as_float(v[c][i + 2])); mx[3] = fmaxf(mx[3], __uint_as_float(v[c][i + 3]));
        }
    const float m_new = fmaxf(m_used, fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3])) * scale_log2);
    const bool grow = __any_sync(0xffffffffu, m_new > m_used + kRescaleThreshold);   // true on the first tile
    float alpha = 1.f;
    if (grow) {
        alpha = ex2f(m_used - m_new);       // 0 on the first tile (m_used = -inf)
        m_used = m_new;
        l *= alpha;
    }
    const float neg_m = -m_used;
    // p = 2^(s*c - m) in place; packed pairs overwrite the first half of each chunk's registers (in the split form the hi
    // pairs; the lo pairs go to lo[]).  The scale-and-shift and the row sums run on packed float pairs (FFMA2 / FADD2: one
    // issue slot for two elements).
    const uint64_t sc2 = f2_pack(scale_log2, scale_log2), nm2 = f2_pack(neg_m, neg_m);
    uint64_t sum2[2] = {0ull, 0ull};       // two (0.f, 0.f) pairs
    uint32_t lo[SPLIT ? NCH : 1][16];
#pragma unroll
    for (int c = 0; c < NCH; ++c)
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
            float t0, t1, t2, t3;
            f2_unpack(f2_fma(f2_pack(__uint_as_float(v[c][i]), __uint_as_float(v[c][i + 1])), sc2, nm2), t0, t1);
            f2_unpack(f2_fma(f2_pack(__uint_as_float(v[c][i + 2]), __uint_as_float(v[c][i + 3])), sc2, nm2), t2, t3);
            const float e0 = ex2f(t0), e1 = ex2f(t1), e2 = ex2f(t2), e3 = ex2f(t3);      // ex2(-inf) = 0
            sum2[0] = f2_add(sum2[0], f2_pack(e0, e1));
            sum2[1] = f2_add(sum2[1], f2_pack(e2, e3));
            if constexpr (SPLIT) {      // p = hi + lo
                const __nv_bfloat162 h01 = __floats2bfloat162_rn(e0, e1), h23 = __floats2bfloat162_rn(e2, e3);
                v[c][i / 2] = *reinterpret_cast<const uint32_t*>(&h01);
                v[c][i / 2 + 1] = *reinterpret_cast<const uint32_t*>(&h23);
                lo[c][i / 2] = pack_bf16x2(e0 - __low2float(h01), e1 - __high2float(h01));
                lo[c][i / 2 + 1] = pack_bf16x2(e2 - __low2float(h23), e3 - __high2float(h23));
            } else {
                v[c][i / 2] = pack_bf16x2(e0, e1);
                v[c][i / 2 + 1] = pack_bf16x2(e2, e3);
            }
        }
    {
        float s0, s1, s2, s3;
        f2_unpack(sum2[0], s0, s1);
        f2_unpack(sum2[1], s2, s3);
        l += (s0 + s1) + (s2 + s3);
    }

    // P and O must no longer be in use by PV(j-1)
    if (j > 0) {
        mbar_wait(bar_pv_done, (j - 1) & 1);
        tc_fence_after();
        if (grow) {
#pragma unroll
            for (int c = 0; c < 2 * NB; ++c) {
                uint32_t o[32];
                tmem_ld_32x32(tO + 32u * c, o);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
                tmem_st_32x32_x32(tO + 32u * c, o);
            }
        }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) pk[i] = (c < NCH) ? v[c < NCH ? c : 0][i] : 0u;     // P = 0 for keys that do not exist
        tmem_st_32x32_x16(tP + 16u * c, pk);
        if constexpr (SPLIT) {
#pragma unroll
            for (int i = 0; i < 16; ++i) pk[i] = (c < NCH) ? lo[c < NCH ? c : 0][i] : 0u;
            tmem_st_32x32_x16(tPlo + 16u * c, pk);
        }
    }
    tmem_st_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(bar_p_full);
}

template <int NB, bool SPLIT>
__global__ void __launch_bounds__(kThreads, AttnCfg<NB, SPLIT>::kMinBlocks)
attn_tc_kernel(const __grid_constant__ AttnMaps<SPLIT> maps, const AttnTcArgs p) {
    using Cfg = AttnCfg<NB, SPLIT>;
    constexpr int kSlots = Cfg::kSlots;
    constexpr int kStages = Cfg::kStages;
    constexpr int kStageBytes = Cfg::kStageBytes;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * kStages + 5];
    __shared__ uint32_t tmem_base_s;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    pdl_launch_dependents();
    const int q0 = blockIdx.x * kQ;
    const int bh = blockIdx.y;
    const int b = bh / p.H, h = bh - b * p.H;
    const int row_base = b * p.T;          // first token row of this image in the [B*T, ld] matrices
    const int nkv = (p.T + kKV - 1) / kKV;

    const uint32_t base = smem_u32(smem_raw);
    if ((base & 1023u) != 0u) __trap();
    const uint32_t sQ = base;
    const uint32_t sKV = base + kSlots * kQBytes;      // stage s at + s * kStageBytes: the K slots, then the V slots
    const uint32_t bar_full = smem_u32(&bars[0]);
    const uint32_t bar_empty = smem_u32(&bars[kStages]);
    const uint32_t bar_q = smem_u32(&bars[2 * kStages]);
    const uint32_t bar_s_full = smem_u32(&bars[2 * kStages + 1]);   // QK^T(j) complete                 (MMA commit)
    const uint32_t bar_s_free = smem_u32(&bars[2 * kStages + 2]);   // S(j) is in registers             (4 warps)
    const uint32_t bar_p_full = smem_u32(&bars[2 * kStages + 3]);   // P(j) (and rescaled O) in TMEM    (4 warps)
    const uint32_t bar_pv_done = smem_u32(&bars[2 * kStages + 4]);  // PV(j) complete                   (MMA commit)

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, 1);
        }
        mbar_init(bar_q, 1);
        mbar_init(bar_s_full, 1);
        mbar_init(bar_s_free, 4);
        mbar_init(bar_p_full, 4);
        mbar_init(bar_pv_done, 1);
        fence_mbar_init();
    }
    if (warp == kMmaWarp) {
        tmem_alloc(smem_u32(&tmem_base_s), Cfg::kTmemCols);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    pdl_wait();       // set-up above overlapped the previous kernel; q/k/v are read from here on

    if (warp == kProducerWarp) {
        // ------------------------------ TMA producer ------------------------------
        if (lane == 0) {
            // slot 1 of a tile: the lo plane at the same columns (split form), or the next 64 columns of the head (NB = 2)
            const CUtensorMap* tm1 = &maps.qkv;
            constexpr int kCol1 = SPLIT ? 0 : 64;
            tma_prefetch_desc(&maps.qkv);
            if constexpr (SPLIT) {
                tm1 = &maps.lo;
                tma_prefetch_desc(tm1);
            }
            mbar_arrive_expect_tx(bar_q, kSlots * kQBytes);
#pragma unroll
            for (int s = 0; s < kSlots; ++s) {
                const CUtensorMap* tm = s ? tm1 : &maps.qkv;
                tma_load_2d(sQ + s * kQBytes, tm, bar_q, h * p.hp + kCol1 * s, row_base + q0);
                tma_load_2d(sQ + s * kQBytes + kBoxBytes, tm, bar_q, h * p.hp + kCol1 * s, row_base + q0 + 64);
            }
            int stage = 0;
            uint32_t phase = 0;
            for (int j = 0; j < nkv; ++j) {
                mbar_wait_relaxed(bar_empty + 8 * stage, phase ^ 1u);
                mbar_arrive_expect_tx(bar_full + 8 * stage, kStageBytes);
                const uint32_t dK = sKV + stage * kStageBytes, dV = dK + kSlots * kTileBytes;
                const int r = row_base + j * kKV;
#pragma unroll
                for (int s = 0; s < kSlots; ++s) {
                    const CUtensorMap* tm = s ? tm1 : &maps.qkv;
                    tma_load_2d(dK + s * kTileBytes, tm, bar_full + 8 * stage, (p.H + h) * p.hp + kCol1 * s, r);
                    tma_load_2d(dK + s * kTileBytes + kBoxBytes, tm, bar_full + 8 * stage, (p.H + h) * p.hp + kCol1 * s, r + 64);
                    tma_load_2d(dV + s * kTileBytes, tm, bar_full + 8 * stage, (2 * p.H + h) * p.hp + kCol1 * s, r);
                    tma_load_2d(dV + s * kTileBytes + kBoxBytes, tm, bar_full + 8 * stage, (2 * p.H + h) * p.hp + kCol1 * s, r + 64);
                }
                if (++stage == kStages) { stage = 0; phase ^= 1u; }
            }
        }
    } else if (warp == kMmaWarp) {
        // ------------------------------ MMA issuer --------------------------------
        // The whole warp runs the loop (warp-uniform control flow, loop state in uniform registers); only the
        // tcgen05 instructions are issued by one elected lane.  Its wake-up-to-issue latency is on the critical
        // path of every tile.
        const uint32_t idesc_qk = umma_idesc_bf16_f32(kQ, kKV);
        const uint32_t idesc_pv = umma_idesc_bf16_f32_bmn(kQ, SPLIT ? 16 * p.k16 : kHP);
        const uint32_t tS = tmem_base + kColS, tP = tmem_base + kColP, tPlo = tmem_base + Cfg::kColPlo, tO = tmem_base + Cfg::kColO;
        const uint64_t dq = umma_desc_sw128_kmajor(sQ);
        const uint64_t dkv0 = umma_desc_sw128_kmajor(sKV);
        constexpr uint32_t kStageStep = kStageBytes >> 4, kVOff = (kSlots * kTileBytes) >> 4, kSlotStep = kTileBytes >> 4;     // descriptor address units (16 B)
        mbar_wait(bar_q, 0);
        // Heads are stored hp (< 64) columns apart, so the 64-column TMA boxes also carry the first columns of the
        // next head.  In QK^T only the columns below 16 * k16 take part: clearing Q's columns [hp, 16 * k16) once makes
        // their products vanish whatever K holds there; V's extra columns only produce columns of O that are never
        // stored.  16-byte chunk c of row r sits at chunk c ^ (r & 7) of the 128-byte swizzled row.
        if (p.hp < 16 * p.k16) {
            const int c_lo = p.hp >> 3, c_hi = 2 * p.k16;      // 16-byte chunks of the head tile
            if constexpr (SPLIT) {
                for (int r = lane; r < 2 * kQ; r += 32)          // rows of Q_hi, then of Q_lo (same swizzle: 1024-byte atoms)
                    for (int c = c_lo; c < c_hi; ++c)
                        asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(sQ + r * 128 + ((c ^ (r & 7)) << 4)), "r"(0u) : "memory");
            } else {
                for (int r = lane; r < kQ; r += 32)              // chunk c lives in box c / 8
                    for (int c = c_lo; c < c_hi; ++c)
                        asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(sQ + (c >> 3) * kQBytes + r * 128 + (((c & 7) ^ (r & 7)) << 4)), "r"(0u) : "memory");
            }
            fence_proxy_async_smem();
            __syncwarp();
        }
        int stage = 0;
        uint32_t phase = 0;
        for (int j = 0; j <= nkv; ++j) {
            if (j < nkv) {
                // S = Q K(j)^T; the softmax warps moved S(j-1) into registers before signalling s_free
                mbar_wait(bar_full + 8 * stage, phase);
                if (j >= 1) mbar_wait(bar_s_free, (j - 1) & 1);
                tc_fence_after();
                if (elect_one()) {
                    const uint64_t dk = dkv0 + static_cast<uint64_t>(stage * kStageStep);
                    if constexpr (SPLIT) {
                        // passes: (q_hi, k_hi), (q_hi, k_lo), (q_lo, k_hi)
#pragma unroll
                        for (int t = 0; t < 3; ++t) {
                            const uint64_t a = dq + (t == 2 ? kSlotStep : 0u), bk = dk + (t == 1 ? kSlotStep : 0u);
                            for (int k = 0; k < p.k16; ++k) umma_bf16_ss(tS, a + 2u * k, bk + 2u * k, idesc_qk, (t | k) ? 1u : 0u);
                        }
                    } else {
                        umma_bf16_ss(tS, dq, dk, idesc_qk, 0u);
                        if (p.k16 > 1) umma_bf16_ss(tS, dq + 2u, dk + 2u, idesc_qk, 1u);
                        if (p.k16 > 2) umma_bf16_ss(tS, dq + 4u, dk + 4u, idesc_qk, 1u);
                        if (p.k16 > 3) umma_bf16_ss(tS, dq + 6u, dk + 6u, idesc_qk, 1u);
                        if (NB > 1) {       // head columns 64 .. 127: the second box of Q and of K
                            for (int k = 4; k < p.k16; ++k)
                                umma_bf16_ss(tS, dq + kSlotStep + 2u * (k - 4), dk + kSlotStep + 2u * (k - 4), idesc_qk, 1u);
                        }
                    }
                    umma_commit(bar_s_full);
                }
                __syncwarp();
            }
            if (j > 0) {
                // O += P(j-1) V(j-1)
                const int ps = (j - 1) % kStages;
                mbar_wait(bar_p_full, (j - 1) & 1);
                tc_fence_after();
                if (elect_one()) {
                    const uint64_t dv = dkv0 + static_cast<uint64_t>(ps * kStageStep + kVOff);
                    // 16 keys per step: 8 packed columns of P, 16 rows (2048 B) of V
                    if constexpr (SPLIT) {
                        // passes: (p_hi, v_hi), (p_hi, v_lo), (p_lo, v_hi)
#pragma unroll
                        for (int t = 0; t < 3; ++t)
#pragma unroll
                            for (int k = 0; k < kKV / 16; ++k)
                                umma_bf16_ts(tO, (t == 2 ? tPlo : tP) + 8u * k, dv + static_cast<uint64_t>((t == 1 ? kSlotStep : 0u) + 128u * k), idesc_pv,
                                             (t | k) ? 1u : (j > 1 ? 1u : 0u));
                    } else {
#pragma unroll
                        for (int nb = 0; nb < NB; ++nb)      // 64 output columns per V box
#pragma unroll
                            for (int k = 0; k < kKV / 16; ++k)
                                umma_bf16_ts(tO + 64u * nb, tP + 8u * k, dv + static_cast<uint64_t>(nb * kSlotStep + 128u * k), idesc_pv,
                                             (k != 0) ? 1u : (j > 1 ? 1u : 0u));
                    }
                    umma_commit(bar_empty + 8 * ps);
                    umma_commit(bar_pv_done);
                }
                __syncwarp();
            }
            if (j < nkv) { if (++stage == kStages) { stage = 0; phase ^= 1u; } }
        }
    } else {
        // ------------------------------ softmax -----------------------------------
        const int quad = warp & 3;                          // TMEM lane quadrant of this warp
        const uint32_t lane_off = static_cast<uint32_t>(quad * 32) << 16;
        const uint32_t tP = tmem_base + lane_off + kColP, tPlo = tmem_base + lane_off + Cfg::kColPlo, tO = tmem_base + lane_off + Cfg::kColO;
        float m_used = -INFINITY;      // running maximum in the scaled log2 domain
        float l = 0.f;                 // running sum of p
        const uint32_t tS = tmem_base + lane_off + kColS;
        for (int j = 0; j < nkv; ++j) {
            const int valid = min(kKV, p.T - j * kKV);      // keys of this tile that exist
            mbar_wait(bar_s_full, j & 1);
            tc_fence_after();
#define VITDET_TILE(NCH, MASK) \
    softmax_tile<NCH, MASK, NB, SPLIT>(tS, tP, tPlo, tO, bar_s_free, bar_pv_done, bar_p_full, lane, j, valid, p.scale_log2, m_used, l)
            if (valid == kKV) {
                VITDET_TILE(4, false);
            } else {
                // last tile of the image: only the chunks with existing keys are loaded and exponentiated
                // (16 of 128 keys at T = 1296); warp-uniform dispatch
                const bool partial = (valid & 31) != 0;
                switch ((valid + 31) >> 5) {
                    case 1: if (partial) VITDET_TILE(1, true); else VITDET_TILE(1, false); break;
                    case 2: if (partial) VITDET_TILE(2, true); else VITDET_TILE(2, false); break;
                    case 3: if (partial) VITDET_TILE(3, true); else VITDET_TILE(3, false); break;
                    default: VITDET_TILE(4, true); break;
                }
            }
#undef VITDET_TILE
        }

        // ---- finalise: O / l -> bf16 context rows (hi and lo planes in the split form) ----
        mbar_wait(bar_pv_done, (nkv - 1) & 1);
        tc_fence_after();
        const int q = q0 + quad * 32 + lane;
        const float inv = 1.f / l;
        const size_t ooff = static_cast<size_t>(row_base + (q < p.T ? q : 0)) * p.ldo + h * p.hp;
#pragma unroll
        for (int c = 0; c < 2 * NB; ++c) {
            uint32_t o[32];
            tmem_ld_32x32(tO + 32u * c, o);
            tmem_ld_wait();
            if (q < p.T) {
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    if (32 * c + 8 * g >= p.hp) break;          // the head holds hp columns; O's further columns are zero
                    uint32_t wh[4], wl[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const float y0 = __uint_as_float(o[8 * g + 2 * e]) * inv, y1 = __uint_as_float(o[8 * g + 2 * e + 1]) * inv;
                        if constexpr (SPLIT) {
                            const __nv_bfloat162 hh = __floats2bfloat162_rn(y0, y1);
                            wh[e] = *reinterpret_cast<const uint32_t*>(&hh);
                            wl[e] = pack_bf16x2(y0 - __low2float(hh), y1 - __high2float(hh));
                        } else {
                            wh[e] = pack_bf16x2(y0, y1);
                        }
                    }
                    *reinterpret_cast<uint4*>(p.ctx + ooff + 32 * c + 8 * g) = make_uint4(wh[0], wh[1], wh[2], wh[3]);
                    if constexpr (SPLIT) *reinterpret_cast<uint4*>(p.ctx_lo + ooff + 32 * c + 8 * g) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == kMmaWarp) {
        tc_fence_after();
        tmem_dealloc(tmem_base, Cfg::kTmemCols);
    }
}

template <int NB, bool SPLIT>
cudaError_t attn_launch(const AttnPlan& plan, const AttnMaps<SPLIT>& maps, void* ctx_lo, cudaStream_t stream) {
    using Cfg = AttnCfg<NB, SPLIT>;
    const AttnDesc& d = plan.desc;
    AttnTcArgs a;
    a.ctx = static_cast<__nv_bfloat16*>(d.ctx);
    a.ldo = d.ldo;
    a.T = d.T;
    a.H = d.H;
    a.hp = d.hp;
    a.k16 = (d.d + 15) / 16;
    a.scale_log2 = d.scale * 1.4426950408889634f;
    a.ctx_lo = static_cast<__nv_bfloat16*>(ctx_lo);
    const size_t smem = Cfg::kSlots * static_cast<size_t>(kQBytes) + static_cast<size_t>(Cfg::kStages) * Cfg::kStageBytes;
    const auto kern = attn_tc_kernel<NB, SPLIT>;
    cudaError_t e = ensure_max_dynamic_smem(reinterpret_cast<const void*>(kern), static_cast<int>(smem));
    if (e != cudaSuccess) return e;
    dim3 grid((d.T + kQ - 1) / kQ, d.B * d.H);
    return launch_kernel(kern, grid, dim3(kThreads), smem, stream, 1, maps, a);
}

}  // namespace

cudaError_t attn_tc_launch(const AttnPlan& plan, cudaStream_t stream) {
    const AttnMaps<false> maps{plan.tmQKV};
    if (plan.desc.hp <= 64) return attn_launch<1, false>(plan, maps, nullptr, stream);
    return attn_launch<2, false>(plan, maps, nullptr, stream);      // 64 < key_dim <= 128: two 64-column boxes per head tile
}

cudaError_t attn_tcs_launch(const AttnPlan& plan, const CUtensorMap& tm_lo, void* ctx_lo, cudaStream_t stream) {
    if (plan.desc.hp > 64) return cudaErrorInvalidValue;      // hi and lo tiles: one 64-column box per head (wider heads: attention.cu)
    return attn_launch<1, true>(plan, AttnMaps<true>{plan.tmQKV, tm_lo}, ctx_lo, stream);
}

}  // namespace vitdet
