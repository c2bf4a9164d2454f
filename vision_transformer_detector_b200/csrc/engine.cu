// Engine behind the C ABI (include/vitdet_b200.h): owns the packed weights and the workspace of one
// detector instance and strings the kernels of this directory into the forward pass that
// create_vision_transformer_detector builds as a Keras graph (reference det.py:498-583):
//   transformer_preprocessor det.py:239-309 -> transformer_encoder det.py:312-414 -> mlp_head
//   det.py:417-495 -> transform_predictions det.py:586-647 + thresholds det.py:2257-2283/1359-1384.
//
// Data layout in HBM (bf16 mode; the fp32 mode uses the same shapes with 4 bytes per element: IEEE float32 for the
// CUDA-core kernels, or two bf16 planes (hi | lo) per buffer for the tensor-core form, see Form):
//   x     f32  [B*T, D4]        residual stream, kept in f32 for the whole batch (145 KB / image)
//   per encoder chunk of Bc images (Mc = Bc*T rows), reused by every chunk:
//   patch bf16 [Mc, P8]         extract_patches output, (row, col, channel) order
//   y     bf16 [Mc, D8]         LayerNorm output (A operand of the QKV GEMM / first MLP GEMM)
//   qkv   bf16 [Mc, 3*H*hp]     q | k | v, hp = key_dim rounded up to 8 elements per head (no 64-wide pad in HBM: the
//                               attention kernel's 64-column TMA boxes start at column head*hp)
//   ctx   bf16 [Mc, H*hp]       attention output, same head pitch
//   u0,u1 bf16 [Mc, w1],[Mc,w2] ping-pong activations of the MLP pyramid
//   head (whole batch, R = B*S rows): s [R, Tp] (Tp = T rounded up to a 16-byte row pitch; for Tp == T this is the
//                               compact [B, T*S] buffer of which the reference's Reshape is a view), h0/h1 [R, u1],[R,u2]
// Weights: every Dense kernel is stored transposed, W[N, K] with K contiguous (both tcgen05 operands
// are K-major), once in bf16 and once in f32; biases in f32.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <condition_variable>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include "../../include/vitdet_b200.h"
#include "common.cuh"
#include "devbuf.h"
#include "kernels.h"

namespace vitdet {

// ------------------------------------------------------------------------------------------------
// error reporting
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

static inline int round_up(int v, int m) { return (v + m - 1) / m * m; }
static size_t a256(size_t v) { return (v + 255) / 256 * 256; }

constexpr int kMaxKeyDim = 128;   // one or two 64-column (128-byte swizzle row) boxes per head in shared memory
constexpr int kMaxKeyDimSplit = 64;     // the split (fp32-accumulate) attention kernel keeps hi and lo tiles: one box per head
// Elements per head in the qkv / ctx matrices: key_dim rounded up to 8 (16-byte rows for TMA and vector stores).  The
// attention kernel's 64-column boxes start at column head * hp, so HBM carries no 64-wide pad (Q's spill columns are
// cleared in shared memory, V's only produce output columns that are never stored).
static inline int head_pitch(int key_dim) { return (key_dim + 7) / 8 * 8; }

// Run-time switches of one handle (vitdet_set_option); the defaults are the product path unless the environment
// variable of the same meaning says otherwise (A/B scripts).
struct Options {
    int fuse_ln = 1;       // VITDET_FUSE_LN=0: stand-alone LayerNorm kernel
    int fuse_tail = 1;     // VITDET_FUSE_TAIL=0: the last three MLP layers as separate GEMM launches
    int gemm_pair = 1;     // VITDET_GEMM_PAIR=0 never / all (2) wherever legal / default: K >= 512 layers
    int fp32_tc = 1;       // VITDET_FP32=simt: the fp32 mode on CUDA-core IEEE kernels instead of split-bf16 tensor-core GEMMs
};

static Options env_options() {
    Options o;
    if (const char* e = getenv("VITDET_FUSE_LN")) o.fuse_ln = strcmp(e, "0") != 0;
    if (const char* e = getenv("VITDET_FUSE_TAIL")) o.fuse_tail = strcmp(e, "0") != 0;
    if (const char* e = getenv("VITDET_GEMM_PAIR")) o.gemm_pair = strcmp(e, "0") == 0 ? 0 : (strcmp(e, "all") == 0 ? 2 : 1);
    if (const char* e = getenv("VITDET_FP32")) o.fp32_tc = strcmp(e, "simt") != 0;
    return o;
}

// ------------------------------------------------------------------------------------------------
// weight packing kernels (run once per set_weight)
// ------------------------------------------------------------------------------------------------
// src: Keras Dense kernel viewed as row-major [K, N].  Element (k, n) goes to row rmap(n), column
// cmap(k) of the transposed, padded destination, where
//   rmap(n) = row_off + (n / gn) * pn + n % gn      cmap(k) = (k / gk) * pk + k % gk
// (identity for plain Dense; gn = key_dim, pn = hp scatters the heads of a q/k/v kernel to their hp-wide slots
// (hp = key_dim rounded up to 8); gk = key_dim, pk = hp does the same for the K axis of attention_output).
__global__ void pack_dense_kernel(const float* __restrict__ src, int K, int N, int gn, int pn, int row_off, int gk,
                                  int pk, __nv_bfloat16* __restrict__ w16, int ld16, long long lo_off,
                                  float* __restrict__ w32, int ld32) {
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= static_cast<long long>(K) * N) return;
    const int k = static_cast<int>(idx / N), n = static_cast<int>(idx - static_cast<long long>(k) * N);
    const int r = row_off + (n / gn) * pn + n % gn;
    const int c = (k / gk) * pk + k % gk;
    const float v = src[idx];
    if (w16) {
        const __nv_bfloat16 hi = __float2bfloat16_rn(v);
        w16[static_cast<size_t>(r) * ld16 + c] = hi;
        // lo plane of the split (fp32-accumulate) form: v = hi + lo up to 2^-18 |v|
        if (lo_off) w16[lo_off + static_cast<size_t>(r) * ld16 + c] = __float2bfloat16_rn(v - __bfloat162float(hi));
    }
    if (w32) w32[static_cast<size_t>(r) * ld32 + c] = v;
}

__global__ void pack_vec_kernel(const float* __restrict__ src, int N, int gn, int pn, int off, float* __restrict__ dst) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    dst[off + (n / gn) * pn + n % gn] = src[n];
}

__global__ void f32_to_bf16_kernel(const float* __restrict__ src, int rows, int cols, int lds,
                                   __nv_bfloat16* __restrict__ dst, int ldd) {
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= static_cast<long long>(rows) * ldd) return;
    const int r = static_cast<int>(idx / ldd), c = static_cast<int>(idx - static_cast<long long>(r) * ldd);
    dst[idx] = __float2bfloat16_rn(c < cols ? src[static_cast<size_t>(r) * lds + c] : 0.f);
}

// float32 rows -> the split (hi, lo) bf16 planes of the fp32-accumulate mode: hi = bf16(x), lo = bf16(x - hi); columns
// [cols, ldd) are written as zero.  8 elements per thread, 16-byte stores.
__global__ void split_rows_kernel(const float* __restrict__ src, long long rows, int cols, int lds, __nv_bfloat16* __restrict__ hi,
                                  __nv_bfloat16* __restrict__ lo, int ldd) {
    const int vec_per_row = ldd >> 3;
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= rows * vec_per_row) return;
    const long long r = idx / vec_per_row;
    const int c0 = static_cast<int>(idx - r * vec_per_row) << 3;
    const float* s = src + r * lds + c0;
    float x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = (c0 + i < cols) ? s[i] : 0.f;
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __nv_bfloat162 hh = __floats2bfloat162_rn(x[2 * i], x[2 * i + 1]);
        const __nv_bfloat162 ll = __floats2bfloat162_rn(x[2 * i] - __low2float(hh), x[2 * i + 1] - __high2float(hh));
        h[i] = *reinterpret_cast<const uint32_t*>(&hh);
        l[i] = *reinterpret_cast<const uint32_t*>(&ll);
    }
    *reinterpret_cast<uint4*>(hi + r * ldd + c0) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(lo + r * ldd + c0) = make_uint4(l[0], l[1], l[2], l[3]);
}

__global__ void pad_rows_f32_kernel(const float* __restrict__ src, int rows, int cols, int lds, float* __restrict__ dst,
                                    int ldd) {
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= static_cast<long long>(rows) * ldd) return;
    const int r = static_cast<int>(idx / ldd), c = static_cast<int>(idx - static_cast<long long>(r) * ldd);
    dst[idx] = c < cols ? src[static_cast<size_t>(r) * lds + c] : 0.f;
}

__global__ void unpad_rows_f32_kernel(const float* __restrict__ src, int rows, int cols, int lds, float* __restrict__ dst) {
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= static_cast<long long>(rows) * cols) return;
    const int r = static_cast<int>(idx / cols), c = static_cast<int>(idx - static_cast<long long>(r) * cols);
    dst[idx] = src[static_cast<size_t>(r) * lds + c];
}

// [B,T,H,d] f32 (q, k, v) -> fused [B*T, 3*H*hp] (bf16 or f32), pads zero.
template <typename T>
__global__ void pack_qkv_kernel(const float* __restrict__ q, const float* __restrict__ k, const float* __restrict__ v,
                                long long rows, int H, int d, int hp, T* __restrict__ dst) {
    const int ld = 3 * H * hp;
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= rows * ld) return;
    const long long r = idx / ld;
    const int c = static_cast<int>(idx - r * ld);
    const int sel = c / (H * hp), hh = (c / hp) % H, j = c % hp;
    float val = 0.f;
    if (j < d) {
        const float* s = sel == 0 ? q : (sel == 1 ? k : v);
        val = s[(r * H + hh) * d + j];
    }
    if (sizeof(T) == 2) reinterpret_cast<__nv_bfloat16*>(dst)[idx] = __float2bfloat16_rn(val);
    else reinterpret_cast<float*>(dst)[idx] = val;
}

template <typename T>
__global__ void unpack_ctx_kernel(const T* __restrict__ ctx, long long rows, int H, int d, int hp, float* __restrict__ out) {
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= rows * H * d) return;
    const long long r = idx / (H * d);
    const int c = static_cast<int>(idx - r * (H * d));
    const int hh = c / d, j = c - hh * d;
    const T* p = ctx + r * (H * hp) + hh * hp + j;
    float val;
    if (sizeof(T) == 2) val = __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(p));
    else val = *reinterpret_cast<const float*>(p);
    out[idx] = val;
}

// context rows kept as (hi, lo) bf16 planes [rows, H*hp] -> float32 [rows, H, d]
__global__ void unpack_ctx_planes_kernel(const __nv_bfloat16* __restrict__ hi, const __nv_bfloat16* __restrict__ lo, long long rows, int H,
                                         int d, int hp, float* __restrict__ out) {
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= rows * H * d) return;
    const long long r = idx / (H * d);
    const int c = static_cast<int>(idx - r * (H * d));
    const int hh = c / d, j = c - hh * d;
    const long long o = r * (H * hp) + hh * hp + j;
    out[idx] = __bfloat162float(hi[o]) + __bfloat162float(lo[o]);
}

static inline int blocks_for(long long n, int bs = 256) { return static_cast<int>((n + bs - 1) / bs); }

// ------------------------------------------------------------------------------------------------
// weights
// ------------------------------------------------------------------------------------------------
// One Dense layer in packed form.
struct DenseW {
    int N = 0, K = 0;          // packed GEMM shape (N includes head-slot pads for qkv, K for attention_output)
    int ld16 = 0, ld32 = 0;
    DevBuf w16, w32, bias;     // w16: hi plane [N, ld16] followed by the lo plane (split form); bias: f32 [round_up(N, 8)]
    long long lo_off() const { return static_cast<long long>(N) * ld16; }
    const void* w16_lo() const { return w16.as<__nv_bfloat16>() + lo_off(); }
    int alloc(int n, int k) {
        N = n; K = k;
        ld16 = round_up(k, 8);
        ld32 = round_up(k, 4);
        RC_TRY(w16.ensure(static_cast<size_t>(n) * ld16 * 2 * 2));
        RC_TRY(w32.ensure(static_cast<size_t>(n) * ld32 * 4));
        RC_TRY(bias.ensure(static_cast<size_t>(round_up(n, 8)) * 4));
        CU_TRY(cudaMemset(w16.p, 0, w16.bytes));
        CU_TRY(cudaMemset(w32.p, 0, w32.bytes));
        CU_TRY(cudaMemset(bias.p, 0, bias.bytes));
        return 0;
    }
};

// How one Keras variable maps into the packed storage.
struct WeightSlot {
    std::string name;
    int ndim = 0;
    int64_t shape[4] = {0, 0, 0, 0};
    int64_t count = 0;
    enum Kind { DENSE_KERNEL, DENSE_BIAS, VEC } kind = VEC;
    DenseW* dense = nullptr;   // DENSE_*
    int K = 0, N = 0;          // source [K, N] view of a kernel / N of a bias
    int gn = 1, pn = 1, row_off = 0, gk = 1, pk = 1;
    float* vec_dst = nullptr;  // VEC: plain f32 copy target (LayerNorm gamma/beta, position embedding, f32-only kernels)
    bool vec_transpose = false;   // VEC kernels kept in f32 as [N, K] (head slot projection, final Dense(6))
    bool set = false;
    std::vector<float> master;    // Keras-layout copy returned by get_weight
};

struct BlockW {
    DevBuf ln1_g, ln1_b, ln2_g, ln2_b;
    DenseW qkv, out;
    std::vector<DenseW> mlp;
};

// ------------------------------------------------------------------------------------------------
// Host staging: a caller's ordinary (pageable) array is copied into page-locked memory by a few threads at
// once — one thread moves ~10 GB/s, far less than the PCIe link the H2D copy then uses — sub-chunk by sub-chunk,
// so that the asynchronous H2D copy of sub-chunk i runs while sub-chunk i+1 is being staged.
// ------------------------------------------------------------------------------------------------
class StagePool {
public:
    explicit StagePool(int workers) {
        for (int i = 0; i < workers; ++i) threads_.emplace_back([this, i] { run(i); });
    }
    ~StagePool() {
        { std::lock_guard<std::mutex> g(m_); stop_ = true; ++gen_; }
        cv_.notify_all();
        for (auto& t : threads_) t.join();
    }
    // Concatenates n pieces into dst: piece k, srcs[k][0, offs[k + 1] - offs[k]), goes to dst + offs[k] - offs[0].  The
    // bytes are split over the workers and the calling thread; returns when all of it is done.
    void copy(char* dst, const char* const* srcs, const size_t* offs, int n) {
        const int parts = static_cast<int>(threads_.size()) + 1;
        const size_t bytes = offs[n] - offs[0];
        const size_t per = parts == 1 || bytes < (1u << 20) ? bytes : ((bytes + parts - 1) / parts + 4095) & ~static_cast<size_t>(4095);
        { std::lock_guard<std::mutex> g(m_); dst_ = dst; srcs_ = srcs; offs_ = offs; n_ = n; per_ = per; }
        if (per == bytes) { slice(0); return; }
        { std::lock_guard<std::mutex> g(m_); pending_ = parts - 1; ++gen_; }
        cv_.notify_all();
        slice(parts - 1);
        std::unique_lock<std::mutex> lk(m_);
        done_.wait(lk, [this] { return pending_ == 0; });
    }
private:
    void slice(int i) {
        const size_t lo = offs_[0] + per_ * static_cast<size_t>(i), hi = std::min(lo + per_, offs_[n_]);
        for (int k = 0; k < n_ && lo < hi; ++k) {
            const size_t a = std::max(lo, offs_[k]), b = std::min(hi, offs_[k + 1]);
            if (a < b) memcpy(dst_ + (a - offs_[0]), srcs_[k] + (a - offs_[k]), b - a);
        }
    }
    void run(int i) {
        unsigned long long seen = 0;
        for (;;) {
            { std::unique_lock<std::mutex> lk(m_); cv_.wait(lk, [&] { return gen_ != seen; }); seen = gen_; if (stop_) return; }
            slice(i);
            { std::lock_guard<std::mutex> g(m_); if (--pending_ == 0) done_.notify_one(); }
        }
    }
    std::vector<std::thread> threads_;
    std::mutex m_;
    std::condition_variable cv_, done_;
    unsigned long long gen_ = 0;
    bool stop_ = false;
    char* dst_ = nullptr; const char* const* srcs_ = nullptr; const size_t* offs_ = nullptr; int n_ = 0; size_t per_ = 0;
    int pending_ = 0;
};

// The records of R detection rows that a host entry point reads back in one copy, each array 256-byte aligned; bytes
// per row: logits 24 | decoded 24 | class_id 4 | class_conf 4 | corners 16 | keep 1 | packed 52 | boxes_original 16,
// the last two only when asked for.
struct RecordBlock {
    size_t R = 0, o_dec = 0, o_id = 0, o_cc = 0, o_cor = 0, o_keep = 0, o_pk = 0, o_box = 0, bytes = 0;
    bool packed = false, boxes = false;
    RecordBlock() = default;
    RecordBlock(size_t rows, bool want_packed, bool want_boxes) : R(rows), packed(want_packed), boxes(want_boxes) {
        o_dec = a256(R * 24); o_id = o_dec + a256(R * 24); o_cc = o_id + a256(R * 4); o_cor = o_cc + a256(R * 4);
        o_keep = o_cor + a256(R * 16); o_pk = o_keep + a256(R);
        o_box = o_pk + (packed ? a256(R * 52) : 0);
        bytes = o_box + (boxes ? a256(R * 16) : 0);
    }
    // the decode outputs inside a DEVICE block at base
    vitdet_detections detections(char* base) const {
        vitdet_detections d = {};
        d.decoded = reinterpret_cast<float*>(base + o_dec);
        d.class_id = reinterpret_cast<int32_t*>(base + o_id);
        d.class_conf = reinterpret_cast<float*>(base + o_cc);
        d.corners = reinterpret_cast<int32_t*>(base + o_cor);
        d.keep = reinterpret_cast<uint8_t*>(base + o_keep);
        if (packed) d.packed = reinterpret_cast<float*>(base + o_pk);
        return d;
    }
    float* boxes_original(char* base) const { return boxes ? reinterpret_cast<float*>(base + o_box) : nullptr; }
    // A HOST copy of the block -> the caller's arrays (each may be null)
    int copy_out(const char* pb, float* logits_host, const vitdet_detections* out_host, float* boxes_host) const {
        if (logits_host) memcpy(logits_host, pb, R * 24);
        if (out_host) {
            if (out_host->decoded) memcpy(out_host->decoded, pb + o_dec, R * 24);
            if (out_host->class_id) memcpy(out_host->class_id, pb + o_id, R * 4);
            if (out_host->class_conf) memcpy(out_host->class_conf, pb + o_cc, R * 4);
            if (out_host->corners) memcpy(out_host->corners, pb + o_cor, R * 16);
            if (out_host->keep) memcpy(out_host->keep, pb + o_keep, R);
            if (out_host->packed) {
                if (!packed) return fail(VITDET_E_INVALID, "collect: the submission did not ask for packed records");
                memcpy(out_host->packed, pb + o_pk, R * 52);
            }
        }
        if (boxes_host) memcpy(boxes_host, pb + o_box, R * 16);
        return 0;
    }
};

// One in-flight host submission (vitdet_submit_host .. vitdet_collect): its own pinned staging, device input and
// record block, so that the H2D copy of submission i+1 overlaps the compute of submission i.  A submission of separate
// images (vitdet_submit_images_host) also owns its letterbox table, copied to dev_table on the compute stream.
struct HostSlot {
    PinnedBuf pin_in, pin_out, pin_table;
    DevBuf dev_in, dev_out, dev_table;
    // a submission of JPEG files (vitdet_submit_jpeg_host): its descriptor block, decode scratch and decoded pixels
    PinnedBuf pin_jpeg;
    DevBuf jpeg_work, jpeg_rgb;
    std::vector<cudaEvent_t> copy_events;      // one per staged sub-chunk of images
    cudaEvent_t done = nullptr;                // recorded after the D2H copy of the record block
    bool busy = false;
    RecordBlock rec;
    float* boxes_host = nullptr;               // where vitdet_collect puts boxes_original, or null
    ~HostSlot() {
        for (auto e : copy_events) cudaEventDestroy(e);
        if (done) cudaEventDestroy(done);
    }
};

// Launch plans of the tensor-core forms for one encoder chunk or for the head, in launch order (see plan_cursor)
struct AttnTcPlan {
    AttnPlan plan;
    CUtensorMap lo;                // Split form: tensor map of the lo plane of qkv
};
struct Plans {
    bool complete = false;         // a whole pass has been recorded
    std::vector<TcGemmPlan> gemm;
    std::vector<AttnTcPlan> attn;
    std::vector<MlpTailPlan> tail;
};

}  // namespace vitdet

using namespace vitdet;

struct vitdet_handle {
    vitdet_config cfg;
    int device = 0;
    int num_sms = 148;
    int gh = 0, gw = 0, T = 0, P = 0, D = 0, H = 0, d = 0, S = 0;
    int hp = 0;                                // head_pitch(d)
    int RP = 0, PK = 0;                 // run pitch of one patch row (round_up(3p, 4)) and padded patch vector p * RP
    int act = ACT_MISH;
    int chunk = 64;
    Options opt;

    // weights
    DenseW proj;
    DevBuf pos;                         // f32 [T]
    std::vector<BlockW> blocks;
    DevBuf head_slot_w, head_slot_b;    // f32 [S, D], [S]
    std::vector<DenseW> head;
    DevBuf tail_w, tail_b;              // f32 [6, U], [6]
    int tail_U = 0;
    std::vector<WeightSlot> slots;
    std::map<std::string, int> slot_index;
    DevBuf stage;                       // device staging for set_weight

    // workspace (grow-only)
    DevBuf x, patch, y, qkv, ctx, u0, u1, s, h0, h1;
    DevBuf tmp32;                       // fp32 tensor-core mode: float32 staging of the patches / LayerNorm rows before their split, planes of the slot matrix
    // cached plans, key (encoder chunk / head, arithmetic form, images in the chunk / batch); cleared when a buffer moves
    std::map<std::tuple<int, int, int>, Plans> plans;

    // debug taps (vitdet_debug_taps): residual stream after the patch embedding and after every block, of the last forward
    bool weights_dirty = false;         // set_weight ran since the last forward: the pack kernels (legacy stream) must finish first
    int s_layout_es = 0;                // element size the slot matrix `s` was last laid out for (its pad columns are zeroed per layout)
    bool taps_on = false;
    DevBuf taps;                        // f32 [(L + 1)][B*T, D4]
    int taps_B = 0;
    const void* head_last = nullptr;    // input of the final Dense(6) in the last forward: [taps_B*S, head_last_ld]
    int head_last_ld = 0, head_last_f32 = 0;

    // profiling (off by default): CUDA events around the launches of the categories in prof_mask
    uint32_t prof_mask = 0;
    struct ProfRec { int cat; cudaEvent_t a, b; };
    std::vector<ProfRec> prof_pending;
    std::vector<cudaEvent_t> prof_pool;
    double prof_ms[32] = {};
    long long prof_n[32] = {};
    long long launches = 0;             // kernels launched by forward_impl since the last reset

    // pinned staging + device buffers for predict_host
    cudaStream_t copy_stream = nullptr;          // H2D copies of the host entry points run here, overlapped with compute
    static constexpr int kHostSlots = 2;
    HostSlot host_slots[kHostSlots];
    int next_slot = 0;
    StagePool* stage_pool = nullptr;             // created on the first pageable submission
    DevBuf images_table;                         // letterbox table of vitdet_forward_images, written in stream order
    // vitdet_decode_jpeg: descriptor block and files staged in pinned memory, device files and decode scratch; jpeg_done,
    // recorded after the last decode, orders their reuse whatever stream the next call runs on
    PinnedBuf jpeg_pin;
    cudaEvent_t jpeg_done = nullptr;
    DevBuf jpeg_files, jpeg_work;
    const long long* jpeg_stats = nullptr;       // repair counters of the last JPEG decode (device)

    ~vitdet_handle() {
        for (auto& r : prof_pending) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
        for (auto e : prof_pool) cudaEventDestroy(e);
        delete stage_pool;
        if (copy_stream) cudaStreamDestroy(copy_stream);
        if (jpeg_done) cudaEventDestroy(jpeg_done);
    }
};

namespace vitdet {

static int check_device(const vitdet_handle* h, const char* fn) {
    int cur = -1;
    CU_TRY(cudaGetDevice(&cur));
    if (cur != h->device)
        return fail(VITDET_E_INVALID, "%s: the handle lives on device %d but the current CUDA device is %d", fn, h->device, cur);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// configuration -> weight table (Keras `model.weights` order and names, see SURVEY §8(a))
// ------------------------------------------------------------------------------------------------
static std::string keras_name(const char* base, int index) {
    // keras.backend.clear_session() (det.py:548) resets the auto-name counters, so the first
    // instance of a layer class is un-suffixed and instance i >= 1 is "<base>_<i>".
    if (index == 0) return base;
    return std::string(base) + "_" + std::to_string(index);
}

static void add_slot(vitdet_handle* h, WeightSlot&& s) {
    s.count = 1;
    for (int i = 0; i < s.ndim; ++i) s.count *= s.shape[i];
    h->slot_index[s.name] = static_cast<int>(h->slots.size());
    h->slots.push_back(std::move(s));
}

static void add_dense_slots(vitdet_handle* h, const std::string& layer, DenseW* w, int K, int N) {
    WeightSlot k;
    k.name = layer + "/kernel"; k.ndim = 2; k.shape[0] = K; k.shape[1] = N;
    k.kind = WeightSlot::DENSE_KERNEL; k.dense = w; k.K = K; k.N = N;
    k.gn = N; k.pn = N; k.gk = K; k.pk = K;
    add_slot(h, std::move(k));
    WeightSlot b;
    b.name = layer + "/bias"; b.ndim = 1; b.shape[0] = N;
    b.kind = WeightSlot::DENSE_BIAS; b.dense = w; b.N = N; b.gn = N; b.pn = N;
    add_slot(h, std::move(b));
}

static int add_vec_slot(vitdet_handle* h, const std::string& name, DevBuf* buf, int ndim, const int64_t* shape,
                        bool transpose = false) {
    WeightSlot v;
    v.name = name; v.ndim = ndim;
    int64_t cnt = 1;
    for (int i = 0; i < ndim; ++i) { v.shape[i] = shape[i]; cnt *= shape[i]; }
    RC_TRY(buf->ensure(static_cast<size_t>(cnt) * 4));
    CU_TRY(cudaMemset(buf->p, 0, buf->bytes));
    v.kind = WeightSlot::VEC; v.vec_dst = buf->as<float>(); v.vec_transpose = transpose;
    if (transpose) { v.K = static_cast<int>(shape[0]); v.N = static_cast<int>(shape[1]); }
    add_slot(h, std::move(v));
    return 0;
}

static int build_weight_table(vitdet_handle* h) {
    const vitdet_config& c = h->cfg;
    const int D = h->D, H = h->H, d = h->d, T = h->T, P = h->P, S = h->S, hp = h->hp;

    // transformer_preprocessor: Dense 'linear_projection' (det.py:297) then PositionEncoding's
    // Embedding(T, 1) 'position_encoding/position_embedding' (det.py:148-151, 291-293).
    // The patch vector is stored with every patch-row run padded from 3p to RP elements (patchify_kernel), so
    // the kernel's K axis is scattered the same way: source row k -> column (k / 3p) * RP + k % 3p, pads zero.
    RC_TRY(h->proj.alloc(D, h->PK));
    add_dense_slots(h, "linear_projection", &h->proj, P, D);
    {
        WeightSlot& ks = h->slots[h->slot_index["linear_projection/kernel"]];
        ks.gk = 3 * c.patch_size; ks.pk = h->RP;
    }
    { const int64_t shp[2] = {T, 1}; RC_TRY(add_vec_slot(h, "position_encoding/position_embedding/embeddings", &h->pos, 2, shp)); }

    h->blocks.resize(c.repeat_times);
    for (int i = 0; i < c.repeat_times; ++i) {
        BlockW& b = h->blocks[i];
        const std::string ln1 = keras_name("layer_normalization", 2 * i);
        const std::string ln2 = keras_name("layer_normalization", 2 * i + 1);
        const std::string mha = keras_name("multi_head_attention", i);
        const int64_t shpD[1] = {D};
        RC_TRY(add_vec_slot(h, ln1 + "/gamma", &b.ln1_g, 1, shpD));
        RC_TRY(add_vec_slot(h, ln1 + "/beta", &b.ln1_b, 1, shpD));
        // MultiHeadAttention (det.py:364-369): q/k/v EinsumDense kernels (D, H, d) + bias (H, d),
        // fused into one [3*H*64, D] GEMM weight; attention_output kernel (H, d, D) + bias (D).
        RC_TRY(b.qkv.alloc(3 * H * hp, D));
        const char* sel[3] = {"query", "key", "value"};
        for (int s = 0; s < 3; ++s) {
            WeightSlot k;
            k.name = mha + "/" + sel[s] + "/kernel"; k.ndim = 3; k.shape[0] = D; k.shape[1] = H; k.shape[2] = d;
            k.kind = WeightSlot::DENSE_KERNEL; k.dense = &b.qkv; k.K = D; k.N = H * d;
            k.gn = d; k.pn = hp; k.row_off = s * H * hp; k.gk = D; k.pk = D;
            add_slot(h, std::move(k));
            WeightSlot bb;
            bb.name = mha + "/" + sel[s] + "/bias"; bb.ndim = 2; bb.shape[0] = H; bb.shape[1] = d;
            bb.kind = WeightSlot::DENSE_BIAS; bb.dense = &b.qkv; bb.N = H * d; bb.gn = d; bb.pn = hp; bb.row_off = s * H * hp;
            add_slot(h, std::move(bb));
        }
        RC_TRY(b.out.alloc(D, H * hp));
        {
            WeightSlot k;
            k.name = mha + "/attention_output/kernel"; k.ndim = 3; k.shape[0] = H; k.shape[1] = d; k.shape[2] = D;
            k.kind = WeightSlot::DENSE_KERNEL; k.dense = &b.out; k.K = H * d; k.N = D;
            k.gn = D; k.pn = D; k.gk = d; k.pk = hp;
            add_slot(h, std::move(k));
            WeightSlot bb;
            bb.name = mha + "/attention_output/bias"; bb.ndim = 1; bb.shape[0] = D;
            bb.kind = WeightSlot::DENSE_BIAS; bb.dense = &b.out; bb.N = D; bb.gn = D; bb.pn = D;
            add_slot(h, std::move(bb));
        }
        RC_TRY(add_vec_slot(h, ln2 + "/gamma", &b.ln2_g, 1, shpD));
        RC_TRY(add_vec_slot(h, ln2 + "/beta", &b.ln2_b, 1, shpD));
        // MLP pyramid (det.py:385-394): widths D * 2^(q-1) ... D.
        b.mlp.resize(c.mlp_quantities);
        int in = D;
        for (int j = 0; j < c.mlp_quantities; ++j) {
            const int units = D << (c.mlp_quantities - 1 - j);
            RC_TRY(b.mlp[j].alloc(units, in));
            add_dense_slots(h, "MLP_" + std::to_string(i + 1) + "_" + std::to_string(j + 1), &b.mlp[j], in, units);
            in = units;
        }
    }

    // mlp_head (det.py:454-493): auto-named 'dense', 'dense_1', ... then 'MLP_Head_no_Sigmoid'.
    int dense_idx = 0;
    {
        const std::string nm = keras_name("dense", dense_idx++);
        const int64_t shpk[2] = {D, S}; const int64_t shpb[1] = {S};
        RC_TRY(add_vec_slot(h, nm + "/kernel", &h->head_slot_w, 2, shpk, true));
        RC_TRY(add_vec_slot(h, nm + "/bias", &h->head_slot_b, 1, shpb));
    }
    const int n_head = c.head_dense_layers * c.head_block_repeats;
    h->head.resize(n_head);
    int in = T, li = 0;
    for (int k = c.head_dense_layers - 1; k >= 0; --k) {
        const int units = c.head_last_units << k;
        for (int r = 0; r < c.head_block_repeats; ++r, ++li) {
            RC_TRY(h->head[li].alloc(units, in));
            add_dense_slots(h, keras_name("dense", dense_idx++), &h->head[li], in, units);
            in = units;
        }
    }
    h->tail_U = in;
    {
        const int64_t shpk[2] = {in, 6}; const int64_t shpb[1] = {6};
        RC_TRY(add_vec_slot(h, "MLP_Head_no_Sigmoid/kernel", &h->tail_w, 2, shpk, true));
        RC_TRY(add_vec_slot(h, "MLP_Head_no_Sigmoid/bias", &h->tail_b, 1, shpb));
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------
// arithmetic forms
// ------------------------------------------------------------------------------------------------
// Bf16:  bf16 operands and stored activations, one tcgen05 pass per Dense (VITDET_MODE_BF16).
// Split: the fp32 mode on the tensor cores (north_star: <= 1e-3 against the float32 reference).  Every float32 activation
//        that feeds a Dense layer or the attention core travels as two bf16 planes (hi = bf16(x), lo = bf16(x - hi)) and
//        every Dense is three tcgen05 passes (hi*hi + hi*lo + lo*hi, float32 accumulation in TMEM) through the same two
//        GEMM kernels as Bf16, with exact expf-based activations in the epilogue; attention is the split instance of
//        attention_tc.cu.  The residual stream, LayerNorm, the head's slot projection and last Dense stay IEEE float32.
//        Buffers are sized as the fp32 mode's (4 bytes per element): the hi plane in the first half, the lo plane in the
//        second (planes_of).
// Ieee:  the fp32 mode on IEEE float32 CUDA-core kernels (gemm_simt.cu, attn_f32): "fp32_tc" = 0, or heads wider than
//        the split attention kernel takes (it holds hi and lo tiles: one 64-column box per head).
enum class Form { Bf16, Split, Ieee };

static Form pick_form(int mode, const Options& o, int key_dim) {
    if (mode == VITDET_MODE_BF16) return Form::Bf16;
    return o.fp32_tc && key_dim <= kMaxKeyDimSplit ? Form::Split : Form::Ieee;
}

struct Planes { __nv_bfloat16* hi; __nv_bfloat16* lo; };
static Planes planes_of(const DevBuf& b) {
    return Planes{b.as<__nv_bfloat16>(), reinterpret_cast<__nv_bfloat16*>(b.as<char>() + (b.bytes / 2 & ~static_cast<size_t>(255)))};
}

// ------------------------------------------------------------------------------------------------
// Dense dispatch
// ------------------------------------------------------------------------------------------------
// One activation matrix as a GEMM operand: bf16 or f32 rows, or the Split form's (hi, lo) planes (lo != nullptr).
struct Operand { void* p = nullptr; void* lo = nullptr; int ld = 0; };

struct DenseCall {
    Operand A;
    const DenseW* w;
    int M;
    const float* pos = nullptr; int pos_period = 1;
    const float* resid = nullptr; int ldr = 0;
    Operand out; int out_f32 = 0; int act = ACT_NONE;     // out.lo: the result is stored as (hi, lo) planes
    // optional fused LayerNorm of the output row (Bf16, N <= 32): see GemmDesc
    const float* ln_gamma = nullptr; const float* ln_beta = nullptr; void* ln_out = nullptr; int ln_ld = 0; float ln_eps = 1e-3f;
};

static GemmDesc make_desc(const DenseCall& c, Form f) {
    GemmDesc g;
    g.A = c.A.p; g.A_lo = c.A.lo; g.lda = c.A.ld;
    g.W = f == Form::Ieee ? c.w->w32.p : c.w->w16.p;
    g.ldw = f == Form::Ieee ? c.w->ld32 : c.w->ld16;
    g.M = c.M; g.N = c.w->N; g.K = c.w->K;
    g.bias = c.w->bias.as<float>();
    g.pos = c.pos; g.pos_period = c.pos_period;
    g.resid = c.resid; g.ldr = c.ldr;
    g.out = c.out.p; g.out_lo = c.out.lo; g.ldc = c.out.ld; g.out_f32 = c.out_f32; g.act = c.act;
    g.ln_gamma = c.ln_gamma; g.ln_beta = c.ln_beta; g.ln_out = c.ln_out; g.ln_ld = c.ln_ld; g.ln_eps = c.ln_eps;
    if (f == Form::Split) { g.split = 1; g.precise = 1; g.W_lo = c.w->w16_lo(); g.out_split = c.out.lo != nullptr; }
    return g;
}

// The CTA-pair form of the GEMM (gemm_tc.cu) serves the layers with enough rows, columns and depth to fill 256 x BN
// cluster tiles; VITDET_GEMM_PAIR=0 forces the single-CTA form everywhere, =all the pair form wherever it
// is legal (A/B measurements and tests).  The pair form has no fused LayerNorm, and no narrow float32 epilogue
// (its float32 layers take the wide one, OUT = 3).
// Measured (B = 64): 3 % faster on the MMA-bound layers (3584 -> 1792 -> 896 -> 448), slower on the K = 28
// layers whose time is the epilogue (the pair couples both CTAs' epilogues), hence the K threshold.
static bool pair_kernel_legal(const GemmDesc& g) { return g.M >= 1024 && g.N >= 128 && !g.ln_out; }

static bool use_pair_kernel(int pair_mode, const GemmDesc& g) {
    if (pair_mode == 0 || !pair_kernel_legal(g)) return false;
    // (the head's M = 17 B rows on the single-CTA kernel instead: 0.239 vs 0.219 ms per step, profiles/r03m_ab.log)
    return pair_mode == 2 || g.K >= 512;
}

// Tensor-core plan of one Dense (Bf16 / Split)
static int plan_dense(TcGemmPlan* plan, const DenseCall& c, Form f, int num_sms, int pair_mode) {
    const GemmDesc g = make_desc(c, f);
    const int rc = tc_gemm_make_plan(plan, g, num_sms, use_pair_kernel(pair_mode, g) ? 1 : 0);
    if (rc) return fail(VITDET_E_INVALID, "tensor-core GEMM plan (M=%d N=%d K=%d lda=%d ldc=%d) failed: %d", g.M, g.N, g.K, g.lda, g.ldc, rc);
    return 0;
}

static int launch_tc(TcGemmPlan plan /*by value: out / resid are patched per launch*/, void* out, const float* resid,
                     cudaStream_t st) {
    plan.desc.out = out;
    plan.desc.resid = resid;
    cudaError_t e = tc_gemm_launch(plan, st);
    if (e != cudaSuccess) return fail(VITDET_E_CUDA, "tc_gemm_launch failed: %s", cudaGetErrorString(e));
    return 0;
}

static int launch_simt(const DenseCall& c, cudaStream_t st) {
    GemmDesc g = make_desc(c, Form::Ieee);
    cudaError_t e = simt_gemm_launch(g, st);
    if (e != cudaSuccess) return fail(VITDET_E_CUDA, "simt_gemm_launch(M=%d N=%d K=%d) failed: %s", g.M, g.N, g.K, cudaGetErrorString(e));
    return 0;
}

// One Dense launch without a plan cache (operator entry points)
static int dense_once(const DenseCall& c, Form f, int num_sms, int pair_mode, cudaStream_t st) {
    if (f == Form::Ieee) return launch_simt(c, st);
    TcGemmPlan plan;
    RC_TRY(plan_dense(&plan, c, f, num_sms, pair_mode));
    return launch_tc(plan, c.out.p, c.resid, st);
}

// The fused LayerNorm needs the whole residual-stream row in one epilogue thread (D <= 32).
static bool ln_is_fused(const vitdet_handle* h) { return h->opt.fuse_ln && h->D <= 32; }
static bool tail_fusion_enabled(const vitdet_handle* h) { return h->opt.fuse_tail != 0; }

// ------------------------------------------------------------------------------------------------
// attention dispatch
// ------------------------------------------------------------------------------------------------
static AttnDesc attn_desc(const Operand& qkv, const Operand& ctx, int B, int T, int H, int d, int hp) {
    AttnDesc ad;
    ad.qkv = qkv.p; ad.ldq = qkv.ld; ad.ctx = ctx.p; ad.ldo = ctx.ld;
    ad.B = B; ad.T = T; ad.H = H; ad.d = d; ad.hp = hp;
    ad.scale = 1.f / sqrtf(static_cast<float>(d));
    return ad;
}

// Tensor-core attention plan; the Split form also maps the lo plane of qkv (same shape and pitch as the hi plane in `ad`).
static int attn_plan(AttnTcPlan* p, const AttnDesc& ad, const void* qkv_lo) {
    int rc = attn_bf16_make_plan(&p->plan, ad);
    if (!rc && qkv_lo) rc = make_tmap_bf16_2d(&p->lo, qkv_lo, ad.B * ad.T, 3 * ad.H * ad.hp, ad.ldq, 64);
    if (rc) return fail(VITDET_E_INVALID, "attention plan (B=%d T=%d H=%d d=%d) failed: %d", ad.B, ad.T, ad.H, ad.d, rc);
    return 0;
}

// ctx_lo: the Split form's lo plane of the context rows; `p` is unused by Ieee
static cudaError_t attn_launch(Form f, const AttnDesc& ad, const AttnTcPlan* p, void* ctx_lo, cudaStream_t st) {
    if (f == Form::Bf16) return attn_tc_launch(p->plan, st);
    if (f == Form::Split) return attn_tcs_launch(p->plan, p->lo, ctx_lo, st);
    return attn_f32_launch(ad, st);
}

// ------------------------------------------------------------------------------------------------
// workspace
// ------------------------------------------------------------------------------------------------
struct Dims {
    int es;          // activation element size
    int D4, D8, Pld, w_qkv, w_ctx, w_u0, w_u1, w_h0, w_h1;
    int Tp;          // row pitch of the slot matrix s [B*S, T]: T rounded up to a 16-byte multiple (pads stay zero)
};

static Dims dims_for(const vitdet_handle* h, Form f) {
    Dims m;
    const vitdet_config& c = h->cfg;
    m.es = f == Form::Bf16 ? 2 : 4;
    m.D4 = round_up(h->D, 4);
    m.D8 = round_up(h->D, 8);
    m.Pld = round_up(h->PK, 8);
    m.Tp = round_up(h->T, f == Form::Bf16 ? 8 : 4);
    m.w_qkv = 3 * h->H * h->hp;
    m.w_ctx = h->H * h->hp;
    // MLP ping-pong: layer j writes buffer j & 1; widest even / odd layer outputs.
    m.w_u0 = 8; m.w_u1 = 8;
    for (int j = 0; j + 1 < c.mlp_quantities; ++j) {
        const int units = round_up(h->D << (c.mlp_quantities - 1 - j), 8);
        if (j & 1) m.w_u1 = units > m.w_u1 ? units : m.w_u1; else m.w_u0 = units > m.w_u0 ? units : m.w_u0;
    }
    m.w_h0 = 8; m.w_h1 = 8;
    for (size_t i = 0; i < h->head.size(); ++i) {
        const int units = round_up(h->head[i].N, 8);
        if (i & 1) m.w_h1 = units > m.w_h1 ? units : m.w_h1; else m.w_h0 = units > m.w_h0 ? units : m.w_h0;
    }
    return m;
}

enum WorkspaceBuf { WS_X, WS_PATCH, WS_Y, WS_QKV, WS_CTX, WS_U0, WS_U1, WS_S, WS_H0, WS_H1, WS_TMP32, WS_COUNT };

// Bytes of every workspace buffer a forward of B images in form f uses.  In the Split form a buffer that holds planes
// keeps the second one at the 256-byte boundary below the middle of the allocation (planes_of); kPlaneSlack keeps that
// boundary above the end of the first plane.  tmp32 (Split only) stages the float32 patches / LayerNorm rows before their
// split, and holds the planes of the slot matrix.
static void workspace_layout(const vitdet_handle* h, int B, Form f, size_t bytes[WS_COUNT]) {
    constexpr size_t kPlaneSlack = 1024;
    const Dims m = dims_for(h, f);
    const size_t Mc = static_cast<size_t>(B < h->chunk ? B : h->chunk) * h->T, R = static_cast<size_t>(B) * h->S;
    const size_t slack = f == Form::Split ? kPlaneSlack : 0;
    bytes[WS_X] = static_cast<size_t>(B) * h->T * m.D4 * 4;
    bytes[WS_PATCH] = Mc * m.Pld * m.es + slack;
    bytes[WS_Y] = Mc * m.D8 * m.es + slack;
    bytes[WS_QKV] = Mc * m.w_qkv * m.es + slack;
    bytes[WS_CTX] = Mc * m.w_ctx * m.es + slack;
    bytes[WS_U0] = Mc * m.w_u0 * m.es + slack;
    bytes[WS_U1] = Mc * m.w_u1 * m.es + slack;
    bytes[WS_S] = R * m.Tp * m.es;
    bytes[WS_H0] = R * m.w_h0 * m.es + slack;
    bytes[WS_H1] = R * m.w_h1 * m.es + slack;
    bytes[WS_TMP32] = 0;
    if (f == Form::Split) {
        const size_t rows = Mc * round_up(h->PK > h->D ? h->PK : h->D, 4) * 4;
        const size_t slots = R * round_up(h->T, 8) * 4 + kPlaneSlack;
        bytes[WS_TMP32] = rows > slots ? rows : slots;
    }
}

static size_t workspace_bytes(const vitdet_handle* h, int B, Form f) {
    size_t bytes[WS_COUNT], tot = 0;
    workspace_layout(h, B, f, bytes);
    for (size_t b : bytes) tot += a256(b);
    return tot;
}

static int ensure_workspace(vitdet_handle* h, int B, Form f) {
    DevBuf* bufs[WS_COUNT] = {&h->x, &h->patch, &h->y, &h->qkv, &h->ctx, &h->u0, &h->u1, &h->s, &h->h0, &h->h1, &h->tmp32};
    size_t need[WS_COUNT];
    workspace_layout(h, B, f, need);
    const Dims m = dims_for(h, f);
    bool moved = false;
    for (int i = 0; i < WS_COUNT; ++i) {
        const void* p = bufs[i]->p;
        const size_t bytes = bufs[i]->bytes;
        RC_TRY(bufs[i]->ensure(need[i]));
        moved = moved || bufs[i]->p != p;
        if (i == WS_S) {
            // the pad columns [T, Tp) of every row are read by the first head GEMM's last k-step and never written
            if (m.Tp != h->T && (h->s.p != p || h->s.bytes != bytes || h->s_layout_es != m.es)) { CU_TRY(cudaMemset(h->s.p, 0, h->s.bytes)); CU_TRY(cudaDeviceSynchronize()); }
            h->s_layout_es = m.es;
        }
    }
    if (moved) h->plans.clear();     // a buffer moved: every cached TMA descriptor is stale
    return 0;
}

// ------------------------------------------------------------------------------------------------
// plan cache: the tensor-core forms' launch plans of one encoder chunk or of the head, in launch order, recorded by the
// first forward pass that needs them and replayed afterwards
// ------------------------------------------------------------------------------------------------
enum PlanPart { kEncoderPlans = 0, kHeadPlans = 1 };

struct PlanCursor {
    Plans* p;
    bool record;                   // first pass: make every plan and append it
    size_t gemm = 0, attn = 0, tail = 0;
};

// part: encoder chunk of n images, or the head of a batch of n
static PlanCursor plan_cursor(vitdet_handle* h, PlanPart part, Form f, int n) {
    Plans& p = h->plans[std::make_tuple(static_cast<int>(part), static_cast<int>(f), n)];
    if (!p.complete) p = Plans();       // (an earlier recording stopped at an error)
    return PlanCursor{&p, !p.complete};
}
// ------------------------------------------------------------------------------------------------
// profiling scopes
// ------------------------------------------------------------------------------------------------
enum ProfCat { PC_PATCHIFY = 0, PC_PROJ, PC_LN, PC_QKV, PC_ATTN, PC_OUT, PC_HEAD_SLOTS, PC_HEAD_GEMM, PC_HEAD_TAIL, PC_MLP0 = 9 };

static const char* prof_cat_name(int c) {
    static const char* base[] = {"patchify", "gemm_linear_projection", "layernorm", "gemm_qkv", "attention",
                                 "gemm_attention_output", "head_slots", "gemm_head", "head_tail_decode"};
    static char buf[32][24];
    if (c < 0 || c >= 32) return "";
    if (c < PC_MLP0) return base[c];
    snprintf(buf[c], sizeof(buf[c]), "gemm_mlp_%d", c - PC_MLP0 + 1);
    return buf[c];
}

static cudaEvent_t prof_event(vitdet_handle* h) {
    if (!h->prof_pool.empty()) { cudaEvent_t e = h->prof_pool.back(); h->prof_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

struct ProfScope {
    vitdet_handle* h; int cat; cudaStream_t st; cudaEvent_t a = nullptr; bool on;
    ProfScope(vitdet_handle* h_, int cat_, cudaStream_t st_) : h(h_), cat(cat_ < 32 ? cat_ : 31), st(st_) {
        ++h->launches;
        on = (h->prof_mask >> cat) & 1u;
        if (on) { a = prof_event(h); cudaEventRecord(a, st); }
    }
    ~ProfScope() {
        if (on) { cudaEvent_t b = prof_event(h); cudaEventRecord(b, st); h->prof_pending.push_back({cat, a, b}); }
    }
};

static int prof_collect(vitdet_handle* h) {
    for (auto& r : h->prof_pending) {
        CU_TRY(cudaEventSynchronize(r.b));
        float ms = 0.f;
        CU_TRY(cudaEventElapsedTime(&ms, r.a, r.b));
        h->prof_ms[r.cat] += ms; h->prof_n[r.cat] += 1;
        h->prof_pool.push_back(r.a); h->prof_pool.push_back(r.b);
    }
    h->prof_pending.clear();
    return 0;
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
// Optional staging information of predict_host: images arrive in sub-chunks of `ready_gran` images,
// sub-chunk i being complete when ready[i] fires; lead_chunks makes the first encoder chunks small so that
// compute starts after one sub-chunk and the rest of the copy hides behind it.
struct ForwardOpts {
    int lead_chunks[2] = {0, 0};      // sizes of the first two encoder chunks (0 = use the regular chunk)
    const cudaEvent_t* ready = nullptr;
    int ready_gran = 0;
};

// The images of a forward, on the device.  F32 / U8: B images of the model's size, one contiguous array of float32 or
// uint8 pixels (the patch kernel normalises uint8 ones, x / 127.5 - 1).  Letterbox: a table of B LetterboxImage entries,
// uint8 images of any size letterboxed inside the patch kernel; boxes_original, if not null, receives the [B * S, 4]
// boxes on the source images.
struct Input {
    enum Kind { F32, U8, Letterbox } kind;
    const void* p;
    float* boxes_original = nullptr;
};

// vitdet_decode_params / vitdet_detections -> the decode kernels' arguments (either may be null: defaults / no outputs)
static void decode_args(const vitdet_decode_params* p, int apply_transform, const vitdet_detections* o, float* logits,
                        DecodeParams* dp, DecodeOut* out) {
    out->logits = logits;
    if (p) {
        dp->obj_thr = p->objectness_threshold; dp->cls_thr = p->classification_threshold;
        dp->strict = p->strict; dp->img_h = p->image_h; dp->img_w = p->image_w; dp->classes = p->classes;
        dp->apply_transform = apply_transform;
        dp->corner_scale = p->corner_scale > 0.f ? p->corner_scale : 1.f;
    }
    if (o) {
        out->decoded = o->decoded; out->class_id = o->class_id; out->class_conf = o->class_conf;
        out->keep = o->keep; out->corners = o->corners; out->packed = o->packed;
    }
}

// One Dense of the forward pass: the tensor-core plan from the cursor (made from `c` on the recording pass), with `out` /
// `resid` patched because they move with the chunk, or the IEEE CUDA-core GEMM.
static int dense(vitdet_handle* h, Form f, PlanCursor& pc, int cat, const DenseCall& c, cudaStream_t st) {
    if (f == Form::Ieee) { ProfScope ps(h, cat, st); return launch_simt(c, st); }
    if (pc.record) {
        TcGemmPlan plan;
        RC_TRY(plan_dense(&plan, c, f, h->num_sms, h->opt.gemm_pair));
        pc.p->gemm.push_back(plan);
    }
    ProfScope ps(h, cat, st);
    return launch_tc(pc.p->gemm[pc.gemm++], c.out.p, c.resid, st);
}

static int forward_impl(vitdet_handle* h, const Input& in, int B, int mode, float* logits,
                        const vitdet_decode_params* dpar, const vitdet_detections* det, cudaStream_t st,
                        const ForwardOpts& opts = ForwardOpts()) {
    if (!h || !in.p || B <= 0) return fail(VITDET_E_INVALID, "forward: bad arguments");
    RC_TRY(check_device(h, "forward"));
    if (mode != VITDET_MODE_BF16 && mode != VITDET_MODE_FP32) return fail(VITDET_E_INVALID, "forward: unknown mode %d", mode);
    for (const WeightSlot& s : h->slots)
        if (!s.set) return fail(VITDET_E_UNSET, "forward: weight '%s' has not been set", s.name.c_str());
    if (h->weights_dirty) { CU_TRY(cudaDeviceSynchronize()); h->weights_dirty = false; }
    const vitdet_config& c = h->cfg;
    const Form f = pick_form(mode, h->opt, h->d);
    RC_TRY(ensure_workspace(h, B, f));
    const Dims m = dims_for(h, f);
    const int T = h->T, L = c.repeat_times, q = c.mlp_quantities;
    // Bf16 with D <= 32: every LayerNorm runs in the epilogue of the GEMM that produces the residual-stream row (projection
    // -> LN1 of block 0; attention output -> LN2; last MLP layer -> LN1 of the next block), and the last three MLP layers
    // of a block run as one kernel when their widths fit it (default model: 224 -> 112 -> 56 -> 28)
    const bool fuse_ln = f == Form::Bf16 && ln_is_fused(h);
    bool fuse_tail = false;
    if (fuse_ln && tail_fusion_enabled(h) && q >= 4) {
        const BlockW& b = h->blocks[0];
        const int N3[3] = {b.mlp[q - 3].N, b.mlp[q - 2].N, b.mlp[q - 1].N};
        const int K3[3] = {b.mlp[q - 3].K, b.mlp[q - 2].K, b.mlp[q - 1].K};
        fuse_tail = mlp_tail_supported(N3, K3);
    }
    const size_t tap_stride = static_cast<size_t>(B) * T * m.D4;      // floats per tap
    if (h->taps_on) { RC_TRY(h->taps.ensure(static_cast<size_t>(L + 1) * tap_stride * 4)); h->taps_B = B; }
    auto tap = [&](int index, const float* xc, int c0, int bc) -> int {
        if (!h->taps_on) return 0;
        CU_TRY(cudaMemcpyAsync(h->taps.as<float>() + index * tap_stride + static_cast<size_t>(c0) * T * m.D4, xc,
                               static_cast<size_t>(bc) * T * m.D4 * 4, cudaMemcpyDeviceToDevice, st));
        return 0;
    };
    // Rows of `cols` values that patchify / LayerNorm / the slot projection write for the next GEMM: into `buf` as bf16
    // (Bf16) or f32 (Ieee) rows, or (Split) f32 rows at `stage` that operand() splits into the planes of `buf`.
    struct Rows { void* p; int ld; int f32; };
    auto rows_out = [&](const DevBuf& buf, const DevBuf& stage, int cols) -> Rows {
        if (f == Form::Bf16) return Rows{buf.p, round_up(cols, 8), 0};
        return Rows{f == Form::Split ? stage.p : buf.p, round_up(cols, 4), 1};
    };
    // `buf` as rows of pitch ld in the form's operand layout (Split: its planes)
    auto act_in = [&](const DevBuf& buf, int ld) -> Operand {
        if (f != Form::Split) return Operand{buf.p, nullptr, ld};
        const Planes pl = planes_of(buf);
        return Operand{pl.hi, pl.lo, ld};
    };
    auto operand = [&](const Rows& r, const DevBuf& buf, long long rows, int cols, Operand* a) -> int {
        if (f != Form::Split) { *a = Operand{r.p, nullptr, r.ld}; return 0; }
        *a = act_in(buf, round_up(cols, 8));
        ++h->launches;
        split_rows_kernel<<<blocks_for(rows * (a->ld >> 3)), 256, 0, st>>>(static_cast<const float*>(r.p), rows, cols, r.ld,
                                                                         static_cast<__nv_bfloat16*>(a->p), static_cast<__nv_bfloat16*>(a->lo), a->ld);
        CU_TRY(cudaGetLastError());
        return 0;
    };
    auto layernorm = [&](const float* x, const DevBuf& gamma, const DevBuf& beta, int Mc, Operand* a) -> int {
        const Rows r = rows_out(h->y, h->tmp32, h->D);
        { ProfScope ps(h, PC_LN, st);
        CU_TRY(layernorm_launch(x, m.D4, gamma.as<float>(), beta.as<float>(), Mc, h->D, c.ln_epsilon, r.p, r.ld, r.f32, st)); }
        return operand(r, h->y, Mc, h->D, a);
    };
    // Output of a Dense that feeds another GEMM or the attention core: rows of `buf` in the form's operand layout
    auto to_act = [&](DenseCall& dc, const DevBuf& buf) {
        dc.out_f32 = f == Form::Ieee;
        dc.out = act_in(buf, round_up(dc.w->N, dc.out_f32 ? 4 : 8));
    };
    // Output into float32 rows [M, ld] (the residual stream, plus itself as the residual when `add`)
    auto to_f32 = [&](DenseCall& dc, float* o, int ld, bool add) {
        dc.out = Operand{o, nullptr, ld}; dc.out_f32 = 1;
        if (add) { dc.resid = o; dc.ldr = ld; }
    };
    auto with_ln = [&](DenseCall& dc, const DevBuf& gamma, const DevBuf& beta) {
        if (fuse_ln) { dc.ln_gamma = gamma.as<float>(); dc.ln_beta = beta.as<float>(); dc.ln_out = h->y.p; dc.ln_ld = m.D8; dc.ln_eps = c.ln_epsilon; }
    };

    for (int c0 = 0, bc = 0, ci = 0; c0 < B; c0 += bc, ++ci) {
        bc = (B - c0) < h->chunk ? (B - c0) : h->chunk;
        if (ci < 2 && opts.lead_chunks[ci] > 0 && opts.lead_chunks[ci] < bc) bc = opts.lead_chunks[ci];
        if (opts.ready) CU_TRY(cudaStreamWaitEvent(st, opts.ready[(c0 + bc + opts.ready_gran - 1) / opts.ready_gran - 1], 0));
        const int Mc = bc * T;
        float* x = h->x.as<float>() + static_cast<size_t>(c0) * T * m.D4;
        PlanCursor pc = plan_cursor(h, kEncoderPlans, f, bc);
        const Rows pr = rows_out(h->patch, h->tmp32, h->PK);
        if (in.kind == Input::Letterbox) {
            ProfScope ps(h, PC_PATCHIFY, st);
            CU_TRY(letterbox_patchify_launch(static_cast<const LetterboxImage*>(in.p) + c0, bc, c.image_h, c.image_w, c.patch_size,
                                             pr.p, pr.ld, h->RP, pr.f32, st));
        } else {
            const int u8 = in.kind == Input::U8;
            const char* img = static_cast<const char*>(in.p) + static_cast<size_t>(c0) * c.image_h * c.image_w * 3 * (u8 ? 1 : 4);
            ProfScope ps(h, PC_PATCHIFY, st);
            CU_TRY(patchify_launch(img, u8, bc, c.image_h, c.image_w, c.patch_size, pr.p, pr.ld, h->RP, pr.f32, st));
        }
        Operand a;
        RC_TRY(operand(pr, h->patch, Mc, h->PK, &a));
        DenseCall pj{a, &h->proj, Mc};
        pj.pos = h->pos.as<float>(); pj.pos_period = T;
        to_f32(pj, x, m.D4, false);
        with_ln(pj, h->blocks[0].ln1_g, h->blocks[0].ln1_b);
        RC_TRY(dense(h, f, pc, PC_PROJ, pj, st));
        RC_TRY(tap(0, x, c0, bc));
        const Operand y_fused{h->y.p, nullptr, m.D8};      // LayerNorm output of a fused epilogue
        for (int i = 0; i < L; ++i) {
            BlockW& b = h->blocks[i];
            a = y_fused;
            if (!fuse_ln) RC_TRY(layernorm(x, b.ln1_g, b.ln1_b, Mc, &a));
            DenseCall qc{a, &b.qkv, Mc};
            to_act(qc, h->qkv);
            RC_TRY(dense(h, f, pc, PC_QKV, qc, st));
            DenseCall oc{act_in(h->ctx, m.w_ctx), &b.out, Mc};      // the attention output is attention_output's A operand
            const AttnDesc ad = attn_desc(qc.out, oc.A, bc, T, h->H, h->d, h->hp);
            if (f != Form::Ieee && pc.record) {
                AttnTcPlan ap;
                RC_TRY(attn_plan(&ap, ad, qc.out.lo));
                pc.p->attn.push_back(ap);
            }
            { ProfScope ps(h, PC_ATTN, st);
            CU_TRY(attn_launch(f, ad, f == Form::Ieee ? nullptr : &pc.p->attn[pc.attn++], oc.A.lo, st)); }
            to_f32(oc, x, m.D4, true);
            with_ln(oc, b.ln2_g, b.ln2_b);
            RC_TRY(dense(h, f, pc, PC_OUT, oc, st));
            a = y_fused;
            if (!fuse_ln) RC_TRY(layernorm(x, b.ln2_g, b.ln2_b, Mc, &a));
            for (int j = 0; j < q; ++j) {
                if (fuse_tail && j == q - 3) {
                    if (pc.record) {
                        MlpTailDesc td;
                        td.A = a.p; td.lda = a.ld; td.M = Mc;
                        for (int l = 0; l < 3; ++l) {
                            DenseW& w = b.mlp[q - 3 + l];
                            td.N[l] = w.N; td.K[l] = w.K; td.W[l] = w.w16.p; td.ldw[l] = w.ld16; td.bias[l] = w.bias.as<float>();
                        }
                        td.x = x; td.ldx = m.D4; td.act = h->act;
                        if (i + 1 < L) {
                            td.ln_gamma = h->blocks[i + 1].ln1_g.as<float>(); td.ln_beta = h->blocks[i + 1].ln1_b.as<float>();
                            td.ln_eps = c.ln_epsilon; td.ln_out = h->y.p; td.ln_ld = m.D8;
                        }
                        MlpTailPlan tp;
                        const int rc = mlp_tail_make_plan(&tp, td, h->num_sms);
                        if (rc) return fail(VITDET_E_INVALID, "mlp_tail_make_plan failed: %d", rc);
                        tp.valid = true;
                        pc.p->tail.push_back(tp);
                    }
                    MlpTailPlan tp = pc.p->tail[pc.tail++];       // by value: the residual-stream pointer is patched per chunk
                    tp.desc.x = x;
                    ProfScope ps(h, PC_MLP0 + j, st);
                    const cudaError_t te = mlp_tail_launch(tp, st);
                    if (te != cudaSuccess) return fail(VITDET_E_CUDA, "mlp_tail_launch failed: %s", cudaGetErrorString(te));
                    break;
                }
                DenseCall mc{a, &b.mlp[j], Mc};
                mc.act = h->act;
                if (j == q - 1) {
                    to_f32(mc, x, m.D4, true);
                    if (i + 1 < L) with_ln(mc, h->blocks[i + 1].ln1_g, h->blocks[i + 1].ln1_b);
                } else {
                    to_act(mc, (j & 1) ? h->u1 : h->u0);
                }
                RC_TRY(dense(h, f, pc, PC_MLP0 + j, mc, st));
                a = mc.out;
            }
            RC_TRY(tap(i + 1, x, c0, bc));
        }
        pc.p->complete = true;
    }

    // mlp_head over the whole batch (det.py:454-493)
    const int R = B * h->S;
    PlanCursor pc = plan_cursor(h, kHeadPlans, f, B);
    const Rows sr{h->s.p, m.Tp, f != Form::Bf16};        // the Split form splits the slot matrix into tmp32's planes
    { ProfScope ps(h, PC_HEAD_SLOTS, st);
    CU_TRY(head_slots_launch(h->x.as<float>(), m.D4, h->head_slot_w.as<float>(), h->head_slot_b.as<float>(), B * T, h->D, h->S,
                             T, sr.ld, sr.p, sr.f32, st)); }
    Operand a;
    RC_TRY(operand(sr, h->tmp32, R, T, &a));
    for (size_t i = 0; i < h->head.size(); ++i) {
        DenseCall hc{a, &h->head[i], R};
        hc.act = h->act;
        DevBuf& ob = (i & 1) ? h->h1 : h->h0;
        // the final Dense(6) reads float32 rows in the Split form
        if (f == Form::Split && i + 1 == h->head.size()) to_f32(hc, ob.as<float>(), round_up(h->head[i].N, 4), false);
        else to_act(hc, ob);
        RC_TRY(dense(h, f, pc, PC_HEAD_GEMM, hc, st));
        a = hc.out;
    }
    pc.p->complete = true;
    DecodeParams dp;
    DecodeOut dout;
    decode_args(dpar, 1 /*the head emits raw logits*/, det, logits, &dp, &dout);
    if (in.kind == Input::Letterbox && in.boxes_original) {
        dout.boxes_original = in.boxes_original;
        dout.letterbox = static_cast<const LetterboxImage*>(in.p);
        dout.slots = h->S;
    }
    const int in_f32 = f != Form::Bf16;
    h->head_last = a.p; h->head_last_ld = a.ld; h->head_last_f32 = in_f32;
    ProfScope ps(h, PC_HEAD_TAIL, st);
    CU_TRY(head_tail_launch(a.p, a.ld, in_f32, h->tail_w.as<float>(), h->tail_b.as<float>(), R, h->tail_U, dp, dout, st));
    return 0;
}

}  // namespace vitdet

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

int vitdet_abi_version(void) { return VITDET_ABI_VERSION; }
const char* vitdet_last_error(void) { return g_err; }

void vitdet_default_config(vitdet_config* c) {
    if (!c) return;
    c->image_h = 608; c->image_w = 608;       // Constants.MODEL_IMAGE_SIZE det.py:22
    c->patch_size = 17; c->embedding_dim = 28; c->num_heads = 8; c->key_dim = 40;     // det.py:499-500
    c->mlp_quantities = 8; c->repeat_times = 8;                                        // det.py:501-502
    c->head_last_units = 136; c->head_dense_layers = 7; c->head_block_repeats = 1;     // det.py:503-504
    c->use_mish = 1;                                                                   // det.py:505
    c->num_slots = 17; c->classes = 80;                                                // det.py:28, :20
    c->ln_epsilon = 1e-3f;                                                             // keras default
}

int vitdet_create(const vitdet_config* cfg, vitdet_handle** out) {
    if (!cfg || !out) return fail(VITDET_E_INVALID, "vitdet_create: null argument");
    *out = nullptr;
    const vitdet_config& c = *cfg;
    if (c.image_h <= 0 || c.image_w <= 0 || c.patch_size <= 0 || c.embedding_dim <= 0 || c.num_heads <= 0 ||
        c.key_dim <= 0 || c.mlp_quantities <= 0 || c.repeat_times <= 0 || c.head_last_units <= 0 ||
        c.head_dense_layers <= 0 || c.head_block_repeats <= 0 || c.num_slots <= 0 || c.classes <= 1)
        return fail(VITDET_E_INVALID, "vitdet_create: every size in the configuration must be positive");
    if (c.key_dim > kMaxKeyDim) return fail(VITDET_E_INVALID, "encoder_key_dim %d > %d is not supported by this build", c.key_dim, kMaxKeyDim);
    if (c.embedding_dim > 2048) return fail(VITDET_E_INVALID, "embedding_dim %d > 2048 is not supported by this build", c.embedding_dim);
    if (c.mlp_quantities > 20 || c.head_dense_layers > 20) return fail(VITDET_E_INVALID, "pyramid depth out of range");

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(VITDET_E_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
    }
    int dev = 0;
    CU_TRY(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, dev));
    if (prop.major != 10) return fail(VITDET_E_NO_DEVICE, "device %d is sm_%d%d; the kernels are built for sm_100a only", dev, prop.major, prop.minor);

    vitdet_handle* h = new vitdet_handle();
    h->cfg = c;
    h->device = dev;
    h->num_sms = prop.multiProcessorCount;
    h->gh = (c.image_h + c.patch_size - 1) / c.patch_size;
    h->gw = (c.image_w + c.patch_size - 1) / c.patch_size;
    h->T = h->gh * h->gw;
    h->P = 3 * c.patch_size * c.patch_size;
    h->RP = round_up(3 * c.patch_size, 4);
    h->PK = c.patch_size * h->RP;
    h->D = c.embedding_dim; h->H = c.num_heads; h->d = c.key_dim; h->S = c.num_slots;
    h->hp = head_pitch(c.key_dim);
    h->act = c.use_mish ? ACT_MISH : ACT_GELU;
    h->opt = env_options();
    int rc = build_weight_table(h);
    if (rc) { delete h; return rc; }
    *out = h;
    return 0;
}

void vitdet_destroy(vitdet_handle* h) { delete h; }

int vitdet_tokens(const vitdet_handle* h) { return h ? h->T : 0; }
int vitdet_patch_dim(const vitdet_handle* h) { return h ? h->P : 0; }
int64_t vitdet_count_params(const vitdet_handle* h) {
    if (!h) return 0;
    int64_t n = 0;
    for (const WeightSlot& s : h->slots) n += s.count;
    return n;
}

int vitdet_num_weights(const vitdet_handle* h) { return h ? static_cast<int>(h->slots.size()) : 0; }

int vitdet_weight_info(const vitdet_handle* h, int index, char* name, int cap, int* ndim, int64_t shape[4]) {
    if (!h || index < 0 || index >= static_cast<int>(h->slots.size())) return fail(VITDET_E_INVALID, "weight_info: bad index %d", index);
    const WeightSlot& s = h->slots[index];
    if (name && cap > 0) { strncpy(name, s.name.c_str(), cap - 1); name[cap - 1] = 0; }
    if (ndim) *ndim = s.ndim;
    if (shape) for (int i = 0; i < 4; ++i) shape[i] = i < s.ndim ? s.shape[i] : 1;
    return 0;
}

int vitdet_set_weight(vitdet_handle* h, const char* name_in, const float* data, int ndim, const int64_t* shape) {
    if (!h || !name_in || !data) return fail(VITDET_E_INVALID, "set_weight: null argument");
    RC_TRY(check_device(h, "set_weight"));
    std::string name(name_in);
    if (name.size() > 2 && name.compare(name.size() - 2, 2, ":0") == 0) name.resize(name.size() - 2);
    auto it = h->slot_index.find(name);
    if (it == h->slot_index.end()) return fail(VITDET_E_NOT_FOUND, "set_weight: unknown weight '%s'", name.c_str());
    WeightSlot& s = h->slots[it->second];
    if (ndim != s.ndim) return fail(VITDET_E_SHAPE, "set_weight('%s'): rank %d, expected %d", name.c_str(), ndim, s.ndim);
    for (int i = 0; i < ndim; ++i)
        if (shape[i] != s.shape[i]) return fail(VITDET_E_SHAPE, "set_weight('%s'): dim %d is %lld, expected %lld", name.c_str(), i, (long long)shape[i], (long long)s.shape[i]);
    RC_TRY(h->stage.ensure(static_cast<size_t>(s.count) * 4));
    CU_TRY(cudaMemcpy(h->stage.p, data, static_cast<size_t>(s.count) * 4, cudaMemcpyHostToDevice));
    const float* src = h->stage.as<float>();
    switch (s.kind) {
        case WeightSlot::DENSE_KERNEL:
            pack_dense_kernel<<<blocks_for(s.count), 256>>>(src, s.K, s.N, s.gn, s.pn, s.row_off, s.gk, s.pk,
                                                            s.dense->w16.as<__nv_bfloat16>(), s.dense->ld16, s.dense->lo_off(),
                                                            s.dense->w32.as<float>(), s.dense->ld32);
            break;
        case WeightSlot::DENSE_BIAS:
            pack_vec_kernel<<<blocks_for(s.N), 256>>>(src, s.N, s.gn, s.pn, s.row_off, s.dense->bias.as<float>());
            break;
        case WeightSlot::VEC:
            if (s.vec_transpose)   // keep as f32 [N, K]
                pack_dense_kernel<<<blocks_for(s.count), 256>>>(src, s.K, s.N, s.N, s.N, 0, s.K, s.K, nullptr, 0, 0, s.vec_dst, s.K);
            else
                CU_TRY(cudaMemcpy(s.vec_dst, src, static_cast<size_t>(s.count) * 4, cudaMemcpyDeviceToDevice));
            break;
    }
    CU_TRY(cudaGetLastError());
    // no device-wide synchronise per tensor (245 of them for the default model): the staging buffer is reused in stream
    // order, and the first forward after a weight change synchronises once (weights_dirty)
    h->weights_dirty = true;
    s.master.assign(data, data + s.count);
    s.set = true;
    return 0;
}

int vitdet_get_weight(const vitdet_handle* h, const char* name_in, float* data, int64_t capacity) {
    if (!h || !name_in || !data) return fail(VITDET_E_INVALID, "get_weight: null argument");
    std::string name(name_in);
    if (name.size() > 2 && name.compare(name.size() - 2, 2, ":0") == 0) name.resize(name.size() - 2);
    auto it = h->slot_index.find(name);
    if (it == h->slot_index.end()) return fail(VITDET_E_NOT_FOUND, "get_weight: unknown weight '%s'", name.c_str());
    const WeightSlot& s = h->slots[it->second];
    if (!s.set) return fail(VITDET_E_UNSET, "get_weight('%s'): weight has not been set", name.c_str());
    if (capacity < s.count) return fail(VITDET_E_SHAPE, "get_weight('%s'): capacity %lld < %lld", name.c_str(), (long long)capacity, (long long)s.count);
    memcpy(data, s.master.data(), static_cast<size_t>(s.count) * 4);
    return 0;
}

int vitdet_profile_enable(vitdet_handle* h, uint32_t category_mask) {
    if (!h) return fail(VITDET_E_INVALID, "profile_enable: null handle");
    h->prof_mask = category_mask;
    return 0;
}

int vitdet_profile_num_categories(const vitdet_handle* h) {
    return h ? PC_MLP0 + h->cfg.mlp_quantities : 0;
}

const char* vitdet_profile_category_name(int category) { return prof_cat_name(category); }

int vitdet_profile_read(vitdet_handle* h, int category, double* total_ms, int64_t* launches, int reset) {
    if (!h || category < 0 || category >= 32) return fail(VITDET_E_INVALID, "profile_read: bad arguments");
    RC_TRY(prof_collect(h));
    if (total_ms) *total_ms = h->prof_ms[category];
    if (launches) *launches = h->prof_n[category];
    if (reset) { h->prof_ms[category] = 0; h->prof_n[category] = 0; }
    return 0;
}

int64_t vitdet_launch_count(vitdet_handle* h, int reset) {
    if (!h) return 0;
    const long long n = h->launches;
    if (reset) h->launches = 0;
    return n;
}

int vitdet_set_option(vitdet_handle* h, const char* key, int value) {
    if (!h || !key) return fail(VITDET_E_INVALID, "set_option: null argument");
    const std::string k(key);
    if (k == "fuse_ln") h->opt.fuse_ln = value != 0;
    else if (k == "fuse_tail") h->opt.fuse_tail = value != 0;
    else if (k == "gemm_pair") { if (value < 0 || value > 2) return fail(VITDET_E_INVALID, "set_option(gemm_pair): 0, 1 or 2"); h->opt.gemm_pair = value; }
    else if (k == "fp32_tc") h->opt.fp32_tc = value != 0;
    else return fail(VITDET_E_NOT_FOUND, "set_option: unknown option '%s'", key);
    h->plans.clear();
    return 0;
}

int vitdet_get_option(const vitdet_handle* h, const char* key, int* value) {
    if (!h || !key || !value) return fail(VITDET_E_INVALID, "get_option: null argument");
    const std::string k(key);
    if (k == "fuse_ln") *value = h->opt.fuse_ln;
    else if (k == "fuse_tail") *value = h->opt.fuse_tail;
    else if (k == "gemm_pair") *value = h->opt.gemm_pair;
    else if (k == "fp32_tc") *value = h->opt.fp32_tc;
    else return fail(VITDET_E_NOT_FOUND, "get_option: unknown option '%s'", key);
    return 0;
}

int vitdet_debug_taps(vitdet_handle* h, int enable) {
    if (!h) return fail(VITDET_E_INVALID, "debug_taps: null handle");
    h->taps_on = enable != 0;
    if (!h->taps_on) h->taps_B = 0;
    return 0;
}

int vitdet_debug_read(vitdet_handle* h, const char* name, float* out_host, int64_t capacity) {
    if (!h || !name || !out_host) return fail(VITDET_E_INVALID, "debug_read: null argument");
    if (!h->taps_on || h->taps_B <= 0) return fail(VITDET_E_UNSET, "debug_read: no forward has run with the taps enabled");
    const std::string k(name);
    CU_TRY(cudaDeviceSynchronize());
    const int B = h->taps_B;
    if (k == "head_last") {
        const int64_t R = static_cast<int64_t>(B) * h->S, U = h->tail_U;
        if (capacity < R * U) return fail(VITDET_E_SHAPE, "debug_read(head_last): capacity %lld < %lld", (long long)capacity, (long long)(R * U));
        const size_t es = h->head_last_f32 ? 4 : 2;
        std::vector<char> raw(static_cast<size_t>(R) * h->head_last_ld * es);
        CU_TRY(cudaMemcpy(raw.data(), h->head_last, raw.size(), cudaMemcpyDeviceToHost));
        for (int64_t r = 0; r < R; ++r)
            for (int64_t u = 0; u < U; ++u) {
                const size_t i = static_cast<size_t>(r) * h->head_last_ld + u;
                out_host[r * U + u] = h->head_last_f32 ? reinterpret_cast<const float*>(raw.data())[i]
                                                       : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(raw.data())[i]);
            }
        return 0;
    }
    int index = -1;
    if (k == "embedded_patches") index = 0;
    else if (k.compare(0, 6, "block_") == 0) index = atoi(k.c_str() + 6);
    if (index < 0 || index > h->cfg.repeat_times || (index == 0 && k != "embedded_patches"))
        return fail(VITDET_E_NOT_FOUND, "debug_read: unknown tap '%s'", name);
    const int D4 = round_up(h->D, 4);
    const int64_t rows = static_cast<int64_t>(B) * h->T;
    if (capacity < rows * h->D) return fail(VITDET_E_SHAPE, "debug_read('%s'): capacity %lld < %lld", name, (long long)capacity, (long long)(rows * h->D));
    CU_TRY(cudaMemcpy2D(out_host, static_cast<size_t>(h->D) * 4, h->taps.as<float>() + static_cast<size_t>(index) * rows * D4,
                        static_cast<size_t>(D4) * 4, static_cast<size_t>(h->D) * 4, static_cast<size_t>(rows), cudaMemcpyDeviceToHost));
    return 0;
}

int vitdet_set_chunk(vitdet_handle* h, int n) {
    if (!h || n <= 0) return fail(VITDET_E_INVALID, "set_chunk: bad argument");
    h->chunk = n;
    return 0;
}

size_t vitdet_workspace_bytes(const vitdet_handle* h, int B, int mode) {
    if (!h || B <= 0) return 0;
    return workspace_bytes(h, B, pick_form(mode, h->opt, h->d));
}

int vitdet_forward(vitdet_handle* h, const float* images_dev, int B, float* logits_dev, int mode, void* stream) {
    if (!logits_dev) return fail(VITDET_E_INVALID, "forward: logits_dev is null");
    return forward_impl(h, Input{Input::F32, images_dev}, B, mode, logits_dev, nullptr, nullptr, static_cast<cudaStream_t>(stream));
}

int vitdet_forward_u8(vitdet_handle* h, const uint8_t* images_dev, int B, float* logits_dev, int mode, const vitdet_decode_params* params,
                      const vitdet_detections* out, void* stream) {
    if (!logits_dev && !(params && out)) return fail(VITDET_E_INVALID, "forward_u8: neither logits_dev nor (params, out) given");
    if ((params == nullptr) != (out == nullptr)) return fail(VITDET_E_INVALID, "forward_u8: params and out go together");
    return forward_impl(h, Input{Input::U8, images_dev}, B, mode, logits_dev, params, out, static_cast<cudaStream_t>(stream));
}

int vitdet_forward_decode(vitdet_handle* h, const float* images_dev, int B, int mode, const vitdet_decode_params* params,
                          float* logits_dev, const vitdet_detections* out, void* stream) {
    if (!params || !out) return fail(VITDET_E_INVALID, "forward_decode: null params / out");
    return forward_impl(h, Input{Input::F32, images_dev}, B, mode, logits_dev, params, out, static_cast<cudaStream_t>(stream));
}

int vitdet_decode(const float* logits_dev, int R, const vitdet_decode_params* p, const vitdet_detections* out, void* stream) {
    if (!logits_dev || !p || !out || R < 0) return fail(VITDET_E_INVALID, "decode: bad arguments");
    if (R == 0) return 0;
    DecodeParams dp;
    DecodeOut o;
    decode_args(p, p->use_transform_predictions ? 1 : 0, out, nullptr, &dp, &o);
    CU_TRY(decode_launch(logits_dev, R, dp, o, static_cast<cudaStream_t>(stream)));
    return 0;
}

int vitdet_iou(const float* label_dev, const float* pred_dev, int64_t R, int width, float* iou_dev, void* stream) {
    if (!label_dev || !pred_dev || !iou_dev || R < 0 || width < 4) return fail(VITDET_E_INVALID, "iou: bad arguments");
    CU_TRY(iou_launch(label_dev, pred_dev, R, width, 1e-8f /* Constants.EPSILON, det.py:24 */, iou_dev, static_cast<cudaStream_t>(stream)));
    return 0;
}

int vitdet_iou_host(const float* label_host, const float* pred_host, int64_t R, int width, float* iou_host) {
    if (!label_host || !pred_host || !iou_host || R < 0 || width < 4) return fail(VITDET_E_INVALID, "iou_host: bad arguments");
    if (R == 0) return 0;
    const size_t nb = static_cast<size_t>(R) * width * 4;
    DevBuf a, b, o;
    RC_TRY(a.ensure(nb)); RC_TRY(b.ensure(nb)); RC_TRY(o.ensure(static_cast<size_t>(R) * 4));
    CU_TRY(cudaMemcpy(a.p, label_host, nb, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(b.p, pred_host, nb, cudaMemcpyHostToDevice));
    RC_TRY(vitdet_iou(a.as<float>(), b.as<float>(), R, width, o.as<float>(), nullptr));
    CU_TRY(cudaMemcpy(iou_host, o.p, static_cast<size_t>(R) * 4, cudaMemcpyDeviceToHost));
    return 0;
}

int vitdet_resize_with_pad_geometry(int h, int w, int th, int tw, int* rh, int* rw, int* ph, int* pw) {
    if (h <= 0 || w <= 0 || th <= 0 || tw <= 0 || !rh || !rw || !ph || !pw) return fail(VITDET_E_INVALID, "resize_with_pad_geometry: bad arguments");
    resize_with_pad_geometry(h, w, th, tw, rh, rw, ph, pw);
    return 0;
}

int vitdet_preprocess_image(const uint8_t* image_dev, int h, int w, float* out_dev, int th, int tw, void* stream) {
    if (!image_dev || !out_dev) return fail(VITDET_E_INVALID, "preprocess_image: null pointer");
    CU_TRY(preprocess_launch(image_dev, h, w, out_dev, th, tw, static_cast<cudaStream_t>(stream)));
    return 0;
}

int vitdet_preprocess_image_host(const uint8_t* image_host, int h, int w, float* out_host, int th, int tw) {
    if (!image_host || !out_host || h <= 0 || w <= 0 || th <= 0 || tw <= 0) return fail(VITDET_E_INVALID, "preprocess_image_host: bad arguments");
    DevBuf in, out;
    RC_TRY(in.ensure(static_cast<size_t>(h) * w * 3));
    RC_TRY(out.ensure(static_cast<size_t>(th) * tw * 3 * 4));
    CU_TRY(cudaMemcpy(in.p, image_host, static_cast<size_t>(h) * w * 3, cudaMemcpyHostToDevice));
    RC_TRY(vitdet_preprocess_image(in.as<uint8_t>(), h, w, out.as<float>(), th, tw, nullptr));
    CU_TRY(cudaMemcpy(out_host, out.p, static_cast<size_t>(th) * tw * 3 * 4, cudaMemcpyDeviceToHost));
    return 0;
}

int vitdet_decode_host(const float* logits_host, int R, const vitdet_decode_params* p, const vitdet_detections* out_host) {
    if (!logits_host || !p || !out_host || R < 0) return fail(VITDET_E_INVALID, "decode_host: bad arguments");
    if (R == 0) return 0;
    // the logits go into the record block's logits rows; the block comes back in one copy
    const RecordBlock rb(static_cast<size_t>(R), out_host->packed != nullptr, false);
    DevBuf buf;
    RC_TRY(buf.ensure(rb.bytes));
    char* b = buf.as<char>();
    CU_TRY(cudaMemcpy(b, logits_host, rb.R * 24, cudaMemcpyHostToDevice));
    const vitdet_detections d = rb.detections(b);
    RC_TRY(vitdet_decode(reinterpret_cast<const float*>(b), R, p, &d, nullptr));
    CU_TRY(cudaDeviceSynchronize());
    std::vector<char> host(rb.bytes);
    CU_TRY(cudaMemcpy(host.data(), b, rb.bytes, cudaMemcpyDeviceToHost));
    return rb.copy_out(host.data(), nullptr, out_host, nullptr);
}

}  // extern "C"

static bool page_locked(const void* p) {
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, p) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    return pinned;
}

// Creates the handle's staging threads on first use
static void ensure_stage_pool(vitdet_handle* h) {
    if (h->stage_pool) return;
    // staging threads (+ the calling thread): a share of the host's cores, divided among the ranks of this node
    // (LOCAL_WORLD_SIZE under torchrun); VITDET_STAGE_THREADS overrides the total
    const int hw = static_cast<int>(std::thread::hardware_concurrency());
    int local_world = 1;
    if (const char* e = getenv("LOCAL_WORLD_SIZE")) local_world = atoi(e) > 0 ? atoi(e) : 1;
    int workers = (hw > 0 ? hw / (2 * local_world) : 6) - 1;
    if (workers > 11) workers = 11;
    if (workers < 1) workers = 1;
    if (const char* e = getenv("VITDET_STAGE_THREADS")) workers = atoi(e) - 1;
    if (hw > 0 && workers > hw - 1) workers = hw - 1;
    if (workers < 0) workers = 0;
    h->stage_pool = new StagePool(workers);
}

// The images of one host submission: image i, src[i][0, offs[i + 1] - offs[i]), goes to byte offs[i] of the slot's device
// input.  F32 / U8: one contiguous array of the model's size.  Letterbox: separate images of any size, whose geometry
// `table` holds; its pixel pointers are filled in here.  `jpeg`: the sources are JPEG files, decoded on the device into
// the slot's pixel arena before the forward.
struct HostImages {
    Input::Kind kind;
    std::vector<const char*> src;
    std::vector<size_t> offs{0};
    std::vector<LetterboxImage> table;
    const JpegBatch* jpeg = nullptr;
    void add(const void* p, size_t bytes) {
        src.push_back(static_cast<const char*>(p));
        offs.push_back(offs.back() + bytes);
    }
};

// Enqueues the decode of a planned batch of JPEG files on st: the descriptor block, through `desc_pin` (page-locked, at
// least jb.desc.size() bytes), to the head of the scratch `work`, then, once files_ready (may be null) has fired, the
// kernels from the concatenated files at files_dev into out.  Its repair counters become the handle's jpeg_stats.
static int jpeg_enqueue(vitdet_handle* h, const JpegBatch& jb, char* desc_pin, const char* files_dev, DevBuf& work, uint8_t* out,
                        cudaEvent_t files_ready, cudaStream_t st) {
    memcpy(desc_pin, jb.desc.data(), jb.desc.size());
    RC_TRY(work.ensure(jb.work_bytes));
    CU_TRY(cudaMemcpyAsync(work.p, desc_pin, jb.desc.size(), cudaMemcpyHostToDevice, st));
    if (files_ready) CU_TRY(cudaStreamWaitEvent(st, files_ready, 0));
    h->launches += kJpegLaunches;
    CU_TRY(jpeg_decode_launch(jb, files_dev, work.p, out, st));
    h->jpeg_stats = reinterpret_cast<const long long*>(work.as<char>() + jb.o_stats);
    return 0;
}

static int submit_host_impl(vitdet_handle* h, HostImages& in, int B, int mode, const vitdet_decode_params* params,
                            int want_packed, float* boxes_host, void* stream, int* ticket) {
    HostSlot& sl = h->host_slots[h->next_slot];
    if (sl.busy) return fail(VITDET_E_INVALID, "submit_host: %d submissions are in flight; collect one first", vitdet_handle::kHostSlots);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool separate = in.kind == Input::Letterbox;
    const size_t in_bytes = in.offs[B];
    sl.rec = RecordBlock(static_cast<size_t>(B) * h->S, want_packed != 0, boxes_host != nullptr);
    sl.boxes_host = boxes_host;
    // a page-locked source is read directly, otherwise the whole submission is staged
    bool pinned = page_locked(in.src[0]);
    for (int i = 1; separate && pinned && i < B; ++i) pinned = page_locked(in.src[i]);
    if (!pinned) RC_TRY(sl.pin_in.ensure(in_bytes));
    RC_TRY(sl.pin_out.ensure(sl.rec.bytes));
    RC_TRY(sl.dev_in.ensure(in_bytes));
    RC_TRY(sl.dev_out.ensure(sl.rec.bytes));
    if (!sl.done) CU_TRY(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
    // Images are copied in sub-chunks of kGran images on a dedicated copy stream, one event per sub-chunk; the encoder
    // runs chunks of 4, 12 and then `chunk` images, each waiting only for its own images: at ~12 images/ms of PCIe
    // against ~4 images/ms of compute every copy but the first 4 images' (0.33 ms) hides behind the previous chunk's
    // compute (measured best of seven schedules, B = 64) — and behind the PREVIOUS submission's compute when the caller
    // keeps two submissions in flight.  A page-locked caller buffer is read directly; a pageable one is staged through
    // the slot's pinned buffer by the staging threads, sub-chunk by sub-chunk, overlapped with the H2D copies.
    // VITDET_E2E_LEAD="g,a,b" overrides the copy granularity and the two lead chunk sizes (tuning experiments).
    int kGran = 4, lead0 = 4, lead1 = 12;
    // uint8 pixels, a quarter of the bytes per image: the same 0.3 ms lead-in with 16 images
    if (in.kind != Input::F32) { kGran = 16; lead0 = 16; lead1 = 0; }
    // with the previous submission still computing, this one's copy has a whole forward pass to finish: no small lead chunks
    if (h->host_slots[(h->next_slot + vitdet_handle::kHostSlots - 1) % vitdet_handle::kHostSlots].busy) { lead0 = 0; lead1 = 0; }
    // nor in the split fp32 form: its three-pass GEMMs lose more on 4- and 12-image chunks than the early start gains
    // (B = 64 on a B200 at 1000 W: 48.5 ms with lead chunks 4, 12 against 45.1 ms without)
    if (pick_form(mode, h->opt, h->d) == Form::Split) { lead0 = 0; lead1 = 0; }
    if (const char* e = getenv("VITDET_E2E_LEAD")) sscanf(e, "%d,%d,%d", &kGran, &lead0, &lead1);
    if (kGran < 1) kGran = 8;
    const int n_sub = (B + kGran - 1) / kGran;
    if (!h->copy_stream) CU_TRY(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    while (static_cast<int>(sl.copy_events.size()) < n_sub) {
        cudaEvent_t e;
        CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        sl.copy_events.push_back(e);
    }
    if (!pinned) ensure_stage_pool(h);
    char* dev_in = sl.dev_in.as<char>();
    for (int i = 0; i < n_sub; ++i) {
        const int i0 = i * kGran, i1 = std::min(B, i0 + kGran);
        const size_t off = in.offs[i0], bytes = in.offs[i1] - off;
        if (!pinned) {
            h->stage_pool->copy(sl.pin_in.as<char>() + off, in.src.data() + i0, in.offs.data() + i0, i1 - i0);
            CU_TRY(cudaMemcpyAsync(dev_in + off, sl.pin_in.as<char>() + off, bytes, cudaMemcpyHostToDevice, h->copy_stream));
        } else if (!separate) {
            CU_TRY(cudaMemcpyAsync(dev_in + off, in.src[i0], bytes, cudaMemcpyHostToDevice, h->copy_stream));
        } else {
            for (int k = i0; k < i1; ++k)
                CU_TRY(cudaMemcpyAsync(dev_in + in.offs[k], in.src[k], in.offs[k + 1] - in.offs[k], cudaMemcpyHostToDevice, h->copy_stream));
        }
        CU_TRY(cudaEventRecord(sl.copy_events[i], h->copy_stream));
    }
    ForwardOpts opts;
    Input input{in.kind, dev_in};
    const char* pixels_dev = dev_in;
    const size_t* pixel_offs = in.offs.data();
    if (in.jpeg) {
        // decode after the last file's copy, on the compute stream, into the slot's arena; the forward then waits for nothing
        const JpegBatch& jb = *in.jpeg;
        RC_TRY(sl.pin_jpeg.ensure(jb.desc.size()));
        RC_TRY(sl.jpeg_rgb.ensure(jb.rgb_bytes));
        RC_TRY(jpeg_enqueue(h, jb, sl.pin_jpeg.as<char>(), dev_in, sl.jpeg_work, sl.jpeg_rgb.as<uint8_t>(), sl.copy_events[n_sub - 1], st));
        pixels_dev = sl.jpeg_rgb.as<char>();
        pixel_offs = jb.rgb_off.data();
    } else {
        if (lead0 > 0 && B > lead0 + lead1) { opts.lead_chunks[0] = lead0; opts.lead_chunks[1] = lead1; }
        else if (lead0 > 0 && B > lead0) opts.lead_chunks[0] = lead0;
        opts.ready = sl.copy_events.data();
        opts.ready_gran = kGran;
    }
    char* dbase = sl.dev_out.as<char>();
    if (separate) {
        // the slot's own table: the pinned copy is not touched again before this submission is collected
        const size_t table_bytes = static_cast<size_t>(B) * sizeof(LetterboxImage);
        RC_TRY(sl.pin_table.ensure(table_bytes));
        RC_TRY(sl.dev_table.ensure(table_bytes));
        LetterboxImage* table = sl.pin_table.as<LetterboxImage>();
        for (int k = 0; k < B; ++k) {
            table[k] = in.table[k];
            table[k].pixels = reinterpret_cast<const uint8_t*>(pixels_dev + pixel_offs[k]);
        }
        CU_TRY(cudaMemcpyAsync(sl.dev_table.p, table, table_bytes, cudaMemcpyHostToDevice, st));
        input.p = sl.dev_table.p;
        input.boxes_original = sl.rec.boxes_original(dbase);
    }
    const vitdet_detections d = sl.rec.detections(dbase);
    RC_TRY(forward_impl(h, input, B, mode, reinterpret_cast<float*>(dbase), params, &d, st, opts));
    CU_TRY(cudaMemcpyAsync(sl.pin_out.p, dbase, sl.rec.bytes, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaEventRecord(sl.done, st));
    sl.busy = true;
    *ticket = h->next_slot;
    h->next_slot = (h->next_slot + 1) % vitdet_handle::kHostSlots;
    return 0;
}

static int collect_impl(vitdet_handle* h, int ticket, float* logits_host, const vitdet_detections* out_host) {
    if (!h || ticket < 0 || ticket >= vitdet_handle::kHostSlots) return fail(VITDET_E_INVALID, "collect: bad ticket %d", ticket);
    HostSlot& sl = h->host_slots[ticket];
    if (!sl.busy) return fail(VITDET_E_INVALID, "collect: ticket %d is not in flight", ticket);
    sl.busy = false;
    CU_TRY(cudaEventSynchronize(sl.done));
    return sl.rec.copy_out(sl.pin_out.as<char>(), logits_host, out_host, sl.boxes_host);
}

// A contiguous host array of B images of the model's size
static int submit_dense_impl(vitdet_handle* h, const void* images_host, Input::Kind kind, int B, int mode, const vitdet_decode_params* params,
                             int want_packed, void* stream, int* ticket) {
    if (!h || !images_host || B <= 0 || !params || !ticket) return fail(VITDET_E_INVALID, "submit_host: bad arguments");
    const size_t img_bytes = static_cast<size_t>(h->cfg.image_h) * h->cfg.image_w * 3 * (kind == Input::U8 ? 1 : 4);
    HostImages in{kind};
    for (int i = 0; i < B; ++i) in.add(static_cast<const char*>(images_host) + i * img_bytes, img_bytes);
    return submit_host_impl(h, in, B, mode, params, want_packed, nullptr, stream, ticket);
}

static int predict_host_impl(vitdet_handle* h, const void* images_host, Input::Kind kind, int B, int mode, const vitdet_decode_params* params,
                             float* logits_host, const vitdet_detections* out_host, void* stream) {
    int ticket = -1;
    RC_TRY(submit_dense_impl(h, images_host, kind, B, mode, params, (out_host && out_host->packed) ? 1 : 0, stream, &ticket));
    return collect_impl(h, ticket, logits_host, out_host);
}

// Checks a list of B images of any size to be letterboxed to the model's input size and fills their table (pixel
// pointers as given); the message of a rejected list names the first bad image.  boxes: boxes_original is requested,
// which needs the decode at the model's size.
static int letterbox_table(const vitdet_handle* h, const char* fn, const vitdet_image* images, int B, const vitdet_decode_params* params,
                           bool boxes, std::vector<LetterboxImage>* table) {
    if (!h || !images || B <= 0) return fail(VITDET_E_INVALID, "%s: %s", fn, !h ? "null handle" : (!images ? "images is null" : "B must be positive"));
    const int th = h->cfg.image_h, tw = h->cfg.image_w;
    if (boxes && (!params || params->image_h != static_cast<float>(th) || params->image_w != static_cast<float>(tw)))
        return fail(VITDET_E_INVALID, "%s: boxes_original needs the decode at the model's input size %d x %d (params image_h / image_w)", fn, th, tw);
    table->resize(B);
    for (int i = 0; i < B; ++i) {
        const vitdet_image& im = images[i];
        if (!im.pixels) return fail(VITDET_E_INVALID, "%s: image %d: null pixel pointer", fn, i);
        if (im.height <= 0 || im.width <= 0) return fail(VITDET_E_INVALID, "%s: image %d: size %d x %d is not positive", fn, i, im.height, im.width);
        if (!letterbox_image(im.pixels, im.height, im.width, th, tw, &(*table)[i]))
            return fail(VITDET_E_INVALID, "%s: image %d: a %d x %d image letterboxed to %d x %d resizes to %d x %d pixels", fn, i, im.height,
                        im.width, th, tw, (*table)[i].rh, (*table)[i].rw);
    }
    return 0;
}

extern "C" {

int vitdet_predict_host(vitdet_handle* h, const float* images_host, int B, int mode, const vitdet_decode_params* params,
                        float* logits_host, const vitdet_detections* out_host, void* stream) {
    return predict_host_impl(h, images_host, Input::F32, B, mode, params, logits_host, out_host, stream);
}

int vitdet_predict_host_u8(vitdet_handle* h, const uint8_t* images_host, int B, int mode, const vitdet_decode_params* params,
                           float* logits_host, const vitdet_detections* out_host, void* stream) {
    return predict_host_impl(h, images_host, Input::U8, B, mode, params, logits_host, out_host, stream);
}

int vitdet_submit_host(vitdet_handle* h, const void* images_host, int images_are_uint8, int B, int mode, const vitdet_decode_params* params,
                       int want_packed, void* stream, int* ticket) {
    return submit_dense_impl(h, images_host, images_are_uint8 ? Input::U8 : Input::F32, B, mode, params, want_packed, stream, ticket);
}

int vitdet_collect(vitdet_handle* h, int ticket, float* logits_host, const vitdet_detections* out_host) {
    return collect_impl(h, ticket, logits_host, out_host);
}

int vitdet_forward_images(vitdet_handle* h, const vitdet_image* images, int B, int mode, const vitdet_decode_params* params,
                          float* logits_dev, const vitdet_detections* out, float* boxes_original_dev, void* stream) {
    if (!logits_dev && !(params && out)) return fail(VITDET_E_INVALID, "forward_images: neither logits_dev nor (params, out) given");
    if ((params == nullptr) != (out == nullptr)) return fail(VITDET_E_INVALID, "forward_images: params and out go together");
    std::vector<LetterboxImage> table;
    RC_TRY(letterbox_table(h, "forward_images", images, B, params, boxes_original_dev != nullptr, &table));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // a pageable source: the copy has taken the table by the time it returns, and it reaches the device in stream order
    const size_t table_bytes = table.size() * sizeof(LetterboxImage);
    RC_TRY(h->images_table.ensure(table_bytes));
    CU_TRY(cudaMemcpyAsync(h->images_table.p, table.data(), table_bytes, cudaMemcpyHostToDevice, st));
    return forward_impl(h, Input{Input::Letterbox, h->images_table.p, boxes_original_dev}, B, mode, logits_dev, params, out, st);
}

int vitdet_submit_images_host(vitdet_handle* h, const vitdet_image* images, int B, int mode, const vitdet_decode_params* params,
                              int want_packed, float* boxes_original_host, void* stream, int* ticket) {
    if (!params || !ticket) return fail(VITDET_E_INVALID, "submit_images_host: params and ticket must not be null");
    HostImages in{Input::Letterbox};
    RC_TRY(letterbox_table(h, "submit_images_host", images, B, params, boxes_original_host != nullptr, &in.table));
    for (int i = 0; i < B; ++i) in.add(images[i].pixels, static_cast<size_t>(images[i].height) * images[i].width * 3);
    return submit_host_impl(h, in, B, mode, params, want_packed, boxes_original_host, stream, ticket);
}

// A caller's list of JPEG files -> the batch plan (every file parsed on the host; a rejected file fails the list, naming it).
// ratios: null (all 1) or per file 1, 2, 4, 8 or 0 (auto for the model's input size).
static int jpeg_files_plan(const vitdet_handle* h, const char* fn, const vitdet_jpeg* files, const int32_t* ratios, int B,
                           const int64_t* out_offsets, JpegBatch* jb) {
    if (!files || B <= 0) return fail(VITDET_E_INVALID, "%s: %s", fn, !files ? "files is null" : "B must be positive");
    std::vector<const uint8_t*> data(B);
    std::vector<int64_t> bytes(B);
    for (int i = 0; i < B; ++i) { data[i] = files[i].data; bytes[i] = files[i].bytes; }
    return jpeg_plan(fn, data.data(), bytes.data(), B, ratios, h->cfg.image_h, h->cfg.image_w, out_offsets, jb);
}

int vitdet_jpeg_info(const uint8_t* data, int64_t bytes, int* height, int* width, int* components) {
    char why[256];
    if (jpeg_info(data, bytes, height, width, components, why, sizeof(why))) return fail(VITDET_E_INVALID, "jpeg_info: %s", why);
    return 0;
}

int vitdet_jpeg_auto_ratio(int height, int width, int target_h, int target_w) {
    if (height <= 0 || width <= 0 || target_h <= 0 || target_w <= 0)
        return fail(VITDET_E_INVALID, "jpeg_auto_ratio: sizes must be positive, got %d x %d to %d x %d", height, width, target_h, target_w);
    return jpeg_auto_ratio(height, width, target_h, target_w);
}

static int decode_jpeg_impl(vitdet_handle* h, const char* fn, const vitdet_jpeg* files, const int32_t* ratios, int B, uint8_t* out_dev,
                            const int64_t* out_offsets, void* stream) {
    if (!h || !out_dev || !out_offsets) return fail(VITDET_E_INVALID, "%s: null handle, out_dev or out_offsets", fn);
    RC_TRY(check_device(h, fn));
    JpegBatch jb;
    RC_TRY(jpeg_files_plan(h, fn, files, ratios, B, out_offsets, &jb));
    for (int i = 0; i < B; ++i)
        if (out_offsets[i] < 0) return fail(VITDET_E_INVALID, "%s: image %d: negative output offset", fn, i);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // the previous decode has read the staging and the device buffers before they are reused, on any stream
    if (h->jpeg_done) CU_TRY(cudaEventSynchronize(h->jpeg_done));
    else CU_TRY(cudaEventCreateWithFlags(&h->jpeg_done, cudaEventDisableTiming));
    // descriptors and files in one pinned block, the files concatenated by the staging threads: the caller's bytes are
    // read before this returns
    const size_t files_bytes = jb.file_off[B];
    RC_TRY(h->jpeg_pin.ensure(jb.desc.size() + files_bytes));
    char* files_pin = h->jpeg_pin.as<char>() + jb.desc.size();
    std::vector<const char*> src(B);
    for (int i = 0; i < B; ++i) src[i] = reinterpret_cast<const char*>(files[i].data);
    ensure_stage_pool(h);
    h->stage_pool->copy(files_pin, src.data(), jb.file_off.data(), B);
    RC_TRY(h->jpeg_files.ensure(files_bytes));
    CU_TRY(cudaMemcpyAsync(h->jpeg_files.p, files_pin, files_bytes, cudaMemcpyHostToDevice, st));
    RC_TRY(jpeg_enqueue(h, jb, h->jpeg_pin.as<char>(), h->jpeg_files.as<char>(), h->jpeg_work, out_dev, nullptr, st));
    CU_TRY(cudaEventRecord(h->jpeg_done, st));
    return 0;
}

int vitdet_decode_jpeg(vitdet_handle* h, const vitdet_jpeg* files, int B, uint8_t* out_dev, const int64_t* out_offsets, void* stream) {
    return decode_jpeg_impl(h, "decode_jpeg", files, nullptr, B, out_dev, out_offsets, stream);
}

int vitdet_decode_jpeg_scaled(vitdet_handle* h, const vitdet_jpeg* files, const int32_t* ratios, int B, uint8_t* out_dev,
                              const int64_t* out_offsets, void* stream) {
    if (!ratios) return fail(VITDET_E_INVALID, "decode_jpeg_scaled: ratios is null");
    return decode_jpeg_impl(h, "decode_jpeg_scaled", files, ratios, B, out_dev, out_offsets, stream);
}

static int submit_jpeg_impl(vitdet_handle* h, const char* fn, const vitdet_jpeg* files, const int32_t* ratios, int B, int mode,
                            const vitdet_decode_params* params, int want_packed, float* boxes_original_host, void* stream, int* ticket) {
    if (!h || !params || !ticket) return fail(VITDET_E_INVALID, "%s: handle, params and ticket must not be null", fn);
    JpegBatch jb;
    RC_TRY(jpeg_files_plan(h, fn, files, ratios, B, nullptr, &jb));
    // the decoded images' sizes; each file's bytes are its image's host source, as the pixels are for separate images
    std::vector<vitdet_image> images(B);
    for (int i = 0; i < B; ++i) images[i] = vitdet_image{files[i].data, jb.height[i], jb.width[i]};
    HostImages in{Input::Letterbox};
    RC_TRY(letterbox_table(h, fn, images.data(), B, params, boxes_original_host != nullptr, &in.table));
    for (int i = 0; i < B; ++i) {
        in.add(files[i].data, static_cast<size_t>(files[i].bytes));
        // boxes_original in the file's pixels: the decoded image's box times file size / decoded size (1 at ratio 1)
        LetterboxImage& g = in.table[i];
        g.file_h = jb.file_height[i];
        g.file_w = jb.file_width[i];
        g.file_hscale = static_cast<float>(g.file_h) / static_cast<float>(g.h);
        g.file_wscale = static_cast<float>(g.file_w) / static_cast<float>(g.w);
    }
    in.jpeg = &jb;
    return submit_host_impl(h, in, B, mode, params, want_packed, boxes_original_host, stream, ticket);
}

int vitdet_submit_jpeg_host(vitdet_handle* h, const vitdet_jpeg* files, int B, int mode, const vitdet_decode_params* params,
                            int want_packed, float* boxes_original_host, void* stream, int* ticket) {
    return submit_jpeg_impl(h, "submit_jpeg_host", files, nullptr, B, mode, params, want_packed, boxes_original_host, stream, ticket);
}

int vitdet_submit_jpeg_host_scaled(vitdet_handle* h, const vitdet_jpeg* files, const int32_t* ratios, int B, int mode,
                                   const vitdet_decode_params* params, int want_packed, float* boxes_original_host, void* stream,
                                   int* ticket) {
    if (!ratios) return fail(VITDET_E_INVALID, "submit_jpeg_host_scaled: ratios is null");
    return submit_jpeg_impl(h, "submit_jpeg_host_scaled", files, ratios, B, mode, params, want_packed, boxes_original_host, stream, ticket);
}

int vitdet_jpeg_stats(vitdet_handle* h, int64_t* stats) {
    if (!h || !stats) return fail(VITDET_E_INVALID, "jpeg_stats: null argument");
    if (!h->jpeg_stats) return fail(VITDET_E_INVALID, "jpeg_stats: no JPEG decode has run on this handle");
    long long v[3];
    CU_TRY(cudaMemcpy(v, h->jpeg_stats, sizeof(v), cudaMemcpyDeviceToHost));
    for (int i = 0; i < 3; ++i) stats[i] = v[i];
    return 0;
}

// ------------------------------------------------------------------------------------------------
// operator-level entry points
// ------------------------------------------------------------------------------------------------
int vitdet_op_dense(const float* A, const float* kernel, const float* bias, const float* resid, float* out, int M, int K,
                    int N, int act, int mode, void* stream) {
    if (!A || !kernel || !out || M <= 0 || K <= 0 || N <= 0) return fail(VITDET_E_INVALID, "op_dense: bad arguments");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int dev = 0, sms = 148;
    CU_TRY(cudaGetDevice(&dev));
    CU_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    DenseW w;
    RC_TRY(w.alloc(N, K));
    pack_dense_kernel<<<blocks_for(static_cast<long long>(K) * N), 256, 0, st>>>(kernel, K, N, N, N, 0, K, K, w.w16.as<__nv_bfloat16>(), w.ld16, w.lo_off(),
                                                                               w.w32.as<float>(), w.ld32);
    if (bias) CU_TRY(cudaMemcpyAsync(w.bias.p, bias, static_cast<size_t>(N) * 4, cudaMemcpyDeviceToDevice, st));
    const int N4 = round_up(N, 4);
    DevBuf a_buf, o_buf, r_buf;
    RC_TRY(o_buf.ensure(static_cast<size_t>(M) * N4 * 4));
    const float* rp = nullptr;
    if (resid) {
        RC_TRY(r_buf.ensure(static_cast<size_t>(M) * N4 * 4));
        pad_rows_f32_kernel<<<blocks_for(static_cast<long long>(M) * N4), 256, 0, st>>>(resid, M, N, N, r_buf.as<float>(), N4);
        rp = r_buf.as<float>();
    }
    // A in the form's operand layout: bf16 rows, (hi, lo) planes, or f32 rows
    const Form f = pick_form(mode, env_options(), 0 /*no attention*/);
    Operand a;
    if (f == Form::Ieee) {
        a = Operand{nullptr, nullptr, round_up(K, 4)};
        RC_TRY(a_buf.ensure(static_cast<size_t>(M) * a.ld * 4));
        a.p = a_buf.p;
        pad_rows_f32_kernel<<<blocks_for(static_cast<long long>(M) * a.ld), 256, 0, st>>>(A, M, K, K, a_buf.as<float>(), a.ld);
    } else {
        a = Operand{nullptr, nullptr, round_up(K, 8)};
        const size_t plane = static_cast<size_t>(M) * a.ld;
        RC_TRY(a_buf.ensure(plane * 2 * (f == Form::Split ? 2 : 1)));
        a.p = a_buf.p;
        if (f == Form::Bf16) {
            f32_to_bf16_kernel<<<blocks_for(static_cast<long long>(plane)), 256, 0, st>>>(A, M, K, K, a_buf.as<__nv_bfloat16>(), a.ld);
        } else {
            a.lo = a_buf.as<__nv_bfloat16>() + plane;
            split_rows_kernel<<<blocks_for(static_cast<long long>(M) * (a.ld >> 3)), 256, 0, st>>>(A, M, K, K, a_buf.as<__nv_bfloat16>(),
                                                                                                 static_cast<__nv_bfloat16*>(a.lo), a.ld);
        }
    }
    DenseCall c{a, &w, M};
    c.resid = rp; c.ldr = N4;
    c.out = Operand{o_buf.p, nullptr, N4}; c.out_f32 = 1; c.act = act;
    RC_TRY(dense_once(c, f, sms, env_options().gemm_pair, st));
    unpad_rows_f32_kernel<<<blocks_for(static_cast<long long>(M) * N), 256, 0, st>>>(o_buf.as<float>(), M, N, N4, out);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(st));
    return 0;
}

int vitdet_op_layernorm(const float* x, const float* gamma, const float* beta, float* y, int M, int D, float eps, void* stream) {
    if (!x || !gamma || !beta || !y || M <= 0 || D <= 0) return fail(VITDET_E_INVALID, "op_layernorm: bad arguments");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int D4 = round_up(D, 4);
    if (D4 == D) {
        CU_TRY(layernorm_launch(x, D, gamma, beta, M, D, eps, y, D, 1, st));
        return 0;
    }
    DevBuf xb, yb;
    RC_TRY(xb.ensure(static_cast<size_t>(M) * D4 * 4));
    RC_TRY(yb.ensure(static_cast<size_t>(M) * D4 * 4));
    pad_rows_f32_kernel<<<blocks_for(static_cast<long long>(M) * D4), 256, 0, st>>>(x, M, D, D, xb.as<float>(), D4);
    CU_TRY(layernorm_launch(xb.as<float>(), D4, gamma, beta, M, D, eps, yb.p, D4, 1, st));
    unpad_rows_f32_kernel<<<blocks_for(static_cast<long long>(M) * D), 256, 0, st>>>(yb.as<float>(), M, D, D4, y);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(st));
    return 0;
}

int vitdet_op_attention(const float* q, const float* k, const float* v, float* out, int B, int T, int H, int d, int mode,
                        void* stream) {
    if (!q || !k || !v || !out || B <= 0 || T <= 0 || H <= 0 || d <= 0 || d > kMaxKeyDim)
        return fail(VITDET_E_INVALID, "op_attention: bad arguments (key_dim must be <= %d)", kMaxKeyDim);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int hp = head_pitch(d);
    const long long rows = static_cast<long long>(B) * T;
    const Form f = pick_form(mode, env_options(), d);
    const int ld = 3 * H * hp;
    // q | k | v as bf16 or f32 rows; the Split form's (hi, lo) planes of them in `planes`, of the context rows in `ctx`
    DevBuf qkv, ctx, planes;
    const size_t es = f == Form::Bf16 ? 2 : 4;
    RC_TRY(qkv.ensure(static_cast<size_t>(rows) * ld * es));
    RC_TRY(ctx.ensure(static_cast<size_t>(rows) * H * hp * es));
    if (f == Form::Bf16) pack_qkv_kernel<__nv_bfloat16><<<blocks_for(rows * ld), 256, 0, st>>>(q, k, v, rows, H, d, hp, qkv.as<__nv_bfloat16>());
    else pack_qkv_kernel<float><<<blocks_for(rows * ld), 256, 0, st>>>(q, k, v, rows, H, d, hp, qkv.as<float>());
    Operand a{qkv.p, nullptr, ld}, o{ctx.p, nullptr, H * hp};
    if (f == Form::Split) {
        RC_TRY(planes.ensure(static_cast<size_t>(rows) * ld * 2 * 2));
        a = Operand{planes.p, planes.as<__nv_bfloat16>() + static_cast<size_t>(rows) * ld, ld};
        o.lo = ctx.as<__nv_bfloat16>() + static_cast<size_t>(rows) * H * hp;
        split_rows_kernel<<<blocks_for(rows * (ld >> 3)), 256, 0, st>>>(qkv.as<float>(), rows, ld, ld, planes.as<__nv_bfloat16>(),
                                                                       static_cast<__nv_bfloat16*>(a.lo), ld);
    }
    const AttnDesc ad = attn_desc(a, o, B, T, H, d, hp);
    AttnTcPlan plan;
    if (f != Form::Ieee) RC_TRY(attn_plan(&plan, ad, a.lo));
    CU_TRY(attn_launch(f, ad, &plan, o.lo, st));
    if (f == Form::Bf16) unpack_ctx_kernel<__nv_bfloat16><<<blocks_for(rows * H * d), 256, 0, st>>>(ctx.as<__nv_bfloat16>(), rows, H, d, hp, out);
    else if (f == Form::Split)
        unpack_ctx_planes_kernel<<<blocks_for(rows * H * d), 256, 0, st>>>(ctx.as<__nv_bfloat16>(), static_cast<const __nv_bfloat16*>(o.lo), rows, H, d, hp, out);
    else unpack_ctx_kernel<float><<<blocks_for(rows * H * d), 256, 0, st>>>(ctx.as<float>(), rows, H, d, hp, out);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(st));
    return 0;
}

__global__ void bf16_rows_to_f32_kernel(const __nv_bfloat16* __restrict__ src, int rows, int cols, int lds, float* __restrict__ dst) {
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= static_cast<long long>(rows) * cols) return;
    const int r = static_cast<int>(idx / cols), c = static_cast<int>(idx - static_cast<long long>(r) * cols);
    dst[idx] = __bfloat162float(src[static_cast<size_t>(r) * lds + c]);
}

int vitdet_op_dense_ex(const float* A, const float* kernel, const float* bias, const float* resid, float* out, int M, int K,
                       int N, int act, const vitdet_dense_ex* ex, void* stream) {
    if (!A || !kernel || !out || !ex || M <= 0 || K <= 0 || N <= 0) return fail(VITDET_E_INVALID, "op_dense_ex: bad arguments");
    if (ex->store_bf16 && (resid || ex->pos || ex->ln_out)) return fail(VITDET_E_INVALID, "op_dense_ex: store_bf16 excludes resid / pos / ln_out");
    if (ex->ln_out && (N > 32 || !ex->ln_gamma || !ex->ln_beta)) return fail(VITDET_E_INVALID, "op_dense_ex: the fused LayerNorm needs N <= 32, gamma and beta");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int dev = 0, sms = 148;
    CU_TRY(cudaGetDevice(&dev));
    CU_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    DenseW w;
    RC_TRY(w.alloc(N, K));
    pack_dense_kernel<<<blocks_for(static_cast<long long>(K) * N), 256, 0, st>>>(kernel, K, N, N, N, 0, K, K, w.w16.as<__nv_bfloat16>(), w.ld16, w.lo_off(),
                                                                               w.w32.as<float>(), w.ld32);
    if (bias) CU_TRY(cudaMemcpyAsync(w.bias.p, bias, static_cast<size_t>(N) * 4, cudaMemcpyDeviceToDevice, st));
    const int N4 = round_up(N, 4), N8 = round_up(N, 8), K8 = round_up(K, 8);
    DevBuf a_buf, o_buf, r_buf, ln_buf;
    RC_TRY(a_buf.ensure(static_cast<size_t>(M) * K8 * 2));
    f32_to_bf16_kernel<<<blocks_for(static_cast<long long>(M) * K8), 256, 0, st>>>(A, M, K, K, a_buf.as<__nv_bfloat16>(), K8);
    const float* rp = nullptr;
    if (resid) {
        RC_TRY(r_buf.ensure(static_cast<size_t>(M) * N4 * 4));
        pad_rows_f32_kernel<<<blocks_for(static_cast<long long>(M) * N4), 256, 0, st>>>(resid, M, N, N, r_buf.as<float>(), N4);
        rp = r_buf.as<float>();
    }
    const int ldc = ex->store_bf16 ? N8 : N4;
    RC_TRY(o_buf.ensure(static_cast<size_t>(M) * ldc * (ex->store_bf16 ? 2 : 4)));
    DenseCall c{Operand{a_buf.p, nullptr, K8}, &w, M};
    c.pos = ex->pos; c.pos_period = ex->pos_period > 0 ? ex->pos_period : 1;
    c.resid = rp; c.ldr = N4;
    c.out = Operand{o_buf.p, nullptr, ldc}; c.out_f32 = ex->store_bf16 ? 0 : 1; c.act = act;
    if (ex->ln_out) {
        RC_TRY(ln_buf.ensure(static_cast<size_t>(M) * N8 * 2));
        c.ln_gamma = ex->ln_gamma; c.ln_beta = ex->ln_beta; c.ln_eps = ex->ln_eps; c.ln_out = ln_buf.p; c.ln_ld = N8;
    }
    if (ex->pair > 0 && !pair_kernel_legal(make_desc(c, Form::Bf16)))
        return fail(VITDET_E_INVALID, "op_dense_ex: the CTA-pair kernel needs M >= 1024, N >= 128 and no fused LayerNorm");
    RC_TRY(dense_once(c, Form::Bf16, sms, ex->pair < 0 ? env_options().gemm_pair : (ex->pair ? 2 : 0), st));
    if (ex->store_bf16) bf16_rows_to_f32_kernel<<<blocks_for(static_cast<long long>(M) * N), 256, 0, st>>>(o_buf.as<__nv_bfloat16>(), M, N, N8, out);
    else unpad_rows_f32_kernel<<<blocks_for(static_cast<long long>(M) * N), 256, 0, st>>>(o_buf.as<float>(), M, N, N4, out);
    if (ex->ln_out) bf16_rows_to_f32_kernel<<<blocks_for(static_cast<long long>(M) * N), 256, 0, st>>>(ln_buf.as<__nv_bfloat16>(), M, N, N8, ex->ln_out);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(st));
    return 0;
}

int vitdet_op_mlp_tail(const float* A, const float* W0, const float* b0, const float* W1, const float* b1, const float* W2,
                       const float* b2, float* x, const float* ln_gamma, const float* ln_beta, float ln_eps, float* ln_out,
                       int M, int K0, int N0, int N1, int N2, int act, void* stream) {
    if (!A || !W0 || !W1 || !W2 || !b0 || !b1 || !b2 || !x || M <= 0) return fail(VITDET_E_INVALID, "op_mlp_tail: bad arguments");
    if (ln_out && (!ln_gamma || !ln_beta)) return fail(VITDET_E_INVALID, "op_mlp_tail: ln_out needs gamma and beta");
    const int N[3] = {N0, N1, N2}, K[3] = {K0, N0, N1};
    if (!mlp_tail_supported(N, K)) return fail(VITDET_E_INVALID, "op_mlp_tail: widths %d -> %d -> %d -> %d are outside what the fused kernel takes", K0, N0, N1, N2);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int dev = 0, sms = 148;
    CU_TRY(cudaGetDevice(&dev));
    CU_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const float* Wk[3] = {W0, W1, W2};
    const float* bk[3] = {b0, b1, b2};
    DenseW w[3];
    for (int l = 0; l < 3; ++l) {
        RC_TRY(w[l].alloc(N[l], K[l]));
        pack_dense_kernel<<<blocks_for(static_cast<long long>(K[l]) * N[l]), 256, 0, st>>>(Wk[l], K[l], N[l], N[l], N[l], 0, K[l], K[l],
                                                                                         w[l].w16.as<__nv_bfloat16>(), w[l].ld16, 0, nullptr, 0);
        CU_TRY(cudaMemcpyAsync(w[l].bias.p, bk[l], static_cast<size_t>(N[l]) * 4, cudaMemcpyDeviceToDevice, st));
    }
    const int K8 = round_up(K0, 8), D4 = round_up(N2, 4), D8 = round_up(N2, 8);
    DevBuf a_buf, x_buf, ln_buf;
    RC_TRY(a_buf.ensure(static_cast<size_t>(M) * K8 * 2));
    RC_TRY(x_buf.ensure(static_cast<size_t>(M) * D4 * 4));
    f32_to_bf16_kernel<<<blocks_for(static_cast<long long>(M) * K8), 256, 0, st>>>(A, M, K0, K0, a_buf.as<__nv_bfloat16>(), K8);
    pad_rows_f32_kernel<<<blocks_for(static_cast<long long>(M) * D4), 256, 0, st>>>(x, M, N2, N2, x_buf.as<float>(), D4);
    MlpTailDesc td;
    td.A = a_buf.p; td.lda = K8; td.M = M;
    for (int l = 0; l < 3; ++l) { td.N[l] = N[l]; td.K[l] = K[l]; td.W[l] = w[l].w16.p; td.ldw[l] = w[l].ld16; td.bias[l] = w[l].bias.as<float>(); }
    td.x = x_buf.as<float>(); td.ldx = D4; td.act = act;
    if (ln_out) {
        RC_TRY(ln_buf.ensure(static_cast<size_t>(M) * D8 * 2));
        td.ln_gamma = ln_gamma; td.ln_beta = ln_beta; td.ln_eps = ln_eps; td.ln_out = ln_buf.p; td.ln_ld = D8;
    }
    MlpTailPlan plan;
    int rc = mlp_tail_make_plan(&plan, td, sms);
    if (rc) return fail(VITDET_E_INVALID, "op_mlp_tail: mlp_tail_make_plan failed: %d", rc);
    cudaError_t te = mlp_tail_launch(plan, st);
    if (te != cudaSuccess) return fail(VITDET_E_CUDA, "op_mlp_tail: launch failed: %s", cudaGetErrorString(te));
    unpad_rows_f32_kernel<<<blocks_for(static_cast<long long>(M) * N2), 256, 0, st>>>(x_buf.as<float>(), M, N2, D4, x);
    if (ln_out) bf16_rows_to_f32_kernel<<<blocks_for(static_cast<long long>(M) * N2), 256, 0, st>>>(ln_buf.as<__nv_bfloat16>(), M, N2, D8, ln_out);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(st));
    return 0;
}

int vitdet_op_head_slots(const float* x, const float* kernel, const float* bias, float* out, int images, int tokens, int D, int S,
                         int mode, void* stream) {
    if (!x || !kernel || !bias || !out || images <= 0 || tokens <= 0 || D <= 0 || S <= 0) return fail(VITDET_E_INVALID, "op_head_slots: bad arguments");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool bf = mode == VITDET_MODE_BF16;
    const int D4 = round_up(D, 4), Tp = round_up(tokens, bf ? 8 : 4);
    const long long M = static_cast<long long>(images) * tokens, R = static_cast<long long>(images) * S;
    DevBuf xb, wt, ob;
    RC_TRY(xb.ensure(static_cast<size_t>(M) * D4 * 4));
    RC_TRY(wt.ensure(static_cast<size_t>(S) * D * 4));
    RC_TRY(ob.ensure(static_cast<size_t>(R) * Tp * (bf ? 2 : 4)));
    CU_TRY(cudaMemsetAsync(ob.p, 0, ob.bytes, st));
    pad_rows_f32_kernel<<<blocks_for(M * D4), 256, 0, st>>>(x, static_cast<int>(M), D, D, xb.as<float>(), D4);
    pack_dense_kernel<<<blocks_for(static_cast<long long>(D) * S), 256, 0, st>>>(kernel, D, S, S, S, 0, D, D, nullptr, 0, 0, wt.as<float>(), D);
    CU_TRY(head_slots_launch(xb.as<float>(), D4, wt.as<float>(), bias, static_cast<int>(M), D, S, tokens, Tp, ob.p, bf ? 0 : 1, st));
    if (bf) bf16_rows_to_f32_kernel<<<blocks_for(R * tokens), 256, 0, st>>>(ob.as<__nv_bfloat16>(), static_cast<int>(R), tokens, Tp, out);
    else unpad_rows_f32_kernel<<<blocks_for(R * tokens), 256, 0, st>>>(ob.as<float>(), static_cast<int>(R), tokens, Tp, out);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(st));
    return 0;
}

int vitdet_op_patchify(const float* images, int B, int H, int W, int p, float* patches, void* stream) {
    if (!images || !patches || B <= 0 || H <= 0 || W <= 0 || p <= 0) return fail(VITDET_E_INVALID, "op_patchify: bad arguments");
    CU_TRY(patchify_launch(images, 0, B, H, W, p, patches, 3 * p * p, 3 * p, 1, static_cast<cudaStream_t>(stream)));
    return 0;
}

}  // extern "C"
