// Memory-bound kernels of the hot path: patch extraction, LayerNorm, the head's per-token slot
// projection, and the fused head tail (Dense(U->6) + sigmoid + clip + scale + thresholds).
// All of them are HBM/L2 streaming kernels: coalesced 16-byte accesses where the layout allows it,
// warp-shuffle reductions, no shared-memory staging (there is no reuse to exploit).
#include <algorithm>

#include "boxops.cuh"
#include "common.cuh"
#include "kernels.h"
#include "launch.h"

namespace vitdet {

namespace {

template <typename T> struct OutT;
template <> struct OutT<float> {
    static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
    static __device__ __forceinline__ void st4(float* p, float a, float b, float c, float d) {
        *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
    }
};
template <> struct OutT<__nv_bfloat16> {
    static __device__ __forceinline__ void st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
    static __device__ __forceinline__ void st4(__nv_bfloat16* p, float a, float b, float c, float d) {
        uint2 o;
        o.x = pack_bf16x2(a, b);
        o.y = pack_bf16x2(c, d);
        *reinterpret_cast<uint2*>(p) = o;
    }
};

// ------------------------------------------------------------------------------------------------
// K1 patchify.  tf.image.extract_patches(sizes=strides=[1,p,p,1], rates=1, padding='SAME')
// (det.py:195-197) followed by Reshape((-1, 3p^2)) (det.py:279-280):
//   grid = ceil(H/p) x ceil(W/p); pad_total = grid*p - size, pad_before = pad_total / 2, zeros;
//   patch vector element (r*p + c)*3 + ch; tokens row-major over the grid.
// Output layout: token row = p runs (one per patch row r) of `rp` elements, rp >= 3p; elements [3p, rp) of a
// run and [p*rp, ldp) of a token row are zero.  The engine uses rp = round_up(3p, 4) (52 for p = 17) so that
// every run starts 8-byte aligned and is written with 4-element vector stores (the projection weight is
// packed with the same zero columns); rp = 3p gives the reference's dense 3p^2 vector.
// One block per (image, token row of the grid).
// Measured and dropped (r02): staging every image row through shared memory with coalesced 16-byte loads and bank-conflict-
// free reads — 0.135 ms against this kernel's 0.118 ms per 64 images (latency-bound at 28 % occupancy, 59 KB of row buffers).
// ------------------------------------------------------------------------------------------------
#ifndef VITDET_PATCH_UNROLL
#define VITDET_PATCH_UNROLL 9
#endif
constexpr int kPatchRowUnroll = VITDET_PATCH_UNROLL;     // patch rows a lane loads before it stores (1 = the r-outer loop)

template <typename T> struct Vec4Store;
template <> struct Vec4Store<float> {
    static __device__ __forceinline__ void st(float* p, float a, float b, float c, float d) {
        *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
    }
};
template <> struct Vec4Store<__nv_bfloat16> {
    static __device__ __forceinline__ void st(__nv_bfloat16* p, float a, float b, float c, float d) {
        uint2 o;
        o.x = pack_bf16x2(a, b);
        o.y = pack_bf16x2(c, d);
        *reinterpret_cast<uint2*>(p) = o;
    }
};

// Pixel fetch of the patch kernel: float32 images are already normalised; uint8 images are normalised on the fly,
// /127.5 then -1 exactly as the reference's input pipeline does (vision_transformer_utilities.py:446-447), so the
// float32 image never exists in HBM and the host->device copy is a quarter of the size.
__device__ __forceinline__ float ld_pixel(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_pixel(const uint8_t* p) { return __fsub_rn(__fdiv_rn(static_cast<float>(__ldg(p)), 127.5f), 1.f); }

template <typename T, bool VEC, typename IN>
__global__ void __launch_bounds__(256)
patchify_kernel(const IN* __restrict__ img, int H, int W, int p, int gh, int gw, int pad_top,
                int pad_left, T* __restrict__ out, int ldp, int rp) {
    pdl_launch_dependents();
    pdl_wait();
    const int py = blockIdx.x;          // token row of the patch grid
    const int b = blockIdx.y;
    const int run = 3 * p;              // source elements per (token, r)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const size_t tok0 = (static_cast<size_t>(b) * gh + py) * gw;
    const int W3 = 3 * W;
    // No integer divisions and no staging: 16 or 32 lanes take one (token, r) run of 3p source floats, the
    // warps stride over the tokens, r is the (uniform) outer loop.  Consecutive tokens read consecutive
    // source bytes, so the misaligned scalar loads hit L1 after the first touch of each sector.
    const int gpr = VEC ? (rp >> 2) : rp;                  // store groups per run (4 elements or 1)
    const int lpr_shift = (VEC && gpr <= 16) ? 4 : 5;      // lanes per run: 16 or 32
    const int runs_per_warp = 32 >> lpr_shift;
    const int sub = lane >> lpr_shift, q0 = lane & ((1 << lpr_shift) - 1);
    if (VEC && kPatchRowUnroll > 1) {
        // A lane keeps its (token, 4-element group) and walks the patch rows, kPatchRowUnroll rows at a time: the 4 x U
        // loads of a step are independent, so a thread has 16 x U bytes in flight instead of 16 (the kernel is bound by
        // the read bytes in flight per SM, not by the LSU).
        const int y_first = py * p - pad_top;
        const IN* img_b = img + static_cast<size_t>(b) * H * W3 - 3 * pad_left;
        // work item = (token, group) flattened over the block (468 items on 256 threads for the default model: 91 % of the
        // lanes busy instead of 61 % with 16 lanes per run); one division per item, outside the row loop
        const int items = gw * gpr;
        for (int idx = threadIdx.x; idx < items; idx += 256) {
            const int px = idx / gpr, q = idx - px * gpr;
            const int x0 = px * run, w = 4 * q;
            T* dst_tok = out + (tok0 + px) * ldp + w;
            bool ok[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int x3 = x0 + w + j - 3 * pad_left;
                ok[j] = (w + j < run) && x3 >= 0 && x3 < W3;
            }
            for (int r0 = 0; r0 < p; r0 += kPatchRowUnroll) {
                float v[kPatchRowUnroll][4];
#pragma unroll
                for (int u = 0; u < kPatchRowUnroll; ++u) {
                    const int y = y_first + r0 + u;
                    const bool y_ok = (r0 + u < p) && (y >= 0) && (y < H);
                    const IN* src = img_b + static_cast<size_t>(y_ok ? y : 0) * W3 + x0 + w;
#pragma unroll
                    for (int j = 0; j < 4; ++j) v[u][j] = (y_ok && ok[j]) ? ld_pixel(src + j) : 0.f;
                }
#pragma unroll
                for (int u = 0; u < kPatchRowUnroll; ++u)
                    if (r0 + u < p) Vec4Store<T>::st(dst_tok + (r0 + u) * rp, v[u][0], v[u][1], v[u][2], v[u][3]);
            }
        }
    } else
    for (int r = 0; r < p; ++r) {
        const int y = py * p + r - pad_top;
        const bool y_ok = (y >= 0) && (y < H);
        const IN* src = img + (static_cast<size_t>(b) * H + (y_ok ? y : 0)) * W3 - 3 * pad_left;
        for (int px = warp * runs_per_warp + sub; px < gw; px += 8 * runs_per_warp) {
            T* dst = out + (tok0 + px) * ldp + r * rp;
            const int x0 = px * run;                       // index into the padded row; source index = x0 + w - 3*pad_left
            for (int q = q0; q < gpr; q += (1 << lpr_shift)) {
                if (VEC) {
                    const int w = 4 * q;
                    float v[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int x3 = x0 + w + j - 3 * pad_left;
                        v[j] = (y_ok && w + j < run && x3 >= 0 && x3 < W3) ? ld_pixel(src + x0 + w + j) : 0.f;
                    }
                    Vec4Store<T>::st(dst + w, v[0], v[1], v[2], v[3]);
                } else {
                    const int x3 = x0 + q - 3 * pad_left;
                    OutT<T>::st(dst + q, (y_ok && q < run && x3 >= 0 && x3 < W3) ? ld_pixel(src + x0 + q) : 0.f);
                }
            }
        }
    }
    const int P = rp * p;
    if (ldp > P) {
        const int padw = ldp - P;
        for (int px = warp; px < gw; px += 8)
            for (int w = lane; w < padw; w += 32) OutT<T>::st(out + (tok0 + px) * ldp + P + w, 0.f);
    }
}

// ------------------------------------------------------------------------------------------------
// Input side ("next" row N4): _get_image_tensor_coco of the reference (vision_transformer_utilities.py:418-449) after
// the file decode: tf.image.resize_with_pad(image, H, W) (bilinear, half-pixel centres, no antialias, zero padding),
// tf.clip_by_value(0, 255), / 127.5, - 1.  The interpolation follows TF's resize_bilinear CPU kernel term by term, without
// FMA contraction.  preprocess_kernel and letterbox_patchify_kernel both evaluate a pixel with the two functions below,
// so the letterboxed patch matrix equals patchify of preprocess_kernel's image bit for bit.
// ------------------------------------------------------------------------------------------------
// Value of a letterbox bar pixel: the zero padding of resize_with_pad after clip, / 127.5, - 1.
constexpr float kLetterboxBar = -1.f;

// Taps of resized coordinate i along one axis: in = (i + 0.5) * scale - 0.5; lower = max(floor(in), 0);
// upper = min(ceil(in), size - 1); lerp = in - floor(in).
struct ResizeTap { int lo, hi; float lerp; };
__device__ __forceinline__ ResizeTap resize_tap(int i, float scale, int size) {
    const float in = __fsub_rn(__fmul_rn(__fadd_rn(static_cast<float>(i), 0.5f), scale), 0.5f);
    const float f = floorf(in);
    return ResizeTap{max(static_cast<int>(f), 0), min(static_cast<int>(ceilf(in)), size - 1), __fsub_rn(in, f)};
}

// One channel of one resized pixel: r0 / r1 are the source rows of the y taps, x0 / x1 the byte offsets of the channel
// at the x taps.  Top and bottom lerp in x, then in y; clip to [0, 255]; / 127.5 - 1.
__device__ __forceinline__ float letterbox_value(const uint8_t* __restrict__ r0, const uint8_t* __restrict__ r1, int x0, int x1,
                                                 float lx, float ly) {
    const float tl = __ldg(r0 + x0), tr = __ldg(r0 + x1), bl = __ldg(r1 + x0), br = __ldg(r1 + x1);
    const float top = __fadd_rn(tl, __fmul_rn(__fsub_rn(tr, tl), lx));
    const float bot = __fadd_rn(bl, __fmul_rn(__fsub_rn(br, bl), lx));
    float v = __fadd_rn(top, __fmul_rn(__fsub_rn(bot, top), ly));
    v = fminf(fmaxf(v, 0.f), 255.f);
    return __fsub_rn(__fdiv_rn(v, 127.5f), 1.f);
}

// K1 for a ragged batch of uint8 images: resize_with_pad to the model's H x W fused into patchify (same output layout
// and work decomposition as the vector form above), so the float32 letterboxed image never exists.  Patch element
// (y, x, c) of the model image is 0 outside it (extract_patches' SAME padding), kLetterboxBar in resize_with_pad's bars,
// and the resized pixel otherwise.  images[b] describes image b of the launch.
// A lane's 4 elements keep their x taps across the patch rows; each row costs one y tap and 16 byte gathers per lane,
// which L1 serves (a 640 x 480 source is 0.9 MB against the 4.4 MB float32 image patchify reads).
#ifndef VITDET_LETTERBOX_UNROLL
#define VITDET_LETTERBOX_UNROLL 4
#endif
constexpr int kLetterboxRowUnroll = VITDET_LETTERBOX_UNROLL;

template <typename T>
__global__ void __launch_bounds__(256)
letterbox_patchify_kernel(const LetterboxImage* __restrict__ images, int H, int W, int p, int gh, int gw, int pad_top,
                          int pad_left, T* __restrict__ out, int ldp, int rp) {
    pdl_launch_dependents();
    pdl_wait();
    const int py = blockIdx.x;
    const int b = blockIdx.y;
    const LetterboxImage im = images[b];
    const int run = 3 * p, gpr = rp >> 2;
    const size_t tok0 = (static_cast<size_t>(b) * gh + py) * gw;
    const size_t src_pitch = static_cast<size_t>(im.w) * 3;
    const int y_first = py * p - pad_top;
    enum { kPad = 0, kBar = 1, kPixel = 2 };
    const int items = gw * gpr;
    for (int idx = threadIdx.x; idx < items; idx += 256) {
        const int px = idx / gpr, q = idx - px * gpr;
        const int w = 4 * q;
        T* dst_tok = out + (tok0 + px) * ldp + w;
        int kind[4], xa[4], xb[4];
        float lx[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int e = w + j, pix = e / 3, ch = e - 3 * pix;
            const int x = px * p + pix - pad_left, rx = x - im.pw;
            kind[j] = (e >= run || x < 0 || x >= W) ? kPad : ((rx < 0 || rx >= im.rw) ? kBar : kPixel);
            const ResizeTap t = resize_tap(kind[j] == kPixel ? rx : 0, im.wscale, im.w);
            xa[j] = 3 * t.lo + ch; xb[j] = 3 * t.hi + ch; lx[j] = t.lerp;
        }
        for (int r0 = 0; r0 < p; r0 += kLetterboxRowUnroll) {
            float v[kLetterboxRowUnroll][4];
#pragma unroll
            for (int u = 0; u < kLetterboxRowUnroll; ++u) {
                const int y = y_first + r0 + u, ry = y - im.ph;
                const bool y_ok = (r0 + u < p) && y >= 0 && y < H;
                const bool in_rows = y_ok && ry >= 0 && ry < im.rh;
                const ResizeTap t = resize_tap(in_rows ? ry : 0, im.hscale, im.h);
                const uint8_t* row0 = im.pixels + static_cast<size_t>(t.lo) * src_pitch;
                const uint8_t* row1 = im.pixels + static_cast<size_t>(t.hi) * src_pitch;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (!y_ok || kind[j] == kPad) v[u][j] = 0.f;
                    else if (!in_rows || kind[j] == kBar) v[u][j] = kLetterboxBar;
                    else v[u][j] = letterbox_value(row0, row1, xa[j], xb[j], lx[j], t.lerp);
                }
            }
#pragma unroll
            for (int u = 0; u < kLetterboxRowUnroll; ++u)
                if (r0 + u < p) Vec4Store<T>::st(dst_tok + (r0 + u) * rp, v[u][0], v[u][1], v[u][2], v[u][3]);
        }
    }
    const int P = rp * p;
    if (ldp > P) {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, padw = ldp - P;
        for (int px = warp; px < gw; px += 8)
            for (int w = lane; w < padw; w += 32) OutT<T>::st(out + (tok0 + px) * ldp + P + w, 0.f);
    }
}

// ------------------------------------------------------------------------------------------------
// K3 LayerNorm over the last axis, eps inside the rsqrt, biased variance, f32 statistics
// (keras.layers.LayerNormalization defaults; det.py:353-357, 375-379).
// LPR lanes cooperate on one row (8 for the 28-wide default stream: four rows per warp, each lane
// one float4; 32 for wide streams).  The row is held in registers between the two reduction
// passes (CH float4 per lane), so x is read exactly once.
// ------------------------------------------------------------------------------------------------
template <int LPR, int CH, typename T>
__global__ void __launch_bounds__(256, CH <= 6 ? 4 : (CH <= 8 ? 3 : 2))      // rows of <= 768 floats: <= 64 registers, 32 resident warps per SM (was 24)
layernorm_kernel(const float* __restrict__ x, int ldx, const float* __restrict__ gamma,
                 const float* __restrict__ beta, int M, int D, float eps, T* __restrict__ y, int ldy) {
    constexpr int ROWS_PER_BLOCK = 256 / LPR;
    pdl_launch_dependents();
    pdl_wait();
    const int sub = threadIdx.x % LPR;
    const int row = blockIdx.x * ROWS_PER_BLOCK + threadIdx.x / LPR;
    const bool row_ok = row < M;
    const float* xr = x + static_cast<size_t>(row_ok ? row : 0) * ldx;

    float4 v[CH];
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < CH; ++i) {
        const int e = 4 * (sub + i * LPR);
        v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row_ok && e < D) {
            if (e + 4 <= D) {
                v[i] = *reinterpret_cast<const float4*>(xr + e);
            } else {
                float t[4] = {0.f, 0.f, 0.f, 0.f};
                for (int j = 0; j < 4 && e + j < D; ++j) t[j] = xr[e + j];
                v[i] = make_float4(t[0], t[1], t[2], t[3]);
            }
        }
        sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float mean = sum / static_cast<float>(D);

    float sq = 0.f;
#pragma unroll
    for (int i = 0; i < CH; ++i) {
        const int e = 4 * (sub + i * LPR);
        const float d0 = (e + 0 < D) ? v[i].x - mean : 0.f;
        const float d1 = (e + 1 < D) ? v[i].y - mean : 0.f;
        const float d2 = (e + 2 < D) ? v[i].z - mean : 0.f;
        const float d3 = (e + 3 < D) ? v[i].w - mean : 0.f;
        sq += (d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3);
    }
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    const float rstd = rsqrtf(sq / static_cast<float>(D) + eps);

    if (!row_ok) return;
    const bool vec_gb = ((reinterpret_cast<uintptr_t>(gamma) | reinterpret_cast<uintptr_t>(beta)) & 15) == 0;
    T* yr = y + static_cast<size_t>(row) * ldy;
#pragma unroll
    for (int i = 0; i < CH; ++i) {
        const int e = 4 * (sub + i * LPR);
        if (e < ldy) {       // pad columns [D, ldy) are written as zero
            float o[4];
            const float xv[4] = {v[i].x, v[i].y, v[i].z, v[i].w};
            if (vec_gb && e + 4 <= D) {
                // wide rows: gamma / beta as one 16-byte load each (8 scalar loads per group made the D = 768 kernel LSU-bound)
                const float4 g4 = __ldg(reinterpret_cast<const float4*>(gamma + e)), b4 = __ldg(reinterpret_cast<const float4*>(beta + e));
                o[0] = (xv[0] - mean) * rstd * g4.x + b4.x; o[1] = (xv[1] - mean) * rstd * g4.y + b4.y;
                o[2] = (xv[2] - mean) * rstd * g4.z + b4.z; o[3] = (xv[3] - mean) * rstd * g4.w + b4.w;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    o[j] = 0.f;
                    if (e + j < D) o[j] = (xv[j] - mean) * rstd * __ldg(gamma + e + j) + __ldg(beta + e + j);
                }
            }
            OutT<T>::st4(yr + e, o[0], o[1], o[2], o[3]);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// mlp_head first stage (det.py:454-463).  One thread per (token, slot).  The reference's Reshape((S, -1)) is a flat
// reinterpretation of the per-image (T, S) matrix as (S, T): flat element f = t*S + s of image b lands in row b*S + f / T,
// column f % T of the slot matrix.  With ldo == T that matrix is the compact buffer itself (out[idx]); a token count that
// is not a multiple of the 16-byte TMA row pitch gets rows of ldo > T elements whose pad columns stay zero.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
head_slots_kernel(const float* __restrict__ x, int ldx, const float* __restrict__ w,
                  const float* __restrict__ bias, long long total, int D, int S, int tokens, int ldo, T* __restrict__ out) {
    pdl_launch_dependents();
    pdl_wait();
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const long long m = idx / S;
    const int s = static_cast<int>(idx - m * S);
    const float* xr = x + m * ldx;
    const float* wr = w + static_cast<size_t>(s) * D;
    float acc = 0.f;
    int d = 0;
    if ((D & 3) == 0) {
        for (; d < D; d += 4) {
            const float4 a = *reinterpret_cast<const float4*>(xr + d);
            const float4 c = __ldg(reinterpret_cast<const float4*>(wr + d));
            acc = fmaf(a.x, c.x, acc);
            acc = fmaf(a.y, c.y, acc);
            acc = fmaf(a.z, c.z, acc);
            acc = fmaf(a.w, c.w, acc);
        }
    }
    for (; d < D; ++d) acc = fmaf(xr[d], __ldg(wr + d), acc);
    long long o = idx;
    if (ldo != tokens) {
        const long long per_image = static_cast<long long>(tokens) * S;
        const long long img = idx / per_image, f = idx - img * per_image;
        o = (img * S + f / tokens) * ldo + f % tokens;
    }
    OutT<T>::st(out + o, acc + __ldg(bias + s));
}

// Wide residual streams (embedding_dim >= 64, e.g. the 768-wide variant): the thread-per-(token, slot) kernel above makes
// every thread walk a whole 3 KB row with 16 bytes in flight (0.70 ms per 32 images at D = 768).  Here a warp owns two
// tokens at a time: the lanes split the row (coalesced 16-byte loads, all in flight at once), every lane accumulates its
// share of all S slot products against a shared-memory copy of the [S, D] kernel (each 16-byte weight read serves both
// tokens), and S butterfly reductions finish the sums.  S is a template parameter so that the accumulators stay in registers.
template <typename T, int S>
__global__ void __launch_bounds__(256)
head_slots_wide_kernel(const float* __restrict__ x, int ldx, const float* __restrict__ w, const float* __restrict__ bias, int M,
                       int D, int tokens, int ldo, T* __restrict__ out) {
    extern __shared__ __align__(16) float hs_smem[];       // [S][D]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int D4 = D >> 2;
    pdl_launch_dependents();
    for (int i = threadIdx.x; i < S * D4; i += 256)        // weights do not depend on the previous kernel
        reinterpret_cast<float4*>(hs_smem)[i] = __ldg(reinterpret_cast<const float4*>(w) + i);
    pdl_wait();
    __syncthreads();
    const float b = lane < S ? __ldg(bias + lane) : 0.f;
    const long long per_image = static_cast<long long>(tokens) * S;
    for (int m0 = 2 * (blockIdx.x * 8 + warp); m0 < M; m0 += 2 * gridDim.x * 8) {
        const bool two = m0 + 1 < M;
        const float4* x0 = reinterpret_cast<const float4*>(x + static_cast<size_t>(m0) * ldx);
        const float4* x1 = reinterpret_cast<const float4*>(x + static_cast<size_t>(two ? m0 + 1 : m0) * ldx);
        float acc0[S], acc1[S];
#pragma unroll
        for (int s = 0; s < S; ++s) { acc0[s] = 0.f; acc1[s] = 0.f; }
#pragma unroll 2
        for (int c = lane; c < D4; c += 32) {
            const float4 a0 = x0[c], a1 = x1[c];
#pragma unroll
            for (int s = 0; s < S; ++s) {
                const float4 ws = reinterpret_cast<const float4*>(hs_smem)[s * D4 + c];
                acc0[s] = fmaf(a0.x, ws.x, fmaf(a0.y, ws.y, fmaf(a0.z, ws.z, fmaf(a0.w, ws.w, acc0[s]))));
                acc1[s] = fmaf(a1.x, ws.x, fmaf(a1.y, ws.y, fmaf(a1.z, ws.z, fmaf(a1.w, ws.w, acc1[s]))));
            }
        }
        float r0 = 0.f, r1 = 0.f;
#pragma unroll
        for (int s = 0; s < S; ++s) {
            float v0 = acc0[s], v1 = acc1[s];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                v0 += __shfl_xor_sync(0xffffffffu, v0, o);
                v1 += __shfl_xor_sync(0xffffffffu, v1, o);
            }
            if (lane == s) { r0 = v0; r1 = v1; }
        }
        if (lane < S) {
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                if (t == 1 && !two) break;
                long long o = static_cast<long long>(m0 + t) * S + lane;
                if (ldo != tokens) {
                    const long long img = o / per_image, f = o - img * per_image;
                    o = (img * S + f / tokens) * ldo + f % tokens;
                }
                OutT<T>::st(out + o, (t ? r1 : r0) + b);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Decode of one slot: transform_predictions (det.py:619-645) + thresholds + corner boxes.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int clip_int(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

__device__ __forceinline__ void decode_slot(const float (&l)[6], long long r, const DecodeParams& dp,
                                            const DecodeOut& o) {
    float dec[6];
    if (dp.apply_transform) {
        transform_slot(l, dp, dec);
    } else {
#pragma unroll
        for (int j = 0; j < 6; ++j) dec[j] = l[j];
    }
    const float id = rintf(dec[1]);                 // tf.round / np.round: half to even
    const float cc = class_confidence(dec[1]);      // det.py:1376, 2279
    bool keep;
    if (dp.strict) keep = (dec[0] > dp.obj_thr) && (cc > dp.cls_thr);        // det.py:1381-1384
    else keep = !(dec[0] < dp.obj_thr) && !(cc < dp.cls_thr);               // det.py:2264, 2282
    if (o.logits) {
#pragma unroll
        for (int j = 0; j < 6; ++j) o.logits[r * 6 + j] = l[j];
    }
    if (o.decoded) {
#pragma unroll
        for (int j = 0; j < 6; ++j) o.decoded[r * 6 + j] = dec[j];
    }
    if (o.class_id) o.class_id[r] = static_cast<int32_t>(id);
    if (o.class_conf) o.class_conf[r] = cc;
    if (o.keep) o.keep[r] = keep ? 1 : 0;
    if (o.corners || o.packed) {
        // det.py:2300-2325: int() truncation toward zero, then clip to the image.
        // boxes are scaled by enlarged_image_scale first (det.py:2294-2297); the clip bounds are the enlarged image's
        // width / height, round(size * scale) (det.py:2237-2252)
        const float s = dp.corner_scale;
        const int iw = static_cast<int>(rintf(dp.img_w * s)), ih = static_cast<int>(rintf(dp.img_h * s));
        const float cx = dec[2] * s, cy = dec[3] * s, bh = dec[4] * s, bw = dec[5] * s;
        const int c0 = clip_int(static_cast<int>(cx - bw / 2.f), 0, iw), c1 = clip_int(static_cast<int>(cy - bh / 2.f), 0, ih);
        const int c2 = clip_int(static_cast<int>(cx + bw / 2.f), 0, iw), c3 = clip_int(static_cast<int>(cy + bh / 2.f), 0, ih);
        if (o.corners) { o.corners[r * 4 + 0] = c0; o.corners[r * 4 + 1] = c1; o.corners[r * 4 + 2] = c2; o.corners[r * 4 + 3] = c3; }
        if (o.packed) {
            // the fixed-size record the ranks all-gather (SURVEY §8e): ints are exact in float32 (< 2^24)
            float* pk = o.packed + r * 13;
#pragma unroll
            for (int j = 0; j < 6; ++j) pk[j] = dec[j];
            pk[6] = id; pk[7] = cc; pk[8] = keep ? 1.f : 0.f;
            pk[9] = static_cast<float>(c0); pk[10] = static_cast<float>(c1); pk[11] = static_cast<float>(c2); pk[12] = static_cast<float>(c3);
        }
    }
    if (o.boxes_original) {
        // the box on the source image: undo resize_with_pad (remove the bar, scale by source size / resized size), then clip
        const LetterboxImage& g = o.letterbox[r / o.slots];
        const float half_h = __fdiv_rn(dec[4], 2.f), half_w = __fdiv_rn(dec[5], 2.f);
        const float pw = static_cast<float>(g.pw), ph = static_cast<float>(g.ph);
        const float sw = static_cast<float>(g.w), sh = static_cast<float>(g.h);
        const float x0 = fminf(fmaxf(__fmul_rn(__fsub_rn(__fsub_rn(dec[2], half_w), pw), g.wscale), 0.f), sw);
        const float y0 = fminf(fmaxf(__fmul_rn(__fsub_rn(__fsub_rn(dec[3], half_h), ph), g.hscale), 0.f), sh);
        const float x1 = fminf(fmaxf(__fmul_rn(__fsub_rn(__fadd_rn(dec[2], half_w), pw), g.wscale), 0.f), sw);
        const float y1 = fminf(fmaxf(__fmul_rn(__fsub_rn(__fadd_rn(dec[3], half_h), ph), g.hscale), 0.f), sh);
        // a reduced decode of a file: on to the file's pixels (a factor of exactly 1 leaves the clipped box as it is)
        const float fw = static_cast<float>(g.file_w), fh = static_cast<float>(g.file_h);
        float* bo = o.boxes_original + r * 4;
        bo[0] = fminf(fmaxf(__fmul_rn(x0, g.file_wscale), 0.f), fw);
        bo[1] = fminf(fmaxf(__fmul_rn(y0, g.file_hscale), 0.f), fh);
        bo[2] = fminf(fmaxf(__fmul_rn(x1, g.file_wscale), 0.f), fw);
        bo[3] = fminf(fmaxf(__fmul_rn(y1, g.file_hscale), 0.f), fh);
    }
}

__device__ __forceinline__ float ld_as_f32(const float* p) { return *p; }
__device__ __forceinline__ float ld_as_f32(const __nv_bfloat16* p) { return __bfloat162float(*p); }

// K9: one warp per (image, slot) row: 6 dot products of length U, shuffle reduction, lane 0 decodes.
template <typename T>
__global__ void __launch_bounds__(256)
head_tail_kernel(const T* __restrict__ h, int ldh, const float* __restrict__ w, const float* __restrict__ bias,
                 int R, int U, DecodeParams dp, DecodeOut o) {
    pdl_launch_dependents();
    pdl_wait();
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= R) return;
    const T* hr = h + static_cast<size_t>(warp) * ldh;
    float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int u = lane; u < U; u += 32) {
        const float a = ld_as_f32(hr + u);
#pragma unroll
        for (int j = 0; j < 6; ++j) acc[j] = fmaf(a, __ldg(w + j * U + u), acc[j]);
    }
#pragma unroll
    for (int j = 0; j < 6; ++j) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], off);
    }
    if (lane == 0) {
        float l[6];
#pragma unroll
        for (int j = 0; j < 6; ++j) l[j] = acc[j] + __ldg(bias + j);
        decode_slot(l, warp, dp, o);
    }
}

__global__ void __launch_bounds__(256)
decode_kernel(const float* __restrict__ logits, int R, DecodeParams dp, DecodeOut o) {
    pdl_launch_dependents();
    pdl_wait();
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    float l[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) l[j] = logits[static_cast<size_t>(r) * 6 + j];
    DecodeOut o2 = o;
    if (o2.logits == logits) o2.logits = nullptr;
    decode_slot(l, r, dp, o2);
}

// ------------------------------------------------------------------------------------------------
// iou_calculator (reference det.py:761-875): element-wise IoU of boxes (cx, cy, h, w) held in the LAST FOUR
// entries of rows of `width` floats.  Same arithmetic and operation order as the reference (edges, strict '<' / '>'
// overlap test, the two middle values of the four sorted edges, I / (U + eps)); __f*_rn intrinsics keep the
// compiler from contracting products and sums into FMAs, so the result is bit-identical to an f32 evaluation.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
iou_kernel(const float* __restrict__ label, const float* __restrict__ pred, long long R, int width, float eps,
           float* __restrict__ iou) {
    pdl_launch_dependents();
    pdl_wait();
    const long long r = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (r >= R) return;
    const float* lb = label + r * width + (width - 4);
    const float* pb = pred + r * width + (width - 4);
    const float lx = lb[0], ly = lb[1], lh = lb[2], lw = lb[3];
    const float px = pb[0], py = pb[1], ph = pb[2], pw = pb[3];
    iou[r] = iou_boxes(lx, ly, lh, lw, px, py, ph, pw, eps);
}

// ------------------------------------------------------------------------------------------------
// Input side, one image: uint8 HWC in, float32 HWC [th, tw, 3] in [-1, 1] out (see resize_tap / letterbox_value).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
preprocess_kernel(const uint8_t* __restrict__ img, int h, int w, float* __restrict__ out, int th, int tw, int rh, int rw,
                  int ph, int pw, float hscale, float wscale) {
    pdl_launch_dependents();
    pdl_wait();
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    if (x >= tw) return;
    float* o = out + (static_cast<size_t>(y) * tw + x) * 3;
    const int ry = y - ph, rx = x - pw;
    if (ry < 0 || ry >= rh || rx < 0 || rx >= rw) {
        o[0] = kLetterboxBar; o[1] = kLetterboxBar; o[2] = kLetterboxBar;
        return;
    }
    const ResizeTap ty = resize_tap(ry, hscale, h), tx = resize_tap(rx, wscale, w);
    const uint8_t* r0 = img + static_cast<size_t>(ty.lo) * w * 3;
    const uint8_t* r1 = img + static_cast<size_t>(ty.hi) * w * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) o[c] = letterbox_value(r0, r1, tx.lo * 3 + c, tx.hi * 3 + c, tx.lerp, ty.lerp);
}

template <int LPR, typename T>
cudaError_t ln_dispatch(const float* x, int ldx, const float* g, const float* b, int M, int D, float eps, T* y,
                        int ldy, cudaStream_t st) {
    const int rows_per_block = 256 / LPR;
    const int grid = (M + rows_per_block - 1) / rows_per_block;
    const int width = ldy > D ? ldy : D;
    const int chunks = (width + 4 * LPR - 1) / (4 * LPR);
    if (chunks <= 1) return launch_kernel(layernorm_kernel<LPR, 1, T>, dim3(grid), dim3(256), 0, st, 1, x, ldx, g, b, M, D, eps, y, ldy);
    else if (chunks <= 2) return launch_kernel(layernorm_kernel<LPR, 2, T>, dim3(grid), dim3(256), 0, st, 1, x, ldx, g, b, M, D, eps, y, ldy);
    else if (chunks <= 4) return launch_kernel(layernorm_kernel<LPR, 4, T>, dim3(grid), dim3(256), 0, st, 1, x, ldx, g, b, M, D, eps, y, ldy);
    else if (chunks <= 6) return launch_kernel(layernorm_kernel<LPR, 6, T>, dim3(grid), dim3(256), 0, st, 1, x, ldx, g, b, M, D, eps, y, ldy);
    else if (chunks <= 8) return launch_kernel(layernorm_kernel<LPR, 8, T>, dim3(grid), dim3(256), 0, st, 1, x, ldx, g, b, M, D, eps, y, ldy);
    else if (chunks <= 16) return launch_kernel(layernorm_kernel<LPR, 16, T>, dim3(grid), dim3(256), 0, st, 1, x, ldx, g, b, M, D, eps, y, ldy);
    return cudaErrorInvalidValue;   // embedding_dim > 2048 is outside what this build supports
}

}  // namespace

template <typename IN>
static cudaError_t patchify_launch_t(const IN* images, int B, int H, int W, int p, void* patches, int ldp, int rp, int out_f32,
                                     cudaStream_t stream) {
    const int gh = (H + p - 1) / p, gw = (W + p - 1) / p;
    const int pad_top = (gh * p - H) / 2, pad_left = (gw * p - W) / 2;
    if (rp < 3 * p || ldp < rp * p) return cudaErrorInvalidValue;
    dim3 grid(gh, B);
    const size_t smem = 0;
    // vector stores need every run (and every token row) to start on a 4-element boundary
    const bool vec = (rp % 4 == 0) && (ldp % 4 == 0) && ((reinterpret_cast<uintptr_t>(patches) & 15) == 0);
    if (out_f32) {
        float* o = static_cast<float*>(patches);
        if (vec) return launch_kernel(patchify_kernel<float, true, IN>, grid, dim3(256), smem, stream, 1, images, H, W, p, gh, gw, pad_top, pad_left, o, ldp, rp);
        return launch_kernel(patchify_kernel<float, false, IN>, grid, dim3(256), smem, stream, 1, images, H, W, p, gh, gw, pad_top, pad_left, o, ldp, rp);
    }
    __nv_bfloat16* o = static_cast<__nv_bfloat16*>(patches);
    if (vec) return launch_kernel(patchify_kernel<__nv_bfloat16, true, IN>, grid, dim3(256), smem, stream, 1, images, H, W, p, gh, gw, pad_top, pad_left, o, ldp, rp);
    return launch_kernel(patchify_kernel<__nv_bfloat16, false, IN>, grid, dim3(256), smem, stream, 1, images, H, W, p, gh, gw, pad_top, pad_left, o, ldp, rp);
}

cudaError_t patchify_launch(const void* images, int in_u8, int B, int H, int W, int p, void* patches, int ldp, int rp, int out_f32,
                            cudaStream_t stream) {
    if (in_u8) return patchify_launch_t(static_cast<const uint8_t*>(images), B, H, W, p, patches, ldp, rp, out_f32, stream);
    return patchify_launch_t(static_cast<const float*>(images), B, H, W, p, patches, ldp, rp, out_f32, stream);
}

cudaError_t layernorm_launch(const float* x, int ldx, const float* gamma, const float* beta, int M, int D, float eps,
                             void* y, int ldy, int out_f32, cudaStream_t stream) {
    if ((ldx % 4) || (ldy % 4) || M <= 0 || D <= 0) return cudaErrorInvalidValue;
    const int width = ldy > D ? ldy : D;
    if (width <= 32) {
        if (out_f32) return ln_dispatch<8, float>(x, ldx, gamma, beta, M, D, eps, static_cast<float*>(y), ldy, stream);
        return ln_dispatch<8, __nv_bfloat16>(x, ldx, gamma, beta, M, D, eps, static_cast<__nv_bfloat16*>(y), ldy, stream);
    }
    if (out_f32) return ln_dispatch<32, float>(x, ldx, gamma, beta, M, D, eps, static_cast<float*>(y), ldy, stream);
    return ln_dispatch<32, __nv_bfloat16>(x, ldx, gamma, beta, M, D, eps, static_cast<__nv_bfloat16*>(y), ldy, stream);
}

cudaError_t head_slots_launch(const float* x, int ldx, const float* w, const float* bias, int M, int D, int S, int tokens,
                              int ldo, void* out, int out_f32, cudaStream_t stream) {
    const long long total = static_cast<long long>(M) * S;
    const int grid = static_cast<int>((total + 255) / 256);
    if (tokens <= 0 || ldo < tokens || M % tokens) return cudaErrorInvalidValue;
    // the reference's head has 17 slots (det.py:454); other slot counts take the generic kernel
    const size_t wide_smem = static_cast<size_t>(S) * D * sizeof(float);
    static const bool wide_ok = !(getenv("VITDET_SLOTS_WIDE") && strcmp(getenv("VITDET_SLOTS_WIDE"), "0") == 0);     // A/B switch
    if (wide_ok && S == 17 && D >= 64 && (D & 3) == 0 && (ldx & 3) == 0 && wide_smem <= 200u * 1024u &&
        (reinterpret_cast<uintptr_t>(w) & 15) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
        const int wgrid = std::min((M + 15) / 16, 2 * 148);
        cudaError_t e;
        if (out_f32) {
            e = ensure_max_dynamic_smem(reinterpret_cast<const void*>(head_slots_wide_kernel<float, 17>), static_cast<int>(wide_smem));
            if (e != cudaSuccess) return e;
            return launch_kernel(head_slots_wide_kernel<float, 17>, dim3(wgrid), dim3(256), wide_smem, stream, 1, x, ldx, w, bias, M, D, tokens,
                                 ldo, static_cast<float*>(out));
        }
        e = ensure_max_dynamic_smem(reinterpret_cast<const void*>(head_slots_wide_kernel<__nv_bfloat16, 17>), static_cast<int>(wide_smem));
        if (e != cudaSuccess) return e;
        return launch_kernel(head_slots_wide_kernel<__nv_bfloat16, 17>, dim3(wgrid), dim3(256), wide_smem, stream, 1, x, ldx, w, bias, M, D,
                             tokens, ldo, static_cast<__nv_bfloat16*>(out));
    }
    if (out_f32)
        return launch_kernel(head_slots_kernel<float>, dim3(grid), dim3(256), 0, stream, 1, x, ldx, w, bias, total, D, S, tokens, ldo,
                             static_cast<float*>(out));
    return launch_kernel(head_slots_kernel<__nv_bfloat16>, dim3(grid), dim3(256), 0, stream, 1, x, ldx, w, bias, total, D, S, tokens, ldo,
                         static_cast<__nv_bfloat16*>(out));
}

cudaError_t head_tail_launch(const void* h, int ldh, int in_f32, const float* w, const float* bias, int R, int U,
                             const DecodeParams& dp, const DecodeOut& out, cudaStream_t stream) {
    const int grid = (R * 32 + 255) / 256;
    if (in_f32)
        return launch_kernel(head_tail_kernel<float>, dim3(grid), dim3(256), 0, stream, 1, static_cast<const float*>(h), ldh, w,
                             bias, R, U, dp, out);
    return launch_kernel(head_tail_kernel<__nv_bfloat16>, dim3(grid), dim3(256), 0, stream, 1,
                         static_cast<const __nv_bfloat16*>(h), ldh, w, bias, R, U, dp, out);
}

void resize_with_pad_geometry(int h, int w, int th, int tw, int* rh, int* rw, int* ph, int* pw) {
    // tf.image.resize_with_pad's size arithmetic, in float32 exactly as TF does it (it is why a 640 x 480 image can
    // come out 607 wide): ratio = max(w / tw, h / th); resized = floor(size / ratio); pad = max(0, floor((target - size / ratio) / 2)).
    const float fh = static_cast<float>(h), fw = static_cast<float>(w), fth = static_cast<float>(th), ftw = static_cast<float>(tw);
    const float ratio = fmaxf(fw / ftw, fh / fth);
    const float rhf = fh / ratio, rwf = fw / ratio;
    *rh = static_cast<int>(floorf(rhf));
    *rw = static_cast<int>(floorf(rwf));
    const int p_h = static_cast<int>(floorf((fth - rhf) / 2.f)), p_w = static_cast<int>(floorf((ftw - rwf) / 2.f));
    *ph = p_h > 0 ? p_h : 0;
    *pw = p_w > 0 ? p_w : 0;
}

bool letterbox_image(const uint8_t* pixels, int h, int w, int th, int tw, LetterboxImage* im) {
    if (h <= 0 || w <= 0 || th <= 0 || tw <= 0) return false;
    im->pixels = pixels; im->h = h; im->w = w;
    resize_with_pad_geometry(h, w, th, tw, &im->rh, &im->rw, &im->ph, &im->pw);
    if (im->rh <= 0 || im->rw <= 0) return false;
    im->hscale = static_cast<float>(h) / static_cast<float>(im->rh);
    im->wscale = static_cast<float>(w) / static_cast<float>(im->rw);
    im->file_h = h; im->file_w = w;
    im->file_hscale = im->file_wscale = 1.f;
    return true;
}

cudaError_t preprocess_launch(const uint8_t* image, int h, int w, float* out, int th, int tw, cudaStream_t stream) {
    LetterboxImage g;
    if (!letterbox_image(image, h, w, th, tw, &g)) return cudaErrorInvalidValue;
    dim3 grid((tw + 255) / 256, th);
    return launch_kernel(preprocess_kernel, grid, dim3(256), 0, stream, 1, image, h, w, out, th, tw, g.rh, g.rw, g.ph, g.pw,
                         g.hscale, g.wscale);
}

cudaError_t letterbox_patchify_launch(const LetterboxImage* images, int B, int H, int W, int p, void* patches, int ldp, int rp,
                                      int out_f32, cudaStream_t stream) {
    const int gh = (H + p - 1) / p, gw = (W + p - 1) / p;
    const int pad_top = (gh * p - H) / 2, pad_left = (gw * p - W) / 2;
    // the vector stores of the patch runs need every run and token row on a 4-element boundary
    if (B <= 0 || rp < 3 * p || ldp < rp * p || rp % 4 || ldp % 4 || (reinterpret_cast<uintptr_t>(patches) & 15))
        return cudaErrorInvalidValue;
    const dim3 grid(gh, B);
    if (out_f32)
        return launch_kernel(letterbox_patchify_kernel<float>, grid, dim3(256), 0, stream, 1, images, H, W, p, gh, gw, pad_top,
                             pad_left, static_cast<float*>(patches), ldp, rp);
    return launch_kernel(letterbox_patchify_kernel<__nv_bfloat16>, grid, dim3(256), 0, stream, 1, images, H, W, p, gh, gw, pad_top,
                         pad_left, static_cast<__nv_bfloat16*>(patches), ldp, rp);
}

cudaError_t iou_launch(const float* label, const float* pred, long long R, int width, float eps, float* iou,
                       cudaStream_t stream) {
    if (R <= 0) return cudaSuccess;
    if (width < 4) return cudaErrorInvalidValue;
    return launch_kernel(iou_kernel, dim3(static_cast<unsigned>((R + 255) / 256)), dim3(256), 0, stream, 1, label, pred, R, width, eps, iou);
}

cudaError_t decode_launch(const float* logits, int R, const DecodeParams& dp, const DecodeOut& out,
                          cudaStream_t stream) {
    return launch_kernel(decode_kernel, dim3((R + 255) / 256), dim3(256), 0, stream, 1, logits, R, dp, out);
}

}  // namespace vitdet
