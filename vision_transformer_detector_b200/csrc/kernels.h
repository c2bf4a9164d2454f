// Internal (C++) declarations of the kernel launchers.  The public boundary is include/vitdet_b200.h.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <vector>

namespace vitdet {

// ------------------------------------------------------------------------------------------------
// Dense layer:  out[M, ldc] = epilogue( A[M,K] (lda) * W[N,K]^T (ldw) )
//   epilogue(acc)[m,n] = act(acc + bias[n] + pos[m % pos_period]) + resid[m,n]
// (the order matches the reference graph: Dense -> activation -> keras.layers.add, det.py:388-412,
//  and Dense -> add(position) for the patch embedding, det.py:297-307).
// Columns [N, round_up(N, vec)) of `out` are written as zero, vec = 8 (bf16) or 4 (f32).
// ------------------------------------------------------------------------------------------------
struct GemmDesc {
    const void* A = nullptr;   // bf16 (tensor-core path) or f32 (SIMT path), row-major, K contiguous
    int lda = 0;
    const void* W = nullptr;   // same element type as A; row n = output unit n, K contiguous
    int ldw = 0;
    int M = 0, N = 0, K = 0;
    const float* bias = nullptr;
    const float* pos = nullptr;
    int pos_period = 1;
    const float* resid = nullptr;   // f32, only with out_f32; may alias `out`
    int ldr = 0;
    void* out = nullptr;
    int ldc = 0;
    int out_f32 = 0;
    int act = 0;               // vitdet::Act
    int block_n = 0;           // 0 = choose
    // Optional fused LayerNormalization of the OUTPUT row (tensor-core kernel, f32 output, N <= 32 only: the
    // epilogue thread holds the whole row): ln_out[m, :] = LN(out[m, :]) * gamma + beta as bf16, pads zero.
    const float* ln_gamma = nullptr;
    const float* ln_beta = nullptr;
    float ln_eps = 1e-3f;
    void* ln_out = nullptr;    // bf16 [M, ln_ld]
    int ln_ld = 0;
    // fp32-accumulate mode on the tensor cores: every float32 value travels as TWO bf16 planes, hi = bf16(x) and
    // lo = bf16(x - hi) (|x - hi - lo| <= 2^-18 |x|), and the product is A_hi W_hi + A_hi W_lo + A_lo W_hi — three passes
    // over K through the same pipeline (the lo*lo term, 2^-18 of the result, is dropped).  split = 1: A_lo / W_lo are the
    // lo planes (same shapes and pitches as A / W).  out_split = 1 (bf16 output only): the result is stored as planes too,
    // out = hi, out_lo = lo.  precise = 1: exact expf / tanhf based activations instead of the ex2/rcp.approx forms.
    int split = 0;
    const void* A_lo = nullptr;
    const void* W_lo = nullptr;
    int out_split = 0;
    void* out_lo = nullptr;
    int precise = 0;
};

struct TcGemmPlan {
    CUtensorMap tmA, tmB;
    CUtensorMap tmC;           // bf16 outputs only: 32 x 32 boxes, 64B swizzle (TMA store from the epilogue)
    CUtensorMap tmA_lo, tmB_lo, tmC_lo;      // the lo planes of the split (fp32-accumulate) mode
    GemmDesc desc;
    int block_n = 0;
    int num_stages = 0;
    int n_tiles = 0;
    int num_tiles = 0;
    int grid = 0;
    size_t smem_bytes = 0;
    int pair = 0;              // 1: built for the CTA-pair form
};

int choose_block_n(int N);
int make_tmap_bf16_2d(CUtensorMap* map, const void* base, int rows, int cols, int ld, int box_rows);
int make_tmap_bf16_2d_ex(CUtensorMap* map, const void* base, int rows, int cols, int ld, int box_cols, int box_rows, int swizzle_bytes);
// pair = 1: the CTA-pair (cta_group::2) form for the large layers, a 256 x BN tile per 2-CTA cluster (gemm_tc.cu).
int tc_gemm_make_plan(TcGemmPlan* plan, const GemmDesc& d, int num_sms, int pair);
cudaError_t tc_gemm_launch(const TcGemmPlan& plan, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------
// Fused tail of the encoder MLP pyramid (mlp_tail.cu): x += act(W2 act(W1 act(W0 A + b0) + b1) + b2) in place on the
// f32 residual stream x, optionally followed by LayerNorm -> bf16 (the next block's first LayerNorm).
// ------------------------------------------------------------------------------------------------
struct MlpTailDesc {
    const void* A = nullptr; int lda = 0;      // bf16 [M, K[0]]
    int M = 0;
    int N[3] = {0, 0, 0}, K[3] = {0, 0, 0};
    const void* W[3] = {nullptr, nullptr, nullptr}; int ldw[3] = {0, 0, 0};     // bf16 [N, K], K contiguous
    const float* bias[3] = {nullptr, nullptr, nullptr};
    float* x = nullptr; int ldx = 0;           // f32 [M, ldx]: residual in, result out
    const float* ln_gamma = nullptr; const float* ln_beta = nullptr; float ln_eps = 1e-3f;
    void* ln_out = nullptr; int ln_ld = 0;     // bf16 [M, ln_ld] or null
    int act = 0;
};
struct MlpTailPlan {
    CUtensorMap tmA, tmW[3];
    MlpTailDesc desc;
    int npad[3], kb[3];
    uint32_t off_w[3], off_act[2];
    size_t smem_bytes = 0;
    int num_tiles = 0, grid = 0;
    bool valid = false;
};
bool mlp_tail_supported(const int N[3], const int K[3]);
int mlp_tail_make_plan(MlpTailPlan* plan, const MlpTailDesc& d, int num_sms);
cudaError_t mlp_tail_launch(const MlpTailPlan& plan, cudaStream_t stream);

// f32 CUDA-core GEMM with the same epilogue (the fp32 parity mode); A, W, out are f32.
// Requires lda, ldw multiples of 4 and zero padding of A and W in columns [K, round_up(K,4)).
cudaError_t simt_gemm_launch(const GemmDesc& d, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------
// Attention.  qkv: [B*T, ldq] with q of head h at columns [h*hp, h*hp+d), k at [(H+h)*hp, ...),
// v at [(2H+h)*hp, ...); ctx: [B*T, H*hp] (columns d..hp-1 of every head written as zero).
// ------------------------------------------------------------------------------------------------
struct AttnDesc {
    const void* qkv = nullptr;
    int ldq = 0;
    void* ctx = nullptr;
    int ldo = 0;
    int B = 0, T = 0, H = 0, d = 0, hp = 0;
    float scale = 1.f;          // 1/sqrt(key_dim), applied to q·k (Keras scales q after its bias)
};
struct AttnPlan {
    CUtensorMap tmQKV;
    AttnDesc desc;
};
int attn_bf16_make_plan(AttnPlan* plan, const AttnDesc& d);
cudaError_t attn_tc_launch(const AttnPlan& plan, cudaStream_t stream);     // tcgen05 kernel, one softmax thread per query row (attention_tc.cu)
cudaError_t attn_f32_launch(const AttnDesc& d, cudaStream_t stream);
// fp32-accumulate mode on the tensor cores (attention_tc.cu, split form): plan.desc.qkv / ctx are the hi planes, tm_lo the tensor map
// of the lo plane of qkv (same shape and pitch), ctx_lo the lo plane of the context rows.
cudaError_t attn_tcs_launch(const AttnPlan& plan, const CUtensorMap& tm_lo, void* ctx_lo, cudaStream_t stream);

// ------------------------------------------------------------------------------------------------
// Memory-bound row kernels
// ------------------------------------------------------------------------------------------------
// tf.image.extract_patches(sizes=strides=p, padding='SAME') + Reshape (det.py:195-197, 279-280).
// images f32 NHWC [B,H,W,3] -> patches [B*gh*gw, ldp]: element r*rp + c*3 + ch (rp >= 3p = run pitch of one
// patch row; rp = 3p is the reference's dense vector), zero padded.
cudaError_t patchify_launch(const void* images, int in_u8 /*1: uint8 pixels, normalised x/127.5-1 on the fly*/, int B, int H, int W, int p,
                            void* patches, int ldp, int rp, int out_f32, cudaStream_t stream);

// One uint8 HWC source image of a ragged batch and how tf.image.resize_with_pad maps it onto the model's input
// (vision_transformer_utilities.py:435-447): resized to rh x rw, placed at (ph, pw) between bars.
struct LetterboxImage {
    const uint8_t* pixels;     // [h, w, 3], dense rows
    int h, w;
    int rh, rw, ph, pw;        // resize_with_pad_geometry
    float hscale, wscale;      // h / rh, w / rw in float32
    // boxes_original goes to a file_h x file_w image of which this one is a reduced decode (a JPEG decoded at 1 / ratio):
    // the box on this image, clipped, times file_h / h (file_w / w) in float32, clipped to the file's size.  Exactly 1
    // and the image's own size otherwise, where the second step changes nothing.
    int file_h, file_w;
    float file_hscale, file_wscale;
};
// Fills *im for an h x w image letterboxed to th x tw (file size = image size); false when a size is not positive or the
// resized image is empty.
bool letterbox_image(const uint8_t* pixels, int h, int w, int th, int tw, LetterboxImage* im);
// patchify of the letterboxed, normalised images without the float32 images: images is a DEVICE table of B entries,
// the output the same patch matrix as patchify_launch's (vector layout only: rp and ldp multiples of 4, 16-byte aligned).
cudaError_t letterbox_patchify_launch(const LetterboxImage* images, int B, int H, int W, int p, void* patches, int ldp, int rp,
                                      int out_f32, cudaStream_t stream);

// keras LayerNormalization(axis=-1), eps=1e-3, biased variance (det.py:353-357, 375-379).
cudaError_t layernorm_launch(const float* x, int ldx, const float* gamma, const float* beta, int M, int D,
                             float eps, void* y, int ldy, int out_f32, cudaStream_t stream);

// mlp_head first stage (det.py:454-463): Dense(D -> S) on every token of M / tokens images, stored as the slot matrix
// [images*S, ldo] (ldo >= tokens; ldo == tokens is the compact [B, T*S] buffer whose row-major view IS the reference's
// Reshape((S,-1))).
cudaError_t head_slots_launch(const float* x, int ldx, const float* w /*[S, D] f32*/, const float* bias,
                              int M, int D, int S, int tokens, int ldo, void* out, int out_f32, cudaStream_t stream);

// Final Dense(U -> 6) 'MLP_Head_no_Sigmoid' (det.py:489-493) fused with transform_predictions
// (det.py:586-647) and the 0.5/0.5 thresholds (det.py:2257-2283 / 1359-1384).
struct DecodeParams {
    float obj_thr = 0.5f, cls_thr = 0.5f;
    int strict = 1;             // 1: keep iff score >  thr (metric copy); 0: keep iff score >= thr (visualise copy)
    float img_h = 608.f, img_w = 608.f;
    int classes = 80;
    int apply_transform = 1;    // 0: rows are already transform_predictions output (det.py:1340-1341)
    float corner_scale = 1.f;   // enlarged_image_scale (det.py:2294-2297)
};
struct DecodeOut {
    float* logits = nullptr;    // [R, 6] raw (optional when decoding given logits)
    float* decoded = nullptr;   // [R, 6] conf, class in [0, classes-1], cx, cy, h, w (pixels)
    int32_t* class_id = nullptr;  // [R] round-half-even(class)
    float* class_conf = nullptr;  // [R] (0.5 - |class - id|) / 0.5
    uint8_t* keep = nullptr;    // [R]
    int32_t* corners = nullptr; // [R, 4] x0, y0, x1, y1 (int truncation then clip; det.py:2300-2325), optional
    float* packed = nullptr;    // [R, 13] decoded[6] | class id | class confidence | keep | corners[4], all as float32 (the gather record)
    // [R, 4] x0, y0, x1, y1 on the source image of row r, letterbox[r / slots] (letterboxed input only), optional
    float* boxes_original = nullptr;
    const LetterboxImage* letterbox = nullptr;
    int slots = 0;
};
cudaError_t head_tail_launch(const void* h, int ldh, int in_f32, const float* w /*[6, U] f32*/, const float* bias,
                             int R, int U, const DecodeParams& dp, const DecodeOut& out, cudaStream_t stream);
cudaError_t decode_launch(const float* logits, int R, const DecodeParams& dp, const DecodeOut& out,
                          cudaStream_t stream);
// Input side (vision_transformer_utilities.py:435-447): uint8 [h, w, 3] -> resize_with_pad(th, tw) -> clip -> /127.5 - 1, f32 [th, tw, 3].
void resize_with_pad_geometry(int h, int w, int th, int tw, int* rh, int* rw, int* ph, int* pw);
cudaError_t preprocess_launch(const uint8_t* image, int h, int w, float* out, int th, int tw, cudaStream_t stream);
// iou_calculator (det.py:761-875): element-wise IoU of (cx, cy, h, w) boxes in the last four entries of `width`-wide rows.
cudaError_t iou_launch(const float* label, const float* pred, long long R, int width, float eps, float* iou,
                       cudaStream_t stream);

// Records the message vitdet_last_error() returns on the calling thread and hands `code` back (engine.cu).
int fail(int code, const char* fmt, ...);

// ------------------------------------------------------------------------------------------------
// Baseline JPEG decode (jpeg.cu), bit-exact with libjpeg-turbo's defaults (ISLOW IDCT, fancy upsampling, jdcolor.c).
// The host parses the headers and cuts the entropy data at RSTn into segments; the device de-stuffs every segment,
// Huffman-decodes it in subsequences of kJpegSubBits bits (speculative pass, kJpegSyncPasses parallel sync passes, one-warp-per-segment
// repair, write pass),
// adds up the DC differences, and runs IDCT, upsampling and colour conversion into dense uint8 (h, w, 3) RGB.
// ------------------------------------------------------------------------------------------------
constexpr int kJpegSubBits = 1024;     // L, a multiple of 32: one checkpoint per 32-bit word
constexpr int kJpegSyncPasses = 8;     // parallel sync passes ahead of the one-warp-per-segment repair
constexpr int kJpegLaunches = 7 + kJpegSyncPasses;     // kernels of one jpeg_decode, whatever the data
// Host header check: 0 and the size and component count, or VITDET_E_INVALID with the reason in why.
int jpeg_info(const uint8_t* data, int64_t bytes, int* height, int* width, int* components, char* why, size_t why_len);
// The device work of a batch of files, planned on the host.  work_bytes of device scratch hold, at these offsets: the
// descriptor block `desc` (images, segments, Huffman tables; copied there by the caller), the compact bit streams, the
// coefficients, the subsequence states, the component planes and three counters (int64: subsequences, subsequences the
// sync passes and the repair re-decoded, symbols they re-decoded).
struct JpegBatch {
    int B = 0, nseg = 0, nsub = 0;
    long long nblocks = 0, npix = 0;
    std::vector<char> desc;
    std::vector<int> height, width;    // of the decoded images: ceil(file size / ratio)
    std::vector<int> file_height, file_width, ratio;
    std::vector<size_t> file_off;      // B + 1: file i is bytes [file_off[i], file_off[i + 1]) of the concatenated files
    std::vector<size_t> rgb_off;       // where image i's pixels go, relative to the output pointer of jpeg_decode
    size_t rgb_bytes = 0;              // with the default layout (out_offsets null): the output's size
    size_t o_compact = 0, o_coef = 0, o_spec = 0, o_check = 0, o_sync = 0, o_start = 0, o_planes = 0, o_stats = 0, work_bytes = 0;
};
// Parses B files (HOST bytes); out_offsets (may be null: images packed 256-byte aligned) place the outputs.  ratios (may be
// null: all 1) decode file i at 1 / ratios[i] scale in the DCT domain (1, 2, 4 or 8; 0: jpeg_auto_ratio for the target
// size).  Fails with VITDET_E_INVALID naming the first file with an invalid ratio, else the first rejected file.
int jpeg_plan(const char* fn, const uint8_t* const* data, const int64_t* bytes, int B, const int32_t* ratios, int target_h,
              int target_w, const int64_t* out_offsets, JpegBatch* b);
// The ratio PIL's draft() picks for an h x w file letterboxed to th x tw: the largest of 8, 4, 2, 1 at most
// min(w / rw, h / rh) for the resized size (rh, rw) of resize_with_pad_geometry; 1 when that size is empty.
int jpeg_auto_ratio(int h, int w, int th, int tw);
// Launches the kJpegLaunches kernels: files_dev holds the concatenated files, work the scratch with b.desc at offset 0.
cudaError_t jpeg_decode_launch(const JpegBatch& b, const char* files_dev, void* work, uint8_t* out, cudaStream_t stream);

}  // namespace vitdet
