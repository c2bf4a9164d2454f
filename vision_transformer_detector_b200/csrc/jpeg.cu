// Baseline JPEG decode on the GPU, bit-exact with libjpeg-turbo's defaults: what PIL's Image.open(f).convert("RGB") and
// tf.image.decode_jpeg return (vision_transformer_utilities.py:418-449).  oracle/jpeg_oracle.py states every stage in numpy.
//
// Host: header parse (SOI, APPn, DQT, DHT, SOF0/1, DRI, SOS, EOI) and the cut of the entropy data at RSTn into segments,
// one descriptor block per batch.  Device, kJpegLaunches kernels whatever the data:
//   1 destuff  one CTA per segment: a run of FF followed by 00 becomes one FF in a compact bit stream; zeroes the
//              segment's blocks
//   2 spec     one thread per subsequence of L = kJpegSubBits bits: decodes from the subsequence's first bit with
//              u = k = 0, keeps its exit state, its block count and a checkpoint at the first symbol boundary at or past
//              every 32-bit word (Weissenberger & Schmidt, Massively Parallel Huffman Decoding on GPUs, ICPP 2018)
//   3 sync     kJpegSyncPasses passes, one thread per subsequence: pass p re-decodes subsequence j from pass p - 1's
//              exit of j - 1 (pass 0 = the speculative pass) until a checkpoint of its speculative run agrees, after
//              which the speculative result holds; a start that pass p - 1 already used keeps its result.  After p passes
//              every subsequence within p hops of one whose speculative run synchronised is exact
//   4 repair   one warp per segment, 32 subsequences at a time: a lane whose start (its left neighbour's exit) is not the
//              one the last pass used re-decodes as above; rounds until no start changes (at most 33), then the block
//              counts are scanned.  Most lanes take the last pass's result without decoding
//   5 write    one thread per subsequence: decodes from its agreed start, writes int16 coefficients (DC as differences)
//   6 dc       one CTA per segment: the DC values, a prefix of the differences per component, reset at every segment
//   7 idct     one thread per block: dequantisation, jidctint.c ISLOW, jdmaster.c's range-limit table -> component planes
//   8 colour   one thread per pixel: jdsample.c fancy upsampling and jdcolor.c ycc_rgb_convert -> (h, w, 3) uint8
// A file may be decoded at 1/2, 1/4 or 1/8 scale in the DCT domain (libjpeg's scale_denom, what PIL's draft() and
// tf.image.decode_jpeg(ratio=) ask for), mixed freely within a batch and in the same launches.  The output is then
// ceil(h / ratio) x ceil(w / ratio).  Each component gets its own DCT scaled size as jdmaster.c sets it: the luma's
// k = 8 / ratio, doubled while both sampling ratios allow, so 4:2:0 chroma keeps 8 x 8 blocks at ratio 2 and is not
// upsampled.  The idct kernel writes 8 x 8 (ISLOW), 4 x 4, 2 x 2 or 1 x 1 (jidctred.c) blocks.  A block whose IDCT is
// 1 x 1 reads its DC alone, so the write and DC kernels store one coefficient for it instead of 64.  The Huffman decode
// is the same at every scale.  The colour kernel upsamples by each component's own expansion factors, fancily only
// where the luma's scaled size is above 1 (jinit_upsampler).  oracle/jpeg_scaled_oracle.py states the reduced decode.
// The state at a symbol boundary is (bit offset, block index u within the MCU, coefficient index k); the exact start of
// subsequence j + 1 is the exit of subsequence j decoded from its exact start, so the result equals a sequential decode by
// construction.  Every decode loop ends at the end of its subsequence (each symbol consumes at least one bit); corrupt data
// decodes under the oracle's clamps: an invalid code is symbol 0 of 16 bits, bits past the end read 0, a run past k = 63
// writes coefficient 63, blocks past a segment's MCU count are dropped and missing ones stay zero.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cub/block/block_scan.cuh>

#include "../../include/vitdet_b200.h"
#include "kernels.h"

namespace vitdet {
namespace {

constexpr int kWordsPerSub = kJpegSubBits / 32;
// Entropy-coded bytes of one restart segment at most: its bit positions, int32 on the device, stay below 2^31 - 8192 (longer
// segments are rejected by the header parse)
constexpr int64_t kMaxSegmentBytes = (int64_t(1) << 28) - 1024;
static_assert(kJpegSubBits % 32 == 0, "one checkpoint per 32-bit word");

__device__ __constant__ uint8_t kNatural[64] = {
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21,
    28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54,
    47, 55, 62, 63};
const uint8_t kNaturalHost[64] = {
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21,
    28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54,
    47, 55, 62, 63};

// A Huffman table in libjpeg's derived form (jdhuff.c): a 9-bit lookahead (code length << 8 | symbol, 0 for longer
// codes), maxcode / valoffset per length, the symbols.
struct JpegHuff {
    uint16_t lut[512];
    int32_t maxcode[18];
    int32_t valoff[18];
    uint8_t vals[256];
};

enum : int { kSpaceYcc = 0, kSpaceRgb = 1, kSpaceGray = 2 };

struct JpegImage {
    int32_t h, w, ncomp, space;      // h, w: the output's size, ceil(file size / ratio)
    int32_t hs[3], vs[3], hmax, vmax, mcux, mcuy;
    int32_t bpm;                     // blocks per MCU
    int8_t blk_c[8], blk_x[8], blk_y[8];   // per block of an MCU: component, column and row in its MCU cell
    int16_t blk_coef[8];             // per block of an MCU: its first coefficient relative to the MCU's
    // coefficients stored per MCU: 64 per block (starting at a multiple of 8: read as 16-byte words), 1 per block whose
    // IDCT reads the DC alone; a multiple of 8 when the MCU holds a 64-coefficient block
    int32_t mcu_coefs;
    int32_t dc[3], ac[3];            // Huffman tables of each component (indices into the batch's table array)
    // per component at the decode's scale (jdmaster.c jpeg_core_output_dimensions): DCT scaled size (8, 4, 2 or 1), plane
    // pitch (mcux * hs * size), scaled width and height, expansion factors to the output (1 or 2; jdsample.c)
    int32_t ks[3], pitch[3], dw[3], dh[3], he[3], ve[3];
    int32_t fancy;                   // jdsample.c fancy upsampling allowed: the luma's scaled size is above 1
    int64_t block0;                  // first coefficient block of the image
    int64_t coef0;                   // first coefficient of the image (a multiple of 8)
    int64_t plane[3];                // byte offset of each component plane
    int64_t out;                     // byte offset of the image's pixels in the output
    int64_t pix0;                    // first pixel of the image in the batch
    uint16_t q[3][64];               // quantisation tables, natural order
};

struct JpegSegment {
    int64_t src;                     // first byte in the concatenated files
    int64_t dst;                     // first byte of its compact stream (8-byte aligned)
    int64_t coef0;                   // first coefficient (its first MCU's)
    int32_t src_len, nbits, nblocks, sub0, image, pad;
};

struct JpegBatchDev {                // the descriptor block's layout
    const JpegImage* img;
    const JpegSegment* seg;
    const JpegHuff* tab;
    int B, nseg, nsub;
};

// ------------------------------------------------------------------------------------------------
// host parse
// ------------------------------------------------------------------------------------------------
struct Parsed {
    int h = 0, w = 0, ncomp = 0, space = kSpaceYcc, ri = 0;
    int hs[3] = {1, 1, 1}, vs[3] = {1, 1, 1}, qid[3] = {0, 0, 0}, cid[3] = {0, 0, 0};
    int td[3] = {0, 0, 0}, ta[3] = {0, 0, 0};
    uint16_t q[4][64];
    bool has_q[4] = {false, false, false, false};
    JpegHuff huff[2][4];
    bool has_huff[2][4] = {{false, false, false, false}, {false, false, false, false}};
    std::vector<int64_t> seg_a, seg_b, seg_stuff;      // byte ranges of the segments in the file, FF00 pairs in each
};

struct Reject {
    char* why; size_t n;
    int operator()(const char* fmt, ...) const {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(why, n, fmt, ap);
        va_end(ap);
        return VITDET_E_INVALID;
    }
};

static bool make_huff(const uint8_t* counts, const uint8_t* syms, int total, bool dc, JpegHuff* t) {
    memset(t, 0, sizeof(*t));
    int code = 0, p = 0;
    for (int l = 0; l < 18; ++l) t->maxcode[l] = -1;
    for (int l = 1; l <= 16; ++l) {
        const int n = counts[l - 1];
        if (n) {
            t->valoff[l] = p - code;
            code += n;
            p += n;
            if (code >= (1 << l)) return false;          // no code may be all ones (jpeg_make_d_derived_tbl)
            t->maxcode[l] = code - 1;
        }
        code <<= 1;
    }
    t->maxcode[17] = 0x7FFFFFFF;
    for (int i = 0; i < total; ++i) {
        if (dc && syms[i] > 15) return false;
        t->vals[i] = syms[i];
    }
    for (int look = 0; look < 512; ++look)
        for (int l = 1; l <= 9; ++l) {
            const int c = look >> (9 - l);
            if (c <= t->maxcode[l]) { t->lut[look] = static_cast<uint16_t>(l << 8 | t->vals[(c + t->valoff[l]) & 255]); break; }
        }
    return true;
}

static int parse(const uint8_t* d, int64_t n, Parsed* P, bool segments, const Reject& rej) {
    if (!d || n < 4 || d[0] != 0xFF || d[1] != 0xD8) return rej("not a JPEG file (no SOI)");
    int64_t p = 2;
    bool frame = false, jfif = false, adobe = false;
    int transform = -1;
    const uint8_t* seg = nullptr;
    int64_t sl = 0;
    for (;;) {
        if (p >= n) return rej("truncated before the scan");
        if (d[p] != 0xFF) return rej("expected a marker at byte %lld", static_cast<long long>(p));
        while (p < n && d[p] == 0xFF) ++p;
        if (p >= n) return rej("truncated before the scan");
        const int m = d[p++];
        if (m == 0xD9) return rej("EOI before any scan");
        if (m == 0xD8 || m == 0x01 || (m >= 0xD0 && m <= 0xD7)) return rej("unexpected marker 0x%02X", m);
        if (p + 2 > n) return rej("truncated before the scan");
        const int ln = d[p] << 8 | d[p + 1];
        if (ln < 2 || p + ln > n) return rej("truncated before the scan");
        seg = d + p + 2;
        sl = ln - 2;
        p += ln;
        if (m == 0xE0) {
            if (sl >= 14 && memcmp(seg, "JFIF\0", 5) == 0) jfif = true;
        } else if (m == 0xEE) {
            if (sl >= 12 && memcmp(seg, "Adobe", 5) == 0) { adobe = true; transform = seg[11]; }
        } else if (m == 0xDB) {
            for (int64_t i = 0; i < sl;) {
                const int pq = seg[i] >> 4, tq = seg[i] & 15;
                if (pq > 1 || tq > 3) return rej("bad quantisation table");
                const int sz = 64 * (pq + 1);
                if (i + 1 + sz > sl) return rej("truncated quantisation table");
                for (int z = 0; z < 64; ++z)
                    P->q[tq][kNaturalHost[z]] = pq ? static_cast<uint16_t>(seg[i + 1 + 2 * z] << 8 | seg[i + 2 + 2 * z]) : seg[i + 1 + z];
                P->has_q[tq] = true;
                i += 1 + sz;
            }
        } else if (m == 0xC4) {
            for (int64_t i = 0; i < sl;) {
                if (i + 17 > sl) return rej("truncated Huffman table");
                const int tc = seg[i] >> 4, th = seg[i] & 15;
                if (tc > 1 || th > 3) return rej("bad Huffman table class or id");
                int total = 0;
                for (int l = 0; l < 16; ++l) total += seg[i + 1 + l];
                if (total > 256) return rej("bad Huffman table: more than 256 symbols");
                if (i + 17 + total > sl) return rej("truncated Huffman table");
                if (!make_huff(seg + i + 1, seg + i + 17, total, tc == 0, &P->huff[tc][th])) return rej("bad Huffman table");
                P->has_huff[tc][th] = true;
                i += 17 + total;
            }
        } else if (m == 0xC0 || m == 0xC1) {
            if (frame) return rej("more than one frame header");
            if (sl < 6) return rej("truncated frame header");
            if (seg[0] != 8) return rej("%d-bit precision (only 8-bit is supported)", seg[0]);
            P->h = seg[1] << 8 | seg[2];
            P->w = seg[3] << 8 | seg[4];
            P->ncomp = seg[5];
            if (P->ncomp != 1 && P->ncomp != 3) return rej("%d components (only 1 or 3 are supported)", P->ncomp);
            if (sl < 6 + 3 * P->ncomp) return rej("truncated frame header");
            for (int c = 0; c < P->ncomp; ++c) {
                P->cid[c] = seg[6 + 3 * c];
                P->hs[c] = seg[7 + 3 * c] >> 4;
                P->vs[c] = seg[7 + 3 * c] & 15;
                P->qid[c] = seg[8 + 3 * c] & 3;
                if (seg[8 + 3 * c] > 3) return rej("bad quantisation table id");
            }
            if (P->h == 0) return rej("height defined by DNL (not supported)");
            if (P->w == 0) return rej("zero width");
            frame = true;
        } else if (m == 0xC2 || m == 0xC6 || m == 0xCA || m == 0xCE) {
            return rej("progressive JPEG (not supported)");
        } else if (m == 0xC3 || m == 0xC7 || m == 0xCB || m == 0xCF) {
            return rej("lossless JPEG (not supported)");
        } else if (m == 0xC5 || m == 0xC9 || m == 0xCC || m == 0xCD) {
            return rej("arithmetic-coded or hierarchical JPEG (not supported)");
        } else if (m == 0xDD) {
            if (sl < 2) return rej("truncated DRI");
            P->ri = seg[0] << 8 | seg[1];
        } else if (m == 0xDC) {
            return rej("DNL marker (not supported)");
        } else if (m == 0xDA) {
            if (!frame) return rej("scan before the frame header");
            break;
        }
    }
    const int ns = sl > 0 ? seg[0] : 0;
    if (sl < 1 + 2 * ns + 3) return rej("truncated scan header");
    if (ns != P->ncomp) return rej("scan does not hold every component (several scans are not supported)");
    for (int i = 0; i < ns; ++i) {
        if (seg[1 + 2 * i] != P->cid[i]) return rej("scan components are not in frame order");
        P->td[i] = seg[2 + 2 * i] >> 4;
        P->ta[i] = seg[2 + 2 * i] & 15;
    }
    if (seg[1 + 2 * ns] != 0 || seg[2 + 2 * ns] != 63 || seg[3 + 2 * ns] != 0) return rej("not a sequential scan");
    if (P->ncomp == 1) {
        P->hs[0] = P->vs[0] = 1;
    } else {
        const bool luma = (P->hs[0] == 1 && P->vs[0] == 1) || (P->hs[0] == 2 && P->vs[0] == 1) || (P->hs[0] == 2 && P->vs[0] == 2);
        if (!luma || P->hs[1] != 1 || P->vs[1] != 1 || P->hs[2] != 1 || P->vs[2] != 1)
            return rej("unsupported sampling factors %dx%d,%dx%d,%dx%d", P->hs[0], P->vs[0], P->hs[1], P->vs[1], P->hs[2], P->vs[2]);
    }
    for (int c = 0; c < ns; ++c) {
        if (P->td[c] > 3 || P->ta[c] > 3 || !P->has_huff[0][P->td[c]] || !P->has_huff[1][P->ta[c]])
            return rej("component %d: Huffman table referenced but never defined", c);
        if (!P->has_q[P->qid[c]]) return rej("component %d: quantisation table referenced but never defined", c);
    }
    if (P->ncomp == 1) P->space = kSpaceGray;
    else if (jfif) P->space = kSpaceYcc;
    else if (adobe) P->space = transform == 0 ? kSpaceRgb : kSpaceYcc;
    else if (P->cid[0] == 82 && P->cid[1] == 71 && P->cid[2] == 66) P->space = kSpaceRgb;
    else P->space = kSpaceYcc;
    // entropy data up to EOI, cut at RSTn.  Inside the data a run of FF followed by 00 is one FF byte (jdhuff.c
    // jpeg_fill_bit_buffer skips fill bytes); a run of FF followed by anything else is a marker.
    int64_t start = p, stuff = 0;
    for (;;) {
        const uint8_t* f = static_cast<const uint8_t*>(memchr(d + p, 0xFF, static_cast<size_t>(n - p)));
        const int64_t e = f ? f - d : n;
        int64_t q = e;
        while (q + 1 < n && d[q + 1] == 0xFF) ++q;
        if (q + 1 >= n) return rej("truncated inside the entropy-coded data (no EOI)");
        const int mk = d[q + 1];
        if (mk == 0x00) { stuff += q - e + 1; p = q + 2; continue; }
        if (e - start > kMaxSegmentBytes)
            return rej("a restart segment holds %lld bytes of entropy-coded data (at most %lld)", static_cast<long long>(e - start),
                       static_cast<long long>(kMaxSegmentBytes));
        if (segments) { P->seg_a.push_back(start); P->seg_b.push_back(e); P->seg_stuff.push_back(stuff); }
        p = q + 2;
        stuff = 0;
        if (mk >= 0xD0 && mk <= 0xD7) { start = p; continue; }
        if (mk == 0xD9) break;
        if (mk == 0xDC) return rej("DNL marker (not supported)");
        if (mk == 0xDA || (mk >= 0xC0 && mk <= 0xCF) || mk == 0xDB || mk == 0xDD) return rej("several scans (not supported)");
        return rej("unexpected marker 0x%02X after the scan", mk);
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------
// device: bit reader and one symbol
// ------------------------------------------------------------------------------------------------
struct Stream {
    const uint32_t* w;
    int nwords;
    int nbits;
};

__device__ __forceinline__ uint32_t word_at(const Stream& s, int i) {
    return i < s.nwords ? __byte_perm(__ldg(s.w + i), 0, 0x0123) : 0u;
}

// 32 bits at pos, MSB first; bits past the end are 0 (the compact stream is zero-padded to its last word)
__device__ __forceinline__ uint32_t peek32(const Stream& s, int pos) {
    const int i = pos >> 5, sh = pos & 31;
    const uint32_t a = word_at(s, i);
    return sh ? (a << sh) | (word_at(s, i + 1) >> (32 - sh)) : a;
}

__device__ __forceinline__ int huff_decode(const JpegHuff* __restrict__ t, uint32_t look, int* len) {
    const uint16_t e = __ldg(t->lut + (look >> 23));
    if (e >> 8) { *len = e >> 8; return e & 255; }
    for (int l = 10; l <= 16; ++l) {
        const int code = static_cast<int>(look >> (32 - l));
        if (code <= __ldg(t->maxcode + l)) { *len = l; return __ldg(t->vals + ((code + __ldg(t->valoff + l)) & 255)); }
    }
    *len = 16;                       // an invalid code: symbol 0, 16 bits
    return 0;
}

__device__ __forceinline__ int extend(uint32_t r, int s) {
    return s && r < (1u << (s - 1)) ? static_cast<int>(r) - (1 << s) + 1 : static_cast<int>(r);
}

struct DecState { int pos, u, k; };

// One symbol from st.  Returns whether it completed a block; *idx / *val the coefficient it writes (idx < 0: none).
__device__ __forceinline__ bool step(const JpegImage& im, const JpegHuff* tabs, const Stream& s, DecState& st, int* idx, int* val) {
    const int c = im.blk_c[st.u];
    const uint32_t look = peek32(s, st.pos);
    int l;
    if (st.k == 0) {
        const int sz = huff_decode(tabs + im.dc[c], look, &l);
        const uint32_t r = sz ? (look << l) >> (32 - sz) : 0u;
        st.pos += l + sz;
        *idx = 0;
        *val = extend(r, sz);
        st.k = 1;
    } else {
        const int rs = huff_decode(tabs + im.ac[c], look, &l);
        const int r = rs >> 4, sz = rs & 15;
        *idx = -1;
        if (sz) {
            st.k += r;
            *idx = kNatural[min(st.k, 63)];
            *val = extend((look << l) >> (32 - sz), sz);
            st.k += 1;
        } else if (r == 15) {
            st.k += 16;
        } else {
            st.k = 64;
        }
        st.pos += l + sz;
    }
    if (st.k >= 64) {
        st.u = st.u + 1 == im.bpm ? 0 : st.u + 1;
        st.k = 0;
        return true;
    }
    return false;
}

__device__ __forceinline__ int pack_state(int u, int k, int blocks) { return u | k << 4 | blocks << 12; }

__device__ __forceinline__ int find_segment(const JpegSegment* seg, int nseg, int g) {
    int lo = 0, hi = nseg - 1;                 // the last segment whose sub0 <= g
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (seg[mid].sub0 <= g) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__device__ __forceinline__ Stream stream_of(const JpegSegment& sg, const char* compact) {
    Stream s;
    s.w = reinterpret_cast<const uint32_t*>(compact + sg.dst);
    s.nbits = sg.nbits;
    s.nwords = (sg.nbits + 31) >> 5;
    return s;
}

// ------------------------------------------------------------------------------------------------
// 1 destuff
// ------------------------------------------------------------------------------------------------
constexpr int kDestuffThreads = 256;

__global__ void __launch_bounds__(kDestuffThreads) jpeg_destuff_kernel(JpegBatchDev b, const uint8_t* __restrict__ files,
                                                                       char* compact, int16_t* coef, long long* stats) {
    using Scan = cub::BlockScan<int, kDestuffThreads>;
    __shared__ typename Scan::TempStorage tmp;
    __shared__ int carry;
    if (blockIdx.x == 0 && threadIdx.x < 3) stats[threadIdx.x] = threadIdx.x == 0 ? b.nsub : 0;
    for (int si = blockIdx.x; si < b.nseg; si += gridDim.x) {
        const JpegSegment sg = b.seg[si];
        const JpegImage& im = b.img[sg.image];
        const int64_t ncoef = static_cast<int64_t>(sg.nblocks / im.bpm) * im.mcu_coefs;
        if (((sg.coef0 | ncoef) & 7) == 0) {
            int4* z = reinterpret_cast<int4*>(coef + sg.coef0);
            for (int64_t i = threadIdx.x; i < ncoef / 8; i += kDestuffThreads) z[i] = make_int4(0, 0, 0, 0);
        } else {                     // DC-only blocks: a segment's coefficients need not fill whole 16-byte words
            for (int64_t i = threadIdx.x; i < ncoef; i += kDestuffThreads) coef[sg.coef0 + i] = 0;
        }
        const uint8_t* src = files + sg.src;
        uint8_t* dst = reinterpret_cast<uint8_t*>(compact + sg.dst);
        if (threadIdx.x == 0) carry = 0;
        __syncthreads();
        for (int base = 0; base < sg.src_len; base += kDestuffThreads * 4) {
            uint8_t v[4];
            int keep = 0;
            const int i0 = base + threadIdx.x * 4;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int i = i0 + t;
                v[t] = i < sg.src_len ? src[i] : 0;
                // a run of FF followed by 00 is one FF: keep its last FF only (a segment never ends inside such a run)
                const bool kept = i < sg.src_len && !(i > 0 && v[t] == 0 && src[i - 1] == 0xFF) &&
                                  !(v[t] == 0xFF && i + 1 < sg.src_len && src[i + 1] == 0xFF);
                keep |= kept << t;
            }
            int off;
            Scan(tmp).ExclusiveSum(__popc(keep), off);
            const int c0 = carry;
            off += c0;
#pragma unroll
            for (int t = 0; t < 4; ++t)
                if ((keep >> t) & 1) dst[off++] = v[t];
            __syncthreads();
            if (threadIdx.x == kDestuffThreads - 1) carry = off;
            __syncthreads();
        }
        // zero padding to the 8-byte aligned end: the bit reader reads whole words
        const int nbytes = sg.nbits >> 3;
        for (int i = nbytes + threadIdx.x; i < ((nbytes + 7) & ~7); i += kDestuffThreads) dst[i] = 0;
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// 2 speculative pass
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) jpeg_spec_kernel(JpegBatchDev b, const char* __restrict__ compact, int2* spec_exit, int2* checks) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= b.nsub) return;
    const JpegSegment& sg = b.seg[find_segment(b.seg, b.nseg, g)];
    const JpegImage& im = b.img[sg.image];
    const Stream s = stream_of(sg, compact);
    const int j = g - sg.sub0;
    const int lo = j * kJpegSubBits, hi = lo + kJpegSubBits, end = min(hi, sg.nbits);
    DecState st{lo, 0, 0};
    int blocks = 0, c = 0, idx, val;
    int2* cp = checks + static_cast<int64_t>(g) * kWordsPerSub;
    while (st.pos < end) {
        blocks += step(im, b.tab, s, st, &idx, &val);
        for (; c < kWordsPerSub && lo + 32 * (c + 1) <= st.pos; ++c) cp[c] = make_int2(st.pos, pack_state(st.u, st.k, blocks));
    }
    for (; c < kWordsPerSub; ++c) cp[c] = make_int2(-1, 0);
    spec_exit[g] = make_int2(st.pos, pack_state(st.u, st.k, blocks));
}

__device__ __forceinline__ DecState unpack_state(int2 e) { return DecState{e.x, e.y & 15, (e.y >> 4) & 255}; }

// Subsequence j (global index g) of a segment decoded from `start`: the exit and (*blocks) the blocks it completes.  From
// the speculative start the speculative result is returned; otherwise decoding stops at the first checkpoint that agrees
// with the speculative run and completes the result from it.  *symbols counts the symbols decoded.
__device__ __forceinline__ DecState redecode(const JpegImage& im, const JpegHuff* tabs, const Stream& s, int g, int j, DecState start,
                             const int2* __restrict__ spec_exit, const int2* __restrict__ checks, int* blocks, unsigned* symbols) {
    const int lo = j * kJpegSubBits, hi = lo + kJpegSubBits, end = min(hi, s.nbits);
    const int2 se = spec_exit[g];
    if (start.pos == lo && start.u == 0 && start.k == 0) { *blocks = se.y >> 12; return unpack_state(se); }
    const int2* cp = checks + static_cast<int64_t>(g) * kWordsPerSub;
    DecState st = start;
    int nb = 0, idx, val, nextb = (st.pos >> 5) * 32 + 32;
    while (st.pos < end) {
        nb += step(im, tabs, s, st, &idx, &val);
        ++*symbols;
        for (; nextb <= st.pos && nextb <= hi; nextb += 32) {
            const int2 c = cp[(nextb - lo) / 32 - 1];
            if (c.x == st.pos && (c.y & 0xFFF) == pack_state(st.u, st.k, 0)) {
                *blocks = nb + (se.y >> 12) - (c.y >> 12);
                return unpack_state(se);
            }
        }
    }
    *blocks = nb;
    return st;
}

__device__ __forceinline__ void count_redecodes(unsigned long long* stats, unsigned redone, unsigned symbols) {
    redone = __reduce_add_sync(0xffffffffu, redone);
    symbols = __reduce_add_sync(0xffffffffu, symbols);
    if ((threadIdx.x & 31) == 0 && redone) { atomicAdd(stats + 1, redone); atomicAdd(stats + 2, symbols); }
}

// ------------------------------------------------------------------------------------------------
// 3 sync pass: out[g] = exit and blocks of subsequence g decoded from prev[g - 1] (from (0, 0, 0) for a segment's first);
// when prev[g - 1] is the start the previous pass used (prevprev[g - 1]), its result prev[g] is kept
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool same_state(int2 a, int2 b) { return a.x == b.x && (a.y & 0xFFF) == (b.y & 0xFFF); }

__global__ void __launch_bounds__(128) jpeg_sync_kernel(JpegBatchDev b, const char* __restrict__ compact, const int2* __restrict__ spec_exit,
                                                        const int2* __restrict__ checks, const int2* __restrict__ prevprev,
                                                        const int2* __restrict__ prev, int2* out, unsigned long long* stats) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned redone = 0, symbols = 0;
    if (g < b.nsub) {
        const JpegSegment& sg = b.seg[find_segment(b.seg, b.nseg, g)];
        const int j = g - sg.sub0;
        if (j > 0 && prevprev && same_state(prev[g - 1], prevprev[g - 1])) {
            out[g] = prev[g];
        } else {
            const DecState start = j == 0 ? DecState{0, 0, 0} : unpack_state(prev[g - 1]);
            redone = !(start.pos == j * kJpegSubBits && start.u == 0 && start.k == 0);
            int blocks;
            const DecState ex = redecode(b.img[sg.image], b.tab, stream_of(sg, compact), g, j, start, spec_exit, checks, &blocks, &symbols);
            out[g] = make_int2(ex.pos, pack_state(ex.u, ex.k, blocks));
        }
    }
    count_redecodes(stats, redone, symbols);
}

// ------------------------------------------------------------------------------------------------
// 4 repair: one warp per segment
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) jpeg_repair_kernel(JpegBatchDev b, const char* __restrict__ compact, const int2* __restrict__ spec_exit,
                                                          const int2* __restrict__ checks, const int2* __restrict__ guesses,
                                                          const int2* __restrict__ results, int4* starts, unsigned long long* stats) {
    const int si = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (si >= b.nseg) return;
    const JpegSegment sg = b.seg[si];
    const JpegImage& im = b.img[sg.image];
    const Stream s = stream_of(sg, compact);
    const int nsub = (sg.nbits + kJpegSubBits - 1) / kJpegSubBits;
    DecState carry{0, 0, 0};
    int base = 0;
    unsigned redone = 0, symbols = 0;
    for (int j0 = 0; j0 < nsub; j0 += 32) {
        const int j = j0 + lane;
        const bool valid = j < nsub;
        const int g = sg.sub0 + j;
        // the start the last sync pass used, and its result
        DecState guess{0, 0, 0};
        if (valid && j > 0) guess = unpack_state(guesses[g - 1]);
        DecState start = lane == 0 ? carry : guess;
        DecState ex{0, 0, 0};
        int blocks = 0;
        bool dirty = valid;
        for (int round = 0; round <= 32; ++round) {
            if (dirty) {
                if (start.pos == guess.pos && start.u == guess.u && start.k == guess.k) {
                    const int2 r = results[g];
                    ex = unpack_state(r);
                    blocks = r.y >> 12;
                } else {
                    ++redone;
                    ex = redecode(im, b.tab, s, g, j, start, spec_exit, checks, &blocks, &symbols);
                }
            }
            // the next start of every lane is its left neighbour's exit
            DecState ns;
            ns.pos = __shfl_up_sync(0xffffffffu, ex.pos, 1);
            ns.u = __shfl_up_sync(0xffffffffu, ex.u, 1);
            ns.k = __shfl_up_sync(0xffffffffu, ex.k, 1);
            const bool changed = valid && lane > 0 && (ns.pos != start.pos || ns.u != start.u || ns.k != start.k);
            if (!__any_sync(0xffffffffu, changed)) break;
            if (changed) start = ns;
            dirty = changed;
        }
        // exclusive prefix of the block counts -> each subsequence's first block in the segment
        int incl = valid ? blocks : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (valid) starts[g] = make_int4(start.pos, start.u, start.k, base + incl - blocks);
        base += __shfl_sync(0xffffffffu, incl, 31);
        const int last = min(31, nsub - 1 - j0);
        carry.pos = __shfl_sync(0xffffffffu, ex.pos, last);
        carry.u = __shfl_sync(0xffffffffu, ex.u, last);
        carry.k = __shfl_sync(0xffffffffu, ex.k, last);
    }
    count_redecodes(stats, redone, symbols);
}

// ------------------------------------------------------------------------------------------------
// 5 write pass
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) jpeg_write_kernel(JpegBatchDev b, const char* __restrict__ compact, const int4* __restrict__ starts, int16_t* coef) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= b.nsub) return;
    const JpegSegment& sg = b.seg[find_segment(b.seg, b.nseg, g)];
    const JpegImage& im = b.img[sg.image];
    const Stream s = stream_of(sg, compact);
    const int j = g - sg.sub0;
    const int end = min((j + 1) * kJpegSubBits, sg.nbits);
    const int4 a = starts[g];
    DecState st{a.x, a.y, a.z};
    int blk = a.w, idx, val;
    if (im.mcu_coefs == im.bpm * 64) {               // every block keeps 64 coefficients, back to back
        int16_t* base = coef + sg.coef0;
        while (st.pos < end && blk < sg.nblocks) {
            const int b_now = blk;
            blk += step(im, b.tab, s, st, &idx, &val);
            if (idx >= 0) base[static_cast<int64_t>(b_now) * 64 + idx] = static_cast<int16_t>(val);
        }
        return;
    }
    // the current block's coefficients: 64, or the DC alone where the component's IDCT reads nothing else
    int u = blk % im.bpm;
    int16_t* mcu = coef + sg.coef0 + static_cast<int64_t>(blk / im.bpm) * im.mcu_coefs;
    int16_t* p = mcu + im.blk_coef[u];
    int last = im.ks[im.blk_c[u]] == 1 ? 0 : 63;
    while (st.pos < end && blk < sg.nblocks) {
        const bool done = step(im, b.tab, s, st, &idx, &val);
        if (idx >= 0 && idx <= last) p[idx] = static_cast<int16_t>(val);
        if (done) {
            ++blk;
            if (++u == im.bpm) { u = 0; mcu += im.mcu_coefs; }
            p = mcu + im.blk_coef[u];
            last = im.ks[im.blk_c[u]] == 1 ? 0 : 63;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// 6 DC values: one CTA per segment
// ------------------------------------------------------------------------------------------------
struct Dc3 { unsigned a, b, c; };
struct Dc3Add { __device__ Dc3 operator()(const Dc3& x, const Dc3& y) const { return Dc3{x.a + y.a, x.b + y.b, x.c + y.c}; } };

constexpr int kDcThreads = 256;

__global__ void __launch_bounds__(kDcThreads) jpeg_dc_kernel(JpegBatchDev b, int16_t* coef) {
    using Scan = cub::BlockScan<Dc3, kDcThreads>;
    __shared__ typename Scan::TempStorage tmp;
    for (int si = blockIdx.x; si < b.nseg; si += gridDim.x) {
        const JpegSegment& sg = b.seg[si];
        const JpegImage& im = b.img[sg.image];
        const int nmcu = sg.nblocks / im.bpm;
        int16_t* base = coef + sg.coef0;
        Dc3 carry{0u, 0u, 0u};
        for (int m0 = 0; m0 < nmcu; m0 += kDcThreads) {
            const int m = m0 + threadIdx.x;
            unsigned sum[3] = {0u, 0u, 0u};
            if (m < nmcu)
                for (int u = 0; u < im.bpm; ++u) sum[im.blk_c[u]] += static_cast<unsigned>(static_cast<int>(base[static_cast<int64_t>(m) * im.mcu_coefs + im.blk_coef[u]]));
            Dc3 pre, tot;
            Scan(tmp).ExclusiveScan(Dc3{sum[0], sum[1], sum[2]}, pre, Dc3{0u, 0u, 0u}, Dc3Add(), tot);
            unsigned run[3] = {carry.a + pre.a, carry.b + pre.b, carry.c + pre.c};
            if (m < nmcu)
                for (int u = 0; u < im.bpm; ++u) {
                    int16_t* p = base + static_cast<int64_t>(m) * im.mcu_coefs + im.blk_coef[u];
                    run[im.blk_c[u]] += static_cast<unsigned>(static_cast<int>(*p));
                    *p = static_cast<int16_t>(run[im.blk_c[u]]);
                }
            carry = Dc3Add()(carry, tot);
            __syncthreads();
        }
    }
}

// ------------------------------------------------------------------------------------------------
// 7 IDCT: jidctint.c jpeg_idct_islow (CONST_BITS 13, PASS1_BITS 2)
// ------------------------------------------------------------------------------------------------
// 64-bit like jidctint.c's JLONG: coefficients of corrupt data or 16-bit quantisation tables overflow 32 bits
using jlong = long long;
__device__ __forceinline__ void idct_1d(jlong s0, jlong s1, jlong s2, jlong s3, jlong s4, jlong s5, jlong s6, jlong s7, jlong* o) {
    jlong z1 = (s2 + s6) * 4433;
    const jlong tmp2 = z1 + s6 * -15137, tmp3 = z1 + s2 * 6270;
    const jlong tmp0 = (s0 + s4) * 8192, tmp1 = (s0 - s4) * 8192;
    const jlong t10 = tmp0 + tmp3, t13 = tmp0 - tmp3, t11 = tmp1 + tmp2, t12 = tmp1 - tmp2;
    jlong t0 = s7, t1 = s5, t2 = s3, t3 = s1;
    z1 = t0 + t3;
    jlong z2 = t1 + t2, z3 = t0 + t2, z4 = t1 + t3;
    const jlong z5 = (z3 + z4) * 9633;
    t0 *= 2446; t1 *= 16819; t2 *= 25172; t3 *= 12299;
    z1 *= -7373; z2 *= -20995; z3 = z3 * -16069 + z5; z4 = z4 * -3196 + z5;
    t0 += z1 + z3; t1 += z2 + z4; t2 += z2 + z3; t3 += z1 + z4;
    o[0] = t10 + t3; o[1] = t11 + t2; o[2] = t12 + t1; o[3] = t13 + t0;
    o[4] = t13 - t0; o[5] = t12 - t1; o[6] = t11 - t2; o[7] = t10 - t3;
}

// jdmaster.c's post-IDCT range-limit table, indexed by (x & RANGE_MASK)
__device__ __forceinline__ uint32_t range_limit(jlong v) {
    const int x = static_cast<int>(v & 1023);
    return x < 128 ? x + 128 : x < 512 ? 255 : x < 896 ? 0 : x - 896;
}

__device__ __forceinline__ int find_image(const JpegImage* img, int B, int64_t v, bool by_pixel) {
    int lo = 0, hi = B - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if ((by_pixel ? img[mid].pix0 : img[mid].block0) <= v) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// jidctred.c jpeg_idct_4x4 / jpeg_idct_2x2 on one column or row (CONST_BITS 13, PASS1_BITS 2): the 4-point form reads
// inputs 0-3 and 5-7, the 2-point form 0, 1, 3, 5 and 7
__device__ __forceinline__ void idct4_1d(jlong s0, jlong s1, jlong s2, jlong s3, jlong s5, jlong s6, jlong s7, jlong* o) {
    const jlong tmp0 = s0 * 16384, tmp2 = s2 * 15137 + s6 * -6270;
    const jlong t10 = tmp0 + tmp2, t12 = tmp0 - tmp2;
    const jlong a = s7 * -1730 + s5 * 11893 + s3 * -17799 + s1 * 8697;
    const jlong c = s7 * -4176 + s5 * -4926 + s3 * 7373 + s1 * 20995;
    o[0] = t10 + c; o[1] = t12 + a; o[2] = t12 - a; o[3] = t10 - c;
}

__device__ __forceinline__ void idct2_1d(jlong s0, jlong s1, jlong s3, jlong s5, jlong s7, jlong* o) {
    const jlong t10 = s0 * 32768, t0 = s7 * -5906 + s5 * 6967 + s3 * -10426 + s1 * 29692;
    o[0] = t10 + t0; o[1] = t10 - t0;
}

// 4 x 4 output of one block: x dequantised, natural order
__device__ __forceinline__ void idct_4x4(const int* x, uint8_t* dst, int pitch) {
    jlong ws[32], o[4];
#pragma unroll
    for (int col = 0; col < 8; ++col) {              // pass 1: columns (column 4 is not read by pass 2)
        if (col == 4) continue;
        idct4_1d(x[col], x[8 + col], x[16 + col], x[24 + col], x[40 + col], x[48 + col], x[56 + col], o);
#pragma unroll
        for (int r = 0; r < 4; ++r) ws[r * 8 + col] = (o[r] + (1 << 11)) >> 12;
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {                    // pass 2: rows
        idct4_1d(ws[r * 8], ws[r * 8 + 1], ws[r * 8 + 2], ws[r * 8 + 3], ws[r * 8 + 5], ws[r * 8 + 6], ws[r * 8 + 7], o);
        *reinterpret_cast<uint32_t*>(dst + static_cast<int64_t>(r) * pitch) =
            range_limit((o[0] + (1 << 18)) >> 19) | range_limit((o[1] + (1 << 18)) >> 19) << 8 |
            range_limit((o[2] + (1 << 18)) >> 19) << 16 | range_limit((o[3] + (1 << 18)) >> 19) << 24;
    }
}

// 2 x 2 output of one block
__device__ __forceinline__ void idct_2x2(const int* x, uint8_t* dst, int pitch) {
    jlong ws[16], o[2];
#pragma unroll
    for (int col = 0; col < 8; ++col) {              // pass 1: columns 0, 1, 3, 5, 7
        if (col != 0 && !(col & 1)) continue;
        idct2_1d(x[col], x[8 + col], x[24 + col], x[40 + col], x[56 + col], o);
        ws[col] = (o[0] + (1 << 12)) >> 13;
        ws[8 + col] = (o[1] + (1 << 12)) >> 13;
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {                    // pass 2: rows
        idct2_1d(ws[r * 8], ws[r * 8 + 1], ws[r * 8 + 3], ws[r * 8 + 5], ws[r * 8 + 7], o);
        *reinterpret_cast<uint16_t*>(dst + static_cast<int64_t>(r) * pitch) =
            static_cast<uint16_t>(range_limit((o[0] + (1 << 19)) >> 20) | range_limit((o[1] + (1 << 19)) >> 20) << 8);
    }
}

// The 4 x 4 and 2 x 2 blocks of a reduced decode, out of line: the 8 x 8 path of jpeg_idct_kernel keeps its registers
__device__ __noinline__ void idct_reduced(const int16_t* __restrict__ blk, const uint16_t* q, int k, uint8_t* dst, int pitch) {
    int x[64];                                       // dequantised as in jpeg_idct_kernel; rows not read stay 0
#pragma unroll
    for (int i = 0; i < 64; ++i) x[i] = 0;
#pragma unroll
    for (int r = 0; r < 8; ++r) {                    // rows the reduced forms read: 0-3, 5-7 (4 x 4), 0, 1, 3, 5, 7 (2 x 2)
        if (r == 4 || (k == 2 && r != 0 && !(r & 1))) continue;
        const int4 v = reinterpret_cast<const int4*>(blk)[r];
        const int w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            x[r * 8 + 2 * t] = static_cast<int16_t>(w[t] & 0xFFFF) * static_cast<int>(q[r * 8 + 2 * t]);
            x[r * 8 + 2 * t + 1] = (w[t] >> 16) * static_cast<int>(q[r * 8 + 2 * t + 1]);
        }
    }
    if (k == 4) idct_4x4(x, dst, pitch);
    else idct_2x2(x, dst, pitch);
}

// five CTAs per SM, as the 8 x 8 path alone compiles to (96 registers)
__global__ void __launch_bounds__(128, 5) jpeg_idct_kernel(JpegBatchDev b, long long nblocks, const int16_t* __restrict__ coef, uint8_t* planes) {
    const long long gb = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (gb >= nblocks) return;
    const JpegImage& im = b.img[find_image(b.img, b.B, gb, false)];
    const long long local = gb - im.block0;
    const int mcu = static_cast<int>(local / im.bpm), u = static_cast<int>(local % im.bpm);
    const int c = im.blk_c[u];
    const int k = im.ks[c], pitch = im.pitch[c];
    const int px = ((mcu % im.mcux) * im.hs[c] + im.blk_x[u]) * k, py = ((mcu / im.mcux) * im.vs[c] + im.blk_y[u]) * k;
    const int16_t* blk = coef + im.coef0 + static_cast<int64_t>(mcu) * im.mcu_coefs + im.blk_coef[u];
    if (k == 1) {                                    // jidctred.c jpeg_idct_1x1: the DC alone, one coefficient stored
        planes[im.plane[c] + static_cast<int64_t>(py) * pitch + px] =
            static_cast<uint8_t>(range_limit((static_cast<jlong>(*blk) * im.q[c][0] + 4) >> 3));
        return;
    }
    if (k < 8) { idct_reduced(blk, im.q[c], k, planes + im.plane[c] + static_cast<int64_t>(py) * pitch + px, pitch); return; }
    int x[64];                                       // dequantised: int16 * uint16 fits 32 bits
    const int4* src = reinterpret_cast<const int4*>(blk);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int4 v = src[i];
        const int w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            x[i * 8 + 2 * t] = static_cast<int16_t>(w[t] & 0xFFFF) * static_cast<int>(im.q[c][i * 8 + 2 * t]);
            x[i * 8 + 2 * t + 1] = (w[t] >> 16) * static_cast<int>(im.q[c][i * 8 + 2 * t + 1]);
        }
    }
    jlong ws[64], o[8];
#pragma unroll
    for (int col = 0; col < 8; ++col) {              // pass 1: columns
        idct_1d(x[col], x[8 + col], x[16 + col], x[24 + col], x[32 + col], x[40 + col], x[48 + col], x[56 + col], o);
#pragma unroll
        for (int r = 0; r < 8; ++r) ws[r * 8 + col] = (o[r] + (1 << 10)) >> 11;
    }
    uint8_t* dst = planes + im.plane[c] + static_cast<int64_t>(py) * pitch + px;
#pragma unroll
    for (int r = 0; r < 8; ++r) {                    // pass 2: rows
        idct_1d(ws[r * 8], ws[r * 8 + 1], ws[r * 8 + 2], ws[r * 8 + 3], ws[r * 8 + 4], ws[r * 8 + 5], ws[r * 8 + 6], ws[r * 8 + 7], o);
        uint2 v;
        v.x = range_limit((o[0] + (1 << 17)) >> 18) | range_limit((o[1] + (1 << 17)) >> 18) << 8 |
              range_limit((o[2] + (1 << 17)) >> 18) << 16 | range_limit((o[3] + (1 << 17)) >> 18) << 24;
        v.y = range_limit((o[4] + (1 << 17)) >> 18) | range_limit((o[5] + (1 << 17)) >> 18) << 8 |
              range_limit((o[6] + (1 << 17)) >> 18) << 16 | range_limit((o[7] + (1 << 17)) >> 18) << 24;
        *reinterpret_cast<uint2*>(dst + static_cast<int64_t>(r) * pitch) = v;
    }
}

// ------------------------------------------------------------------------------------------------
// 8 upsampling (jdsample.c) and colour conversion (jdcolor.c)
// ------------------------------------------------------------------------------------------------
// One chroma sample of output pixel (x, y): pl is the component's plane at its DCT scaled size, dw x dh samples, expanded by
// (he, ve) to the output.  jinit_upsampler replicates when fancy upsampling is off (the luma's scaled size is 1) or the
// component is at most 2 samples wide.
__device__ __forceinline__ int chroma(const uint8_t* pl, int pitch, int he, int ve, bool fancy, int dw, int dh, int x, int y) {
    if (he == 1 && ve == 1) return pl[static_cast<int64_t>(y) * pitch + x];
    const int i = x >> 1;
    if (!fancy || dw <= 2) return pl[static_cast<int64_t>(y / ve) * pitch + i];     // plain replication
    const bool even = (x & 1) == 0;
    const int nb = min(max(even ? i - 1 : i + 1, 0), dw - 1);
    const bool first = even && i == 0, last = !even && i == dw - 1;
    if (ve == 1) {                                                         // h2v1_fancy_upsample
        const uint8_t* r = pl + static_cast<int64_t>(y) * pitch;
        const int near = r[i], far = r[nb];
        if (first || last) return near;
        return even ? (near * 3 + far + 1) >> 2 : (near * 3 + far + 2) >> 2;
    }
    const int r = y >> 1, r2 = min(max((y & 1) ? r + 1 : r - 1, 0), dh - 1);   // h2v2_fancy_upsample, context rows replicated
    const uint8_t* a = pl + static_cast<int64_t>(r) * pitch;
    const uint8_t* c = pl + static_cast<int64_t>(r2) * pitch;
    const int t = a[i] * 3 + c[i], o = a[nb] * 3 + c[nb];
    if (first) return (t * 4 + 8) >> 4;
    if (last) return (t * 4 + 7) >> 4;
    return even ? (t * 3 + o + 8) >> 4 : (t * 3 + o + 7) >> 4;
}

__global__ void __launch_bounds__(256) jpeg_color_kernel(JpegBatchDev b, long long npix, const uint8_t* __restrict__ planes, uint8_t* out) {
    const long long gp = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (gp >= npix) return;
    const JpegImage& im = b.img[find_image(b.img, b.B, gp, true)];
    const int64_t local = gp - im.pix0;
    const int y = static_cast<int>(local / im.w), x = static_cast<int>(local % im.w);
    const int Y = planes[im.plane[0] + static_cast<int64_t>(y) * im.pitch[0] + x];
    uint8_t* o = out + im.out + local * 3;
    if (im.space == kSpaceGray) { o[0] = o[1] = o[2] = static_cast<uint8_t>(Y); return; }
    const int cb = chroma(planes + im.plane[1], im.pitch[1], im.he[1], im.ve[1], im.fancy, im.dw[1], im.dh[1], x, y);
    const int cr = chroma(planes + im.plane[2], im.pitch[2], im.he[2], im.ve[2], im.fancy, im.dw[2], im.dh[2], x, y);
    if (im.space == kSpaceRgb) { o[0] = static_cast<uint8_t>(Y); o[1] = static_cast<uint8_t>(cb); o[2] = static_cast<uint8_t>(cr); return; }
    const int xb = cb - 128, xr = cr - 128;
    const int r = Y + ((91881 * xr + 32768) >> 16);
    const int g = Y + ((-22554 * xb + 32768 - 46802 * xr) >> 16);
    const int bl = Y + ((116130 * xb + 32768) >> 16);
    o[0] = static_cast<uint8_t>(min(max(r, 0), 255));
    o[1] = static_cast<uint8_t>(min(max(g, 0), 255));
    o[2] = static_cast<uint8_t>(min(max(bl, 0), 255));
}

inline size_t a256(size_t v) { return (v + 255) & ~static_cast<size_t>(255); }

}  // namespace

int jpeg_info(const uint8_t* data, int64_t bytes, int* height, int* width, int* components, char* why, size_t why_len) {
    Parsed P;
    const int rc = parse(data, bytes, &P, false, Reject{why, why_len});
    if (rc) return rc;
    if (height) *height = P.h;
    if (width) *width = P.w;
    if (components) *components = P.ncomp;
    return 0;
}

int jpeg_auto_ratio(int h, int w, int th, int tw) {
    int rh, rw, ph, pw;
    resize_with_pad_geometry(h, w, th, tw, &rh, &rw, &ph, &pw);
    if (rh <= 0 || rw <= 0) return 1;
    const int scale = std::min(w / rw, h / rh);
    return scale >= 8 ? 8 : scale >= 4 ? 4 : scale >= 2 ? 2 : 1;
}

int jpeg_plan(const char* fn, const uint8_t* const* data, const int64_t* bytes, int B, const int32_t* ratios, int target_h,
              int target_w, const int64_t* out_offsets, JpegBatch* b) {
    for (int i = 0; ratios && i < B; ++i)
        if (ratios[i] != 0 && ratios[i] != 1 && ratios[i] != 2 && ratios[i] != 4 && ratios[i] != 8)
            return fail(VITDET_E_INVALID, "%s: file %d: ratio %d (expected 1, 2, 4, 8 or 0 for auto)", fn, i, ratios[i]);
    std::vector<JpegImage> imgs(B);
    std::vector<JpegSegment> segs;
    std::vector<JpegHuff> tabs;
    b->B = B;
    b->height.assign(B, 0);
    b->width.assign(B, 0);
    b->file_height.assign(B, 0);
    b->file_width.assign(B, 0);
    b->ratio.assign(B, 1);
    b->file_off.assign(B + 1, 0);
    b->rgb_off.assign(B, 0);
    size_t compact = 0, planes = 0, rgb = 0, coefs = 0;
    long long nblocks = 0, npix = 0;
    int nsub = 0;
    char why[256];
    for (int i = 0; i < B; ++i) {
        if (!data[i] || bytes[i] <= 0) return fail(VITDET_E_INVALID, "%s: file %d: no bytes", fn, i);
        Parsed P;                    // every file's own state: restart interval, tables, markers seen
        if (parse(data[i], bytes[i], &P, true, Reject{why, sizeof(why)})) return fail(VITDET_E_INVALID, "%s: file %d: %s", fn, i, why);
        b->file_off[i + 1] = b->file_off[i] + static_cast<size_t>(bytes[i]);
        JpegImage& im = imgs[i];
        memset(&im, 0, sizeof(im));
        int ratio = ratios ? ratios[i] : 1;
        if (ratio == 0) ratio = jpeg_auto_ratio(P.h, P.w, target_h, target_w);
        // the output ceil(h / ratio) x ceil(w / ratio); the luma's DCT scaled size k = 8 / ratio
        const int k = 8 / ratio;
        im.h = (P.h + ratio - 1) / ratio; im.w = (P.w + ratio - 1) / ratio; im.ncomp = P.ncomp; im.space = P.space;
        im.hmax = im.vmax = 1;
        for (int c = 0; c < P.ncomp; ++c) {
            im.hs[c] = P.hs[c]; im.vs[c] = P.vs[c];
            im.hmax = std::max(im.hmax, P.hs[c]); im.vmax = std::max(im.vmax, P.vs[c]);
            memcpy(im.q[c], P.q[P.qid[c]], sizeof(im.q[c]));
            im.dc[c] = static_cast<int>(tabs.size()); tabs.push_back(P.huff[0][P.td[c]]);
            im.ac[c] = static_cast<int>(tabs.size()); tabs.push_back(P.huff[1][P.ta[c]]);
        }
        im.mcux = (P.w + 8 * im.hmax - 1) / (8 * im.hmax);
        im.mcuy = (P.h + 8 * im.vmax - 1) / (8 * im.vmax);
        im.bpm = 0;
        for (int c = 0; c < P.ncomp; ++c)
            for (int by = 0; by < im.vs[c]; ++by)
                for (int bx = 0; bx < im.hs[c]; ++bx) { im.blk_c[im.bpm] = c; im.blk_x[im.bpm] = bx; im.blk_y[im.bpm] = by; ++im.bpm; }
        // jdmaster.c jpeg_core_output_dimensions: each component's DCT scaled size starts at k and doubles while both
        // sampling ratios allow it (4:2:0 chroma at ratio 2 takes 8 x 8 blocks and needs no upsampling); its scaled size
        // is ceil(size * samp * scaled size / (max samp * 8)); jdsample.c expands it by max samp * k / (samp * scaled size)
        im.fancy = k > 1;
        for (int c = 0; c < P.ncomp; ++c) {
            int ss = k;
            while (ss < 8 && (im.hmax * k) % (im.hs[c] * ss * 2) == 0 && (im.vmax * k) % (im.vs[c] * ss * 2) == 0) ss *= 2;
            im.ks[c] = ss;
            im.pitch[c] = im.mcux * im.hs[c] * ss;
            im.dw[c] = static_cast<int>((static_cast<long long>(P.w) * im.hs[c] * ss + im.hmax * 8 - 1) / (im.hmax * 8));
            im.dh[c] = static_cast<int>((static_cast<long long>(P.h) * im.vs[c] * ss + im.vmax * 8 - 1) / (im.vmax * 8));
            im.he[c] = im.hmax * k / (im.hs[c] * ss);
            im.ve[c] = im.vmax * k / (im.vs[c] * ss);
        }
        im.mcu_coefs = 0;
        bool full = false;
        for (int u = 0; u < im.bpm; ++u) {
            const bool dc_only = im.ks[im.blk_c[u]] == 1;
            if (!dc_only) im.mcu_coefs = (im.mcu_coefs + 7) & ~7;
            im.blk_coef[u] = static_cast<int16_t>(im.mcu_coefs);
            im.mcu_coefs += dc_only ? 1 : 64;
            full |= !dc_only;
        }
        if (full) im.mcu_coefs = (im.mcu_coefs + 7) & ~7;
        const long long nmcu = static_cast<long long>(im.mcux) * im.mcuy;
        im.block0 = nblocks;
        im.coef0 = static_cast<int64_t>(coefs);
        coefs += (static_cast<size_t>(nmcu) * im.mcu_coefs + 7) & ~static_cast<size_t>(7);
        for (int c = 0; c < P.ncomp; ++c) {
            im.plane[c] = static_cast<int64_t>(planes);
            planes += a256(static_cast<size_t>(nmcu) * im.hs[c] * im.vs[c] * im.ks[c] * im.ks[c]);
        }
        im.pix0 = npix;
        b->rgb_off[i] = out_offsets ? static_cast<size_t>(out_offsets[i]) : rgb;
        im.out = static_cast<int64_t>(b->rgb_off[i]);
        rgb += a256(static_cast<size_t>(im.h) * im.w * 3);
        const long long ri = P.ri ? P.ri : nmcu;
        const long long nseg = (nmcu + ri - 1) / ri;
        for (long long s = 0; s < nseg; ++s) {
            JpegSegment sg;
            memset(&sg, 0, sizeof(sg));
            const bool have = s < static_cast<long long>(P.seg_a.size());   // extra RSTn segments dropped, missing ones empty
            sg.src = static_cast<int64_t>(b->file_off[i]) + (have ? P.seg_a[s] : 0);
            sg.src_len = have ? static_cast<int32_t>(P.seg_b[s] - P.seg_a[s]) : 0;
            const long long clen = have ? P.seg_b[s] - P.seg_a[s] - P.seg_stuff[s] : 0;
            sg.nbits = static_cast<int32_t>(clen * 8);
            sg.dst = static_cast<int64_t>(compact);
            compact += (static_cast<size_t>(clen) + 7) & ~static_cast<size_t>(7);
            sg.coef0 = im.coef0 + s * ri * im.mcu_coefs;
            sg.nblocks = static_cast<int32_t>((std::min(nmcu, (s + 1) * ri) - s * ri) * im.bpm);
            sg.sub0 = nsub;
            sg.image = i;
            nsub += (sg.nbits + kJpegSubBits - 1) / kJpegSubBits;
            segs.push_back(sg);
        }
        nblocks += nmcu * im.bpm;
        npix += static_cast<long long>(im.h) * im.w;
        b->height[i] = im.h;
        b->width[i] = im.w;
        b->file_height[i] = P.h;
        b->file_width[i] = P.w;
        b->ratio[i] = ratio;
    }
    b->nseg = static_cast<int>(segs.size());
    b->nsub = nsub;
    b->nblocks = nblocks;
    b->npix = npix;
    b->rgb_bytes = rgb;
    const size_t o_seg = a256(sizeof(JpegImage) * B), o_tab = o_seg + a256(sizeof(JpegSegment) * segs.size());
    const size_t desc_bytes = o_tab + sizeof(JpegHuff) * tabs.size();
    b->desc.assign(desc_bytes, 0);
    memcpy(b->desc.data(), imgs.data(), sizeof(JpegImage) * B);
    memcpy(b->desc.data() + o_seg, segs.data(), sizeof(JpegSegment) * segs.size());
    memcpy(b->desc.data() + o_tab, tabs.data(), sizeof(JpegHuff) * tabs.size());
    b->o_compact = a256(desc_bytes);
    b->o_coef = b->o_compact + a256(compact);
    b->o_spec = b->o_coef + a256(coefs * sizeof(int16_t));
    b->o_check = b->o_spec + a256(sizeof(int2) * nsub);
    b->o_sync = b->o_check + a256(sizeof(int2) * kWordsPerSub * static_cast<size_t>(nsub));
    b->o_start = b->o_sync + 3 * a256(sizeof(int2) * nsub);
    b->o_planes = b->o_start + a256(sizeof(int4) * nsub);
    b->o_stats = b->o_planes + a256(planes);
    b->work_bytes = b->o_stats + 256;
    return 0;
}

cudaError_t jpeg_decode_launch(const JpegBatch& b, const char* files_dev, void* work, uint8_t* out, cudaStream_t st) {
    char* w = static_cast<char*>(work);
    JpegBatchDev d;
    const size_t o_seg = a256(sizeof(JpegImage) * b.B), o_tab = o_seg + a256(sizeof(JpegSegment) * b.nseg);
    d.img = reinterpret_cast<const JpegImage*>(w);
    d.seg = reinterpret_cast<const JpegSegment*>(w + o_seg);
    d.tab = reinterpret_cast<const JpegHuff*>(w + o_tab);
    d.B = b.B; d.nseg = b.nseg; d.nsub = b.nsub;
    char* compact = w + b.o_compact;
    int16_t* coef = reinterpret_cast<int16_t*>(w + b.o_coef);
    int2* spec = reinterpret_cast<int2*>(w + b.o_spec);
    int2* checks = reinterpret_cast<int2*>(w + b.o_check);
    int2* sync[3];                   // pass p writes sync[p % 3], reads the two before it
    for (int i = 0; i < 3; ++i) sync[i] = reinterpret_cast<int2*>(w + b.o_sync + i * a256(sizeof(int2) * b.nsub));
    int4* starts = reinterpret_cast<int4*>(w + b.o_start);
    uint8_t* planes = reinterpret_cast<uint8_t*>(w + b.o_planes);
    long long* stats = reinterpret_cast<long long*>(w + b.o_stats);
    // grids of at least one CTA: the launch count does not depend on the data.  Plain stream-ordered launches: these
    // kernels read their predecessor's output from their first instruction.
    const unsigned seg_grid = static_cast<unsigned>(std::max(1, std::min(b.nseg, 1 << 20)));
    const unsigned sub_grid = static_cast<unsigned>(std::max(1, (b.nsub + 127) / 128));
    jpeg_destuff_kernel<<<seg_grid, kDestuffThreads, 0, st>>>(d, reinterpret_cast<const uint8_t*>(files_dev), compact, coef, stats);
    jpeg_spec_kernel<<<sub_grid, 128, 0, st>>>(d, compact, spec, checks);
    unsigned long long* counters = reinterpret_cast<unsigned long long*>(stats);
    for (int p = 1; p <= kJpegSyncPasses; ++p)
        jpeg_sync_kernel<<<sub_grid, 128, 0, st>>>(d, compact, spec, checks, p == 1 ? nullptr : p == 2 ? spec : sync[(p - 2) % 3],
                                                   p == 1 ? spec : sync[(p - 1) % 3], sync[p % 3], counters);
    jpeg_repair_kernel<<<std::max(1, (b.nseg + 3) / 4), 128, 0, st>>>(d, compact, spec, checks, sync[(kJpegSyncPasses - 1) % 3],
                                                                       sync[kJpegSyncPasses % 3], starts, counters);
    jpeg_write_kernel<<<sub_grid, 128, 0, st>>>(d, compact, starts, coef);
    jpeg_dc_kernel<<<seg_grid, kDcThreads, 0, st>>>(d, coef);
    jpeg_idct_kernel<<<static_cast<unsigned>(std::max(1LL, (b.nblocks + 127) / 128)), 128, 0, st>>>(d, b.nblocks, coef, planes);
    jpeg_color_kernel<<<static_cast<unsigned>(std::max(1LL, (b.npix + 255) / 256)), 256, 0, st>>>(d, b.npix, planes, out);
    return cudaGetLastError();
}

}  // namespace vitdet
