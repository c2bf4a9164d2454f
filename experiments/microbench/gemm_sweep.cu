// Kernel-level timing sweep of the library's GEMM launchers (links against libvitdet_b200.so): time vs rows, n-tiles and
// block_n for the small layers of the default model, to separate fixed launch cost from per-tile cost.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -I vision_transformer_detector_b200/csrc -I include \
//        -o /tmp/gemm_sweep experiments/microbench/gemm_sweep.cu -L vision_transformer_detector_b200 -lvitdet_b200 \
//        -Xlinker -rpath -Xlinker $PWD/vision_transformer_detector_b200
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cuda_bf16.h>
#include "kernels.h"

using namespace vitdet;

static void* dalloc(size_t bytes, int fill) {
    void* p; cudaMalloc(&p, bytes); cudaMemset(p, fill, bytes); return p;
}

struct Case { const char* name; int M, K, N, act, out_f32, resid, ln, pair, block_n; int ld = 0; };

static float time_plan(const TcGemmPlan& plan, int reps) {
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int i = 0; i < 3; ++i) tc_gemm_launch(plan, 0);
    cudaEventRecord(e0);
    for (int i = 0; i < reps; ++i) tc_gemm_launch(plan, 0);
    cudaEventRecord(e1);
    cudaError_t err = cudaDeviceSynchronize();
    if (err != cudaSuccess) { printf("error %s\n", cudaGetErrorString(err)); exit(1); }
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    return ms / reps * 1000.f;
}

int main() {
    const int Mmax = 82944;
    void* A = dalloc(size_t(Mmax) * 3584 * 2, 0);
    void* W = dalloc(size_t(3584) * 3584 * 2, 0);
    void* out = dalloc(size_t(Mmax) * 3584 * 2, 0);
    float* bias = (float*)dalloc(4096 * 4, 0);
    float* x = (float*)dalloc(size_t(Mmax) * 32 * 4, 0);
    void* ln = dalloc(size_t(Mmax) * 32 * 2, 0);
    float* g = (float*)dalloc(128, 0);
    std::vector<Case> cases;
    // one tile per CTA or less: the latency of a launch (fill + drain), back to back with programmatic dependent launch
    for (int M : {128, 148 * 128, 2 * 148 * 128, 4 * 148 * 128}) {
        cases.push_back({"qkv 28->192 (1 n-tile)", M, 28, 192, 0, 0, 0, 0, 0, 192});
        cases.push_back({"mlp_5 448->224 mish", M, 448, 224, 1, 0, 0, 0, 0, 0});
        cases.push_back({"out 320->28 f32+res+ln", M, 320, 28, 0, 1, 1, 1, 0, 0});
        cases.push_back({"mlp_4 896->448 mish pair", M, 896, 448, 1, 0, 0, 0, 1, 0});
    }
    for (int M : {82944}) {
        cases.push_back({"qkv 28->960", M, 28, 960, 0, 0, 0, 0, 0, 0});
        cases.push_back({"mlp_1 28->3584 mish", M, 28, 3584, 1, 0, 0, 0, 0, 0});
        cases.push_back({"mlp_5 448->224 mish", M, 448, 224, 1, 0, 0, 0, 0, 0});
        cases.push_back({"out 320->28 f32+res+ln", M, 320, 28, 0, 1, 1, 1, 0, 0});
        cases.push_back({"mlp_4 896->448 mish pair", M, 896, 448, 1, 0, 0, 0, 1, 0});
    }
    for (int bn : {64, 96, 128, 192, 256}) cases.push_back({"qkv 28->960 block_n", 82944, 28, 960, 0, 0, 0, 0, 0, bn});
    for (int N : {192, 384, 576, 768, 960}) cases.push_back({"28->N bn192", 82944, 28, N, 0, 0, 0, 0, 0, 192});
    for (int K : {28, 64, 128, 256}) cases.push_back({"K->960", 82944, K, 960, 0, 0, 0, 0, 0, 0});
    for (int bn : {32, 64, 128, 224}) cases.push_back({"mlp_5 block_n", 82944, 448, 224, 1, 0, 0, 0, 0, bn});
    // is the K = 28 case slow because of the 64-byte row pitch or because of the out-of-bounds half of the TMA box?
    cases.push_back({"qkv K=28 pitch 32", 82944, 28, 960, 0, 0, 0, 0, 0, 0, 32});
    cases.push_back({"qkv K=28 pitch 64", 82944, 28, 960, 0, 0, 0, 0, 0, 0, 64});
    cases.push_back({"qkv K=32 pitch 32", 82944, 32, 960, 0, 0, 0, 0, 0, 0, 32});
    cases.push_back({"qkv K=32 pitch 64", 82944, 32, 960, 0, 0, 0, 0, 0, 0, 64});
    cases.push_back({"qkv K=64 pitch 64", 82944, 64, 960, 0, 0, 0, 0, 0, 0, 64});
    cases.push_back({"mlp_1 K=28 pitch 32", 82944, 28, 3584, 1, 0, 0, 0, 0, 0, 32});
    cases.push_back({"mlp_1 K=28 pitch 64", 82944, 28, 3584, 1, 0, 0, 0, 0, 0, 64});
    cases.push_back({"mlp_1 K=64 pitch 64", 82944, 64, 3584, 1, 0, 0, 0, 0, 0, 64});
    for (const Case& c : cases) {
        GemmDesc d;
        const int K8 = c.ld ? c.ld : (c.K + 7) / 8 * 8;
        d.A = A; d.lda = K8; d.W = W; d.ldw = K8; d.M = c.M; d.N = c.N; d.K = c.K; d.bias = bias; d.act = c.act; d.block_n = c.block_n;
        if (c.out_f32) {
            d.out = x; d.ldc = 28; d.out_f32 = 1;
            if (c.resid) { d.resid = x; d.ldr = 28; }
            if (c.ln) { d.ln_gamma = g; d.ln_beta = g; d.ln_out = ln; d.ln_ld = 32; }
        } else {
            d.out = out; d.ldc = (c.N + 7) / 8 * 8;
        }
        TcGemmPlan plan;
        int r = tc_gemm_make_plan(&plan, d, 148, c.pair);
        if (r) { printf("%-28s plan error %d\n", c.name, r); continue; }
        const float us = time_plan(plan, 20);
        printf("%-28s M %6d K %4d N %4d bn %3d stages %d tiles %5d (%.1f / CTA): %7.1f us  %6.0f clk/tile@1.8GHz\n", c.name, c.M, c.K, c.N,
               plan.block_n, plan.num_stages, plan.num_tiles, plan.num_tiles / double(plan.grid), us,
               us * 1800.0 / (plan.num_tiles / double(plan.grid)));
    }
    return 0;
}
