// Runs ONE kernel of the library back to back for a few seconds so that nvidia-smi can sample the SM clock and the board
// power under exactly that kernel (scripts/gpu_power_probe.sh).  Cases: the dominant 3584 -> 1792 pair GEMM, the 28 -> 3584
// Mish layer, and a store-only stand-in is not needed — the attention kernel is sampled through bench.py.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <cuda_bf16.h>
#include "kernels.h"
using namespace vitdet;

int main(int argc, char** argv) {
    const char* which = argc > 1 ? argv[1] : "mlp_2";
    const double seconds = argc > 2 ? atof(argv[2]) : 3.0;
    const int M = 82944;
    void *A, *W, *out; float* bias;
    cudaMalloc(&A, size_t(M) * 3584 * 2); cudaMalloc(&W, size_t(3584) * 3584 * 2); cudaMalloc(&out, size_t(M) * 3584 * 2); cudaMalloc(&bias, 4096 * 4);
    // small non-zero operands: the tensor pipe's power depends on the data toggling
    {
        size_t n = size_t(M) * 3584;
        __nv_bfloat16* h = (__nv_bfloat16*)malloc(n * 2);
        unsigned s = 12345u;
        for (size_t i = 0; i < n; ++i) { s = s * 1664525u + 1013904223u; h[i] = __float2bfloat16(((s >> 8) & 0xffff) / 65536.f - 0.5f); }
        cudaMemcpy(A, h, n * 2, cudaMemcpyHostToDevice);
        cudaMemcpy(W, h, size_t(3584) * 3584 * 2, cudaMemcpyHostToDevice);
        free(h);
        cudaMemset(bias, 0, 4096 * 4);
    }
    GemmDesc d; d.A = A; d.W = W; d.out = out; d.bias = bias; d.M = M; d.act = 1;
    bool pair = false;
    if (!strcmp(which, "mlp_2")) { d.K = 3584; d.N = 1792; pair = true; }
    else if (!strcmp(which, "mlp_3")) { d.K = 1792; d.N = 896; pair = true; }
    else if (!strcmp(which, "mlp_1")) { d.K = 28; d.N = 3584; }
    else if (!strcmp(which, "qkv")) { d.K = 28; d.N = 960; d.act = 0; }
    else { printf("unknown case\n"); return 1; }
    d.lda = (d.K + 7) / 8 * 8; d.ldw = d.lda; d.ldc = d.N;
    TcGemmPlan plan;
    int r = tc_gemm_make_plan(&plan, d, 148, pair);
    if (r) { printf("plan error %d\n", r); return 1; }
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    auto t0 = std::chrono::steady_clock::now();
    long launches = 0; float ms_total = 0.f;
    while (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() < seconds) {
        cudaEventRecord(e0);
        for (int i = 0; i < 50; ++i) tc_gemm_launch(plan, 0);
        cudaEventRecord(e1);
        if (cudaDeviceSynchronize() != cudaSuccess) { printf("launch failed\n"); return 1; }
        float ms; cudaEventElapsedTime(&ms, e0, e1); ms_total += ms; launches += 50;
    }
    const double us = ms_total * 1000.0 / launches;
    printf("%s: %ld launches, %.1f us per launch, %.0f TFLOP/s\n", which, launches, us, 2.0 * M * d.K * d.N / (us * 1e-6) / 1e12);
    return 0;
}
