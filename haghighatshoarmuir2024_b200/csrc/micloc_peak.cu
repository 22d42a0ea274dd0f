// micloc_peak.cu -- FP32 FMA-pipe micro-benchmark: the measured denominator of the
// hot path's roofline (SURVEY.md 8d: the chain is bound by the FP32 FMA pipe, and
// MEASURED_PEAKS.json only holds HBM and bf16-tensor figures).
//
//   variant 0: scalar FFMA, 16 independent accumulators per thread
//   variant 1: packed fma.rn.f32x2 (FFMA2), 8 independent 2-wide accumulators
// Both run `iters` x 16 FMA per thread on a grid of sm_count x 8 CTAs x 256 threads.
#include <cuda_runtime.h>

#include "micloc_common.h"

namespace micloc {

__global__ void __launch_bounds__(256)
k_peak_ffma(float *out, int iters, float a, float b) {
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = (float)(threadIdx.x + i);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) acc[i] = fmaf(acc[i], a, b);
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += acc[i];
    if (s == 123.456f) out[0] = s;   // never true; keeps the loop alive
}

__global__ void __launch_bounds__(256)
k_peak_ffma2(float *out, int iters, float a, float b) {
    unsigned long long acc[8], av, bv;
    asm("mov.b64 %0, {%1, %1};" : "=l"(av) : "f"(a));
    asm("mov.b64 %0, {%1, %1};" : "=l"(bv) : "f"(b));
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float lo = (float)(threadIdx.x + i), hi = lo + 0.5f;
        asm("mov.b64 %0, {%1, %2};" : "=l"(acc[i]) : "f"(lo), "f"(hi));
    }
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
            asm volatile("fma.rn.f32x2 %0, %0, %1, %2;" : "+l"(acc[i]) : "l"(av), "l"(bv));
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        float lo, hi;
        asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(acc[i]));
        s += lo + hi;
    }
    if (s == 123.456f) out[0] = s;
}

// variant 2: FP64 DFMA, 8 independent accumulators (is the FP64 pipe a usable second arithmetic pipe on this part?)
__global__ void __launch_bounds__(256)
k_peak_dfma(float *out, int iters, double a, double b) {
    double acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = (double)(threadIdx.x + i);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = fma(acc[i], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += acc[i];
    if (s == 123.456) out[0] = (float)s;
}

}  // namespace micloc

using namespace micloc;

extern "C" int micloc_fp32_peak(int device, int variant, double *tflops) {
    if (!tflops || variant < 0 || variant > 2) return set_error(MICLOC_ERR_CONFIG, "bad arguments");
    MICLOC_CUDA(cudaSetDevice(device));
    int sms = 0;
    MICLOC_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    float *out = nullptr;
    MICLOC_CUDA(cudaMalloc(&out, sizeof(float)));
    cudaEvent_t e0, e1;
    MICLOC_CUDA(cudaEventCreate(&e0));
    MICLOC_CUDA(cudaEventCreate(&e1));
    const int iters = 1 << 16, grid = sms * 8;
    double best = 0.0;
    for (int rep = 0; rep < 6; ++rep) {
        MICLOC_CUDA(cudaEventRecord(e0, 0));
        if (variant == 0) k_peak_ffma<<<grid, 256>>>(out, iters, 0.999f, 0.001f);
        else if (variant == 1) k_peak_ffma2<<<grid, 256>>>(out, iters, 0.999f, 0.001f);
        else k_peak_dfma<<<grid, 256>>>(out, iters / 4, 0.999, 0.001);
        MICLOC_CUDA(cudaEventRecord(e1, 0));
        MICLOC_CUDA(cudaEventSynchronize(e1));
        float ms = 0.f;
        MICLOC_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        count_launch(1);
        // flop counted: 16 FP32 FMA per iteration (variants 0, 1), 8 FP64 FMA (variant 2)
        const double fl = variant == 2 ? 2.0 * 8.0 * (double)(iters / 4) * 256.0 * (double)grid
                                       : 2.0 * 16.0 * (double)iters * 256.0 * (double)grid;
        const double tf = fl / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
    MICLOC_CUDA(cudaGetLastError());
    *tflops = best;
    return MICLOC_OK;
}
