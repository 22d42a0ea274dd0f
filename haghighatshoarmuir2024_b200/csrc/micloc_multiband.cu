// micloc_multiband.cu -- what surrounds the per-band SNN chains of a multi-band localiser (SURVEY.md 8f rank 4):
//
//   filterbank on the raw frame    micloc/filterbank.py:25-46 (ButterworthFilterbank.evolve: one band-pass per band on
//                                  every microphone, zero state); int32 `T x 8` wav frames with the channels beyond
//                                  the microphones dropped, micloc/localization_demo_snn.py:141-145
//   activity detection             micloc/localization_demo_snn.py:151-163 (rms of the whole frame against a threshold)
//   power summed over the bands    micloc/localization_demo_snn.py:172-189 (power_grid += mean |y|^2, argmax)
//   DoA estimators                 micloc/xylo_snn_localization.py:400-444 ("peak", "periodic_ml", "trimmed_periodic_ml")
//
// In the reference's float path the filterbank comes BEFORE each band's STHT, so the F chains see F different inputs:
// the per-band chain (STHT included) stays the fused kernel of micloc_fused_tc.cu, launched once per band on the rows
// this file's filterbank kernel writes; the Xylo path, whose filterbank follows one shared STHT, fans out inside
// micloc_xylo.cu.
#include <cuda_runtime.h>
#include <math.h>

#include "micloc_common.h"

namespace micloc {

template <typename T> __device__ __forceinline__ float fb_to_f32(T v) { return (float)v; }

// one thread per (clip, microphone): reads its sample once, steps the F band-pass cascades, writes F rows.
// out [F][B][T][M] float32; sumsq [B] (nullable) += sum over the clip's kept channels of x^2 (float64)
template <typename IN_T>
__global__ void __launch_bounds__(128)
k_filterbank(const IN_T *__restrict__ audio, float *__restrict__ out, double *__restrict__ sumsq,
             const __grid_constant__ FilterbankParams fp, long long B, long long T, int in_ch, int M) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * M) return;
    const long long b = i / M;
    const int m = (int)(i % M);
    const IN_T *src = audio + b * T * in_ch + m;
    BiquadState st[8];
#pragma unroll
    for (int f = 0; f < 8; ++f) biquad_reset(st[f]);
    double ss = 0.0;
    float part = 0.f;
    for (long long t = 0; t < T; ++t) {
        const float x = fb_to_f32<IN_T>(src[t * in_ch]);
        part = fmaf(x, x, part);
        if ((t & 255) == 255) { ss += (double)part; part = 0.f; }
#pragma unroll
        for (int f = 0; f < 8; ++f)          // (unrolled with a predicate: the states stay in registers)
            if (f < fp.F) out[((long long)f * B + b) * T * M + t * M + m] = biquad_step(fp.sos[f], fp.nsec, st[f], x);
    }
    if (sumsq) atomicAdd(sumsq + b, ss + (double)part);
}

struct FuseParams {
    int F, G;
    const int32_t *band_flags[8];              // multi-band stream batches: each band's per-slot flags, or all null
};

// one CTA per clip: power_sum[g] = sum_f power[f][b][g] (bands added in order, float64 like the reference's
// power_grid), first argmax, periodic ML = angle(mean(p e^{j doa})), trimmed periodic ML = the same over
// arange(-G/2 // 2, G/2 // 2 + 1) - argmax with numpy's negative-index wrap (an index below -G is the reference's
// IndexError: flags bit 1, estimate NaN).  rows_b (nullable, multi-band stream batches): a clip with rows_b[b] == 0
// has no power rows and is not written.  With band_flags, flags[b] is first set to the OR of the bands' bit 0;
// without, the caller zeroes flags.
__global__ void __launch_bounds__(256)
k_power_fuse(const float *__restrict__ power, const double *__restrict__ doa_list, float *__restrict__ power_sum,
             int32_t *__restrict__ doa, double *__restrict__ ml, double *__restrict__ trimmed, int32_t *__restrict__ flags,
             const int32_t *__restrict__ rows_b, const __grid_constant__ FuseParams fp, long long B) {
    extern __shared__ double s_p[];            // [G] summed pattern
    __shared__ double s_red[3][8];
    __shared__ int s_idx[8];
    __shared__ int s_arg;
    const long long b = blockIdx.x;
    if (rows_b && rows_b[b] == 0) return;      // (uniform across the block: before any barrier)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = fp.G;
    double best = -1.0; int bi = 0x7fffffff;
    double re = 0.0, im = 0.0;
    for (int g = tid; g < G; g += blockDim.x) {
        double p = 0.0;
        for (int f = 0; f < fp.F; ++f) p += (double)power[((long long)f * B + b) * G + g];
        s_p[g] = p;
        if (power_sum) power_sum[b * G + g] = (float)p;
        if (p > best) { best = p; bi = g; }
        if (doa_list) { double s, c; sincos(doa_list[g], &s, &c); re += p * c; im += p * s; }
    }
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
        re += __shfl_xor_sync(0xffffffffu, re, o);
        im += __shfl_xor_sync(0xffffffffu, im, o);
    }
    if (lane == 0) { s_red[0][warp] = best; s_idx[warp] = bi; s_red[1][warp] = re; s_red[2][warp] = im; }
    __syncthreads();
    if (tid == 0) {
        const int nw = blockDim.x >> 5;
        for (int w = 1; w < nw; ++w) {
            if (s_red[0][w] > best || (s_red[0][w] == best && s_idx[w] < bi)) { best = s_red[0][w]; bi = s_idx[w]; }
            re += s_red[1][w]; im += s_red[2][w];
        }
        s_arg = bi;
        if (doa) doa[b] = bi;
        if (flags && fp.band_flags[0]) {
            int v = 0;
            for (int f = 0; f < fp.F; ++f) v |= fp.band_flags[f][b] & 1;
            flags[b] = v;
        }
        if (ml && doa_list) ml[b] = atan2(im / G, re / G);
    }
    __syncthreads();
    if (trimmed && doa_list && warp == 0) {
        const int arg = s_arg;
        const int nd = G / 2;
        // np.arange(-nd // 2, nd // 2 + 1): python floor division of the negated count
        const int lo = -((nd + 1) / 2), hi = nd / 2;         // inclusive bounds
        double tr = 0.0, ti = 0.0;
        bool bad = false;
        for (int k = lo + lane; k <= hi; k += 32) {
            int idx = k - arg;
            if (idx < -G) { bad = true; continue; }
            if (idx < 0) idx += G;
            double s, c; sincos(doa_list[idx], &s, &c);
            tr += s_p[idx] * c; ti += s_p[idx] * s;
        }
        for (int o = 16; o > 0; o >>= 1) {
            tr += __shfl_xor_sync(0xffffffffu, tr, o);
            ti += __shfl_xor_sync(0xffffffffu, ti, o);
        }
        bad = __any_sync(0xffffffffu, bad);
        if (lane == 0) {
            const int n = hi - lo + 1;
            trimmed[b] = bad ? nan("") : atan2(ti / n, tr / n);
            if (bad && flags) atomicOr(flags + b, 2);
        }
    }
}

}  // namespace micloc

int micloc::filterbank_params(int32_t F, int32_t n_sections, const double *sos, FilterbankParams *out) {
    if (F < 1 || F > 8) return set_error(MICLOC_ERR_CONFIG, "filterbank of %d bands (1..8 supported)", F);
    if (n_sections < 1 || n_sections > kMaxSections) return set_error(MICLOC_ERR_CONFIG, "n_sections must be 1..%d", kMaxSections);
    FilterbankParams fp{};
    fp.F = F; fp.nsec = n_sections;
    for (int f = 0; f < F; ++f) MICLOC_TRY(sos_to_f32(sos + (size_t)f * n_sections * 6, n_sections, &fp.sos[f][0][0]));
    *out = fp;
    return MICLOC_OK;
}

int micloc::launch_power_fuse(const float *power, int F, long long B, int G, const double *doa_list, float *power_sum,
                              int32_t *doa, double *ml, double *trimmed, int32_t *flags, const int32_t *rows_b,
                              const int32_t *const *band_flags, cudaStream_t st) {
    FuseParams fp{};
    fp.F = F; fp.G = G;
    for (int f = 0; band_flags && f < F; ++f) fp.band_flags[f] = band_flags[f];
    const size_t smem = (size_t)G * sizeof(double);
    if (smem > 48 * 1024) MICLOC_CUDA(cudaFuncSetAttribute(k_power_fuse, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_power_fuse<<<(unsigned)B, 256, smem, st>>>(power, doa_list, power_sum, doa, ml, trimmed, flags, rows_b, fp, B);
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}

using namespace micloc;

extern "C" int micloc_filterbank(const void *audio_dev, int dtype, int64_t B, int64_t T, int32_t in_channels, int32_t M,
                                 int32_t F, int32_t n_sections, const double *sos, float *out_dev, double *sumsq_dev,
                                 int device, void *stream) {
    if (!audio_dev || !out_dev || !sos) return set_error(MICLOC_ERR_SHAPE, "null argument");
    if (B < 1 || T < 1 || M < 1) return set_error(MICLOC_ERR_SHAPE, "empty batch");
    if (in_channels < M)
        return set_error(MICLOC_ERR_SHAPE, "number of channels in the input siganl %d should be the same as the number of microphones %d!", in_channels, M);
    FilterbankParams fp;
    MICLOC_TRY(filterbank_params(F, n_sections, sos, &fp));
    MICLOC_CUDA(cudaSetDevice(device));
    cudaStream_t st = (cudaStream_t)stream;
    if (sumsq_dev) MICLOC_CUDA(cudaMemsetAsync(sumsq_dev, 0, (size_t)B * sizeof(double), st));
    const unsigned grid = (unsigned)((B * M + 127) / 128);
    if (dtype == MICLOC_F32) k_filterbank<float><<<grid, 128, 0, st>>>((const float *)audio_dev, out_dev, sumsq_dev, fp, B, T, in_channels, M);
    else if (dtype == MICLOC_I16) k_filterbank<int16_t><<<grid, 128, 0, st>>>((const int16_t *)audio_dev, out_dev, sumsq_dev, fp, B, T, in_channels, M);
    else if (dtype == MICLOC_I32) k_filterbank<int32_t><<<grid, 128, 0, st>>>((const int32_t *)audio_dev, out_dev, sumsq_dev, fp, B, T, in_channels, M);
    else return set_error(MICLOC_ERR_SHAPE, "dtype must be MICLOC_F32, MICLOC_I16 or MICLOC_I32");
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}

extern "C" int micloc_power_fuse(const float *power_dev, int32_t F, int64_t B, int32_t G, const double *doa_list_dev,
                                 float *power_sum_dev, int32_t *doa_dev, double *periodic_ml_dev, double *trimmed_ml_dev,
                                 int32_t *flags_dev, int device, void *stream) {
    if (!power_dev) return set_error(MICLOC_ERR_SHAPE, "null argument");
    if (F < 1 || B < 1 || G < 1) return set_error(MICLOC_ERR_SHAPE, "empty input");
    if ((periodic_ml_dev || trimmed_ml_dev) && !doa_list_dev) return set_error(MICLOC_ERR_SHAPE, "the ML estimators need doa_list");
    MICLOC_CUDA(cudaSetDevice(device));
    cudaStream_t st = (cudaStream_t)stream;
    if (flags_dev) MICLOC_CUDA(cudaMemsetAsync(flags_dev, 0, (size_t)B * sizeof(int32_t), st));
    return launch_power_fuse(power_dev, F, B, G, doa_list_dev, power_sum_dev, doa_dev, periodic_ml_dev, trimmed_ml_dev,
                             flags_dev, nullptr, nullptr, st);
}
