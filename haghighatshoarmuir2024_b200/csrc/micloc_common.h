// micloc_common.h -- host-side helpers shared by the API translation units.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/micloc_b200.h"
#include "micloc_device.cuh"

namespace micloc {

int set_error(int code, const char *fmt, ...);
void count_launch(int n);

#define MICLOC_CUDA(expr)                                                                         \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess)                                                                    \
            return ::micloc::set_error(MICLOC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,           \
                                       cudaGetErrorString(_e), __FILE__, __LINE__);               \
    } while (0)

#define MICLOC_TRY(expr)          \
    do {                          \
        int _rc = (expr);         \
        if (_rc != 0) return _rc; \
    } while (0)

// device scratch that only grows
struct DevBuf {
    void *ptr = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return 0;
        if (ptr) cudaFree(ptr);
        ptr = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&ptr, bytes);
        if (e != cudaSuccess)
            return set_error(MICLOC_ERR_CUDA, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
        cap = bytes;
        return 0;
    }
    void release() { if (ptr) cudaFree(ptr); ptr = nullptr; cap = 0; }
};

// Layout of the fused kernel's per-context counter block (32-bit words, device memory):
//   [0, 1024)            FIR warps placed per (SM, sub-partition): word 4*smid + smsp   (reset per launch)
//   [kSlotPair]          dynamic clip-pair counter                                      (reset per launch)
//   (kSlotPair, kSlotDbg) CTAs arrived per SM                                            (reset per launch)
//   [kSlotDbg, +64)      32 x 64-bit debug counters (MICLOC_ROLE_TIMING builds)
//   [kSlotCta, ...)      16 x 64-bit words per CTA for the first 512 CTAs (MICLOC_ROLE_TIMING builds)
constexpr int kSlotPair = 1024;
constexpr int kSlotDbg = 1280;
constexpr int kSlotCta = 1536;
constexpr size_t kSlotWords = kSlotCta + 2 * 16 * 512;
constexpr int kSlotResetWords = kSlotDbg;

int setup_stht(ChainParams &p, const double *h, int K, float **d_taps);
}  // namespace micloc

// what a stream (micloc_stream.cu) takes over from its parent context; valid until the context's bf_mat is replaced
struct micloc_snn_params {
    micloc::ChainParams chain;
    const void *taps_dev;       // float [n_taps]
    const void *bf_f32_dev;     // float [2M][G]
    const void *bf_f64_dev;     // double [2M][G]
    int device;
};
int micloc_snn_get_params(micloc_snn *ctx, micloc_snn_params *out);

namespace micloc {
int sos_to_f32(const double *sos, int nsec, float *out);
// the float32 band-pass sections of a filterbank of F <= 8 bands (micloc_multiband.cu)
struct FilterbankParams {
    int F, nsec;
    float sos[8][kMaxSections][5];
};
// checks F (1..8) and n_sections (1..kMaxSections), converts sos [F][n_sections][6] (host, float64)
int filterbank_params(int32_t F, int32_t n_sections, const double *sos, FilterbankParams *out);
// k_power_fuse over power [F][B][G]; rows_b (nullable): clip b with rows_b[b] == 0 is not written;
// band_flags (nullable, F device pointers [B]): flags[b] = OR of their bit 0 before the estimator bit is added
int launch_power_fuse(const float *power, int F, long long B, int G, const double *doa_list, float *power_sum,
                      int32_t *doa, double *ml, double *trimmed, int32_t *flags, const int32_t *rows_b,
                      const int32_t *const *band_flags, cudaStream_t st);
// power[b][g] = w_g^T gram_b w_g * inv_T (float64, stored as float32) and doa[b] = first argmax over g, for gram
// [B][C2][C2] float64.  The one place that picks the power kernel (micloc_snn_run_taps and the stream batches):
//   k_power_wide               C2 >= 32 and Gram + steering tile in <= 200 KB of shared memory (M <= 72), unless
//                              MICLOC_POWER_NARROW or rows_b
//   k_power_argmax<true>       otherwise while the Gram matrix fits the block's shared memory (M <= 84 on sm_100)
//   k_power_argmax<false>      beyond: Gram rows read from global memory
// rows_b (nullable): clip b averages over rows_b[b] rows (inv_T unused), a clip with no rows is not written.
// nchunk > 1: DoA slices on separate CTAs into cv / ci [B][nchunk], k_argmax_chunks then writes doa.
int launch_power(const double *gram, const double *Wd, float *power, int32_t *doa, int C2, int G, long long B,
                 double inv_T, const int32_t *rows_b, int nchunk, double *cv, int *ci, cudaStream_t st);
int launch_stht_any(const ChainParams &p, const float *d_taps, const void *audio, int dtype, float *q,
                    long long B, long long T, cudaStream_t st);
// time segments of the band-pass + RZCC kernel (k_chain_blk): segment s keeps samples [s*seg_len, (s+1)*seg_len) and
// runs from `warm` samples before them to `tail` samples after them; seg_len and warm are multiples of kSeg
struct ChainSegs { int seg_len, warm, tail, nseg; };
// one segment per chain: the sequential recurrence
inline ChainSegs sequential_chain(long long T) { return {(int)((T + kSeg - 1) & ~(long long)(kSeg - 1)), 0, 0, 1}; }
int launch_chain_any(const ChainParams &p, const ChainSegs &segs, const void *audio, int dtype, const float *q,
                     const float *band_sos, int nb, float *z, int8_t *spikes, int32_t *flags, long long B, long long T,
                     cudaStream_t st);
int launch_fused(const ChainParams &p, const float *d_taps, const double *d_Wd, const void *audio, int dtype,
                 long long B, long long T, int8_t *spikes, float *power, int32_t *doa, int32_t *flags,
                 unsigned int *sm_slots, int sm_count, cudaStream_t st);
bool fused_supported(const ChainParams &p);
// tensor-core variant (micloc_fused_tc.cu): STHT as a tcgen05 Toeplitz GEMM; the default where it applies
namespace tc {
int launch_fused(const ChainParams &p, const float *d_taps, const double *d_Wd, const void *audio, int dtype,
                 long long B, long long T, int8_t *spikes, float *power, int32_t *doa, int32_t *flags,
                 unsigned int *sm_slots, int sm_count, cudaStream_t st);
bool fused_supported(const ChainParams &p);
}  // namespace tc

}  // namespace micloc
