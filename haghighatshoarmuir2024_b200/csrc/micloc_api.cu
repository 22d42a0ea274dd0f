// micloc_api.cu -- C-ABI of the float SNN chain (include/micloc_b200.h).
// Host-side only: validates arguments the way the reference raises, owns device
// constants and scratch, and launches the kernels in micloc_staged.cuh /
// micloc_fused.cuh on the caller's stream.
#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/micloc_b200.h"
#include "micloc_common.h"
#include "micloc_staged.cuh"

using namespace micloc;

// ---------------------------------------------------------------------------
// error handling / bookkeeping
// ---------------------------------------------------------------------------
static thread_local std::string g_err;
static std::atomic<long long> g_launches{0};

int micloc::set_error(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
void micloc::count_launch(int n) { g_launches.fetch_add(n); }

extern "C" const char *micloc_last_error(void) { return g_err.c_str(); }
extern "C" int micloc_version(void) { return MICLOC_VERSION; }
extern "C" int64_t micloc_launch_count(void) { return g_launches.load(); }

// ---------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------
struct micloc_snn {
    int device = 0;
    ChainParams p{};
    float *d_taps = nullptr;       // [n_taps]
    float *d_sos = nullptr;        // [1][kMaxSections][5]
    float *d_W = nullptr;          // [C2][G] f32
    double *d_Wd = nullptr;        // [C2][G] f64
    unsigned int *d_sm_slots = nullptr;  // [3][kSlotWords]: per-SM CTA arrival counters + clip-pair counter of the fused
                                         // kernel (+ debug counters); one set per concurrently running launch: set 0 for
                                         // micloc_snn_run on the caller's stream, sets 1 and 2 for run_host's two streams
    cudaEvent_t ev_last = nullptr;       // recorded behind the last launch of micloc_snn_run / run_taps / gram: run_host's
                                         // private streams wait for it before they touch the shared scratch
    DevBuf q, spikes, vmem, gram, flags, part, chunkbuf;
    DevBuf rz, rzd, rspk, rflag;            // one clip's worth of scratch of the overflow path (heal_overflow)
    long long refined = 0;                  // clips redone with the unbounded encoder so far
    int32_t *h_flags_all = nullptr;         // pinned host copy of a run_host batch's flags
    size_t h_flags_cap = 0;
    // host staging for run_host
    DevBuf h_audio[2], h_spk[2], h_pow[2], h_doa[2], h_flg[2];
    cudaStream_t hs[2] = {nullptr, nullptr};
    bool timing = false;
    std::vector<cudaEvent_t> ev;   // [2*i], [2*i+1] bracket the kernels of the i-th timed run
    size_t ev_used = 0;            // events recorded since the last micloc_snn_last_kernel_ms
    int last_kernels = 0;
    int sm_count = 148;
    double pole_radius = 1.0;      // largest pole modulus of the band-pass: how fast it forgets (time-segmented kernels)
};

// Time segments of the sequential stages (k_chain_blk / k_neuron_seg): the chain's, and neuron segments of
// seg_len_neuron samples that start nwarm samples early.
struct SegPlan { ChainSegs chain; int seg_len_neuron, nwarm, nseg_neuron; };
static SegPlan sequential_plan(long long T) { return {sequential_chain(T), (int)T, 0, 1}; }

// Few long clips (BASELINE config 5) are cut into time segments; everything else runs sequentially.
static SegPlan plan_segments(const micloc_snn *c, long long B, long long T, int nb) {
    const ChainParams &p = c->p;
    if (getenv("MICLOC_NO_SEGMENTS")) return sequential_plan(T);
    const long long chains = B * p.C2 * nb;
    if (chains >= 16384 || T < 32768) return sequential_plan(T);  // enough sequential chains to fill the GPU already
    if (!(c->pole_radius > 0.0 && c->pole_radius < 0.9995)) return sequential_plan(T);
    // band-pass transient below 1e-9 of full scale, the decision latency of the RZCC encoder on top
    int warm = (int)std::ceil(std::log(1e-9) / std::log(c->pole_radius)) + 2 * rzcc_lag(p.w);
    warm = (warm + 31) & ~31;
    // The chains are latency-bound (one dependent recurrence per thread): what counts is threads in flight, not work.
    // Aim at ONE full wave of the block-wise chain kernel -- 3 CTAs of 128 threads per SM (its register budget) -- and
    // never more: a few CTAs beyond the wave would run alone for a whole segment.  A segment is never shorter than its
    // own warm-up (2.1 x the sequential work at worst).
    long long want = (3ll * kChainBlkThreads * c->sm_count) / chains;        // segments per chain that fill the GPU
    if (want < 1) want = 1;
    long long seg = (T + want - 1) / want;
    if (seg < warm) seg = warm;
    seg = (seg + 31) & ~31ll;
    if (seg * 2 > T) return sequential_plan(T);
    SegPlan sp;
    sp.chain = {(int)seg, warm, rzcc_lag(p.w) + kSeg, (int)((T + seg - 1) / seg)};
    // alpha kernel h[n] = c n a^n: below 1e-12 of its peak
    sp.nwarm = (int)std::ceil(std::log(1e-12) / std::log((double)p.na)) + p.nL + 64;
    sp.seg_len_neuron = 1024 > 4 * sp.nwarm ? 1024 : 4 * sp.nwarm;
    sp.nseg_neuron = (int)((T + sp.seg_len_neuron - 1) / sp.seg_len_neuron);
    return sp;
}

static int upload_bf(micloc_snn *c, const double *bf, int G) {
    const int C2 = c->p.C2;
    std::vector<float> wf((size_t)C2 * G);
    for (size_t i = 0; i < wf.size(); ++i) wf[i] = (float)bf[i];
    if (c->d_W) cudaFree(c->d_W);
    if (c->d_Wd) cudaFree(c->d_Wd);
    c->d_W = nullptr; c->d_Wd = nullptr;
    MICLOC_CUDA(cudaMalloc(&c->d_W, wf.size() * sizeof(float)));
    MICLOC_CUDA(cudaMalloc(&c->d_Wd, wf.size() * sizeof(double)));
    MICLOC_CUDA(cudaMemcpy(c->d_W, wf.data(), wf.size() * sizeof(float), cudaMemcpyHostToDevice));
    MICLOC_CUDA(cudaMemcpy(c->d_Wd, bf, wf.size() * sizeof(double), cudaMemcpyHostToDevice));
    c->p.G = G;
    return MICLOC_OK;
}

// Shared by the SNN and the Xylo front end: fills the STHT part of ChainParams and
// uploads the compacted taps.  Taps below 1e-12 * max|h| are treated as zero (the
// Hilbert kernel's even taps are exact zeros or ~1e-19 FFT residue).
int micloc::setup_stht(ChainParams &p, const double *h, int K, float **d_taps) {
    if (K < 1 || K > 8192) return set_error(MICLOC_ERR_CONFIG, "kernel_len %d out of range [1, 8192]", K);
    double mx = 0.0;
    for (int k = 0; k < K; ++k) mx = std::fmax(mx, std::fabs(h[k]));
    const double thr = mx * 1e-12;
    int first = -1, last = -1;
    bool same_parity = true;
    for (int k = 0; k < K; ++k)
        if (std::fabs(h[k]) > thr) {
            if (first < 0) first = k;
            else if (((k - first) & 1) != 0) same_parity = false;
            last = k;
        }
    if (first < 0) { first = 0; last = 0; }
    const int stride = (same_parity && last > first) ? 2 : 1;
    int n = (last - first) / stride + 1;
    const int npad = (n + kFirJB - 1) / kFirJB * kFirJB;
    std::vector<float> taps(npad, 0.f);
    for (int j = 0; j < n; ++j) taps[j] = (float)h[first + stride * j];
    p.K = K; p.half = K / 2;
    p.tap_stride = stride; p.tap_first = first; p.n_taps = npad;
    p.span = first + stride * (npad - 1);
    p.tap_max = (float)mx;
    MICLOC_CUDA(cudaMalloc(d_taps, npad * sizeof(float)));
    MICLOC_CUDA(cudaMemcpy(*d_taps, taps.data(), npad * sizeof(float), cudaMemcpyHostToDevice));
    return MICLOC_OK;
}

int micloc::sos_to_f32(const double *sos, int nsec, float *out /* [kMaxSections][5] */) {
    if (nsec < 1 || nsec > kMaxSections)
        return set_error(MICLOC_ERR_CONFIG, "n_sections %d out of range [1, %d]", nsec, kMaxSections);
    for (int k = 0; k < kMaxSections * 5; ++k) out[k] = 0.f;
    for (int k = 0; k < nsec; ++k) {
        const double a0 = sos[k * 6 + 3];
        if (a0 == 0.0) return set_error(MICLOC_ERR_CONFIG, "sos section %d has a0 == 0", k);
        out[k * 5 + 0] = (float)(sos[k * 6 + 0] / a0);
        out[k * 5 + 1] = (float)(sos[k * 6 + 1] / a0);
        out[k * 5 + 2] = (float)(sos[k * 6 + 2] / a0);
        out[k * 5 + 3] = (float)(sos[k * 6 + 4] / a0);
        out[k * 5 + 4] = (float)(sos[k * 6 + 5] / a0);
    }
    return MICLOC_OK;
}

extern "C" int micloc_snn_create(const micloc_snn_config *cfg, int device, micloc_snn **out) {
    if (!cfg || !out) return set_error(MICLOC_ERR_CONFIG, "null config");
    *out = nullptr;
    if (cfg->num_mic < 1 || cfg->num_mic > 128)
        return set_error(MICLOC_ERR_CONFIG, "num_mic %d out of range [1, 128]", cfg->num_mic);
    if (!cfg->stht_kernel || !cfg->sos || !cfg->bf_mat) return set_error(MICLOC_ERR_CONFIG, "null array in config");
    if (cfg->robust_width < 1)
        return set_error(MICLOC_ERR_CONFIG, "`distance` must be greater or equal to 1");  // scipy find_peaks
    if (cfg->neuron_len < 1 || !(cfg->neuron_decay > 0.0 && cfg->neuron_decay < 1.0))
        return set_error(MICLOC_ERR_CONFIG, "bad neuron kernel (len %d, decay %g)", cfg->neuron_len, cfg->neuron_decay);
    if (cfg->num_doa < 1) return set_error(MICLOC_ERR_CONFIG, "num_doa must be >= 1");
    MICLOC_CUDA(cudaSetDevice(device));
    micloc_snn *c = new micloc_snn();
    c->device = device;
    ChainParams &p = c->p;
    p.M = cfg->num_mic; p.C2 = 2 * cfg->num_mic;
    int rc = setup_stht(p, cfg->stht_kernel, cfg->kernel_len, &c->d_taps);
    if (rc) { micloc_snn_destroy(c); return rc; }
    p.nsec = cfg->n_sections;
    rc = sos_to_f32(cfg->sos, cfg->n_sections, &p.sos[0][0]);
    if (rc) { micloc_snn_destroy(c); return rc; }
    c->pole_radius = 0.0;
    for (int k = 0; k < cfg->n_sections; ++k) {
        const double a1 = cfg->sos[k * 6 + 4] / cfg->sos[k * 6 + 3], a2 = cfg->sos[k * 6 + 5] / cfg->sos[k * 6 + 3];
        const double disc = a1 * a1 - 4.0 * a2;
        const double r = disc < 0.0 ? std::sqrt(a2) : (std::fabs(a1) + std::sqrt(disc)) / 2.0;
        if (r > c->pole_radius) c->pole_radius = r;
    }
    p.w = cfg->robust_width; p.bipolar = cfg->bipolar ? 1 : 0;
    p.na = (float)cfg->neuron_decay; p.nc = (float)cfg->neuron_scale; p.nL = cfg->neuron_len;
    p.ncT = (float)(cfg->neuron_scale * std::pow(cfg->neuron_decay, (double)cfg->neuron_len));
    p.nLf = (float)cfg->neuron_len;
    if (cudaMalloc(&c->d_sos, sizeof(float) * kMaxSections * 5) != cudaSuccess ||
        cudaMemcpy(c->d_sos, &p.sos[0][0], sizeof(float) * kMaxSections * 5, cudaMemcpyHostToDevice) != cudaSuccess) {
        micloc_snn_destroy(c);
        return set_error(MICLOC_ERR_CUDA, "cudaMalloc(sos) failed");
    }
    rc = upload_bf(c, cfg->bf_mat, cfg->num_doa);
    if (rc) { micloc_snn_destroy(c); return rc; }
    if (cudaMalloc(&c->d_sm_slots, 3 * kSlotWords * sizeof(unsigned int)) != cudaSuccess ||
        cudaMemset(c->d_sm_slots, 0, 3 * kSlotWords * sizeof(unsigned int)) != cudaSuccess ||
        cudaEventCreateWithFlags(&c->ev_last, cudaEventDisableTiming) != cudaSuccess) {
        micloc_snn_destroy(c);
        return set_error(MICLOC_ERR_CUDA, "cudaMalloc(sm_slots) failed");
    }
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    *out = c;
    return MICLOC_OK;
}

extern "C" int micloc_snn_destroy(micloc_snn *c) {
    if (!c) return MICLOC_OK;
    cudaSetDevice(c->device);
    cudaFree(c->d_taps); cudaFree(c->d_sos); cudaFree(c->d_W); cudaFree(c->d_Wd); cudaFree(c->d_sm_slots);
    c->q.release(); c->spikes.release(); c->vmem.release(); c->gram.release(); c->flags.release(); c->part.release(); c->chunkbuf.release();
    c->rz.release(); c->rzd.release(); c->rspk.release(); c->rflag.release();
    if (c->h_flags_all) cudaFreeHost(c->h_flags_all);
    for (int i = 0; i < 2; ++i) {
        c->h_audio[i].release(); c->h_spk[i].release(); c->h_pow[i].release(); c->h_doa[i].release(); c->h_flg[i].release();
        if (c->hs[i]) cudaStreamDestroy(c->hs[i]);
    }
    for (cudaEvent_t e : c->ev) cudaEventDestroy(e);
    if (c->ev_last) cudaEventDestroy(c->ev_last);
    delete c;
    return MICLOC_OK;
}

int micloc_snn_get_params(micloc_snn *c, micloc_snn_params *out) {
    if (!c || !out) return set_error(MICLOC_ERR_CONFIG, "null context");
    out->chain = c->p; out->taps_dev = c->d_taps; out->bf_f32_dev = c->d_W; out->bf_f64_dev = c->d_Wd; out->device = c->device;
    return MICLOC_OK;
}

extern "C" int micloc_snn_set_bf(micloc_snn *c, const double *bf, int32_t G) {
    if (!c || !bf || G < 1) return set_error(MICLOC_ERR_CONFIG, "bad bf_mat");
    MICLOC_CUDA(cudaSetDevice(c->device));
    MICLOC_CUDA(cudaDeviceSynchronize());
    return upload_bf(c, bf, G);
}

// Debug: busy cycles per warp role of the fused kernel (FIR slot 0, FIR slot 1, front, neuron) and
// the number of warps that reported, summed since the previous call; all zero unless the library
// was built with -DMICLOC_ROLE_TIMING.
extern "C" int micloc_snn_debug_counters(micloc_snn *c, uint64_t out[32]) {
    if (!c || !out) return set_error(MICLOC_ERR_CONFIG, "null argument");
    MICLOC_CUDA(cudaSetDevice(c->device));
    MICLOC_CUDA(cudaDeviceSynchronize());
    MICLOC_CUDA(cudaMemcpy(out, c->d_sm_slots + kSlotDbg, 32 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    MICLOC_CUDA(cudaMemset(c->d_sm_slots + kSlotDbg, 0, 32 * sizeof(uint64_t)));
    return MICLOC_OK;
}

// Debug: (start ns, end ns, SM id, role rotation, busy cycles of the 4 roles) of the first `n` CTAs of the last fused launch (MICLOC_ROLE_TIMING builds).
extern "C" int micloc_snn_debug_cta_times(micloc_snn *c, uint64_t *out, int32_t n) {
    if (!c || !out || n < 1 || n > 512) return set_error(MICLOC_ERR_CONFIG, "bad argument");
    MICLOC_CUDA(cudaSetDevice(c->device));
    MICLOC_CUDA(cudaDeviceSynchronize());
    MICLOC_CUDA(cudaMemcpy(out, c->d_sm_slots + kSlotCta, (size_t)n * 16 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return MICLOC_OK;
}

extern "C" int micloc_snn_enable_timing(micloc_snn *c, int enable) {
    if (!c) return set_error(MICLOC_ERR_CONFIG, "null context");
    c->timing = enable != 0;
    c->ev_used = 0;
    return MICLOC_OK;
}

// record one event of a (start, stop) pair on `st`; pairs accumulate until they are read
static int timing_mark(micloc_snn *c, cudaStream_t st) {
    if (!c->timing) return MICLOC_OK;
    if (c->ev_used == c->ev.size()) {
        if (c->ev.size() >= 16384) return MICLOC_OK;   // stop recording, keep running
        cudaEvent_t e;
        MICLOC_CUDA(cudaEventCreate(&e));
        c->ev.push_back(e);
    }
    MICLOC_CUDA(cudaEventRecord(c->ev[c->ev_used++], st));
    return MICLOC_OK;
}

extern "C" int micloc_snn_last_kernel_ms(micloc_snn *c, float *ms, int32_t *n_kernels) {
    if (!c || !c->timing) return set_error(MICLOC_ERR_CONFIG, "timing not enabled");
    double total = 0.0;
    const size_t pairs = c->ev_used / 2;
    for (size_t i = 0; i < pairs; ++i) {
        float v = 0.f;
        MICLOC_CUDA(cudaEventSynchronize(c->ev[2 * i + 1]));
        MICLOC_CUDA(cudaEventElapsedTime(&v, c->ev[2 * i], c->ev[2 * i + 1]));
        total += v;
    }
    c->ev_used = 0;
    if (ms) *ms = (float)total;
    if (n_kernels) *n_kernels = (int)pairs;
    return MICLOC_OK;
}

// ---------------------------------------------------------------------------
// launches
// ---------------------------------------------------------------------------
template <typename IN_T>
static int launch_stht(const ChainParams &p, const float *d_taps, const IN_T *audio, float *q,
                       long long B, long long T, cudaStream_t st) {
    if (p.tap_stride == 2 && p.M > 8 && p.tap_max * kStTapScale < 60000.f && stht_tc_smem(p.n_taps) <= 112 * 1024 &&
        T < (1ll << 30) && !getenv("MICLOC_STHT_FP32")) {
        // wide arrays: polyphase Toeplitz product on the tensor cores
        const int ntiles_tc = (int)((T + 32 * kStMB - 1) / (32 * kStMB));
        const size_t smem_tc = stht_tc_smem(p.n_taps);
        MICLOC_CUDA(cudaFuncSetAttribute(k_stht_tc<IN_T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tc));
        k_stht_tc<IN_T><<<dim3((unsigned)(B * ntiles_tc), (unsigned)((p.M + kStMics - 1) / kStMics)), kStThreads, smem_tc, st>>>(
            audio, q, d_taps, p, T, ntiles_tc);
        count_launch(1);
        MICLOC_CUDA(cudaGetLastError());
        return MICLOC_OK;
    }
    const int TT = 512;
    const int MG = p.M < 8 ? p.M : 8;
    const int ntiles = (int)((T + TT - 1) / TT);
    const size_t smem = (size_t)(((p.n_taps + 3) & ~3) + MG * fir_row_pitch(TT, p.span)) * sizeof(float);
    if (smem > 227 * 1024) return set_error(MICLOC_ERR_UNSUPPORTED, "STHT tile needs %zu B of shared memory", smem);
    dim3 grid((unsigned)(B * ntiles), (unsigned)((p.M + MG - 1) / MG));
    if (p.tap_stride == 2) {
        MICLOC_CUDA(cudaFuncSetAttribute(k_stht<IN_T, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_stht<IN_T, 2><<<grid, 256, smem, st>>>(audio, q, d_taps, p, T, TT, ntiles, MG);
    } else {
        MICLOC_CUDA(cudaFuncSetAttribute(k_stht<IN_T, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_stht<IN_T, 1><<<grid, 256, smem, st>>>(audio, q, d_taps, p, T, TT, ntiles, MG);
    }
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}

int micloc::launch_stht_any(const ChainParams &p, const float *d_taps, const void *audio, int dtype, float *q,
                            long long B, long long T, cudaStream_t st) {
    return dtype == MICLOC_I16 ? launch_stht<int16_t>(p, d_taps, (const int16_t *)audio, q, B, T, st)
                               : launch_stht<float>(p, d_taps, (const float *)audio, q, B, T, st);
}

int micloc::launch_chain_any(const ChainParams &p, const ChainSegs &segs, const void *audio, int dtype, const float *q,
                             const float *band_sos, int nb, float *z, int8_t *spikes, int32_t *flags,
                             long long B, long long T, cudaStream_t st) {
    // k_chain_blk counts time in int, up to one block of kSeg samples past the end
    if (T >= (1ll << 31) - kSeg) return set_error(MICLOC_ERR_SHAPE, "T = %lld too long for the chain kernel", T);
    MICLOC_CUDA(cudaMemsetAsync(spikes, 0, (size_t)B * T * p.C2 * nb, st));     // the kernel stores spikes only
    const long long n = B * segs.nseg * p.C2 * nb;
    const unsigned grid = (unsigned)((n + kChainBlkThreads - 1) / kChainBlkThreads);
    auto launch = [&](auto kernel, auto *x) {
        kernel<<<grid, kChainBlkThreads, 0, st>>>(x, q, band_sos, z, spikes, flags, p, B, T, nb, segs.seg_len, segs.warm,
                                                  segs.tail, segs.nseg);
    };
    if (dtype == MICLOC_I16)
        launch(p.nsec == 2 ? k_chain_blk<int16_t, 2> : k_chain_blk<int16_t, 0>, (const int16_t *)audio);
    else
        launch(p.nsec == 2 ? k_chain_blk<float, 2> : k_chain_blk<float, 0>, (const float *)audio);
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}

static int check_run_args(micloc_snn *c, const void *audio, int dtype, int64_t B, int64_t T) {
    if (!c) return set_error(MICLOC_ERR_CONFIG, "null context");
    if (!audio) return set_error(MICLOC_ERR_SHAPE, "null audio pointer");
    if (dtype != MICLOC_F32 && dtype != MICLOC_I16) return set_error(MICLOC_ERR_SHAPE, "dtype must be MICLOC_F32 or MICLOC_I16");
    if (B < 1 || T < 1) return set_error(MICLOC_ERR_SHAPE, "empty batch (B=%lld, T=%lld)", (long long)B, (long long)T);
    if (T > (1ll << 30)) return set_error(MICLOC_ERR_SHAPE, "T too large");
    return MICLOC_OK;
}

static int run_power(micloc_snn *c, const float *vmem, long long B, long long T, float *power, int32_t *doa,
                     cudaStream_t st) {
    const ChainParams &p = c->p;
    MICLOC_TRY(c->gram.reserve((size_t)B * p.C2 * p.C2 * sizeof(double)));
    dim3 gg((unsigned)B, (unsigned)((p.C2 * p.C2 + 255) / 256));
    const bool few_long = (long long)gg.x * gg.y < 2ll * c->sm_count && T >= 65536 && !getenv("MICLOC_NO_SEGMENTS");
    if (p.C2 >= 32 && T >= 256 && !getenv("MICLOC_NO_SEGMENTS")) {
        // wide arrays (BASELINE config 5: 128 channels): the Gram matrix is a real GEMM -- a tiled float32 product over
        // time slabs, summed in float64; clips go through in groups that bound the slab buffer to 1 GB
        const int nblk = (p.C2 + kGtTile - 1) / kGtTile, nblocks = nblk * (nblk + 1) / 2;
        const long long slab_len = kGtFlush;                                 // float32 sums of 1024 samples, float64 across slabs
        const long long nslab = (T + slab_len - 1) / slab_len;
        if (nslab > 65535) return set_error(MICLOC_ERR_UNSUPPORTED, "clip too long for the tiled Gram kernel");
        const size_t per_clip = (size_t)nslab * p.C2 * p.C2 * sizeof(double);
        long long bgrp = (long long)(((size_t)1 << 30) / per_clip);
        if (bgrp < 1) bgrp = 1;
        if (bgrp > B) bgrp = B;
        if (bgrp > 65535) bgrp = 65535;
        MICLOC_TRY(c->part.reserve((size_t)bgrp * per_clip));
        // tensor-core form (fp16 hi + lo of the membrane values x 2^12): needs |v| <= sum |h| < 15 to stay in fp16 range
        double habs = 0.0, an = 1.0;
        for (int n = 0; n < p.nL; ++n) { habs += (double)p.nc * n * an; an *= (double)p.na; }
        const bool tc = p.C2 >= 64 && habs < 15.0 && !getenv("MICLOC_GRAM_FP32");
        for (long long b0 = 0; b0 < B; b0 += bgrp) {
            const long long nb = B - b0 < bgrp ? B - b0 : bgrp;
            if (tc && nblk == 1)
                k_gram_tc<true><<<dim3((unsigned)nb, (unsigned)nblocks, (unsigned)nslab), 256, 0, st>>>(
                    vmem + (size_t)b0 * T * p.C2, (double *)c->part.ptr, p.C2, nb, T, 0, slab_len);
            else if (tc)
                k_gram_tc<false><<<dim3((unsigned)nb, (unsigned)nblocks, (unsigned)nslab), 256, 0, st>>>(
                    vmem + (size_t)b0 * T * p.C2, (double *)c->part.ptr, p.C2, nb, T, 0, slab_len);
            else
                k_gram_tiled<<<dim3((unsigned)nb, (unsigned)nblocks, (unsigned)nslab), 256, 0, st>>>(
                    vmem + (size_t)b0 * T * p.C2, (double *)c->part.ptr, p.C2, nb, T, 0, slab_len);
            const long long ne = nb * p.C2 * p.C2;
            k_gram_reduce<<<(unsigned)((ne + 31) / 32), 256, 0, st>>>((const double *)c->part.ptr,
                                                                       (double *)c->gram.ptr + (size_t)b0 * p.C2 * p.C2, p.C2, nb, (int)nslab);
            count_launch(2);
        }
    } else if (few_long) {
        // few long clips: time slabs so that the sum fills the GPU
        int nslab = (int)((4ll * c->sm_count + (long long)gg.x * gg.y - 1) / ((long long)gg.x * gg.y));
        if (nslab > 64) nslab = 64;
        const long long slab_len = (T + nslab - 1) / nslab;
        MICLOC_TRY(c->part.reserve((size_t)nslab * B * p.C2 * p.C2 * sizeof(double)));
        gg.z = (unsigned)nslab;
        k_gram_slab<<<gg, 256, 0, st>>>(vmem, (double *)c->part.ptr, p.C2, B, T, 0, slab_len);
        const long long ne = B * p.C2 * p.C2;
        k_gram_reduce<<<(unsigned)((ne + 31) / 32), 256, 0, st>>>((const double *)c->part.ptr, (double *)c->gram.ptr, p.C2, B, nslab);
        count_launch(2);
    } else {
        k_gram<<<gg, 256, 0, st>>>(vmem, (double *)c->gram.ptr, p.C2, T, 0);
        count_launch(1);
    }
    // few clips: slices of the DoA grid on separate CTAs (one CTA per clip would run G x C2^2 float64 FMAs on one SM)
    int nchunk = 1;
    if (B < c->sm_count && (long long)p.G * p.C2 * p.C2 >= (1ll << 20)) {
        nchunk = (int)((c->sm_count + B - 1) / B);
        const int max_chunk = (p.G + 31) / 32;
        if (nchunk > max_chunk) nchunk = max_chunk;
        if (nchunk < 1) nchunk = 1;
    }
    double *cv = nullptr; int *ci = nullptr;
    if (nchunk > 1) {
        MICLOC_TRY(c->chunkbuf.reserve((size_t)B * nchunk * (sizeof(double) + sizeof(int))));
        cv = (double *)c->chunkbuf.ptr;
        ci = (int *)(cv + (size_t)B * nchunk);
    }
    return launch_power((const double *)c->gram.ptr, c->d_Wd, power, doa, p.C2, p.G, B, 1.0 / (double)T, nullptr, nchunk,
                        cv, ci, st);
}

int micloc::launch_power(const double *gram, const double *Wd, float *power, int32_t *doa, int C2, int G, long long B,
                         double inv_T, const int32_t *rows_b, int nchunk, double *cv, int *ci, cudaStream_t st) {
    const size_t smem = (size_t)C2 * C2 * sizeof(double);
    const size_t smem_w = smem + ((size_t)C2 * 32 + (size_t)kPwSlices * 32) * sizeof(double);
    const dim3 grid((unsigned)B, (unsigned)nchunk);
    if (!rows_b && C2 >= 32 && smem_w <= 200 * 1024 && !getenv("MICLOC_POWER_NARROW")) {
        // wide arrays: a warp per slice of Gram rows x 32 DoAs (one thread per DoA leaves most of the CTA idle)
        MICLOC_CUDA(cudaFuncSetAttribute(k_power_wide, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_w));
        k_power_wide<<<grid, 32 * kPwSlices, smem_w, st>>>(gram, Wd, power, doa, C2, G, inv_T, nchunk, cv, ci);
    } else {
        // the Gram matrix in shared memory while it fits next to the kernel's static reduction scratch
        int dev = 0, optin = 0;
        cudaFuncAttributes fa{};
        MICLOC_CUDA(cudaGetDevice(&dev));
        MICLOC_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        MICLOC_CUDA(cudaFuncGetAttributes(&fa, k_power_argmax<true>));
        if (smem + fa.sharedSizeBytes <= (size_t)optin) {
            MICLOC_CUDA(cudaFuncSetAttribute(k_power_argmax<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k_power_argmax<true><<<grid, 256, smem, st>>>(gram, Wd, power, doa, C2, G, inv_T, nchunk, cv, ci, rows_b);
        } else {
            k_power_argmax<false><<<grid, 256, 0, st>>>(gram, Wd, power, doa, C2, G, inv_T, nchunk, cv, ci, rows_b);
        }
    }
    count_launch(1);
    if (nchunk > 1 && doa) {
        k_argmax_chunks<<<(unsigned)((B + 31) / 32), 32, 0, st>>>(cv, ci, doa, B, nchunk);
        count_launch(1);
    }
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}

// reads the clip flags back (synchronises `st`) and calls fn(i) for every clip i with bit 0 set, up to the first error
template <typename Fn>
static int for_flagged(const int32_t *flg, long long B, cudaStream_t st, Fn &&fn) {
    std::vector<int32_t> hf((size_t)B);
    MICLOC_CUDA(cudaMemcpyAsync(hf.data(), flg, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MICLOC_CUDA(cudaStreamSynchronize(st));
    for (long long i = 0; i < B; ++i)
        if (hf[(size_t)i] & 1) MICLOC_TRY(fn(i));
    return MICLOC_OK;
}

// ---------------------------------------------------------------------------
// RZCC overflow (flags bit 0): the streaming encoder of the staged / fused kernels buffers kClusterMax candidates per
// cluster and follows flat tops of kPlateauMax exact zeros (digital silence: the float32 band-pass output underflows
// to exact 0).  The staged entry points redo the spikes of such a clip HERE with the unbounded float64 encoder
// (micloc_rzcc_encode_f64 on the clip's band-pass output) and clear the bit; costs one flag read-back + stream sync.
// ---------------------------------------------------------------------------
static int heal_overflow(micloc_snn *c, const void *audio, int dtype, const float *q, float *z_dev, int8_t *spk,
                         int32_t *flg, long long B, long long T, cudaStream_t st) {
    const ChainParams &p = c->p;
    const size_t n_c = (size_t)T * p.C2, esz = dtype == MICLOC_I16 ? 2 : 4;
    return for_flagged(flg, B, st, [&](long long i) -> int {
        MICLOC_TRY(c->rzd.reserve(n_c * sizeof(double)));
        const float *z = z_dev ? z_dev + (size_t)i * n_c : nullptr;
        if (!z) {      // the band-pass output was not kept: once more for this clip
            MICLOC_TRY(c->rz.reserve(n_c * sizeof(float)));
            MICLOC_TRY(c->rspk.reserve(n_c));
            MICLOC_TRY(c->rflag.reserve(sizeof(int32_t)));
            MICLOC_TRY(launch_chain_any(p, sequential_chain(T), (const char *)audio + (size_t)i * T * p.M * esz, dtype,
                                        q + (size_t)i * T * p.M, c->d_sos, 1, (float *)c->rz.ptr, (int8_t *)c->rspk.ptr,
                                        (int32_t *)c->rflag.ptr, 1, T, st));
            z = (const float *)c->rz.ptr;
        }
        k_f32_to_f64<<<(unsigned)((n_c + 255) / 256), 256, 0, st>>>(z, (double *)c->rzd.ptr, (long long)n_c);
        count_launch(1);
        MICLOC_CUDA(cudaGetLastError());
        MICLOC_TRY(micloc_rzcc_encode_f64((const double *)c->rzd.ptr, 1, T, p.C2, p.w, p.bipolar, spk + (size_t)i * n_c,
                                          c->device, st));
        MICLOC_CUDA(cudaMemsetAsync(flg + i, 0, sizeof(int32_t), st));
        c->refined++;
        return MICLOC_OK;
    });
}

// The staged front end: flags reset -> STHT (q) -> band-pass (z, optional) + RZCC (spk) -> overflow heal -> neuron filter
// (vm; skipped when null).  Clips that a segmented chain could not vouch for (or whose cluster overflowed) are first
// redone sequentially: the sequential kernel's own overflow flag is then the clip's.
static int run_front(micloc_snn *c, const SegPlan &sp, const void *audio, int dtype, long long B, long long T, float *q,
                     float *z, int8_t *spk, int32_t *flg, float *vm, cudaStream_t st) {
    const ChainParams &p = c->p;
    MICLOC_CUDA(cudaMemsetAsync(flg, 0, (size_t)B * sizeof(int32_t), st));
    MICLOC_TRY(launch_stht_any(p, c->d_taps, audio, dtype, q, B, T, st));
    MICLOC_TRY(launch_chain_any(p, sp.chain, audio, dtype, q, c->d_sos, 1, z, spk, flg, B, T, st));
    if (sp.chain.nseg > 1) {
        const size_t esz = dtype == MICLOC_I16 ? 2 : 4;
        MICLOC_TRY(for_flagged(flg, B, st, [&](long long i) {
            MICLOC_CUDA(cudaMemsetAsync(flg + i, 0, sizeof(int32_t), st));
            return launch_chain_any(p, sequential_chain(T), (const char *)audio + (size_t)i * T * p.M * esz, dtype,
                                    q + (size_t)i * T * p.M, c->d_sos, 1, z ? z + (size_t)i * T * p.C2 : nullptr,
                                    spk + (size_t)i * T * p.C2, flg + i, 1, T, st);
        }));
    }
    MICLOC_TRY(heal_overflow(c, audio, dtype, q, z, spk, flg, B, T, st));
    if (!vm) return MICLOC_OK;
    const long long n = B * sp.nseg_neuron * p.C2;
    k_neuron_seg<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(spk, vm, p, B, T, sp.seg_len_neuron, sp.nwarm, sp.nseg_neuron);
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}

extern "C" int micloc_snn_run_taps(micloc_snn *c, const void *audio, int dtype, int64_t B, int64_t T,
                                   float *q_dev, float *z_dev, int8_t *spikes_dev, float *vmem_dev,
                                   float *y_dev, float *power_dev, int32_t *doa_dev, int32_t *flags_dev,
                                   void *stream) {
    MICLOC_TRY(check_run_args(c, audio, dtype, B, T));
    MICLOC_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const ChainParams &p = c->p;
    const size_t n_q = (size_t)B * T * p.M, n_c = (size_t)B * T * p.C2;
    float *q = q_dev; int8_t *spk = spikes_dev; float *vm = vmem_dev; int32_t *flg = flags_dev;
    if (!q) { MICLOC_TRY(c->q.reserve(n_q * sizeof(float))); q = (float *)c->q.ptr; }
    if (!spk) { MICLOC_TRY(c->spikes.reserve(n_c)); spk = (int8_t *)c->spikes.ptr; }
    if (!vm) { MICLOC_TRY(c->vmem.reserve(n_c * sizeof(float))); vm = (float *)c->vmem.ptr; }
    if (!flg) { MICLOC_TRY(c->flags.reserve((size_t)B * sizeof(int32_t))); flg = (int32_t *)c->flags.ptr; }
    MICLOC_TRY(timing_mark(c, st));
    const long long l0 = g_launches.load();
    const bool need_vmem = vmem_dev || y_dev || power_dev || doa_dev;
    MICLOC_TRY(run_front(c, plan_segments(c, B, T, 1), audio, dtype, B, T, q, z_dev, spk, flg, need_vmem ? vm : nullptr, st));
    if (power_dev || doa_dev) MICLOC_TRY(run_power(c, vm, B, T, power_dev, doa_dev, st));
    if (y_dev) {
        const int slab = 256;
        dim3 grid((unsigned)((p.G + 127) / 128), (unsigned)((T + slab - 1) / slab), (unsigned)B);
        if (B > 65535) return set_error(MICLOC_ERR_UNSUPPORTED, "dense output supports B <= 65535");
        if (p.C2 <= 16) k_dense<16><<<grid, 128, 0, st>>>(vm, c->d_W, y_dev, p.C2, p.G, T, slab);
        else k_dense<0><<<grid, 128, 0, st>>>(vm, c->d_W, y_dev, p.C2, p.G, T, slab);
        count_launch(1);
        MICLOC_CUDA(cudaGetLastError());
    }
    MICLOC_TRY(timing_mark(c, st));
    c->last_kernels = (int)(g_launches.load() - l0);
    MICLOC_CUDA(cudaEventRecord(c->ev_last, st));
    return MICLOC_OK;
}

extern "C" int micloc_snn_gram(micloc_snn *c, const void *audio, int dtype, int64_t B, int64_t T,
                               int64_t t_start, double *gram_dev, void *stream) {
    MICLOC_TRY(check_run_args(c, audio, dtype, B, T));
    if (!gram_dev || t_start < 0 || t_start >= T) return set_error(MICLOC_ERR_SHAPE, "bad gram output / t_start");
    MICLOC_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const ChainParams &p = c->p;
    const size_t n_q = (size_t)B * T * p.M, n_c = (size_t)B * T * p.C2;
    MICLOC_TRY(c->q.reserve(n_q * sizeof(float)));
    MICLOC_TRY(c->spikes.reserve(n_c));
    MICLOC_TRY(c->vmem.reserve(n_c * sizeof(float)));
    MICLOC_TRY(c->flags.reserve((size_t)B * sizeof(int32_t)));
    MICLOC_TRY(run_front(c, sequential_plan(T), audio, dtype, B, T, (float *)c->q.ptr, nullptr, (int8_t *)c->spikes.ptr,
                         (int32_t *)c->flags.ptr, (float *)c->vmem.ptr, st));
    dim3 gg((unsigned)B, (unsigned)((p.C2 * p.C2 + 255) / 256));
    k_gram<<<gg, 256, 0, st>>>((const float *)c->vmem.ptr, gram_dev, p.C2, T, t_start);
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    MICLOC_CUDA(cudaEventRecord(c->ev_last, st));
    return MICLOC_OK;
}

// `slot_set` picks the counter block of the fused kernel: launches that may overlap in time (the two
// staging streams of micloc_snn_run_host) must not share the dynamic clip-pair counter.
static int snn_run_impl(micloc_snn *c, const void *audio, int dtype, int64_t B, int64_t T,
                        int8_t *spikes_dev, float *power_dev, int32_t *doa_dev, int32_t *flags_dev,
                        int fused, void *stream, int slot_set) {
    if (!fused)
        return micloc_snn_run_taps(c, audio, dtype, B, T, nullptr, nullptr, spikes_dev, nullptr, nullptr,
                                   power_dev, doa_dev, flags_dev, stream);
    MICLOC_TRY(check_run_args(c, audio, dtype, B, T));
    MICLOC_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    int32_t *flg = flags_dev;
    if (!flg) { MICLOC_TRY(c->flags.reserve((size_t)B * sizeof(int32_t))); flg = (int32_t *)c->flags.ptr; }
    MICLOC_TRY(timing_mark(c, st));
    const long long l0 = g_launches.load();
    MICLOC_CUDA(cudaMemsetAsync(flg, 0, (size_t)B * sizeof(int32_t), st));
    MICLOC_TRY(launch_fused(c->p, c->d_taps, c->d_Wd, audio, dtype, B, T, spikes_dev, power_dev, doa_dev, flg,
                            c->d_sm_slots + (size_t)slot_set * kSlotWords, c->sm_count, st));
    MICLOC_TRY(timing_mark(c, st));
    c->last_kernels = (int)(g_launches.load() - l0);
    if (slot_set == 0) MICLOC_CUDA(cudaEventRecord(c->ev_last, st));
    return MICLOC_OK;
}

extern "C" int micloc_snn_run(micloc_snn *c, const void *audio, int dtype, int64_t B, int64_t T,
                              int8_t *spikes_dev, float *power_dev, int32_t *doa_dev, int32_t *flags_dev,
                              int fused, void *stream) {
    return snn_run_impl(c, audio, dtype, B, T, spikes_dev, power_dev, doa_dev, flags_dev, fused, stream, 0);
}

// ---------------------------------------------------------------------------
// The fused kernel only REPORTS an overflowed clip (flags bit 0): micloc_snn_run stays stream-ordered.  micloc_snn_refine
// is its synchronising companion: it reads the flags back and reruns every flagged clip through the staged kernels,
// which heal the overflow themselves (heal_overflow).  micloc_snn_run_host calls it on its own.
// ---------------------------------------------------------------------------
extern "C" int micloc_snn_refine(micloc_snn *c, const void *audio, int dtype, int64_t B, int64_t T, int8_t *spikes_dev,
                                 float *power_dev, int32_t *doa_dev, int32_t *flags_dev, int64_t *n_refined, void *stream) {
    MICLOC_TRY(check_run_args(c, audio, dtype, B, T));
    if (n_refined) *n_refined = 0;
    if (!flags_dev) return set_error(MICLOC_ERR_SHAPE, "refine needs the flags of the run");
    MICLOC_CUDA(cudaSetDevice(c->device));
    const ChainParams &p = c->p;
    const size_t esz = dtype == MICLOC_I16 ? 2 : 4;
    const bool timing = c->timing;
    c->timing = false;                                   // the rerun is not a timed run of its own
    long long n = 0;
    const int rc = for_flagged(flags_dev, B, (cudaStream_t)stream, [&](long long i) {
        ++n;
        return micloc_snn_run_taps(c, (const char *)audio + (size_t)i * T * p.M * esz, dtype, 1, T, nullptr, nullptr,
                                   spikes_dev ? spikes_dev + (size_t)i * T * p.C2 : nullptr, nullptr, nullptr,
                                   power_dev ? power_dev + (size_t)i * p.G : nullptr, doa_dev ? doa_dev + i : nullptr,
                                   flags_dev + i, stream);
    });
    c->timing = timing;
    if (n_refined) *n_refined = n;
    return rc;
}

extern "C" int64_t micloc_snn_refined_count(micloc_snn *c) { return c ? c->refined : 0; }

// ---------------------------------------------------------------------------
// end-to-end with host buffers: two chunks in flight on two private streams
// ---------------------------------------------------------------------------
extern "C" int micloc_snn_run_host(micloc_snn *c, const void *audio_host, int dtype, int64_t B, int64_t T,
                                   int8_t *spikes_host, float *power_host, int32_t *doa_host,
                                   int32_t *flags_host, int fused) {
    MICLOC_TRY(check_run_args(c, audio_host, dtype, B, T));
    MICLOC_CUDA(cudaSetDevice(c->device));
    const ChainParams &p = c->p;
    const size_t esz = dtype == MICLOC_I16 ? 2 : 4;
    const size_t clip_in = (size_t)T * p.M * esz, clip_spk = (size_t)T * p.C2;
    // chunk so that two chunks of input stay under ~1 GiB and every chunk fills the GPU
    long long chunk = (long long)((512ull << 20) / clip_in);
    if (const char *e = getenv("MICLOC_HOST_CHUNK_CLIPS")) {   // tests: force several chunks on small batches
        const long long v = atoll(e);
        if (v > 0) chunk = v;
    }
    if (chunk < 1) chunk = 1;
    if (chunk > B) chunk = B;
    if ((size_t)B > c->h_flags_cap) {
        if (c->h_flags_all) cudaFreeHost(c->h_flags_all);
        c->h_flags_all = nullptr; c->h_flags_cap = 0;
        MICLOC_CUDA(cudaHostAlloc((void **)&c->h_flags_all, (size_t)B * sizeof(int32_t), cudaHostAllocDefault));
        c->h_flags_cap = (size_t)B;
    }
    for (int i = 0; i < 2; ++i) {
        if (!c->hs[i]) MICLOC_CUDA(cudaStreamCreateWithFlags(&c->hs[i], cudaStreamNonBlocking));
        MICLOC_TRY(c->h_audio[i].reserve((size_t)chunk * clip_in));
        if (spikes_host) MICLOC_TRY(c->h_spk[i].reserve((size_t)chunk * clip_spk));
        MICLOC_TRY(c->h_pow[i].reserve((size_t)chunk * p.G * sizeof(float)));
        MICLOC_TRY(c->h_doa[i].reserve((size_t)chunk * sizeof(int32_t)));
        MICLOC_TRY(c->h_flg[i].reserve((size_t)chunk * sizeof(int32_t)));
    }
    // whatever micloc_snn_run / run_taps / gram left running on the caller's stream owns the context scratch until it
    // is done: both private streams wait for it
    for (int i = 0; i < 2; ++i) MICLOC_CUDA(cudaStreamWaitEvent(c->hs[i], c->ev_last, 0));
    // the staged path shares one scratch set, so its chunks are serialised on stream 0
    int slot = 0;
    for (long long b0 = 0; b0 < B; b0 += chunk, slot ^= fused ? 1 : 0) {
        const long long nb = (B - b0 < chunk) ? (B - b0) : chunk;
        cudaStream_t st = c->hs[slot];
        MICLOC_CUDA(cudaMemcpyAsync(c->h_audio[slot].ptr, (const char *)audio_host + (size_t)b0 * clip_in,
                                    (size_t)nb * clip_in, cudaMemcpyHostToDevice, st));
        int8_t *d_spk = spikes_host ? (int8_t *)c->h_spk[slot].ptr : nullptr;
        float *d_pow = power_host ? (float *)c->h_pow[slot].ptr : nullptr;
        int rc = snn_run_impl(c, c->h_audio[slot].ptr, dtype, nb, T, d_spk, d_pow, (int32_t *)c->h_doa[slot].ptr,
                              (int32_t *)c->h_flg[slot].ptr, fused, st, 1 + slot);
        if (rc) return rc;
        if (spikes_host)
            MICLOC_CUDA(cudaMemcpyAsync(spikes_host + (size_t)b0 * clip_spk, d_spk, (size_t)nb * clip_spk,
                                        cudaMemcpyDeviceToHost, st));
        if (power_host)
            MICLOC_CUDA(cudaMemcpyAsync(power_host + (size_t)b0 * p.G, d_pow, (size_t)nb * p.G * sizeof(float),
                                        cudaMemcpyDeviceToHost, st));
        if (doa_host)
            MICLOC_CUDA(cudaMemcpyAsync(doa_host + b0, c->h_doa[slot].ptr, (size_t)nb * sizeof(int32_t),
                                        cudaMemcpyDeviceToHost, st));
        if (flags_host)
            MICLOC_CUDA(cudaMemcpyAsync(flags_host + b0, c->h_flg[slot].ptr, (size_t)nb * sizeof(int32_t),
                                        cudaMemcpyDeviceToHost, st));
        MICLOC_CUDA(cudaMemcpyAsync(c->h_flags_all + b0, c->h_flg[slot].ptr, (size_t)nb * sizeof(int32_t),
                                    cudaMemcpyDeviceToHost, st));       // the library's own copy (pinned): overflow check below
    }
    MICLOC_CUDA(cudaStreamSynchronize(c->hs[0]));
    MICLOC_CUDA(cudaStreamSynchronize(c->hs[1]));
    // clips whose RZCC clusters overflowed the streaming encoder are redone one by one through the staged kernels (rare)
    if (fused) {
        cudaStream_t st = c->hs[0];
        const int32_t *fl = (const int32_t *)c->h_flags_all;
        for (long long i = 0; i < B; ++i) {
            if (!(fl[i] & 1)) continue;
            MICLOC_CUDA(cudaMemcpyAsync(c->h_audio[0].ptr, (const char *)audio_host + (size_t)i * clip_in, clip_in,
                                        cudaMemcpyHostToDevice, st));
            int8_t *d_spk = spikes_host ? (int8_t *)c->h_spk[0].ptr : nullptr;
            float *d_pow = power_host ? (float *)c->h_pow[0].ptr : nullptr;
            MICLOC_TRY(micloc_snn_run_taps(c, c->h_audio[0].ptr, dtype, 1, T, nullptr, nullptr, d_spk, nullptr, nullptr, d_pow,
                                           (int32_t *)c->h_doa[0].ptr, (int32_t *)c->h_flg[0].ptr, st));
            if (spikes_host) MICLOC_CUDA(cudaMemcpyAsync(spikes_host + (size_t)i * clip_spk, d_spk, clip_spk, cudaMemcpyDeviceToHost, st));
            if (power_host) MICLOC_CUDA(cudaMemcpyAsync(power_host + (size_t)i * p.G, d_pow, (size_t)p.G * sizeof(float), cudaMemcpyDeviceToHost, st));
            if (doa_host) MICLOC_CUDA(cudaMemcpyAsync(doa_host + i, c->h_doa[0].ptr, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
            if (flags_host) MICLOC_CUDA(cudaMemcpyAsync(flags_host + i, c->h_flg[0].ptr, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
            MICLOC_CUDA(cudaStreamSynchronize(st));
        }
    }
    return MICLOC_OK;
}

// ---------------------------------------------------------------------------
// Beamformer.apply_to_signal (micloc/beamformer.py:260-292)
// ---------------------------------------------------------------------------
extern "C" int micloc_hilbert_beamform(micloc_snn *c, const void *audio, int dtype, int64_t B, int64_t T,
                                       const double *bf_re, const double *bf_im, int32_t G, float *y_dev,
                                       float *power_dev, int32_t *doa_dev, void *stream) {
    MICLOC_TRY(check_run_args(c, audio, dtype, B, T));
    if (!bf_re || !bf_im || G < 1 || !y_dev) return set_error(MICLOC_ERR_SHAPE, "bad beamforming matrix / output");
    if (B > 65535) return set_error(MICLOC_ERR_UNSUPPORTED, "hilbert_beamform supports B <= 65535");
    MICLOC_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const ChainParams &p = c->p;
    const size_t n_q = (size_t)B * T * p.M, n_c = (size_t)B * T * p.C2;
    MICLOC_TRY(c->q.reserve(n_q * sizeof(float)));
    MICLOC_TRY(c->vmem.reserve(n_c * sizeof(float)));   // holds z
    MICLOC_TRY(c->spikes.reserve(n_c));
    MICLOC_TRY(c->flags.reserve((size_t)B * sizeof(int32_t)));
    MICLOC_TRY(c->part.reserve((size_t)2 * p.M * G * sizeof(float)));
    std::vector<float> w((size_t)2 * p.M * G);
    for (size_t i = 0; i < (size_t)p.M * G; ++i) { w[i] = (float)bf_re[i]; w[(size_t)p.M * G + i] = (float)bf_im[i]; }
    MICLOC_CUDA(cudaMemcpyAsync(c->part.ptr, w.data(), w.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    MICLOC_CUDA(cudaStreamSynchronize(st));  // w is a stack-owned vector
    float *z = (float *)c->vmem.ptr;
    MICLOC_TRY(launch_stht_any(p, c->d_taps, audio, dtype, (float *)c->q.ptr, B, T, st));
    MICLOC_TRY(launch_chain_any(p, sequential_chain(T), audio, dtype, (float *)c->q.ptr, c->d_sos, 1, z,
                                (int8_t *)c->spikes.ptr, (int32_t *)c->flags.ptr, B, T, st));
    const int slab = 256;
    dim3 grid((unsigned)((G + 127) / 128), (unsigned)((T + slab - 1) / slab), (unsigned)B);
    const float *bfr = (const float *)c->part.ptr, *bfi = bfr + (size_t)p.M * G;
    k_cproject<<<grid, 128, 0, st>>>(z, bfr, bfi, (float2 *)y_dev, p.M, G, T, slab);
    count_launch(1);
    if (power_dev || doa_dev) {
        k_cpower_argmax<<<(unsigned)B, 256, 0, st>>>((const float2 *)y_dev, power_dev, doa_dev, G, T);
        count_launch(1);
    }
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}

// ---------------------------------------------------------------------------
// DoA histogram of a batch (the only thing that crosses GPUs: SURVEY.md 8e)
// ---------------------------------------------------------------------------
namespace micloc {
__global__ void __launch_bounds__(256)
k_doa_hist(const int32_t *__restrict__ doa, long long B, int G, unsigned long long *__restrict__ hist) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B) return;
    const int g = doa[i];
    if (g >= 0 && g < G) atomicAdd(hist + g, 1ull);
}
}  // namespace micloc

extern "C" int micloc_doa_histogram(const int32_t *doa_dev, int64_t B, int32_t G, int64_t *hist_dev, int device,
                                    void *stream) {
    if (!doa_dev || !hist_dev || B < 0 || G < 1) return set_error(MICLOC_ERR_SHAPE, "bad histogram arguments");
    if (B == 0) return MICLOC_OK;
    MICLOC_CUDA(cudaSetDevice(device));
    k_doa_hist<<<(unsigned)((B + 255) / 256), 256, 0, (cudaStream_t)stream>>>(doa_dev, B, G,
                                                                             (unsigned long long *)hist_dev);
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}
