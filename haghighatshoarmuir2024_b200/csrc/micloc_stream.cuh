// micloc_stream.cuh -- the slot book and frame assembly shared by the stream batches: the float SNN chain's stream and
// multi-band batches (micloc_stream.cu), the Xylo integer chain's (micloc_xylo.cu) and the Hilbert beamformer's
// (micloc_hilbert.cu).  The rule of where a slot stands and what a push, flush or reset does to it lives here once; each
// batch keeps its chain state and flags next to it.  The bank front (BankFront: band context checks, filterbank
// assembly, DoA list and power fusion) serves the multi-band SNN and the Hilbert batches.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "micloc_common.h"

namespace micloc {

// where a slot stands: samples pushed (N), samples returned as final (F), 0 once flushed.  Positions stay below
// 2^31 - 4096 (the host refuses a push beyond), so the kernels count time in int.
struct SlotPos { int N, F, active, pad; };

// [K-1 history rows | frame rows] of every slot: cur [S][hist + n][M].  History = the last hist rows of the previous
// push's buffer prev [S][hist + n_prev][M], zeros for a slot that starts (N == 0); frame rows converted to OUT_T
// (float for the float chain, double for the Xylo chain's exact front end: int32 wav samples are not float-exact),
// channels >= M dropped.
template <typename IN_T, typename OUT_T = float>
__global__ void __launch_bounds__(256)
k_stream_assemble(const IN_T *__restrict__ frames, const OUT_T *__restrict__ prev, OUT_T *__restrict__ cur,
                  const SlotPos *__restrict__ pos, long long S, int n, int n_prev, int in_ch, int M, int hist) {
    const long long rows = (long long)hist + n;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S * rows * M) return;
    const int m = (int)(i % M);
    const long long r = (i / M) % rows, s = i / (rows * M);
    OUT_T v;
    if (r < hist) v = pos[s].N > 0 ? prev[(s * (hist + n_prev) + n_prev + r) * M + m] : (OUT_T)0;
    else v = (OUT_T)frames[(s * n + (r - hist)) * in_ch + m];
    cur[i] = v;
}

// Multi-band frame assembly: one thread per (slot, microphone) steps the F band-pass cascades of the filterbank
// (biquad_cascade with the float32 sections of k_filterbank, so band f's rows are micloc_filterbank's bits for the whole
// recording) from its state in fb_state [F][S][M], and writes band f's [hist_f history rows | frame] buffer cur[f]
// [S][hist_f + n][M] directly; history from the band's previous buffer prev[f] [S][hist_f + n_prev][M].  A slot at
// N == 0 (new or reset) starts from zero filter state and zero history.  sumsq [S] (nullable, zeroed by the caller)
// += sum of x^2 over the frame's kept channels, float32 partials of 256 samples added in float64 as in k_filterbank.
struct MbAssembleParams {
    FilterbankParams fb;
    const float *prev[8];
    float *cur[8];
    int hist[8];
};

// NF = F is a template argument: the bands stay in registers, and the unrolled loop body stays small enough for the
// instruction cache.  A predicated loop over 8 bands inside a 16-sample unroll did not (20 k instructions): 3.5 ms per
// push at 1024 slots against 2.0 ms at 4096 slots in this form (F = 3, one B200).
template <typename IN_T, int NF>
__global__ void __launch_bounds__(128)
k_mb_stream_assemble(const IN_T *__restrict__ frames, BiquadState *__restrict__ fb_state, double *__restrict__ sumsq,
                     const SlotPos *__restrict__ pos, const __grid_constant__ MbAssembleParams ap, long long S, int n,
                     int n_prev, int in_ch, int M) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S * M) return;
    const long long s = i / M;
    const int m = (int)(i % M);
    const bool fresh = pos[s].N == 0;
    BiquadState st[NF];
    float *row[NF];                       // band f's first frame row of this (slot, microphone)
#pragma unroll
    for (int f = 0; f < NF; ++f) {
        if (fresh) biquad_reset(st[f]);
        else st[f] = fb_state[f * S * M + i];
        const int hist = ap.hist[f];
        float *cur = ap.cur[f] + s * ((long long)hist + n) * M + m;
        const float *prev = ap.prev[f] + (s * ((long long)hist + n_prev) + n_prev) * M + m;
#pragma unroll 4
        for (int r = 0; r < hist; ++r) cur[(long long)r * M] = fresh ? 0.f : prev[(long long)r * M];
        row[f] = cur + (long long)hist * M;
    }
    // the frame in blocks of 8 samples, the next block's loads issued before the current one is filtered
    constexpr int kBlk = 8;
    const IN_T *src = frames + s * (long long)n * in_ch + m;
    float nx[kBlk];
    auto load = [&](int t0) {
#pragma unroll
        for (int u = 0; u < kBlk; ++u) nx[u] = t0 + u < n ? (float)src[(long long)(t0 + u) * in_ch] : 0.f;
    };
    double ss = 0.0;
    float part = 0.f;
    load(0);
    for (int t0 = 0; t0 < n; t0 += kBlk) {
        float x[kBlk];
#pragma unroll
        for (int u = 0; u < kBlk; ++u) x[u] = nx[u];
        if (t0 + kBlk < n) load(t0 + kBlk);
#pragma unroll
        for (int u = 0; u < kBlk; ++u) {
            const int t = t0 + u;
            if (t < n) {
                part = fmaf(x[u], x[u], part);
                if ((t & 255) == 255) { ss += (double)part; part = 0.f; }
#pragma unroll
                for (int f = 0; f < NF; ++f)
                    row[f][(long long)t * M] = biquad_cascade<kNsecRuntime>(ap.fb.sos[f], ap.fb.nsec, st[f], x[u]);
            }
        }
    }
    if (sumsq) atomicAdd(sumsq + s, ss + (double)part);
#pragma unroll
    for (int f = 0; f < NF; ++f) fb_state[f * S * M + i] = st[f];
}

template <typename IN_T>
static void launch_mb_assemble(int F, unsigned grid, cudaStream_t st, const void *frames, BiquadState *fb_state,
                               double *sumsq, const SlotPos *pos, const MbAssembleParams &ap, long long S, int n,
                               int n_prev, int in_ch, int M) {
    static decltype(&k_mb_stream_assemble<IN_T, 1>) const ks[8] = {
        k_mb_stream_assemble<IN_T, 1>, k_mb_stream_assemble<IN_T, 2>, k_mb_stream_assemble<IN_T, 3>,
        k_mb_stream_assemble<IN_T, 4>, k_mb_stream_assemble<IN_T, 5>, k_mb_stream_assemble<IN_T, 6>,
        k_mb_stream_assemble<IN_T, 7>, k_mb_stream_assemble<IN_T, 8>};
    ks[F - 1]<<<grid, 128, 0, st>>>((const IN_T *)frames, fb_state, sumsq, pos, ap, S, n, n_prev, in_ch, M);
}

// The slots of one stream batch.  The chain kernel of a push or flush reads pos[pcur] and writes every slot's new
// position to pos[pcur ^ 1] and its number of final rows to m; the owner then calls pushed() / flushed(), which flip
// pcur and advance the host mirror N / F / active the same way, so that n_out is known without a device
// synchronisation.  Every band of a multi-band batch runs its chain on the same book: their kernels write identical
// positions.  Reset and flush take slot lists through upload(); reset_done() synchronises the stream, whether a list
// was given or not.  A push never synchronises.
struct SlotBook {
    long long S = 0, max_frame = 0;
    int D = 0;                      // output latency in samples
    SlotPos *pos[2] = {nullptr, nullptr};
    int pcur = 0;
    int32_t *m = nullptr;           // [S] final rows of the last push / flush
    int32_t *sel = nullptr;         // [S] slot list of the last upload (1 = listed)
    std::vector<long long> N, F;    // host mirror of the positions
    std::vector<char> active;
    std::vector<int32_t> sel_h;     // staging of the slot lists
    int xcur = 0;                   // assembly buffer xcur holds the newest [history | frame] rows (n_prev frame rows)
    long long n_prev = 0;

    int create(int32_t num_streams, int64_t max_frame_len) {
        if (num_streams < 1 || num_streams > 65535) return set_error(MICLOC_ERR_SHAPE, "num_streams %d out of range [1, 65535]", num_streams);
        if (max_frame_len < 1 || max_frame_len > (1ll << 24)) return set_error(MICLOC_ERR_SHAPE, "max_frame_len out of range");
        S = num_streams; max_frame = max_frame_len;
        N.assign((size_t)S, 0); F.assign((size_t)S, 0); active.assign((size_t)S, 1);
        const size_t bytes = (size_t)S * sizeof(int32_t);
        if (cudaMalloc(&pos[0], S * sizeof(SlotPos)) != cudaSuccess || cudaMalloc(&pos[1], S * sizeof(SlotPos)) != cudaSuccess ||
            cudaMalloc(&m, bytes) != cudaSuccess || cudaMalloc(&sel, bytes) != cudaSuccess)
            return set_error(MICLOC_ERR_CUDA, "cudaMalloc(slot positions) failed");
        return MICLOC_OK;
    }

    void destroy() { cudaFree(pos[0]); cudaFree(pos[1]); cudaFree(m); cudaFree(sel); }

    // slots_host [n_slots] (NULL = every slot) -> sel on the device; synchronises `st`: the staging vector is reused by
    // the next call
    int upload(const int32_t *slots_host, int32_t n_slots, cudaStream_t st) {
        if (slots_host && n_slots < 0) return set_error(MICLOC_ERR_SHAPE, "n_slots %d < 0", n_slots);
        for (int32_t i = 0; slots_host && i < n_slots; ++i)
            if (slots_host[i] < 0 || slots_host[i] >= S)
                return set_error(MICLOC_ERR_SHAPE, "slot %d out of range [0, %lld)", slots_host[i], S);
        sel_h.assign((size_t)S, slots_host ? 0 : 1);
        for (int32_t i = 0; slots_host && i < n_slots; ++i) sel_h[(size_t)slots_host[i]] = 1;
        MICLOC_CUDA(cudaMemcpyAsync(sel, sel_h.data(), (size_t)S * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        MICLOC_CUDA(cudaStreamSynchronize(st));
        return MICLOC_OK;
    }

    // the frame arguments of a push against the book
    int check_push(int dtype, int64_t n, int32_t in_channels, int M) const {
        if (n < 1 || n > max_frame) return set_error(MICLOC_ERR_SHAPE, "frame of %lld samples (stream takes 1..%lld)", (long long)n, max_frame);
        if (in_channels < M)
            return set_error(MICLOC_ERR_SHAPE, "number of channels in the input siganl %d should be the same as the number of microphones %d!", in_channels, M);
        if (dtype != MICLOC_F32 && dtype != MICLOC_I16 && dtype != MICLOC_I32)
            return set_error(MICLOC_ERR_SHAPE, "dtype must be MICLOC_F32, MICLOC_I16 or MICLOC_I32");
        for (long long s = 0; s < S; ++s)
            if (active[(size_t)s] && N[(size_t)s] + n >= (1ll << 31) - 4096)
                return set_error(MICLOC_ERR_SHAPE, "stream position exceeds 2^31 samples: reset the stream");
        return MICLOC_OK;
    }

    // k_stream_assemble of the frames into xbuf[xcur ^ 1]
    template <typename OUT_T>
    int assemble(OUT_T *const xbuf[2], const void *frames, int dtype, int64_t n, int32_t in_channels, int M, int hist,
                 cudaStream_t st) {
        const int nxt = xcur ^ 1;
        const unsigned ga = (unsigned)((S * (hist + n) * M + 255) / 256);
        const OUT_T *prev = xbuf[xcur];
        if (dtype == MICLOC_F32)
            k_stream_assemble<float, OUT_T><<<ga, 256, 0, st>>>((const float *)frames, prev, xbuf[nxt], pos[pcur], S, (int)n, (int)n_prev, in_channels, M, hist);
        else if (dtype == MICLOC_I16)
            k_stream_assemble<int16_t, OUT_T><<<ga, 256, 0, st>>>((const int16_t *)frames, prev, xbuf[nxt], pos[pcur], S, (int)n, (int)n_prev, in_channels, M, hist);
        else
            k_stream_assemble<int32_t, OUT_T><<<ga, 256, 0, st>>>((const int32_t *)frames, prev, xbuf[nxt], pos[pcur], S, (int)n, (int)n_prev, in_channels, M, hist);
        count_launch(1);
        MICLOC_CUDA(cudaGetLastError());
        assembled(n);
        return MICLOC_OK;
    }

    // after the assembly of a frame of n samples into xbuf[xcur ^ 1]: that buffer becomes the newest
    void assembled(long long n) { xcur ^= 1; n_prev = n; }

    // after the owner's reset kernels (listed = a slot list was uploaded): waits for them, the listed slots restart at 0
    int reset_done(bool listed, cudaStream_t st) {
        MICLOC_CUDA(cudaStreamSynchronize(st));
        for (size_t s = 0; s < (size_t)S; ++s)
            if (!listed || sel_h[s]) { N[s] = 0; F[s] = 0; active[s] = 1; }
        return MICLOC_OK;
    }

    // after the chain kernels of a push of n samples: n_out_host [S] = samples that became final
    void pushed(long long n, int64_t *n_out_host) {
        pcur ^= 1;
        for (size_t s = 0; s < (size_t)S; ++s) {
            n_out_host[s] = 0;
            if (!active[s]) continue;
            N[s] += n;
            const long long f = N[s] - D > F[s] ? N[s] - D : F[s];
            n_out_host[s] = f - F[s];
            F[s] = f;
        }
    }

    // after the chain kernels of a flush of the uploaded slots: they return the rest and stop
    void flushed(int64_t *n_out_host) {
        pcur ^= 1;
        for (size_t s = 0; s < (size_t)S; ++s) {
            n_out_host[s] = 0;
            if (!active[s] || !sel_h[s]) continue;
            n_out_host[s] = N[s] - F[s];
            F[s] = N[s];
            active[s] = 0;
        }
    }
};

struct BandShape { int device, M, G; };

// The band contexts ctxs [F] of a multi-band batch (`kind` in the errors): F in 1..8, none null, all on band 0's device
// with its M and G.  read(f, shape) reads band f's context for the caller and gives its shape, or an error code.
template <typename Read>
int check_bands(const char *kind, micloc_snn *const *ctxs, int32_t F, Read read) {
    if (F < 1 || F > 8) return set_error(MICLOC_ERR_CONFIG, "%s of %d bands (1..8 supported)", kind, F);
    BandShape b0{}, b{};
    for (int f = 0; f < F; ++f) {
        if (!ctxs[f]) return set_error(MICLOC_ERR_CONFIG, "null context of band %d", f);
        MICLOC_TRY(read(f, b));
        if (f == 0) b0 = b;
        if (b.device != b0.device)
            return set_error(MICLOC_ERR_CONFIG, "band %d's context is on device %d, band 0's on device %d", f, b.device, b0.device);
        if (b.M != b0.M || b.G != b0.G)
            return set_error(MICLOC_ERR_SHAPE, "band %d's context has %d microphones and %d DoAs, band 0's %d and %d", f,
                             b.M, b.G, b0.M, b0.G);
    }
    return MICLOC_OK;
}

// What sits in front of F band chains on one slot book (multi-band SNN and Hilbert stream batches): the filterbank with
// its state, the DoA list of the estimators and the per-band power that k_power_fuse adds up.
struct BankFront {
    int F = 0, M = 0, G = 0;
    long long S = 0;
    FilterbankParams fb{};
    BiquadState *fb_state = nullptr;    // [F][S][M] filterbank state (never read at N == 0), null: no filterbank
    double *doa_list = nullptr;         // [G] on the device, null: no ML estimators
    float *power = nullptr;             // [F][S][G] per-band power when the caller passes no power_dev

    // sos [F][n_sections][6] and doa_list [G] on the host, either may be NULL
    int create(int F_, int M_, int G_, long long S_, int32_t n_sections, const double *sos, const double *doa_list_host) {
        if (sos) MICLOC_TRY(filterbank_params(F_, n_sections, sos, &fb));
        F = F_; M = M_; G = G_; S = S_;
        if (cudaMalloc(&power, (size_t)F * S * G * sizeof(float)) != cudaSuccess ||
            (sos && cudaMalloc(&fb_state, (size_t)F * S * M * sizeof(BiquadState)) != cudaSuccess) ||
            (doa_list_host && (cudaMalloc(&doa_list, (size_t)G * sizeof(double)) != cudaSuccess ||
                               cudaMemcpy(doa_list, doa_list_host, (size_t)G * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess)))
            return set_error(MICLOC_ERR_CUDA, "filterbank front set-up failed");
        return MICLOC_OK;
    }

    void destroy() { cudaFree(fb_state); cudaFree(doa_list); cudaFree(power); }

    // k_mb_stream_assemble of the frames into every band's xbuf[bk.xcur ^ 1]; sumsq [S] (nullable) is zeroed first
    template <typename Band>
    int assemble(SlotBook &bk, const Band *band, const void *frames, int dtype, int64_t n, int32_t in_channels,
                 double *sumsq, cudaStream_t st) {
        MbAssembleParams ap{};
        ap.fb = fb;
        for (int f = 0; f < F; ++f) {
            ap.prev[f] = band[f].xbuf[bk.xcur]; ap.cur[f] = band[f].xbuf[bk.xcur ^ 1]; ap.hist[f] = band[f].hist;
        }
        if (sumsq) MICLOC_CUDA(cudaMemsetAsync(sumsq, 0, (size_t)S * sizeof(double), st));
        const unsigned grid = (unsigned)((S * M + 127) / 128);
        auto launch = dtype == MICLOC_F32 ? launch_mb_assemble<float> : dtype == MICLOC_I16 ? launch_mb_assemble<int16_t>
                                                                                        : launch_mb_assemble<int32_t>;
        launch(F, grid, st, frames, fb_state, sumsq, bk.pos[bk.pcur], ap, S, (int)n, (int)bk.n_prev, in_channels, M);
        count_launch(1);
        MICLOC_CUDA(cudaGetLastError());
        bk.assembled(n);
        return MICLOC_OK;
    }

    // k_power_fuse over power [F][S][G]: sum over the bands, argmax, estimators (rows_b, band_flags: launch_power_fuse)
    int fuse(const float *power_fb, float *power_grid, int32_t *doa, double *ml, double *trimmed, int32_t *flags,
             const int32_t *rows_b, const int32_t *const *band_flags, cudaStream_t st) const {
        return launch_power_fuse(power_fb, F, S, G, doa_list, power_grid, doa, ml, trimmed, flags, rows_b, band_flags, st);
    }
};

}  // namespace micloc
