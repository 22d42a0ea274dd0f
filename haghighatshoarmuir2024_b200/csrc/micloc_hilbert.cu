// micloc_hilbert.cu -- the Hilbert beamformer at batch scale (micloc_hilbert_localize).
//
// s_t = zr_t + i zi_t, the band-passed analytic signal, in the real layout z = [zr | zi] ([T][2M]) that k_chain_blk
// produces.  Everything the Beamformer needs from a clip is its real 2M x 2M Gram matrix G = sum_{t >= t_start} z_t z_t^T:
//   power[g] = (u_g^T G u_g + v_g^T G v_g) / n_rows,  u = [wr; wi], v = [-wi; wr]   (y_t = sum_m s_tm conj(w_m))
//   cov      = S^H S = (Grr + Gii) + i (Gri - Gir)                                  (design_from_template)
// so the dense y [T][G] of micloc_hilbert_beamform is never formed.
//
// A channel's z is k_chain_blk's: the same input (ClipChannelInput: np.roll of the microphone, or the STHT output) and
// the same band-pass (biquad_cascade), so z equals run_taps' z tap bit for bit on the sequential plan.
//
// Kernels per chunk of clips (launch count independent of the chunk's size):
//   2M <= 16:  k_stht / k_stht_tc -> k_hilbert_gram (roll + band-pass + float64 Gram, z stays on chip) -> k_hilbert_finish
//   2M >  16:  k_stht / k_stht_tc -> k_hilbert_z (roll + band-pass -> z) -> k_gram_tiled -> k_hilbert_finish
// k_gram_tc is not used: its fp16 scaling assumes |v| < 15 (membrane values); z of int16 audio is in the thousands.
//
// HILBERT STREAM BATCHES (micloc_hilbert_streams_*): S live recordings through F band chains, state carried across
// pushes.  A batch is a SlotBook (latency D = 0) and a BankFront (micloc_stream.cuh, shared with the multi-band SNN
// batch; it has no filterbank state without a filterbank) plus, per band, the [K-1 history | frame] buffers, the STHT
// output and one BiquadState per (slot, channel) of the band-pass.  A slot at N == 0 (new or reset) starts from zero
// filter state, so reset only rewrites positions.  Per push, whatever S:
//   k_mb_stream_assemble (filterbank) or k_stream_assemble (none)                                         1
//   per band: STHT, k_hilbert_gram_stream (2M <= 16) or k_hilbert_z_stream + k_gram_tiled (2M > 16)        2 or 3
//             k_hilbert_finish when cov, power or a fused output is asked for                              +1
//   k_power_fuse when power_grid, doa, the estimators or flags are asked for                               +1
#include <cuda_runtime.h>

#include <cmath>

#include "micloc_common.h"
#include "micloc_staged.cuh"
#include "micloc_stream.cuh"

namespace micloc {

constexpr int kHbLanes = 16;                 // lanes per (clip, segment) unit of k_hilbert_gram: lane c < 2M is channel c
constexpr int kHbThreads = 128;
constexpr int kHbUnits = kHbThreads / kHbLanes;
constexpr int kHbPitch = kHbLanes + 1;       // column 16 stays zero: Gram entries beyond 2M(2M+1)/2 read it
constexpr int kHbEntries = (kHbLanes * (kHbLanes + 1) / 2 + kHbLanes - 1) / kHbLanes;   // upper-triangle entries per lane

// Time segments (see hilbert_segments): segment s keeps [s seg_len, (s+1) seg_len) and runs the band-pass from `warm` samples
// before it from zero state (warm = 0 without band-pass: z is then exact in every segment).
struct HbSegs { int seg_len, warm, nseg; };

// The float64 Gram matrix of one 16-lane unit (lane c < 2M is channel c): lane `lane` owns the entries
// e = lane + 16 k of the upper triangle, row-major (beyond the triangle: column 16, which stays zero).  A block of kSeg
// band-passed samples is staged in the unit's shared rows zu as float64, then every lane adds its <= 9 entries over the
// block's rows [i0, i1) (float64 FMAs in time order).  The one-shot and the stream kernels accumulate through it.
struct HbGram {
    int ei[kHbEntries], ej[kHbEntries];
    double acc[kHbEntries];

    __device__ __forceinline__ HbGram(double (*zu)[kHbPitch], int lane, int C2) {
        for (int i = 0; i < kSeg; ++i) zu[i][kHbLanes] = 0.0;   // (each lane writes the same zero)
        const int npair = C2 * (C2 + 1) / 2;
#pragma unroll
        for (int k = 0; k < kHbEntries; ++k) {
            int e = lane + kHbLanes * k, i = 0;
            if (e < npair) {
                while (e >= C2 - i) { e -= C2 - i; ++i; }
                ei[k] = i; ej[k] = i + e;
            } else {
                ei[k] = ej[k] = kHbLanes;
            }
            acc[k] = 0.0;
        }
    }
    __device__ __forceinline__ void add_block(double (*zu)[kHbPitch], int lane, int C2, unsigned hmask,
                                              const float (&v)[kSeg], int i0, int i1) {
        __syncwarp(hmask);                               // the previous block's reads are done
#pragma unroll
        for (int i = 0; i < kSeg; ++i) zu[i][lane] = lane < C2 ? (double)v[i] : 0.0;
        __syncwarp(hmask);
        for (int i = i0; i < i1; ++i) {
#pragma unroll
            for (int k = 0; k < kHbEntries; ++k) acc[k] = fma(zu[i][ei[k]], zu[i][ej[k]], acc[k]);
        }
    }
    // the upper triangle into out [2M][2M], as k_gram_tiled writes a partial sum
    __device__ __forceinline__ void store(double *out, int C2) const {
#pragma unroll
        for (int k = 0; k < kHbEntries; ++k)
            if (ei[k] < kHbLanes) out[ei[k] * C2 + ej[k]] = acc[k];
    }
};

// ---------------------------------------------------------------------------
// 2M <= 16: one unit of 16 lanes per (clip, segment).  Each block of kSeg samples: lane c band-passes channel c into
// registers and stages it in shared memory as float64; then every lane adds its <= 9 upper-triangle entries of the Gram
// matrix over the block's rows t >= t_start (float64 FMAs in time order).  part[seg][b][i][j] (i <= j) as k_gram_tiled
// writes it; z goes to HBM only as the optional debug tap.
// ---------------------------------------------------------------------------
template <typename IN_T, int NSEC>
__global__ void __launch_bounds__(kHbThreads)
k_hilbert_gram(const IN_T *__restrict__ audio, const float *__restrict__ q, const float *__restrict__ band_sos,
               float *__restrict__ z_out, double *__restrict__ part, const __grid_constant__ ChainParams p, long long B,
               long long T64, int t_start, int seg_len, int warm, int nseg) {
    __shared__ double zs[kHbUnits][kSeg][kHbPitch];
    const int unit_l = threadIdx.x / kHbLanes, lane = threadIdx.x % kHbLanes;
    const long long unit = (long long)blockIdx.x * kHbUnits + unit_l;
    const bool live = unit < B * nseg;
    const long long b = live ? unit / nseg : 0;
    const int seg = live ? (int)(unit % nseg) : 0;
    const int C2 = p.C2, T = (int)T64;
    const int c = lane < C2 ? lane : C2 - 1;             // idle lanes shadow the last channel and stage zeros
    const unsigned hmask = 0xffffu << (threadIdx.x & 16);
    double (*zu)[kHbPitch] = zs[unit_l];
    HbGram gm(zu, lane, C2);

    const int start = seg * seg_len, end = min(T, start + seg_len);
    const int t_begin = max(0, start - warm);
    const int t_stop = live ? end : t_begin;
    const int t_lo = max(start, t_start);                // rows of the Gram sum
    const ClipChannelInput<IN_T> src(audio, q, p, b, c, T, t_begin);
    float sos[kMaxSections][5];
    load_sos(sos, band_sos);
    BiquadState bq; biquad_reset(bq);
    const int nsec = p.nsec;
    float x[kSeg];
    src.load(t_begin, t_stop, x);
    for (int ts = t_begin; ts < t_stop; ts += kSeg) {
        float v[kSeg];
#pragma unroll
        for (int i = 0; i < kSeg; ++i) v[i] = biquad_cascade<NSEC>(sos, nsec, bq, x[i]);
        if (ts + kSeg < t_stop) src.load(ts + kSeg, t_stop, x);
        if (ts + kSeg <= start) continue;                // warm-up only (uniform across the unit)
        if (z_out && lane < C2) {
            float *zo = z_out + ((long long)b * T + ts) * C2 + lane;
#pragma unroll
            for (int i = 0; i < kSeg; ++i)
                if (ts + i >= start && ts + i < end) zo[(long long)i * C2] = v[i];
        }
        const int i0 = max(0, t_lo - ts), i1 = min(kSeg, end - ts);
        if (i0 >= i1) continue;
        gm.add_block(zu, lane, C2, hmask, v, i0, i1);
    }
    if (!live) return;
    gm.store(part + ((long long)seg * B + b) * C2 * C2, C2);
}

// ---------------------------------------------------------------------------
// 2M > 16: z of every (clip, segment, channel) to HBM; k_gram_tiled then sums it.
// ---------------------------------------------------------------------------
template <typename IN_T, int NSEC>
__global__ void __launch_bounds__(kChainBlkThreads)
k_hilbert_z(const IN_T *__restrict__ audio, const float *__restrict__ q, const float *__restrict__ band_sos,
            float *__restrict__ z_out, const __grid_constant__ ChainParams p, long long B, long long T64, int seg_len,
            int warm, int nseg) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int C2 = p.C2, T = (int)T64;
    if (idx >= B * nseg * C2) return;
    const int c = (int)(idx % C2);
    const int seg = (int)((idx / C2) % nseg);
    const long long b = idx / ((long long)C2 * nseg);
    const int start = seg * seg_len, end = min(T, start + seg_len);
    const int t_begin = max(0, start - warm);
    const ClipChannelInput<IN_T> src(audio, q, p, b, c, T, t_begin);
    float sos[kMaxSections][5];
    load_sos(sos, band_sos);
    BiquadState bq; biquad_reset(bq);
    const int nsec = p.nsec;
    float x[kSeg];
    src.load(t_begin, end, x);
    for (int ts = t_begin; ts < end; ts += kSeg) {
        float v[kSeg];
#pragma unroll
        for (int i = 0; i < kSeg; ++i) v[i] = biquad_cascade<NSEC>(sos, nsec, bq, x[i]);
        if (ts + kSeg < end) src.load(ts + kSeg, end, x);
        float *zo = z_out + ((long long)b * T + ts) * C2 + c;
#pragma unroll
        for (int i = 0; i < kSeg; ++i)
            if (ts + i >= start && ts + i < end) zo[(long long)i * C2] = v[i];
    }
}

// ---------------------------------------------------------------------------
// One CTA per clip: G = sum of the nslab partial sums part[slab][b] (upper triangle, slab order: deterministic), then
//   cov[i][j] = (G[i][j] + G[M+i][M+j], G[i][M+j] - G[M+i][j])
//   power[g]  = (u^T G u + v^T G v) * inv_n,  u = W[:, g] = [wr; wi], v = [-wi; wr]   (float64, stored as float32)
//   doa       = first argmax.
// kSmem: G in shared memory (2M <= 128); otherwise in the global scratch `gram` [B][2M][2M].
// ---------------------------------------------------------------------------
template <bool kSmem>
__global__ void __launch_bounds__(256)
k_hilbert_finish(const double *__restrict__ part, int nslab, double *__restrict__ gram, const double *__restrict__ W,
                 int M, int G, long long B, double inv_n, double *__restrict__ cov, float *__restrict__ power,
                 int32_t *__restrict__ doa) {
    extern __shared__ __align__(16) double hf_sm[];
    __shared__ double red_v[256];
    __shared__ int red_i[256];
    const long long b = blockIdx.x;
    const int C2 = 2 * M;
    double *Gs = kSmem ? hf_sm : gram + b * C2 * C2;
    for (int e = threadIdx.x; e < C2 * C2; e += blockDim.x) {
        const int i = e / C2, j = e % C2;
        const int lo = i < j ? i : j, hi = i < j ? j : i;
        double s = 0.0;
        for (int k = 0; k < nslab; ++k) s += part[((long long)k * B + b) * C2 * C2 + lo * C2 + hi];
        Gs[e] = s;
    }
    __syncthreads();
    if (cov)
        for (int e = threadIdx.x; e < M * M; e += blockDim.x) {
            const int i = e / M, j = e % M;
            cov[(b * M * M + e) * 2] = Gs[i * C2 + j] + Gs[(M + i) * C2 + M + j];
            cov[(b * M * M + e) * 2 + 1] = Gs[i * C2 + M + j] - Gs[(M + i) * C2 + j];
        }
    if (!power && !doa) return;
    double best = -1.0; int besti = 0x7fffffff;
    for (int g = threadIdx.x; g < G; g += blockDim.x) {
        double acc = 0.0;
        for (int i = 0; i < C2; ++i) {
            double ru = 0.0, rv = 0.0;
            for (int j = 0; j < C2; ++j) {
                const double gij = Gs[i * C2 + j];
                const double uj = W[(long long)j * G + g];
                const double vj = j < M ? -W[(long long)(M + j) * G + g] : W[(long long)(j - M) * G + g];
                ru = fma(gij, uj, ru);
                rv = fma(gij, vj, rv);
            }
            const double ui = W[(long long)i * G + g];
            const double vi = i < M ? -W[(long long)(M + i) * G + g] : W[(long long)(i - M) * G + g];
            acc = fma(ui, ru, fma(vi, rv, acc));
        }
        acc *= inv_n;
        if (power) power[b * G + g] = (float)acc;
        if (acc > best) { best = acc; besti = g; }      // ascending g: first maximum kept
    }
    red_v[threadIdx.x] = best; red_i[threadIdx.x] = besti;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) {
            const double ov = red_v[threadIdx.x + s]; const int oi = red_i[threadIdx.x + s];
            if (ov > red_v[threadIdx.x] || (ov == red_v[threadIdx.x] && oi < red_i[threadIdx.x])) {
                red_v[threadIdx.x] = ov; red_i[threadIdx.x] = oi;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0 && doa) doa[b] = red_i[0];
}

// Time segments when the B clips of a chunk are too few chains to fill the GPU: about 3 x 128 chains per SM; a segment
// is never shorter than its band-pass warm-up (transient below 1e-9 of full scale), and never more than half the clip.
static HbSegs hilbert_segments(long long B, long long T, int lanes, bool bandpass, double pole_radius, int sm_count) {
    const HbSegs seq{(int)((T + kSeg - 1) & ~(long long)(kSeg - 1)), 0, 1};
    const long long chains = B * lanes;
    if (chains >= 3ll * kChainBlkThreads * sm_count || T < 32768) return seq;
    int warm = 0;
    if (bandpass) {
        if (!(pole_radius > 0.0 && pole_radius < 0.9995)) return seq;
        warm = (int)std::ceil(std::log(1e-9) / std::log(pole_radius));
        warm = (warm + kSeg - 1) & ~(kSeg - 1);
    }
    long long want = (3ll * kChainBlkThreads * sm_count) / chains;
    if (want < 1) want = 1;
    long long seg = (T + want - 1) / want;
    if (seg < warm) seg = warm;
    seg = (seg + kSeg - 1) & ~(long long)(kSeg - 1);
    if (seg * 2 > T) return seq;
    return {(int)seg, warm, (int)((T + seg - 1) / seg)};
}

template <typename IN_T, int NSEC>
static void launch_front(bool narrow, const IN_T *audio, const float *q, const float *sos, float *z, double *part,
                         const ChainParams &p, long long B, long long T, long long t_start, const HbSegs &sg,
                         cudaStream_t st) {
    if (narrow) {
        const long long units = B * sg.nseg;
        k_hilbert_gram<IN_T, NSEC><<<(unsigned)((units + kHbUnits - 1) / kHbUnits), kHbThreads, 0, st>>>(
            audio, q, sos, z, part, p, B, T, (int)t_start, sg.seg_len, sg.warm, sg.nseg);
    } else {
        const long long n = B * sg.nseg * p.C2;
        k_hilbert_z<IN_T, NSEC><<<(unsigned)((n + kChainBlkThreads - 1) / kChainBlkThreads), kChainBlkThreads, 0, st>>>(
            audio, q, sos, z, p, B, T, sg.seg_len, sg.warm, sg.nseg);
    }
}

template <typename IN_T>
static void launch_front_t(bool narrow, int nsec, const IN_T *audio, const float *q, const float *sos, float *z,
                           double *part, const ChainParams &p, long long B, long long T, long long t_start,
                           const HbSegs &sg, cudaStream_t st) {
    if (nsec == 0) launch_front<IN_T, 0>(narrow, audio, q, sos, z, part, p, B, T, t_start, sg, st);
    else if (nsec == 2) launch_front<IN_T, 2>(narrow, audio, q, sos, z, part, p, B, T, t_start, sg, st);
    else launch_front<IN_T, kNsecRuntime>(narrow, audio, q, sos, z, part, p, B, T, t_start, sg, st);
}

int hilbert_localize(const HilbertCtx &hc, HilbertScratch &s, const void *audio, int dtype, long long B, long long T,
                     long long t_start, int bandpass, float *z_dev, double *cov_dev, float *power_dev, int32_t *doa_dev,
                     cudaStream_t st) {
    const ChainParams &p = hc.p;
    const int C2 = p.C2;
    const bool narrow = C2 <= kHbLanes;
    const bool bp = bandpass != 0;
    ChainParams pz = p;
    if (!bp) pz.nsec = 0;
    const long long nslab_w = (T - t_start + kGtFlush - 1) / kGtFlush;     // k_gram_tiled's slabs (wide arrays)
    if (!narrow && nslab_w > 65535) return set_error(MICLOC_ERR_UNSUPPORTED, "clip too long for the tiled Gram kernel");
    // chunks of clips: STHT output, z (wide arrays, unless the caller keeps it) and the slab sums within ~1 GB
    const size_t esz = dtype == MICLOC_I16 ? 2 : 4;
    const size_t q_clip = (size_t)T * p.M * sizeof(float);
    const size_t z_clip = (!narrow && !z_dev) ? (size_t)T * C2 * sizeof(float) : 0;
    const size_t slab_clip = narrow ? 0 : (size_t)nslab_w * C2 * C2 * sizeof(double);
    long long chunk = (long long)(((size_t)1 << 30) / (q_clip + z_clip + slab_clip));
    if (chunk < 1) chunk = 1;
    if (chunk > 65535) chunk = 65535;
    if (chunk > B) chunk = B;
    // the chains of one chunk are what has to fill the GPU: time segments are planned for the chunk
    const HbSegs sg = hilbert_segments(chunk, T, narrow ? kHbLanes : C2, bp, hc.pole_radius, hc.sm_count);
    const long long nslab = narrow ? sg.nseg : nslab_w;
    const size_t part_clip = (size_t)nslab * C2 * C2 * sizeof(double);
    MICLOC_TRY(s.q.reserve((size_t)chunk * q_clip));
    if (z_clip) MICLOC_TRY(s.z.reserve((size_t)chunk * z_clip));
    MICLOC_TRY(s.part.reserve((size_t)chunk * part_clip));
    const bool smem = (size_t)C2 * C2 * sizeof(double) <= 128 * 1024;
    if (!smem) MICLOC_TRY(s.gram.reserve((size_t)chunk * C2 * C2 * sizeof(double)));
    const size_t smem_b = smem ? (size_t)C2 * C2 * sizeof(double) : 0;
    if (smem) MICLOC_CUDA(cudaFuncSetAttribute(k_hilbert_finish<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               (int)smem_b));
    const double inv_n = 1.0 / (double)(T - t_start);
    for (long long b0 = 0; b0 < B; b0 += chunk) {
        const long long nb = B - b0 < chunk ? B - b0 : chunk;
        const void *a = (const char *)audio + (size_t)b0 * T * p.M * esz;
        float *q = (float *)s.q.ptr;
        float *z = z_dev ? z_dev + (size_t)b0 * T * C2 : (narrow ? nullptr : (float *)s.z.ptr);
        double *part = (double *)s.part.ptr;
        MICLOC_TRY(launch_stht_any(p, hc.d_taps, a, dtype, q, nb, T, st));
        if (dtype == MICLOC_I16)
            launch_front_t<int16_t>(narrow, pz.nsec, (const int16_t *)a, q, hc.d_sos, z, part, pz, nb, T, t_start, sg, st);
        else
            launch_front_t<float>(narrow, pz.nsec, (const float *)a, q, hc.d_sos, z, part, pz, nb, T, t_start, sg, st);
        count_launch(1);
        if (!narrow) {
            const int nblk = (C2 + kGtTile - 1) / kGtTile, nblocks = nblk * (nblk + 1) / 2;
            k_gram_tiled<<<dim3((unsigned)nb, (unsigned)nblocks, (unsigned)nslab), 256, 0, st>>>(
                z, part, C2, nb, T, t_start, kGtFlush);
            count_launch(1);
        }
        const size_t o = (size_t)b0;
        double *cov = cov_dev ? cov_dev + o * p.M * p.M * 2 : nullptr;
        float *pw = power_dev ? power_dev + o * hc.G : nullptr;
        int32_t *dd = doa_dev ? doa_dev + o : nullptr;
        if (smem)
            k_hilbert_finish<true><<<(unsigned)nb, 256, smem_b, st>>>(part, (int)nslab, nullptr, hc.d_W, p.M, hc.G, nb,
                                                                      inv_n, cov, pw, dd);
        else
            k_hilbert_finish<false><<<(unsigned)nb, 256, 0, st>>>(part, (int)nslab, (double *)s.gram.ptr, hc.d_W, p.M,
                                                                  hc.G, nb, inv_n, cov, pw, dd);
        count_launch(1);
        MICLOC_CUDA(cudaGetLastError());
    }
    return MICLOC_OK;
}

// ---------------------------------------------------------------------------
// Stream forms.  Channel c of slot s reads the band's [hist | frame] rows: in-phase x[t - K/2] at row hist - K/2 + i,
// quadrature q at row hist + i (i = t - N, as k_stream_blk), and continues its band-pass from state [S][2M] (zero
// state at N == 0).  The filter stops after the frame's n samples: the state the next push continues from.
// ---------------------------------------------------------------------------
struct StreamChannelInput {
    const float *src;
    int M, n;
    __device__ __forceinline__ StreamChannelInput(const float *xbuf, const float *q, const ChainParams &p, long long s,
                                                  int c, int hist, int n_)
        : M(p.M), n(n_) {
        const long long base = s * ((long long)hist + n) * M;
        src = c < M ? xbuf + base + (long long)(hist - p.half) * M + c : q + base + (long long)hist * M + (c - M);
    }
    // x[i] = input of frame row i0 + i, 0 past the frame
    __device__ __forceinline__ void load(int i0, float (&x)[kSeg]) const {
        const float *pp = src + (long long)i0 * M;
        if (n - i0 >= kSeg) {
#pragma unroll
            for (int i = 0; i < kSeg; ++i) { x[i] = *pp; pp += M; }
        } else {
#pragma unroll
            for (int i = 0; i < kSeg; ++i) x[i] = i < n - i0 ? pp[(long long)i * M] : 0.f;
        }
    }
};

// v = band-pass of the block's nv valid inputs (zeros beyond, the state untouched by them)
template <int NSEC>
__device__ __forceinline__ void stream_bandpass(const float (&sos)[kMaxSections][5], int nsec, BiquadState &bq,
                                                const float (&x)[kSeg], int nv, float (&v)[kSeg]) {
    if (nv == kSeg) {
#pragma unroll
        for (int i = 0; i < kSeg; ++i) v[i] = biquad_cascade<NSEC>(sos, nsec, bq, x[i]);
    } else {
#pragma unroll
        for (int i = 0; i < kSeg; ++i) v[i] = i < nv ? biquad_cascade<NSEC>(sos, nsec, bq, x[i]) : 0.f;
    }
}

// 2M <= 16: one 16-lane unit per slot (k_hilbert_gram's body through HbGram); part [S][2M][2M] is the single partial
// sum k_hilbert_finish reads.  Every band's launch writes the same next positions and row counts m = n.
template <int NSEC>
__global__ void __launch_bounds__(kHbThreads)
k_hilbert_gram_stream(const float *__restrict__ xbuf, const float *__restrict__ q, const float *__restrict__ band_sos,
                      BiquadState *__restrict__ state, const SlotPos *__restrict__ pos_in, SlotPos *__restrict__ pos_out,
                      int32_t *__restrict__ m_out, float *__restrict__ z_out, double *__restrict__ part,
                      const __grid_constant__ ChainParams p, long long S, int n, int hist) {
    __shared__ double zs[kHbUnits][kSeg][kHbPitch];
    const int unit_l = threadIdx.x / kHbLanes, lane = threadIdx.x % kHbLanes;
    const long long unit = (long long)blockIdx.x * kHbUnits + unit_l;
    const bool live = unit < S;
    const long long s = live ? unit : 0;
    const int C2 = p.C2;
    const int c = lane < C2 ? lane : C2 - 1;             // idle lanes shadow the last channel and stage zeros
    const unsigned hmask = 0xffffu << (threadIdx.x & 16);
    double (*zu)[kHbPitch] = zs[unit_l];
    HbGram gm(zu, lane, C2);
    const SlotPos ps = pos_in[s];
    BiquadState bq;
    if (ps.N == 0) biquad_reset(bq);
    else bq = state[s * C2 + c];
    float sos[kMaxSections][5];
    load_sos(sos, band_sos);
    const int nsec = p.nsec;
    const StreamChannelInput src(xbuf, q, p, s, c, hist, n);
    const int t_stop = live ? n : 0;
    float x[kSeg];
    if (t_stop > 0) src.load(0, x);
    for (int ts = 0; ts < t_stop; ts += kSeg) {
        const int nv = min(kSeg, t_stop - ts);
        float v[kSeg];
        stream_bandpass<NSEC>(sos, nsec, bq, x, nv, v);
        if (ts + kSeg < t_stop) src.load(ts + kSeg, x);
        if (z_out && lane < C2) {
            float *zo = z_out + (s * n + ts) * C2 + lane;
#pragma unroll
            for (int i = 0; i < kSeg; ++i)
                if (i < nv) zo[(long long)i * C2] = v[i];
        }
        gm.add_block(zu, lane, C2, hmask, v, 0, nv);
    }
    if (!live) return;
    if (lane < C2) state[s * C2 + lane] = bq;
    if (lane == 0) { pos_out[s] = SlotPos{ps.N + n, ps.N + n, 1, 0}; m_out[s] = n; }
    gm.store(part + s * C2 * C2, C2);
}

// 2M > 16: one thread per (slot, channel) writes z [S][n][2M]; k_gram_tiled and k_hilbert_finish follow
template <int NSEC>
__global__ void __launch_bounds__(kChainBlkThreads)
k_hilbert_z_stream(const float *__restrict__ xbuf, const float *__restrict__ q, const float *__restrict__ band_sos,
                   BiquadState *__restrict__ state, const SlotPos *__restrict__ pos_in, SlotPos *__restrict__ pos_out,
                   int32_t *__restrict__ m_out, float *__restrict__ z_out, const __grid_constant__ ChainParams p,
                   long long S, int n, int hist) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int C2 = p.C2;
    if (idx >= S * C2) return;
    const int c = (int)(idx % C2);
    const long long s = idx / C2;
    const SlotPos ps = pos_in[s];
    BiquadState bq;
    if (ps.N == 0) biquad_reset(bq);
    else bq = state[idx];
    float sos[kMaxSections][5];
    load_sos(sos, band_sos);
    const int nsec = p.nsec;
    const StreamChannelInput src(xbuf, q, p, s, c, hist, n);
    float x[kSeg];
    src.load(0, x);
    for (int ts = 0; ts < n; ts += kSeg) {
        const int nv = min(kSeg, n - ts);
        float v[kSeg];
        stream_bandpass<NSEC>(sos, nsec, bq, x, nv, v);
        if (ts + kSeg < n) src.load(ts + kSeg, x);
        float *zo = z_out + (s * n + ts) * C2 + c;
#pragma unroll
        for (int i = 0; i < kSeg; ++i)
            if (i < nv) zo[(long long)i * C2] = v[i];
    }
    state[idx] = bq;
    if (c == 0) { pos_out[s] = SlotPos{ps.N + n, ps.N + n, 1, 0}; m_out[s] = n; }
}

// the listed slots (sel == nullptr: all) restart at sample 0
__global__ void __launch_bounds__(256)
k_hilbert_stream_reset(SlotPos *__restrict__ pos, const int32_t *__restrict__ sel, long long S) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s < S && (!sel || sel[s])) pos[s] = SlotPos{0, 0, 1, 0};
}

}  // namespace micloc

using namespace micloc;

// one band of a Hilbert stream batch
struct HilbertStreamBand {
    HilbertCtx hc;                  // the context's chain constants, taps and band-pass; d_W is the batch's own copy
    int hist = 0;                   // K - 1
    float *xbuf[2] = {nullptr, nullptr}, *q = nullptr;
    BiquadState *state = nullptr;   // [S][2M] band-pass state
    double *W = nullptr;            // [2M][G] copy of the context's complex steering matrix
};

struct micloc_hilbert_streams {
    int device = 0;
    SlotBook book;
    BankFront front;                // fb_state null: no filterbank, the single band takes the raw frames
    HilbertStreamBand band[8];
    float *z = nullptr;                 // [S][max_frame][2M] z scratch of the wide path
    double *part = nullptr;             // [nslab][S][2M][2M] Gram partial sums (reused band after band)
    double *gram = nullptr;             // [S][2M][2M] k_hilbert_finish's Gram when it does not fit shared memory
};

extern "C" int micloc_hilbert_streams_destroy(micloc_hilbert_streams *hs) {
    if (!hs) return MICLOC_OK;
    cudaSetDevice(hs->device);
    hs->book.destroy();
    for (int f = 0; f < hs->front.F; ++f) {
        HilbertStreamBand &b = hs->band[f];
        cudaFree(b.xbuf[0]); cudaFree(b.xbuf[1]); cudaFree(b.q); cudaFree(b.state); cudaFree(b.W);
    }
    hs->front.destroy();
    cudaFree(hs->z); cudaFree(hs->part); cudaFree(hs->gram);
    delete hs;
    return MICLOC_OK;
}

extern "C" int micloc_hilbert_streams_reset(micloc_hilbert_streams *hs, const int32_t *slots_host, int32_t n_slots,
                                            void *stream) {
    if (!hs) return set_error(MICLOC_ERR_CONFIG, "null stream");
    MICLOC_CUDA(cudaSetDevice(hs->device));
    cudaStream_t st = (cudaStream_t)stream;
    SlotBook &bk = hs->book;
    if (slots_host) MICLOC_TRY(bk.upload(slots_host, n_slots, st));
    k_hilbert_stream_reset<<<(unsigned)((bk.S + 255) / 256), 256, 0, st>>>(bk.pos[bk.pcur], slots_host ? bk.sel : nullptr, bk.S);
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    return bk.reset_done(slots_host != nullptr, st);
}

static int nslab_of(int C2, long long n) { return C2 <= kHbLanes ? 1 : (int)((n + kGtFlush - 1) / kGtFlush); }

extern "C" int micloc_hilbert_streams_create(micloc_snn *const *ctxs, int32_t F, int32_t n_sections, const double *sos,
                                             const double *doa_list, int32_t num_streams, int64_t max_frame_len,
                                             micloc_hilbert_streams **out) {
    if (!ctxs || !out) return set_error(MICLOC_ERR_CONFIG, "null argument");
    *out = nullptr;
    if (!sos && F > 1) return set_error(MICLOC_ERR_CONFIG, "%d bands need a filterbank (sos == NULL takes one band)", F);
    HilbertCtx hc[8];
    int dev[8];
    MICLOC_TRY(check_bands("Hilbert stream batch", ctxs, F, [&](int f, BandShape &b) -> int {
        MICLOC_TRY(hilbert_ctx(ctxs[f], &hc[f], &dev[f]));
        if (!hc[f].d_W) return set_error(MICLOC_ERR_CONFIG, "band %d has no Hilbert steering matrix (micloc_hilbert_set_bf)", f);
        b = {dev[f], hc[f].p.M, hc[f].G};
        return MICLOC_OK;
    }));
    MICLOC_CUDA(cudaSetDevice(dev[0]));
    micloc_hilbert_streams *hs = new micloc_hilbert_streams();
    hs->device = dev[0];
    int rc = hs->book.create(num_streams, max_frame_len);
    if (!rc) rc = hs->front.create(F, hc[0].p.M, hc[0].G, num_streams, n_sections, sos, doa_list);
    const size_t S = (size_t)num_streams, M = (size_t)hc[0].p.M, C2 = 2 * M, G = (size_t)hc[0].G;
    const bool narrow = (int)C2 <= kHbLanes;
    for (int f = 0; f < F && !rc; ++f) {
        HilbertStreamBand &b = hs->band[f];
        b.hc = hc[f];
        b.hist = hc[f].p.K - 1;
        const size_t rows = (size_t)b.hist + (size_t)max_frame_len;
        if (!(cudaMalloc(&b.xbuf[0], S * rows * M * sizeof(float)) == cudaSuccess &&
              cudaMalloc(&b.xbuf[1], S * rows * M * sizeof(float)) == cudaSuccess &&
              cudaMalloc(&b.q, S * rows * M * sizeof(float)) == cudaSuccess &&
              cudaMalloc(&b.state, S * C2 * sizeof(BiquadState)) == cudaSuccess &&
              cudaMalloc(&b.W, C2 * G * sizeof(double)) == cudaSuccess))
            rc = set_error(MICLOC_ERR_CUDA, "cudaMalloc(Hilbert stream batch) failed");
        else if (cudaMemcpy(b.W, hc[f].d_W, C2 * G * sizeof(double), cudaMemcpyDeviceToDevice) != cudaSuccess)
            rc = set_error(MICLOC_ERR_CUDA, "copy of band %d's steering matrix failed", f);
        b.hc.d_W = b.W;
    }
    const size_t nslab = (size_t)nslab_of((int)C2, max_frame_len);
    if (!rc && !(cudaMalloc(&hs->part, nslab * S * C2 * C2 * sizeof(double)) == cudaSuccess &&
                 (narrow || cudaMalloc(&hs->z, S * (size_t)max_frame_len * C2 * sizeof(float)) == cudaSuccess) &&
                 (C2 * C2 * sizeof(double) <= 128 * 1024 || cudaMalloc(&hs->gram, S * C2 * C2 * sizeof(double)) == cudaSuccess)))
        rc = set_error(MICLOC_ERR_CUDA, "cudaMalloc(Hilbert stream batch) failed");
    if (!rc) rc = micloc_hilbert_streams_reset(hs, nullptr, 0, nullptr);
    if (rc) { micloc_hilbert_streams_destroy(hs); return rc; }
    *out = hs;
    return MICLOC_OK;
}

extern "C" int micloc_hilbert_streams_latency(micloc_hilbert_streams *hs) { return hs ? hs->book.D : 0; }

// band f's chain over the newest [history | frame] buffers: STHT, band-pass + Gram (z to z_f when given), then cov and
// power from the Gram; the caller flips the book
template <int NSEC>
static int hilbert_stream_band(micloc_hilbert_streams *hs, int f, long long n, float *z_f, double *cov_f, float *power_f,
                               cudaStream_t st) {
    HilbertStreamBand &b = hs->band[f];
    const SlotBook &bk = hs->book;
    const ChainParams &p = b.hc.p;
    const long long S = bk.S;
    const int C2 = p.C2;
    const float *xb = b.xbuf[bk.xcur];
    MICLOC_TRY(launch_stht_any(p, b.hc.d_taps, xb, MICLOC_F32, b.q, S, b.hist + n, st));
    const SlotPos *pin = bk.pos[bk.pcur];
    SlotPos *pout = bk.pos[bk.pcur ^ 1];
    const int nslab = nslab_of(C2, n);
    if (C2 <= kHbLanes) {
        k_hilbert_gram_stream<NSEC><<<(unsigned)((S + kHbUnits - 1) / kHbUnits), kHbThreads, 0, st>>>(
            xb, b.q, b.hc.d_sos, b.state, pin, pout, bk.m, z_f, hs->part, p, S, (int)n, b.hist);
        count_launch(1);
    } else {
        float *z = z_f ? z_f : hs->z;
        k_hilbert_z_stream<NSEC><<<(unsigned)((S * C2 + kChainBlkThreads - 1) / kChainBlkThreads), kChainBlkThreads, 0, st>>>(
            xb, b.q, b.hc.d_sos, b.state, pin, pout, bk.m, z, p, S, (int)n, b.hist);
        const int nblk = (C2 + kGtTile - 1) / kGtTile, nblocks = nblk * (nblk + 1) / 2;
        k_gram_tiled<<<dim3((unsigned)S, (unsigned)nblocks, (unsigned)nslab), 256, 0, st>>>(z, hs->part, C2, S, n, 0, kGtFlush);
        count_launch(2);
    }
    MICLOC_CUDA(cudaGetLastError());
    if (!cov_f && !power_f) return MICLOC_OK;
    const double inv_n = 1.0 / (double)n;
    if (!hs->gram) {
        const size_t smem_b = (size_t)C2 * C2 * sizeof(double);
        MICLOC_CUDA(cudaFuncSetAttribute(k_hilbert_finish<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
        k_hilbert_finish<true><<<(unsigned)S, 256, smem_b, st>>>(hs->part, nslab, nullptr, b.W, p.M, b.hc.G, S, inv_n, cov_f,
                                                                 power_f, nullptr);
    } else {
        k_hilbert_finish<false><<<(unsigned)S, 256, 0, st>>>(hs->part, nslab, hs->gram, b.W, p.M, b.hc.G, S, inv_n, cov_f,
                                                             power_f, nullptr);
    }
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}

extern "C" int micloc_hilbert_streams_push(micloc_hilbert_streams *hs, const void *frames_dev, int dtype, int64_t n,
                                           int32_t in_channels, float *z_dev, double *cov_dev, float *power_dev,
                                           float *power_grid_dev, int32_t *doa_dev, double *periodic_ml_dev,
                                           double *trimmed_ml_dev, double *sumsq_dev, int32_t *flags_dev,
                                           int64_t *n_out_host, void *stream) {
    if (!hs || !frames_dev || !n_out_host) return set_error(MICLOC_ERR_SHAPE, "null argument");
    SlotBook &bk = hs->book;
    BankFront &fr = hs->front;
    MICLOC_TRY(bk.check_push(dtype, n, in_channels, fr.M));
    MICLOC_TRY(check_doa_list(fr.doa_list, periodic_ml_dev, trimmed_ml_dev));
    if (sumsq_dev && !fr.fb_state) return set_error(MICLOC_ERR_SHAPE, "sumsq needs the filterbank (sos != NULL at create)");
    MICLOC_CUDA(cudaSetDevice(hs->device));
    cudaStream_t st = (cudaStream_t)stream;
    const long long S = bk.S;
    if (fr.fb_state) MICLOC_TRY(fr.assemble(bk, hs->band, frames_dev, dtype, n, in_channels, sumsq_dev, st));
    else MICLOC_TRY(bk.assemble(hs->band[0].xbuf, frames_dev, dtype, n, in_channels, fr.M, hs->band[0].hist, st));
    const bool fuse = power_grid_dev || doa_dev || periodic_ml_dev || trimmed_ml_dev || flags_dev;
    float *power = power_dev ? power_dev : (fuse ? fr.power : nullptr);
    for (int f = 0; f < fr.F; ++f) {
        float *z_f = z_dev ? z_dev + (size_t)f * S * n * 2 * fr.M : nullptr;
        double *cov_f = cov_dev ? cov_dev + (size_t)f * S * fr.M * fr.M * 2 : nullptr;
        float *pw_f = power ? power + (size_t)f * S * fr.G : nullptr;
        const int nsec = hs->band[f].hc.p.nsec;
        MICLOC_TRY(nsec == 2 ? hilbert_stream_band<2>(hs, f, n, z_f, cov_f, pw_f, st)
                             : hilbert_stream_band<kNsecRuntime>(hs, f, n, z_f, cov_f, pw_f, st));
    }
    bk.pushed(n, n_out_host);
    if (!fuse) return MICLOC_OK;
    if (flags_dev) MICLOC_CUDA(cudaMemsetAsync(flags_dev, 0, (size_t)S * sizeof(int32_t), st));
    return fr.fuse(power, power_grid_dev, doa_dev, periodic_ml_dev, trimmed_ml_dev, flags_dev, nullptr, nullptr, st);
}
