// micloc_device.cuh -- device-side building blocks shared by the staged and the
// fused kernels of the SNN-localisation hot path (sm_100a).
//
// Reference sites restated (paths under /root/reference):
//   STHT FIR                    micloc/snn_beamformer.py:325-327
//   band-pass (as SOS cascade)  micloc/snn_beamformer.py:330-331
//   RZCC                        micloc/spike_encoder.py:115-137 (+ scipy find_peaks)
//   neuron alpha kernel         micloc/snn_beamformer.py:342-364
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace micloc {

constexpr int kMaxSections = 4;   // biquads per band-pass
constexpr int kClusterMax = 8;    // RZCC candidates buffered per open cluster
constexpr int kFirR = 16;         // consecutive outputs per thread in the FIR
constexpr int kFirJB = 8;         // taps per register block

// Constants of one SNN chain; lives in __grid_constant__ kernel parameters.
struct ChainParams {
    int M;            // microphones
    int C2;           // 2*M real channels (in-phase | quadrature)
    int K;            // STHT kernel length
    int half;         // K/2: circular shift of the in-phase branch
    int tap_stride;   // 1 (dense) or 2 (Hilbert: every other tap is zero)
    int tap_first;    // index k0 of the first kept tap
    int n_taps;       // kept taps, padded with zeros to a multiple of kFirJB
    int span;         // largest look-back = tap_first + tap_stride*(n_taps-1)
    float tap_max;    // largest |tap| (the tensor-core STHT keeps taps x 2^14 in fp16)
    int nsec;         // biquad sections
    float sos[kMaxSections][5];  // b0 b1 b2 a1 a2
    int w;            // RZCC distance (>=1)
    int bipolar;
    float na;         // neuron decay a
    float nc;         // neuron scale c
    float ncT;        // c * a^L
    float nLf;        // (float)L
    int nL;           // neuron kernel length L
    int G;
};

// ---------------------------------------------------------------------------
// input sample fetch (float32 or int16 PCM; int16 is used at face value)
// ---------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<int16_t>(int16_t v) { return (float)v; }

// padded index inside one mic row of the FIR tile: 4 extra floats per 32 so
// that lanes reading float4 at a 16-float pitch hit distinct bank groups.
__host__ __device__ __forceinline__ int fir_pad(int l) { return l + ((l >> 5) << 2); }

// ---------------------------------------------------------------------------
// STHT FIR building blocks (used by k_stht and by the fused kernel)
// ---------------------------------------------------------------------------
template <int STRIDE> struct FirGeom {
    static constexpr int WIN = kFirR + STRIDE * (kFirJB - 1);
    static constexpr int NV = (WIN + 3) / 4;
};

__host__ __device__ inline int fir_row_pitch(int TT, int span) {
    const int lrow = TT + span + 8;
    return (lrow + ((lrow >> 5) << 2) + 4 + 3) & ~3;
}

template <int STRIDE>
__device__ __forceinline__ void fir_accumulate(const float *__restrict__ row, const float *__restrict__ taps_s,
                                               int n_taps, int span, int k0, int chunk,
                                               float (&acc)[kFirR]) {
    constexpr int WIN = FirGeom<STRIDE>::WIN;
    constexpr int NV = FirGeom<STRIDE>::NV;
#pragma unroll
    for (int i = 0; i < kFirR; ++i) acc[i] = 0.f;
    const int nblk = n_taps / kFirJB;
    // l index of the window start for tap block 0; it moves back by STRIDE*JB per block
    int lmin = span + kFirR * chunk - k0 - STRIDE * (kFirJB - 1);
#pragma unroll 1
    for (int jb = 0; jb < nblk; ++jb, lmin -= STRIDE * kFirJB) {

        float g[kFirJB];
        {
            const float4 g0 = *reinterpret_cast<const float4 *>(taps_s + jb * kFirJB);
            const float4 g1 = *reinterpret_cast<const float4 *>(taps_s + jb * kFirJB + 4);
            g[0] = g0.x; g[1] = g0.y; g[2] = g0.z; g[3] = g0.w;
            g[4] = g1.x; g[5] = g1.y; g[6] = g1.z; g[7] = g1.w;
        }
        float wv[NV * 4];
#pragma unroll
        for (int v = 0; v < NV; ++v) {
            const float4 x4 = *reinterpret_cast<const float4 *>(row + fir_pad(lmin + 4 * v));
            wv[4 * v + 0] = x4.x; wv[4 * v + 1] = x4.y; wv[4 * v + 2] = x4.z; wv[4 * v + 3] = x4.w;
        }
#pragma unroll
        for (int jj = 0; jj < kFirJB; ++jj)
#pragma unroll
            for (int i = 0; i < kFirR; ++i)
                acc[i] = fmaf(g[jj], wv[i + STRIDE * (kFirJB - 1 - jj)], acc[i]);
        (void)WIN;
    }
}

// fill rows[mm][fir_pad(l)] = x[b][t0 - span + l][m0 + mm] for l < lrow (zero outside the clip)
template <typename IN_T>
__device__ __forceinline__ void fir_fill_rows(float *rows, int pitch, const IN_T *__restrict__ clip,
                                              long long T, int M, int m0, int mg, long long t0,
                                              int span, int lrow) {
    for (int l = threadIdx.x; l < lrow; l += blockDim.x) {
        const long long t = t0 - span + l;
        const bool ok = (t >= 0) && (t < T);
        const IN_T *src = clip + (ok ? t : 0) * M + m0;
        const int pl = fir_pad(l);
        for (int mm = 0; mm < mg; ++mm) rows[mm * pitch + pl] = ok ? to_f32<IN_T>(src[mm]) : 0.f;
    }
}

// ---------------------------------------------------------------------------
// biquad cascade, direct form II transposed, one sample
// ---------------------------------------------------------------------------
struct BiquadState { float s1[kMaxSections]; float s2[kMaxSections]; };

__device__ __forceinline__ void biquad_reset(BiquadState &st) {
#pragma unroll
    for (int k = 0; k < kMaxSections; ++k) { st.s1[k] = 0.f; st.s2[k] = 0.f; }
}

__device__ __forceinline__ float biquad_step(const float (&sos)[kMaxSections][5], int nsec,
                                             BiquadState &st, float x) {
#pragma unroll
    for (int k = 0; k < kMaxSections; ++k) {
        if (k < nsec) {
            const float y = fmaf(sos[k][0], x, st.s1[k]);
            st.s1[k] = fmaf(sos[k][1], x, fmaf(-sos[k][3], y, st.s2[k]));
            st.s2[k] = fmaf(sos[k][2], x, -sos[k][4] * y);
            x = y;
        }
    }
    return x;
}

// ---------------------------------------------------------------------------
// RZCC: streaming find_peaks(cumsum(z), distance=w) for one channel
// (micloc/spike_encoder.py:115-137 + scipy _local_maxima_1d / _select_by_peak_distance).
//
// Candidates: a peak of the cumulative sum sits where z goes + -> (zeros) -> -, at
// the midpoint of the flat top; a valley (peak of -cumsum, spike_encoder.py:131-135)
// where z goes - -> (zeros) -> +.  First and last sample are never peaks.  The
// height of a candidate is the cumulative sum on the flat top, i.e. the running sum
// BEFORE the sample that ends it.  Heights are only ever compared inside one cluster
// (< kClusterMax*w samples) and the cumulative sum of a band-passed signal stays
// bounded, so a float32 running sum orders them as the reference's float64 one does.
//
// Clusters: candidates of one polarity closer than w samples form a cluster; it is
// closed once w samples pass without a new candidate (checked every kSeg samples)
// and is then resolved by scipy's greedy rule (highest first, it removes every
// candidate nearer than w; ties -> later position).  A cluster that overflows, or a
// flat top of more than kPlateauMax exact zeros, sets `overflow` (the clip is
// flagged; micloc_rzcc_encode_f64 is the unbounded encoder).
//
// Two front ends feed the same cluster logic and give identical spikes:
//   rzcc_detect         one sample at a time (stream kernel)
//   rzcc_segment_masks  kSeg samples at once from sign / zero bit masks and the
//                       per-sample running sums (k_chain_blk, fused kernels)
// ---------------------------------------------------------------------------
constexpr int kSeg = 32;          // samples between two cluster close checks
constexpr int kPlateauMax = 16;   // longest run of exact zeros inside a flat top the streaming encoder follows

struct RzccState {
    float csum;               // running cumulative sum
    int r;                    // index of the last non-zero sample (-1: none yet)
    int sgn;                  // 1 when that sample was positive
    int n0, n1;               // open cluster sizes: valleys, peaks
    int last0, last1;         // position of the newest candidate of each open cluster
    int overflow;
    __device__ __forceinline__ int n(int pol) const { return pol ? n1 : n0; }
    __device__ __forceinline__ int last(int pol) const { return pol ? last1 : last0; }
    __device__ __forceinline__ void set_n(int pol, int v) { if (pol) n1 = v; else n0 = v; }
    __device__ __forceinline__ void set_last(int pol, int v) { if (pol) last1 = v; else last0 = v; }
};

__device__ __forceinline__ void rzcc_reset(RzccState &s) {
    s.csum = 0.f; s.r = -1; s.sgn = 0;
    s.n0 = s.n1 = 0; s.last0 = s.last1 = 0; s.overflow = 0;
}

// Cluster buffers of one channel.  `stride` is the distance between consecutive
// entries (1 for a private array, 32 for arrays interleaved across the lanes of a
// warp in shared memory).
// HT = float (float32 chain) or double (the Xylo chain's exact front end, heights of a float64 np.cumsum).
// CAP = candidates buffered per open cluster.
template <typename HT, int CAP = kClusterMax> struct RzccStoreT {
    int *cl_pos;              // [2][CAP]
    HT *cl_h;                 // [2][CAP]  height, sign-adjusted so that higher wins
    int stride;
};
using RzccStore = RzccStoreT<float>;

// scipy's greedy distance rule on one closed cluster of n >= 2 candidates: returns the bit mask of
// the candidates that stay.  Rare (band-limited signals give single-candidate clusters), so it is
// kept out of line: the fused kernel's instruction footprint matters more than this call.
template <typename HT, int CAP>
static __device__ __noinline__ unsigned rzcc_select(const int *cp, const HT *ch, int stride, int n, int w) {
    static_assert(CAP <= 32, "one bit per candidate");
    unsigned und = (CAP == 32 && n == 32) ? 0xffffffffu : (1u << n) - 1u, kept = 0u;
    while (und) {
        int best = -1; HT hb = (HT)0;
        for (int i = 0; i < n; ++i)
            if ((und >> i) & 1u) {
                const HT h = ch[i * stride];
                if (best < 0 || h >= hb) { best = i; hb = h; }
            }
        const int pb = cp[best * stride];
        kept |= 1u << best;
        for (int i = 0; i < n; ++i) {
            int d = cp[i * stride] - pb;
            d = d < 0 ? -d : d;
            if (d < w) und &= ~(1u << i);
        }
    }
    return kept;
}

// POL 1 = peaks (+1 spikes), 0 = valleys (-1 spikes); compile-time so that the cluster state stays in
// named registers
template <int POL, typename Emit, typename HT, int CAP>
__device__ __forceinline__ void rzcc_resolve(RzccState &s, const RzccStoreT<HT, CAP> &st, int w, Emit &&emit) {
    const int n = POL ? s.n1 : s.n0;
    const int *cp = st.cl_pos + POL * CAP * st.stride;
    const HT *ch = st.cl_h + POL * CAP * st.stride;
    constexpr int sign = POL ? 1 : -1;
    if (POL) s.n1 = 0; else s.n0 = 0;
    if (n == 1) { emit(cp[0], sign); return; }
    unsigned kept = rzcc_select<HT, CAP>(cp, ch, st.stride, n, w);
    while (kept) {
        const int i = __ffs(kept) - 1;
        kept &= kept - 1;
        emit(cp[i * st.stride], sign);
    }
}

// a new candidate (candidates of one polarity arrive in time order)
template <int POL, typename Emit, typename HT, int CAP>
__device__ __forceinline__ void rzcc_push(RzccState &s, const RzccStoreT<HT, CAP> &st, int pos, HT h, int w, Emit &&emit) {
    if ((POL ? s.n1 : s.n0) > 0 && pos - (POL ? s.last1 : s.last0) >= w) rzcc_resolve<POL>(s, st, w, emit);
    const int n = POL ? s.n1 : s.n0;
    if (n == CAP) { s.overflow = 1; return; }
    st.cl_pos[(POL * CAP + n) * st.stride] = pos;
    st.cl_h[(POL * CAP + n) * st.stride] = h;
    if (POL) { s.last1 = pos; s.n1 = n + 1; } else { s.last0 = pos; s.n0 = n + 1; }
}

template <typename Emit, typename HT, int CAP>
__device__ __forceinline__ void rzcc_push(RzccState &s, const RzccStoreT<HT, CAP> &st, int pol, int pos, HT h, int w,
                                          Emit &&emit) {
    if (pol) rzcc_push<1>(s, st, pos, h, w, emit); else rzcc_push<0>(s, st, pos, h, w, emit);
}

// every kSeg samples (t_end = last sample seen): close the clusters that can no longer
// grow; everything when `final`.  A spike at position p is emitted at the latest by the
// close check at t_end >= p + kPlateauMax/2 + (kClusterMax-1)*(w-1) + w + kSeg - 1.
template <typename Emit, typename HT, int CAP>
__device__ __forceinline__ void rzcc_close(RzccState &s, const RzccStoreT<HT, CAP> &st, int w, int t_end, bool final,
                                           Emit &&emit) {
    if (s.n1 > 0 && (final || t_end - s.last1 >= w)) rzcc_resolve<1>(s, st, w, emit);
    if (s.n0 > 0 && (final || t_end - s.last0 >= w)) rzcc_resolve<0>(s, st, w, emit);
}

// candidate test for sample t with value class (nz, positive) and the running sum before it
template <typename Emit, typename HT, int CAP>
__device__ __forceinline__ void rzcc_sample(RzccState &s, const RzccStoreT<HT, CAP> &st, int bipolar, int w, int t, bool nz,
                                            bool positive, HT cprev, Emit &&emit) {
    const bool ev = nz && (s.r >= 1) && (positive != (s.sgn != 0)) && (bipolar || s.sgn);
    if (ev) {
        if (t - 1 - s.r > kPlateauMax) s.overflow = 1;
        else rzcc_push(s, st, s.sgn, (s.r + t - 1) >> 1, s.sgn ? cprev : -cprev, w, emit);
    }
    if (nz) { s.r = t; s.sgn = positive ? 1 : 0; }
}

// The reference's np.cumsum runs in float64 and stops moving once |z| < ulp(sum) / 2: find_peaks then sees a flat top
// although z still alternates.  That happens in digital silence, where the band-pass output is the filter's decaying
// tail (below 2^-53 of the sum after ~40 ms; in float32 it then never reaches 0 but settles into a denormal limit
// cycle whose sign changes would spike forever).  The float32 chains therefore treat such a sample as an exact zero:
// half an ulp of the float64 sum = 2^(exponent(sum) - 53).
__device__ __forceinline__ bool rzcc_flat(float z, float cprev) {
    const float hu = __uint_as_float(__float_as_uint(cprev) & 0x7f800000u) * 1.1102230246251565e-16f;
    return z == 0.f || fabsf(z) < hu;
}
constexpr float kFlatTrigger = 4.5e-16f;      // a segment whose smallest |z| is below this x |sum| takes the per-sample path

// one sample at a time
template <typename Emit>
__device__ __forceinline__ void rzcc_detect(RzccState &s, const RzccStore &st, int bipolar, int w, int t, float z,
                                            Emit &&emit) {
    const float cprev = s.csum;
    s.csum = cprev + z;
    rzcc_sample(s, st, bipolar, w, t, !rzcc_flat(z, cprev), z > 0.f, cprev, emit);
}

// kSeg samples ts .. ts+nvalid-1 at once.  Bit (31-i) of `neg` / `zero` says that sample ts+i is
// negative (IEEE sign bit) / exactly zero; cs[i*cs_stride] is the running sum after sample ts+i and
// `carry` the running sum before sample ts.
template <typename Emit>
__device__ __forceinline__ void rzcc_segment_masks(RzccState &s, const RzccStore &st, int bipolar, int w, int ts,
                                                   int nvalid, unsigned neg, unsigned zero, const float *cs,
                                                   int cs_stride, float carry, Emit &&emit) {
    if (zero == 0u && nvalid == kSeg && s.r == ts - 1) {
        // no exact zeros and no open flat top: a candidate sits right before every sign change
        const unsigned prev = (neg >> 1) | (s.sgn ? 0u : 0x80000000u);
        unsigned d = neg ^ prev;
        if (ts == 0) d &= 0x3fffffffu;          // sample 0 has no predecessor and cannot start a flat top
        // peaks: + -> - (the sample that confirms it is negative); valleys: - -> +
        unsigned dp = d & neg, dv = bipolar ? (d & ~neg) : 0u;
        while (dp) {
            const int i = __clz(dp);
            dp &= ~(0x80000000u >> i);
            rzcc_push<1>(s, st, ts + i - 1, i ? cs[(i - 1) * cs_stride] : carry, w, emit);
        }
        while (dv) {
            const int i = __clz(dv);
            dv &= ~(0x80000000u >> i);
            rzcc_push<0>(s, st, ts + i - 1, -(i ? cs[(i - 1) * cs_stride] : carry), w, emit);
        }
        s.r = ts + kSeg - 1;
        s.sgn = (neg & 1u) ? 0 : 1;
    } else {
        for (int i = 0; i < nvalid; ++i) {
            const bool nz = !((zero >> (31 - i)) & 1u);
            const bool positive = nz && !((neg >> (31 - i)) & 1u);
            rzcc_sample(s, st, bipolar, w, ts + i, nz, positive, i ? cs[(i - 1) * cs_stride] : carry, emit);
        }
    }
}

// number of samples after which the spike raster is final (see rzcc_close)
__host__ __device__ inline int rzcc_lag(int w) { return (kClusterMax - 1) * (w - 1) + w + kSeg + kPlateauMax / 2; }

// ---------------------------------------------------------------------------
// neuron (synapse + membrane) alpha kernel h[n] = c*n*a^n, n < L, as two
// two-state recurrences: the full alpha response minus its tail, the tail being
// the same response driven by the spike train delayed by L.
// ---------------------------------------------------------------------------
struct NeuronState { float p1, p2, q1, q2; };

__device__ __forceinline__ void neuron_reset(NeuronState &n) { n.p1 = n.p2 = n.q1 = n.q2 = 0.f; }

// s = spike at t, sd = spike at t-L (0 before the clip starts)
__device__ __forceinline__ float neuron_step(const ChainParams &p, NeuronState &n, float s, float sd) {
    n.p2 = p.na * (n.p2 + n.p1);
    n.p1 = __fadd_rn(__fmul_rn(p.na, n.p1), s);      // not fused: the fused kernel adds +-1 under a predicate
    n.q2 = p.na * (n.q2 + n.q1);
    n.q1 = __fadd_rn(__fmul_rn(p.na, n.q1), sd);
    const float tail = fmaf(p.nLf, n.q1, n.q2);
    return fmaf(-p.ncT, tail, p.nc * n.p2);
}

}  // namespace micloc
