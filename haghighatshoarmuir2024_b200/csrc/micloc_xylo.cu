// micloc_xylo.cu -- Xylo-quantised integer chain (BASELINE config 3).
//
// Reference sites (paths under /root/reference):
//   Demo.spike_encoding   micloc/xylo_snn_localization.py:315-356  STHT -> hstack(I,Q) -> Butterworth
//                         filterbank (micloc/filterbank.py:40-44) -> RZCC with the band-0 encoder ->
//                         pos/neg split
//   Demo.xylo_process     micloc/xylo_snn_localization.py:358-377  rockpool XyloSim hidden layer:
//                         integer LIF (bit-shift decay, int8 weights, 16-bit state, subtractive
//                         multi-spike reset); rec["Spikes"] = hidden raster
//   extract_rate / peak   micloc/xylo_snn_localization.py:379-427, micloc/utils.py:84-121 as used by
//                         paper_plots/target_xylo_localization.py:594-605
//
// Two front ends produce the signed spike raster int8 [B][T][2M*F]:
//   fast  (exact = 0): float32 STHT FIR (k_stht) + float32 SOS band filters + streaming RZCC (k_chain_blk)
//   exact (exact = 1): float64 throughout with the reference's own operation order -- lfilter's
//                      direct-form-II-transposed FIR / IIR (product rounded, then added, oldest tap
//                      first) and find_peaks on a float64 np.cumsum -- so that the spikes, and with
//                      them every integer downstream, are bit-identical to numpy/scipy.
// The integer network then runs as ONE kernel, one thread per (clip, hidden neuron) looping over
// time with I_syn / V_mem / spike count in registers; the input spikes of a clip are turned into
// per-step event masks in shared memory and each event is one predicated add of an int16 weight.
// Xylo stream batches (end of this file) run the same exact front end and network on many continuous recordings, with
// the chain and neuron state carried across pushes (STREAM / STATE forms of the kernels).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <type_traits>
#include <vector>

#include "micloc_common.h"
#include "micloc_stream.cuh"

namespace micloc {

// ---------------------------------------------------------------------------
// exact float64 front end
// ---------------------------------------------------------------------------
constexpr int kF64Tile = 256;   // outputs per CTA and microphone
constexpr int kF64MG = 8;       // microphones per CTA

// q[b][t][m] = lfilter(h, [1], x)[t][m] in float64, summed exactly as scipy's DF2T delay line does:
// ((x[t-K+1] h[K-1] + x[t-K+2] h[K-2]) + ...) + x[t] h[0], every product rounded before its add.
template <typename IN_T>
__global__ void __launch_bounds__(kF64Tile)
k_stht_f64(const IN_T *__restrict__ audio, const double *__restrict__ h, double *__restrict__ q,
           int M, int K, long long T, int ntiles) {
    extern __shared__ __align__(16) double smd[];
    double *hs = smd;                                   // [K]
    double *xs = smd + K;                               // [mg][kF64Tile + K - 1], microphone-major
    const int pitch = kF64Tile + K - 1;
    const long long b = blockIdx.x / ntiles;
    const long long t0 = (long long)(blockIdx.x % ntiles) * kF64Tile;
    const int m0 = blockIdx.y * kF64MG;
    const int mg = min(kF64MG, M - m0);
    const IN_T *clip = audio + b * T * M;
    for (int i = threadIdx.x; i < K; i += blockDim.x) hs[i] = h[i];
    for (int e = threadIdx.x; e < pitch * mg; e += blockDim.x) {
        const int l = e / mg, mm = e % mg;
        const long long t = t0 - (K - 1) + l;
        xs[mm * pitch + l] = (t >= 0 && t < T) ? (double)clip[t * M + m0 + mm] : 0.0;
    }
    __syncthreads();
    const long long t = t0 + threadIdx.x;
    if (t >= T) return;
    // the microphones of the group are independent dependency chains: walk them together
    const double *xr = xs + threadIdx.x;                    // xr[mm*pitch + j] = x[t - (K-1) + j][m0 + mm]
    double acc[kF64MG];
#pragma unroll
    for (int mm = 0; mm < kF64MG; ++mm) acc[mm] = mm < mg ? __dmul_rn(xr[mm * pitch], hs[K - 1]) : 0.0;
#pragma unroll 2
    for (int j = 1; j < K; ++j) {
        const double hj = hs[K - 1 - j];
#pragma unroll
        for (int mm = 0; mm < kF64MG; ++mm)
            if (mm < mg) acc[mm] = __dadd_rn(acc[mm], __dmul_rn(xr[mm * pitch + j], hj));
    }
#pragma unroll
    for (int mm = 0; mm < kF64MG; ++mm)
        if (mm < mg) q[(b * T + t) * M + m0 + mm] = acc[mm];
}

// ---- the same sum for a Hilbert kernel (every other tap exactly 0.0), register-blocked ------------------------------
// A zero tap contributes x * 0.0 = +-0, and acc + (+-0) == acc for every acc != 0: the terms of the non-zero taps,
// added in the same order (oldest first, product rounded, then added), give the same float64 bit pattern (an acc that
// is exactly zero may differ in the SIGN of zero only, which nothing downstream can see: sums and comparisons).
// Each thread owns kSR consecutive outputs of one microphone and slides a register window along the taps: per tap
// kSR x (DMUL + DADD) against 2 LDS.64-equivalents, i.e. the float64 pipe is the only limit (the dense kernel above
// spends one shared-memory load per multiply-add).  Lanes of a warp own consecutive output blocks of one microphone;
// rows are padded by 2 doubles per 8 so that the lanes' 128-bit loads fall into distinct bank groups.
constexpr int kSR = 8;                 // outputs per thread
constexpr int kSTile = 256;            // outputs per CTA and microphone = 32 lanes x kSR
__host__ __device__ __forceinline__ int f64_pad(int p) { return p + ((p >> 3) << 1); }

template <bool FIRST>
__device__ __forceinline__ void stht_f64_taps4(double (&acc)[kSR], const double (&W)[2 * kSR], const double (&g)[4]) {
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int r = 0; r < kSR; ++r) {
            const double prod = __dmul_rn(W[2 * u + r], g[u]);
            acc[r] = (FIRST && u == 0) ? prod : __dadd_rn(acc[r], prod);
        }
}

// g[i] = h[K - 1 - 2 i], i < ntap (ntap a multiple of 4): the non-zero taps, oldest sample first
template <typename IN_T>
__global__ void __launch_bounds__(256)
k_stht_f64_sparse(const IN_T *__restrict__ audio, const double *__restrict__ g, double *__restrict__ q,
                  int M, int K, int ntap, long long T, int ntiles, long long t_first = 0) {
    extern __shared__ __align__(16) double smd[];
    double *gs = smd;                                   // [ntap]
    const int npos = kSTile + K - 1;                    // positions per row: x[t0 - (K-1) + p]
    const int pitch = (f64_pad(npos) + 9) & ~1;
    double *xs = smd + ntap;                            // [mg][pitch], microphone-major
    const long long b = blockIdx.x / ntiles;
    const long long t0 = t_first + (long long)(blockIdx.x % ntiles) * kSTile;   // (t_first: outputs before it are not wanted)
    const int m0 = blockIdx.y * kF64MG;
    const int mg = min(kF64MG, M - m0);
    const IN_T *clip = audio + b * T * M;
    for (int i = threadIdx.x; i < ntap; i += blockDim.x) gs[i] = g[i];
    for (int e = threadIdx.x; e < npos * mg; e += blockDim.x) {
        const int l = e / mg, mm = e % mg;
        const long long t = t0 - (K - 1) + l;
        xs[mm * pitch + f64_pad(l)] = (t >= 0 && t < T) ? (double)clip[t * M + m0 + mm] : 0.0;
    }
    __syncthreads();
    const int mm = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (mm >= mg) return;
    // output r of this thread is t = t0 + kSR*lane + r; tap i reads position kSR*lane + r + 2i
    const double *row = xs + mm * pitch;
    double acc[kSR], W[2 * kSR], gg[4];
    auto load8 = [&](int grp, double *dst) {            // the 8 positions of group `grp` are contiguous and 16-byte aligned
        const double2 *p2 = reinterpret_cast<const double2 *>(row + 10 * grp);
#pragma unroll
        for (int v = 0; v < 4; ++v) { const double2 d = p2[v]; dst[2 * v] = d.x; dst[2 * v + 1] = d.y; }
    };
    load8(lane, W);
    const int nit = ntap >> 2;
#pragma unroll 1
    for (int I = 0; I < nit; ++I) {
        load8(lane + I + 1, W + kSR);
        {
            const double2 a = reinterpret_cast<const double2 *>(gs + 4 * I)[0], c = reinterpret_cast<const double2 *>(gs + 4 * I)[1];
            gg[0] = a.x; gg[1] = a.y; gg[2] = c.x; gg[3] = c.y;
        }
        if (I == 0) stht_f64_taps4<true>(acc, W, gg); else stht_f64_taps4<false>(acc, W, gg);
#pragma unroll
        for (int r = 0; r < kSR; ++r) W[r] = W[kSR + r];
    }
    const long long tb = t0 + kSR * lane;
#pragma unroll
    for (int r = 0; r < kSR; ++r)
        if (tb + r < T) q[(b * T + tb + r) * M + m0 + mm] = acc[r];
}

// ---- band filters -> np.cumsum -> find_peaks in float64, one WARP per clip, one lane per (band, channel) ------------
// The chain is sequential in time and bit-exactness forbids re-association, so its speed is the number of chains in
// flight: a warp needs 5 KB of shared memory (64-step tiles of q and of the in-phase samples x[(t - K/2) mod T], loaded
// coalesced) and its candidate clusters live in per-thread local memory, i.e. 32 clips per SM.  The band filter runs in
// lfilter's operation order (as k_iir_f64), the running sum is np.cumsum's left-to-right float64 sum, and peaks are
// detected on that sum itself (acc > prev / acc < prev with scipy's plateau-midpoint rule, as k_rzcc_scan does), not
// on the sign of z: once |z| drops below half an ulp of the sum (decaying filters in digital silence) the sum stops
// moving although z still alternates, and find_peaks sees one flat top.  Clusters are resolved by the streaming
// encoder of micloc_device.cuh with float64 heights; a cluster of more than kF64Cluster candidates flags the clip
// (bit 0) and the host redoes it with the unbounded kernels.  z never reaches HBM.
constexpr int kF64Cluster = 32;         // candidates buffered per open cluster (noisy order-1 bands chain up to ~12)
constexpr int kChainTile = 64;          // time steps staged per warp
constexpr int kChainWarps = 8;          // clips per CTA

using F64Store = RzccStoreT<double, kF64Cluster>;

// cluster of POL candidates closed: one candidate stays; of two (always nearer than w) the higher one, the later one on
// a tie; three or more go through the greedy rule of micloc_device.cuh
template <int POL, typename Emit>
__device__ __forceinline__ void f64_resolve(RzccState &s, const F64Store &st, int w, Emit &&emit) {
    const int n = POL ? s.n1 : s.n0;
    if (n <= 2) {
        const int *cp = st.cl_pos + POL * kF64Cluster;
        const double *ch = st.cl_h + POL * kF64Cluster;
        const int keep = (n == 2 && ch[1] >= ch[0]) ? 1 : 0;
        emit(cp[keep], POL ? 1 : -1);
        if (POL) s.n1 = 0; else s.n0 = 0;
        return;
    }
    rzcc_resolve<POL>(s, st, w, emit);
}
template <int POL, typename Emit>
__device__ __forceinline__ void f64_push(RzccState &s, const F64Store &st, int pos, double h, int w, Emit &&emit) {
    if ((POL ? s.n1 : s.n0) > 0 && pos - (POL ? s.last1 : s.last0) >= w) f64_resolve<POL>(s, st, w, emit);
    const int n = POL ? s.n1 : s.n0;
    if (n == kF64Cluster) { s.overflow = 1; return; }
    st.cl_pos[POL * kF64Cluster + n] = pos;
    st.cl_h[POL * kF64Cluster + n] = h;
    if (POL) { s.last1 = pos; s.n1 = n + 1; } else { s.last0 = pos; s.n0 = n + 1; }
}

// Stream form (STREAM = true, Xylo stream batches): warp b is slot b, its lanes' chain state is parked in global memory
// between pushes, and time runs in the slot's ABSOLUTE positions [N, N + n): the 64-step tiles start at the same
// samples as in a one-shot clip of the whole recording.  A push may end inside a tile; the clusters are then checked
// for closing there too, which emits nothing a later check would not (a cluster closed that way can no longer grow).
// Spikes go to the slot's ring at their absolute position; the rows [F, N + n - D) are final and copied out.
constexpr int kF64FlatTop = 64;         // flat-top allowance of the stream latency (samples)

struct XyloChanState {                  // one per (slot, band, channel)
    double zs[5];                       // band-filter delays (NBA <= 5)
    double cs;                          // running sum
    int rise, fall;                     // start of the running sum's current flat top / bottom (-1: none)
    RzccState rz;
    int cl_pos[2 * kF64Cluster];
    double cl_h[2 * kF64Cluster];
};

struct XyloChainStream {
    XyloChanState *state;               // [S][CT]
    const SlotPos *pos_in;
    SlotPos *pos_out;
    int32_t *m_out;                     // [S] final rows of this call
    const int32_t *close_sel;           // flush: 1 = close this slot like a clip end; nullptr: push
    int8_t *ring;                       // [S][ring_len][CT] spikes at (absolute position mod ring_len)
    int ring_len;                       // power of two >= max_frame_len + D
    int hist;                           // rows of the assembled buffer before the frame (K - 1)
    int rows;                           // row stride of the output raster (n + D)
    int D;                              // latency
};

template <typename IN_T, int NBA, bool STREAM = false>
__global__ void __launch_bounds__(32 * kChainWarps, 3)
k_xylo_chain_f64(const IN_T *__restrict__ audio, const double *__restrict__ q, const double *__restrict__ ba_b,
                 const double *__restrict__ ba_a, int8_t *__restrict__ spikes, int32_t *__restrict__ flags,
                 int M, int half, int nba, int F, int w, int bipolar, long long B, long long T,
                 const XyloChainStream sa = XyloChainStream{}) {
    // STREAM: audio = assembled rows [S][hist + T][M] (float64), q the same rows' STHT, T = frame rows (0: flush)
    using XS_T = typename std::conditional<STREAM, double, float>::type;
    extern __shared__ __align__(16) double smd[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nw = STREAM ? (int)(blockDim.x >> 5) : kChainWarps;   // (the stream form stages float64 in-phase rows)
    const long long b = (long long)blockIdx.x * nw + warp;
    if (b >= B) return;
    const int C2 = 2 * M, CT = C2 * F;
    const int passes = (CT + 31) >> 5;
    double *qs = smd + (size_t)warp * kChainTile * M;                                                       // [tile][M]
    XS_T *xs = reinterpret_cast<XS_T *>(smd + (size_t)nw * kChainTile * M) + (size_t)warp * kChainTile * M;   // [tile][M]
    const long long rows_in = STREAM ? sa.hist + T : T;
    const IN_T *clip = audio + b * rows_in * M;
    const double *qc = q + b * rows_in * M;

    long long tstart = 0, tstop = T;
    bool flush = false;
    int F0 = 0, F1 = 0;
    if constexpr (STREAM) {
        const SlotPos sp = sa.pos_in[b];
        flush = sa.close_sel != nullptr;
        const bool run = sp.active && (!flush || sa.close_sel[b] != 0);
        const int N0 = sp.N;
        const int t_end = (run && !flush) ? N0 + (int)T : N0;
        F0 = sp.F;
        F1 = !run ? F0 : (flush ? N0 : max(t_end - sa.D, F0));
        if (lane == 0) {
            sa.pos_out[b] = SlotPos{t_end, F1, (run && flush) ? 0 : sp.active, 0};
            sa.m_out[b] = F1 - F0;
        }
        if (!run) return;
        tstart = N0; tstop = t_end;
    }

    // per-pass chain state (CT <= 64: at most two (band, channel) per lane)
    // (parked in local memory between tiles: only the pass at work lives in registers)
    struct Save { double zs[NBA]; double cs; int rise, fall; RzccState rz; } sv[2];
    int cl_pos[2][2 * kF64Cluster];
    double cl_h[2][2 * kF64Cluster];
    int q_pos[kChainTile + 1];          // candidates of the tile at work, in time order (+ the scratch slot behind a full queue)
    double q_h[kChainTile + 1];
#pragma unroll 1
    for (int ps = 0; ps < 2; ++ps) {
        if constexpr (STREAM) {
            const int cc = lane + 32 * ps;
            if (cc < CT) {
                const XyloChanState &g = sa.state[b * CT + cc];
#pragma unroll
                for (int k = 0; k < NBA; ++k) sv[ps].zs[k] = g.zs[k];
                sv[ps].cs = g.cs; sv[ps].rise = g.rise; sv[ps].fall = g.fall;
                sv[ps].rz = g.rz;
                for (int i = 0; i < sv[ps].rz.n0; ++i) { cl_pos[ps][i] = g.cl_pos[i]; cl_h[ps][i] = g.cl_h[i]; }
                for (int i = 0; i < sv[ps].rz.n1; ++i) {
                    cl_pos[ps][kF64Cluster + i] = g.cl_pos[kF64Cluster + i];
                    cl_h[ps][kF64Cluster + i] = g.cl_h[kF64Cluster + i];
                }
            }
        } else {
#pragma unroll
            for (int k = 0; k < NBA; ++k) sv[ps].zs[k] = 0.0;
            sv[ps].cs = 0.0; sv[ps].rise = sv[ps].fall = -1;
            rzcc_reset(sv[ps].rz);
        }
    }
    int8_t *const sbase = STREAM ? sa.ring + b * (long long)sa.ring_len * CT : spikes + b * T * CT;
    const int rmask = sa.ring_len - 1;
    // tiles of kChainTile ABSOLUTE samples (the first and last of a stream push may be partial)
    for (long long t0 = tstart; t0 < tstop;) {
        const int len = (int)min((long long)(kChainTile - (int)(t0 & (kChainTile - 1))), tstop - t0);
        __syncwarp();
        for (int e = lane; e < len * M; e += 32) {
            const int i = e / M, m = e - i * M;
            if constexpr (STREAM) {
                const long long r = sa.hist + (t0 - tstart) + i;              // row of sample t0 + i
                qs[e] = qc[r * M + m];
                xs[e] = clip[(r - half) * M + m];                             // causal x[t - K/2] (zeros before the slot starts)
            } else {
                qs[e] = qc[t0 * M + e];
                long long src = t0 + i - half;                       // np.roll: x[(t - K/2) mod T]
                if (src < 0) { src %= T; if (src < 0) src += T; }
                xs[e] = (float)clip[src * M + m];
            }
        }
        __syncwarp();
#pragma unroll 1
        for (int ps = 0; ps < passes; ++ps) {
            const int cc = lane + 32 * ps;
            if (cc < CT) {
                const int c = cc % C2, band = cc / C2;
                const bool inphase = c < M;
                const int col = inphase ? c : c - M;
                const F64Store store{cl_pos[ps], cl_h[ps], 1};
                int8_t *out = sbase + cc;
                auto emit = [&](int pos, int sign) {
                    if constexpr (STREAM) out[(long long)(pos & rmask) * CT] = (int8_t)sign;
                    else out[(long long)pos * CT] = (int8_t)sign;
                };
                double bb[NBA], aa[NBA], zs[NBA];
#pragma unroll
                for (int k = 0; k < NBA; ++k) {
                    bb[k] = k < nba ? ba_b[band * nba + k] : 0.0;
                    aa[k] = k < nba ? ba_a[band * nba + k] : 0.0;
                    zs[k] = sv[ps].zs[k];
                }
                RzccState s = sv[ps].rz;
                double acc = sv[ps].cs;
                int rs = sv[ps].rise, fl = sv[ps].fall;    // start of the running sum's current flat top / bottom (-1: none)
                // (a) the sequential part, the same instructions in every lane: filter, running sum, candidate
                //     detection; candidates are only queued here
                int nq = 0;
                unsigned long long qpol = 0ull;
#pragma unroll 4
                for (int i = 0; i < len; ++i) {
                    const double x = inphase ? (double)xs[i * M + col] : qs[i * M + col];
                    const double y = __dadd_rn(zs[0], __dmul_rn(bb[0], x));
#pragma unroll
                    for (int k = 0; k < NBA - 1; ++k)
                        zs[k] = __dsub_rn(__dadd_rn(zs[k + 1], __dmul_rn(x, bb[k + 1])), __dmul_rn(y, aa[k + 1]));
                    const double prev = acc;
                    acc = __dadd_rn(acc, y);
                    const int t = (int)t0 + i;
                    // candidate test without branches (the lanes' events fall on different samples): slot nq of the
                    // queue is written at every step and kept when the step closed a flat top (peak) or bottom (valley)
                    const bool up = acc > prev, down = acc < prev;           // sample 0 has no predecessor: rs = fl = -1 there
                    const bool peak = down && rs >= 0, valley = up && fl >= 0 && bipolar;
                    q_pos[nq] = ((peak ? rs : fl) + t - 1) >> 1;
                    q_h[nq] = peak ? prev : -prev;
                    qpol |= (unsigned long long)peak << nq;
                    nq += (peak || valley) ? 1 : 0;
                    rs = up ? t : (down ? -1 : rs);
                    fl = down ? t : (up ? -1 : fl);
                    if (t == 0) { rs = -1; fl = -1; }
                }
                // (b) the queued candidates enter the clusters, the lanes of the warp in step (each lane's events fall
                //     on different samples: handled where they occur, every one of them would run with one lane active)
                const unsigned am = __activemask();
                for (int j = 0; __any_sync(am, j < nq); ++j)
                    if (j < nq) {
                        if ((qpol >> j) & 1ull) f64_push<1>(s, store, q_pos[j], q_h[j], w, emit);
                        else f64_push<0>(s, store, q_pos[j], q_h[j], w, emit);
                    }
                {
                    // a cluster is closed once no later candidate can fall within w of its newest one: a candidate
                    // still to come sits at the midpoint of a flat stretch that began at rs / fl
                    const int t = (int)t0 + len - 1;
                    const int e1 = rs >= 0 ? (rs + t) >> 1 : t, e0 = fl >= 0 ? (fl + t) >> 1 : t;
                    if (s.n1 > 0 && e1 - s.last1 >= w) f64_resolve<1>(s, store, w, emit);
                    if (s.n0 > 0 && e0 - s.last0 >= w) f64_resolve<0>(s, store, w, emit);
                }
                if (!STREAM && t0 + len == tstop) {
                    rzcc_close(s, store, w, (int)(T - 1), true, emit);
                    if (s.overflow) atomicOr(flags + b, 1);
                }
#pragma unroll
                for (int k = 0; k < NBA; ++k) sv[ps].zs[k] = zs[k];
                sv[ps].rz = s; sv[ps].cs = acc; sv[ps].rise = rs; sv[ps].fall = fl;
            }
        }
        t0 += len;
    }
    if constexpr (STREAM) {
        // flush: close like a clip end.  Push: every spike below F1 must have been emitted -- the earliest position a
        // spike can still take is the first candidate of an open cluster or the midpoint of an open flat top / bottom
        // and a sample after the push; if that lies below F1 (or a cluster overflowed) the slot is flagged (bit 0).
        // Then the final rows [F0, F1) of the lane's channels leave the ring (which is cleared behind them).
#pragma unroll 1
        for (int ps = 0; ps < passes; ++ps) {
            const int cc = lane + 32 * ps;
            if (cc >= CT) continue;
            const F64Store store{cl_pos[ps], cl_h[ps], 1};
            int8_t *ring = sbase + cc;
            auto emit = [&](int pos, int sign) { ring[(long long)(pos & rmask) * CT] = (int8_t)sign; };
            RzccState s = sv[ps].rz;
            const int t_end = (int)tstop;
            if (flush) {
                if (t_end > 0) rzcc_close(s, store, w, t_end - 1, true, emit);
            } else {
                int h = t_end;
                if (s.n1 > 0) h = min(h, cl_pos[ps][kF64Cluster]);
                if (s.n0 > 0) h = min(h, cl_pos[ps][0]);
                if (sv[ps].rise >= 0) h = min(h, (sv[ps].rise + t_end - 1) >> 1);
                if (bipolar && sv[ps].fall >= 0) h = min(h, (sv[ps].fall + t_end - 1) >> 1);
                if (h < F1) s.overflow = 1;
            }
            if (s.overflow) atomicOr(flags + b, 1);
            XyloChanState &g = sa.state[b * CT + cc];
#pragma unroll
            for (int k = 0; k < NBA; ++k) g.zs[k] = sv[ps].zs[k];
            g.cs = sv[ps].cs; g.rise = sv[ps].rise; g.fall = sv[ps].fall;
            g.rz = s;
            for (int i = 0; i < s.n0; ++i) { g.cl_pos[i] = cl_pos[ps][i]; g.cl_h[i] = cl_h[ps][i]; }
            for (int i = 0; i < s.n1; ++i) {
                g.cl_pos[kF64Cluster + i] = cl_pos[ps][kF64Cluster + i];
                g.cl_h[kF64Cluster + i] = cl_h[ps][kF64Cluster + i];
            }
            int8_t *o = spikes + b * (long long)sa.rows * CT + cc;
#pragma unroll 4
            for (int t = F0; t < F1; ++t) {
                int8_t *r = ring + (long long)(t & rmask) * CT;
                o[(long long)(t - F0) * CT] = *r;
                *r = 0;
            }
        }
    }
}

constexpr int kMaxBa = 9;       // len(b) of a band filter (order-4 band-pass at most)

// z[b][t][band*2M + c] = lfilter(b_band, a_band, hstack(I, Q))[t][c] in float64, DF2T evaluated in
// scipy's order: y = z0 + b0 x; z[k] = (z[k+1] + x b[k+1]) - y a[k+1], the last delay being
// x b[N-1] - y a[N-1] (= the same expression with z[N-1] == 0).  One thread per (clip, band,
// channel), sequential in time.  NBA = len(b) rounded up to 3, 5 or 9 (coefficients zero-padded).
template <typename IN_T, int NBA>
__global__ void __launch_bounds__(128)
k_iir_f64(const IN_T *__restrict__ audio, const double *__restrict__ q, const double *__restrict__ ba_b,
          const double *__restrict__ ba_a, double *__restrict__ z, int M, int half, int nba, int nb,
          long long B, long long T) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int C2 = 2 * M, CT = C2 * nb;
    if (idx >= B * CT) return;
    const long long b = idx / CT;
    const int cc = (int)(idx % CT);
    const int band = cc / C2, c = cc % C2;
    double bb[NBA], aa[NBA], zs[NBA];
#pragma unroll
    for (int k = 0; k < NBA; ++k) {
        bb[k] = k < nba ? ba_b[band * nba + k] : 0.0;
        aa[k] = k < nba ? ba_a[band * nba + k] : 0.0;
        zs[k] = 0.0;
    }
    const bool inphase = c < M;
    const IN_T *xa = audio + b * T * M + (inphase ? c : 0);
    const double *xq = q + b * T * M + (inphase ? 0 : c - M);
    double *zo = z + b * T * CT + cc;
    long long src = ((-(long long)half) % T + T) % T;   // (t - K/2) mod T at t = 0 (np.roll)
    for (long long t = 0; t < T; ++t) {
        double x;
        if (inphase) { x = (double)xa[src * M]; if (++src == T) src = 0; }
        else x = xq[t * M];
        const double y = __dadd_rn(zs[0], __dmul_rn(bb[0], x));
#pragma unroll
        for (int k = 0; k < NBA - 1; ++k)
            zs[k] = __dsub_rn(__dadd_rn(zs[k + 1], __dmul_rn(x, bb[k + 1])), __dmul_rn(y, aa[k + 1]));
        zo[t * CT] = y;
    }
}

template <typename IN_T>
static void launch_iir_f64(const IN_T *audio, const double *q, const double *ba_b, const double *ba_a, double *z,
                           int M, int half, int nba, int nb, long long B, long long T, cudaStream_t st) {
    const long long nthr = B * 2 * M * nb;
    const unsigned grid = (unsigned)((nthr + 127) / 128);
    if (nba <= 3) k_iir_f64<IN_T, 3><<<grid, 128, 0, st>>>(audio, q, ba_b, ba_a, z, M, half, nba, nb, B, T);
    else if (nba <= 5) k_iir_f64<IN_T, 5><<<grid, 128, 0, st>>>(audio, q, ba_b, ba_a, z, M, half, nba, nb, B, T);
    else k_iir_f64<IN_T, kMaxBa><<<grid, 128, 0, st>>>(audio, q, ba_b, ba_a, z, M, half, nba, nb, B, T);
}

// ---------------------------------------------------------------------------
// integer LIF network (XyloSim hidden layer)
// ---------------------------------------------------------------------------
constexpr int kLifTile = 256;   // time steps staged in shared memory at once

// bit-shift decay: v -= v >> dash (arithmetic), by at least one towards zero.  For v < 0 the shift
// never reaches 0, for v > 0 it is raised to 1, for v == 0 it stays 0: dv = max(v >> dash, min(v, 1)).
__device__ __forceinline__ int xylo_decay(int v, int dash) { return v - max(v >> dash, min(v, 1)); }
__device__ __forceinline__ int xylo_sat16(int v) { return max(-32768, min(32767, v)); }

// spikes: SIGNED_IN ? int8 [B][T][CI] in {-1,0,+1} (bipolar: input channel c is the positive part of
// column c, channel CI + c its negative part) : int8 [B][T][N_in] in {0,1}.
// grid = (B, neuron chunks); block = chunk size rounded up to a warp.
// one time step of one hidden neuron; returns the number of spikes it fired (th2 = 2 * th)
template <bool SAT_ISYN>
__device__ __forceinline__ int xylo_step(int &isyn, int &vmem, int in, int ds, int dm, int bs, int th, int th2,
                                         int max_spikes) {
    isyn = xylo_decay(isyn, ds) + in;
    if (SAT_ISYN) isyn = xylo_sat16(isyn);
    int v = xylo_sat16(xylo_decay(vmem, dm) + isyn + bs);
    const bool fire = v >= th, multi = v >= th2;     // two independent compares
    int ns = fire ? 1 : 0;
    v -= fire ? th : 0;                              // the common single spike, predicated
    if (multi) {                                     // rare: several spikes in one step
        while (v >= th && ns < max_spikes) { v -= th; ++ns; }
    }
    vmem = v;
    return ns;
}

// The same step for the tensor-core-input kernel, which is bound by the integer ALU pipe (half rate): no clamps when the
// host has proved them idle (SAT_ISYN / SAT_V), no bias add without a bias, and the common single spike as two
// predicated ops.  Identical results.
template <bool SAT_ISYN, bool SAT_V, bool HAS_BIAS>
__device__ __forceinline__ void xylo_step_lean(int &isyn, int &vmem, int &count, int in, int ds, int dm, int bs, int th,
                                               int max_spikes, int &ns_out) {
    isyn = xylo_decay(isyn, ds) + in;
    if (SAT_ISYN) isyn = xylo_sat16(isyn);
    int v = xylo_decay(vmem, dm) + isyn;
    if (HAS_BIAS) v += bs;
    if (SAT_V) v = xylo_sat16(v);
    int ns = 0;
    if (v >= th) { v -= th; ns = 1; }                  // predicated
    if (v >= th) {                                     // rare: several spikes in one step
        while (v >= th && ns < max_spikes) { v -= th; ++ns; }
    }
    count += ns;
    vmem = v;
    ns_out = ns;
}

// named barriers (ids 1..4): full[buf] = masks of a tile are ready, empty[buf] = they have been consumed
// (the forms without .aligned: a warp need not arrive converged)
__device__ __forceinline__ void bar_sync_named(int id, int count) { asm volatile("barrier.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void bar_arrive_named(int id, int count) { asm volatile("barrier.arrive %0, %1;" ::"r"(id), "r"(count) : "memory"); }

// Warp-specialised: the LAST warp of the CTA is the producer, it stages the raw spike bytes of tile
// k+1 and turns them into per-step event masks while the neuron warps run tile k (two mask buffers,
// handed over with named barriers).  Neuron threads: one (clip, hidden neuron) each, state in registers.
// SAT_ISYN = false when the host proved that I_syn cannot leave the int16 range
// (2^dash_syn * (sum_i |w_i| + 1) <= 32767 for every neuron).
constexpr int kLifMinBlocks = 3;     // CTAs of 512 threads per SM the register budget is cut for
// STATE (Xylo stream batches): clip b runs over its first rows_b[b] rows only (T is then the row stride), from the
// I_syn / V_mem it left in nstate [B][N] at its previous call, and leaves them there; counts are those of this call
// (not written for a clip with no rows).
template <bool SIGNED_IN, int W, bool SAT_ISYN, bool RASTER, bool STATE = false>
__global__ void __launch_bounds__(512, kLifMinBlocks)
k_xylo_lif(const int8_t *__restrict__ spikes, int CI, int bipolar, int N_in, const int16_t *__restrict__ w,
           const int16_t *__restrict__ thr, const int8_t *__restrict__ dash_syn, const int8_t *__restrict__ dash_mem,
           const int16_t *__restrict__ bias, int max_spikes, int N, int npb, long long T,
           uint8_t *__restrict__ raster, int32_t *__restrict__ counts, const int32_t *__restrict__ rows_b = nullptr,
           int2 *__restrict__ nstate = nullptr) {
    extern __shared__ __align__(16) unsigned char sm_raw[];
    int16_t *w_s = reinterpret_cast<int16_t *>(sm_raw);                            // [N_in][npb_pad]
    const int npb_pad = (npb + 7) & ~7;
    unsigned int *masks = reinterpret_cast<unsigned int *>(sm_raw + (((size_t)N_in * npb_pad * 2 + 15) & ~(size_t)15));   // [2][kLifTile][W]
    int8_t *raw = reinterpret_cast<int8_t *>(masks + 2 * kLifTile * W);           // [kLifTile][row], producer only
    const int row = SIGNED_IN ? CI : N_in;

    const long long b = blockIdx.x;
    const int n0 = blockIdx.y * npb;
    const int tid = threadIdx.x;
    const int nthreads = blockDim.x;
    const int n_cons = nthreads - 32;                     // neuron threads
    const long long Tb = STATE ? (long long)rows_b[b] : T;                // steps of this clip
    const int ntiles = (int)((Tb + kLifTile - 1) / kLifTile);
    for (int e = tid; e < N_in * npb; e += nthreads) {
        const int i = e / npb, j = e % npb;
        w_s[i * npb_pad + j] = (n0 + j < N) ? w[(long long)i * N + n0 + j] : (int16_t)0;
    }
    __syncthreads();

    if (tid >= n_cons) {
        // ---------------- producer warp ----------------
        const int lane = tid - n_cons;
        const int8_t *src = spikes + b * T * row;
        for (int k = 0; k < ntiles; ++k) {
            const long long t0 = (long long)k * kLifTile;
            const int len = (int)min((long long)kLifTile, Tb - t0);
            {   // raw spike bytes of the tile (coalesced; 16-byte vectors when aligned)
                const int8_t *g = src + t0 * row;
                const int nbytes = len * row;
                if ((reinterpret_cast<uintptr_t>(g) & 15) == 0) {
                    const int nv = nbytes >> 4;
                    for (int v = lane; v < nv; v += 32)
                        reinterpret_cast<int4 *>(raw)[v] = __ldg(reinterpret_cast<const int4 *>(g) + v);
                    for (int e = (nv << 4) + lane; e < nbytes; e += 32) raw[e] = g[e];
                } else {
                    for (int e = lane; e < nbytes; e += 32) raw[e] = g[e];
                }
            }
            __syncwarp();
            if (k >= 2) bar_sync_named(3 + (k & 1), nthreads);       // buffer k&1 has been consumed (tile k-2)
            unsigned int *mk = masks + (k & 1) * kLifTile * W;
            const int len8 = (len + 7) & ~7;                         // the consumers read whole groups of 8 steps
            for (int s = lane; s < len8; s += 32) {
                unsigned int m[W];
#pragma unroll
                for (int q = 0; q < W; ++q) m[q] = 0u;
                if (s < len) {
                    const int8_t *r = raw + s * row;
                    for (int c = 0; c < row; ++c) {
                        const int v = r[c];
                        int bit = -1;
                        if (SIGNED_IN) { if (v > 0) bit = c; else if (v < 0 && bipolar) bit = CI + c; }
                        else if (v != 0) bit = c;
                        if (bit >= 0) {
#pragma unroll
                            for (int q = 0; q < W; ++q)
                                if ((bit >> 5) == q) m[q] |= 1u << (bit & 31);
                        }
                    }
                }
#pragma unroll
                for (int q = 0; q < W; ++q) mk[s * W + q] = m[q];
            }
            __threadfence_block();
            bar_arrive_named(1 + (k & 1), nthreads);                 // masks of tile k are ready
        }
        return;
    }

    // ---------------- neuron threads ----------------
    const int n = n0 + tid;
    const bool live = tid < npb && n < N;
    int isyn = 0, vmem = 0, count = 0;
    if (STATE && live) { const int2 v = nstate[b * N + n]; isyn = v.x; vmem = v.y; }
    const int th = live ? thr[n] : 0x3fffffff;
    const int th2 = 2 * th;
    const int ds = live ? dash_syn[n] : 0, dm = live ? dash_mem[n] : 0;
    const int bs = (live && bias) ? bias[n] : 0;
    const unsigned wn_addr = (unsigned)__cvta_generic_to_shared(w_s + tid);   // this neuron's column of the weight tile
    const int row_bytes = npb_pad * 2;
    uint8_t *rp = (RASTER && live) ? raster + b * T * N + n : nullptr;

    for (int k = 0; k < ntiles; ++k) {
        const int len = (int)min((long long)kLifTile, Tb - (long long)k * kLifTile);
        bar_sync_named(1 + (k & 1), nthreads);                       // wait for the masks of tile k
        if (live) {
            const unsigned int *mk = masks + (k & 1) * kLifTile * W;
#pragma unroll 1
            for (int s0 = 0; s0 < len; s0 += 8) {
                // (A) weighted input of 8 steps: per step a warp-uniform loop over the input events, one add
                //     of an int16 weight each.  It does not depend on the neuron state, so its shared-memory
                //     latency stays off the recurrence
                int wsum[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    int acc = 0;
#pragma unroll
                    for (int q = 0; q < W; ++q) {
                        unsigned int m = mk[(s0 + u) * W + q];       // the same word for the whole CTA: a broadcast
                        while (m) {
                            const int i = 31 - __clz(m);             // highest pending event
                            m ^= 1u << i;
                            int wv;
                            asm("ld.shared.s16 %0, [%1];" : "=r"(wv) : "r"(wn_addr + (unsigned)((i + 32 * q) * row_bytes)));
                            acc += wv;
                        }
                    }
                    wsum[u] = acc;
                }
                // (B) the integer LIF recurrence of the 8 steps, state in registers
                if (s0 + 8 <= len) {
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int ns = xylo_step<SAT_ISYN>(isyn, vmem, wsum[u], ds, dm, bs, th, th2, max_spikes);
                        count += ns;
                        if (RASTER) { *rp = (uint8_t)ns; rp += N; }
                    }
                } else {
#pragma unroll
                    for (int u = 0; u < 8; ++u)
                        if (s0 + u < len) {
                            const int ns = xylo_step<SAT_ISYN>(isyn, vmem, wsum[u], ds, dm, bs, th, th2, max_spikes);
                            count += ns;
                            if (RASTER) { *rp = (uint8_t)ns; rp += N; }
                        }
                }
            }
        }
        if (k + 2 < ntiles) bar_arrive_named(3 + (k & 1), nthreads); // buffer k&1 may be refilled (tile k+2)
    }
    if (STATE && live) nstate[b * N + n] = make_int2(isyn, vmem);
    if (live && counts && (!STATE || Tb > 0)) counts[b * N + n] = count;
}


// ---------------------------------------------------------------------------
// The same network with the weighted input on the tensor cores.  The input current of a step, sum_i spike_i[t] w[i][n],
// IS a matrix product (binary spikes [T][N_in] x int8 weights [N_in][N]).  Every neuron warp computes it for its own 32
// neurons, exactly, with int8 mma.sync.m16n8k32 (A = weights of 16 neurons x 32 inputs, held in registers for the
// whole clip; B = 8 time steps x 32 inputs from the tile's binary spike rows; int32 accumulators): 6 MMAs per tile of
// 24 steps.  The accumulator layout spreads a neuron's steps over four lanes, so the sums pass through a warp-private
// int16 [neuron][step] buffer in shared memory (48-byte rows: the 32-bit stores and the 128-bit loads are both
// conflict-free) and a neuron thread fetches the inputs of 8 steps with one load.  Per step that is ~2 instructions
// instead of the ~12 of the event loop above (bit scan + address + load + add per event), at identical integer
// results.  The producer warp only turns the signed spike bytes of the next tile into binary rows.
// Needs N_in <= 32 and |sum| < 2^15 (checked by the host); otherwise the event-loop kernel runs.
// ---------------------------------------------------------------------------
constexpr int kMmaTile = 24;     // time steps per tile: 3 MMA column blocks
constexpr int kLifMmaMinBlocks = 2;

__device__ __forceinline__ void mma_s8_16x8x32(int (&d)[4], const unsigned (&a)[4], unsigned b0, unsigned b1) {
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.s8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
                 : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1), "r"(0));
}

__device__ __forceinline__ int imad_pipe(int a, int b, int c) {
    int r;
    asm("mad.lo.s32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}
constexpr int kTrPitch = 28;      // int32 words per neuron row of the hand-over buffer: 24 steps + 4 (conflict-free 128-bit reads)
// STATE: as in k_xylo_lif (per-clip row counts rows_b, I_syn / V_mem carried in nstate, counts of this call).  A group of
// 8 steps that straddles a clip's last row takes the tail path, so the multi-spike redo never sees a step beyond it.
template <bool SIGNED_IN, bool SAT_ISYN, bool SAT_V, bool HAS_BIAS, bool RASTER, bool STATE = false>
__global__ void __launch_bounds__(512, kLifMmaMinBlocks)
k_xylo_lif_mma(const int8_t *__restrict__ spikes, int CI, int bipolar, int N_in, const int8_t *__restrict__ w8, int w_shift,
               const int16_t *__restrict__ thr, const int8_t *__restrict__ dash_syn, const int8_t *__restrict__ dash_mem,
               const int16_t *__restrict__ bias, int max_spikes, int N, int npb, long long T,
               uint8_t *__restrict__ raster, int32_t *__restrict__ counts, const int32_t *__restrict__ rows_b = nullptr,
               int2 *__restrict__ nstate = nullptr) {
    extern __shared__ __align__(16) unsigned char sm_raw[];
    uint8_t *Sb = sm_raw;                                                                // [2][kMmaTile][32] binary spikes
    int *tr_all = reinterpret_cast<int *>(sm_raw + 2 * kMmaTile * 32);                   // [neuron warps][32][kTrPitch]
    const int row = SIGNED_IN ? CI : N_in;

    const long long b = blockIdx.x;
    const int n0 = blockIdx.y * npb;
    const int tid = threadIdx.x;
    const int nthreads = blockDim.x;
    const int n_cons = nthreads - 32;
    const long long Tb = STATE ? (long long)rows_b[b] : T;                // steps of this clip
    const int ntiles = (int)((Tb + kMmaTile - 1) / kMmaTile);
    for (int e = tid; e < 2 * kMmaTile * 32; e += nthreads) Sb[e] = 0;       // columns beyond the inputs stay zero
    __syncthreads();

    if (tid >= n_cons) {
        // ---------------- producer warp: signed spike bytes -> binary rows ----------------
        // lane = time step of the tile; a row (<= 32 bytes, even length) travels as 16-bit words, prefetched one tile ahead
        const int lane = tid - n_cons;
        const int8_t *src = spikes + b * T * row;
        constexpr int kPreW = 16;
        unsigned short pre[kPreW];
        auto prefetch = [&](int k) {
            const long long t = (long long)k * kMmaTile + lane;
            const bool valid = k < ntiles && lane < kMmaTile && t < Tb;
            const unsigned short *gp = reinterpret_cast<const unsigned short *>(src + t * row);
#pragma unroll
            for (int j = 0; j < kPreW; ++j) pre[j] = (valid && 2 * j < row) ? __ldg(gp + j) : (unsigned short)0;
        };
        prefetch(0);
        for (int k = 0; k < ntiles; ++k) {
            if (k >= 2) bar_sync_named(3 + (k & 1), nthreads);       // rows k&1 have been read (tile k-2)
            if (lane < kMmaTile) {
                uint8_t *S = Sb + ((k & 1) * kMmaTile + lane) * 32;
#pragma unroll
                for (int j = 0; j < kPreW; ++j) {
                    if (2 * j < row) {
                        const int v0 = (int)(signed char)(pre[j] & 0xff), v1 = (int)(signed char)(pre[j] >> 8);   // zero behind the clip end
                        if (SIGNED_IN) {
                            *reinterpret_cast<unsigned short *>(S + 2 * j) = (unsigned short)((v0 > 0 ? 1 : 0) | (v1 > 0 ? 0x100 : 0));
                            if (bipolar) { S[CI + 2 * j] = v0 < 0 ? 1 : 0; S[CI + 2 * j + 1] = v1 < 0 ? 1 : 0; }
                        } else {
                            *reinterpret_cast<unsigned short *>(S + 2 * j) = (unsigned short)((v0 != 0 ? 1 : 0) | (v1 != 0 ? 0x100 : 0));
                        }
                    }
                }
            }
            __threadfence_block();
            bar_arrive_named(1 + (k & 1), nthreads);                 // rows of tile k are ready
            prefetch(k + 1);                                         // next tile's bytes on their way
        }
        return;
    }

    // ---------------- neuron warps ----------------
    const int lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, tq = lane & 3;
    const int n = n0 + tid;
    const bool live = tid < npb && n < N;
    int isyn = 0, vmem = 0, count = 0;
    if (STATE && live) { const int2 v = nstate[b * N + n]; isyn = v.x; vmem = v.y; }
    const int th = live ? thr[n] : 0x3fffffff;
    const int ds = live ? dash_syn[n] : 0, dm = live ? dash_mem[n] : 0;
    const int bs = (live && bias) ? bias[n] : 0;
    uint8_t *rp = (RASTER && live) ? raster + b * T * N + n : nullptr;
    int *tr = tr_all + (size_t)warp * 32 * kTrPitch;
    const int one = (w_shift >> 31) + 1, neg_one = -one;      // 1 and -1 (w_shift >= 0), but not to the compiler
    // A fragments of this warp's two blocks of 16 neurons: a0 = (neuron g, inputs 4 tq ..), a1 = (neuron g + 8, same),
    // a2 / a3 = inputs 16 + 4 tq ..
    unsigned af[2][4];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int nl = 32 * warp + 16 * r + g + 8 * (q & 1);   // neuron inside this CTA's chunk
            unsigned v = 0u;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int i = 16 * (q >> 1) + 4 * tq + e;
                const int wv = (i < N_in && nl < npb && n0 + nl < N) ? (int)w8[(long long)i * N + n0 + nl] : 0;
                v |= ((unsigned)wv & 0xffu) << (8 * e);
            }
            af[r][q] = v;
        }

    for (int k = 0; k < ntiles; ++k) {
        const int len = (int)min((long long)kMmaTile, Tb - (long long)k * kMmaTile);
        bar_sync_named(1 + (k & 1), nthreads);                       // wait for the binary rows of tile k
        const uint8_t *S = Sb + (k & 1) * kMmaTile * 32;
        unsigned bf[kMmaTile / 8][2];
#pragma unroll
        for (int sb = 0; sb < kMmaTile / 8; ++sb) {
            bf[sb][0] = *reinterpret_cast<const unsigned *>(S + (8 * sb + g) * 32 + 4 * tq);
            bf[sb][1] = *reinterpret_cast<const unsigned *>(S + (8 * sb + g) * 32 + 16 + 4 * tq);
        }
        if (k + 2 < ntiles) bar_arrive_named(3 + (k & 1), nthreads); // rows k&1 may be refilled (tile k+2)
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int sb = 0; sb < kMmaTile / 8; ++sb) {
                int d[4];
                mma_s8_16x8x32(d, af[r], bf[sb][0], bf[sb][1]);
                // d0, d1 = (neuron g, steps 2 tq, 2 tq + 1); d2, d3 = neuron g + 8
                *reinterpret_cast<int2 *>(tr + (16 * r + g) * kTrPitch + 8 * sb + 2 * tq) = make_int2(d[0] << w_shift, d[1] << w_shift);
                *reinterpret_cast<int2 *>(tr + (16 * r + g + 8) * kTrPitch + 8 * sb + 2 * tq) = make_int2(d[2] << w_shift, d[3] << w_shift);
            }
        __syncwarp();
        if (live) {
            const int *wt = tr + lane * kTrPitch;
#pragma unroll 1
            for (int s0 = 0; s0 < len; s0 += 8) {
                const int4 p0 = *reinterpret_cast<const int4 *>(wt + s0), p1 = *reinterpret_cast<const int4 *>(wt + s0 + 4);
                const int in[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
                if (s0 + 8 <= len) {
                    // eight steps with at most ONE spike each (the common case: two predicated ops per step, no branch);
                    // a step that would fire again (V >= 2 threshold, rare) only raises a flag, and the group is then
                    // redone from its saved state by the exact multi-spike loop
                    const int isyn0 = isyn, vmem0 = vmem, count0 = count;
                    bool again = false;
                    unsigned fired = 0u;
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        // (the adds as IMADs by a register that holds 1 / -1: they issue on the FMA pipe, which idles, instead
                        //  of the half-rate integer ALU pipe that bounds this loop)
                        isyn = imad_pipe(in[u], one, imad_pipe(max(isyn >> ds, min(isyn, 1)), neg_one, isyn));
                        if (SAT_ISYN) isyn = xylo_sat16(isyn);
                        int v = imad_pipe(isyn, one, imad_pipe(max(vmem >> dm, min(vmem, 1)), neg_one, vmem));
                        if (HAS_BIAS) v += bs;
                        if (SAT_V) v = xylo_sat16(v);
                        if (v >= th) { v = imad_pipe(th, neg_one, v); count = imad_pipe(one, one, count); if (RASTER) fired |= 1u << u; }
                        again |= v >= th;
                        vmem = v;
                    }
                    if (again) {
                        isyn = isyn0; vmem = vmem0; count = count0;
#pragma unroll 1
                        for (int u = 0; u < 8; ++u) {
                            int ns;
                            xylo_step_lean<SAT_ISYN, SAT_V, HAS_BIAS>(isyn, vmem, count, in[u], ds, dm, bs, th, max_spikes, ns);
                            if (RASTER) { *rp = (uint8_t)ns; rp += N; }
                        }
                    } else if (RASTER) {
#pragma unroll
                        for (int u = 0; u < 8; ++u) { *rp = (uint8_t)((fired >> u) & 1u); rp += N; }
                    }
                } else {
#pragma unroll 1
                    for (int u = 0; u < 8; ++u)
                        if (s0 + u < len) {
                            int ns;
                            xylo_step_lean<SAT_ISYN, SAT_V, HAS_BIAS>(isyn, vmem, count, in[u], ds, dm, bs, th, max_spikes, ns);
                            if (RASTER) { *rp = (uint8_t)ns; rp += N; }
                        }
                }
            }
        }
        __syncwarp();                                                // the next tile overwrites this warp's buffer
    }
    if (STATE && live) nstate[b * N + n] = make_int2(isyn, vmem);
    if (live && counts && (!STATE || Tb > 0)) counts[b * N + n] = count;
}

// One CTA per clip: S[g] = sum_f counts[f*G + g]; doa = first argmax S; doa_peak = first argmax of the
// 'full' box-car sums of S, minus win/2, modulo G (micloc/utils.py:84-121 on integers).
__global__ void __launch_bounds__(128)
k_xylo_doa(const int32_t *__restrict__ counts, int G, int F, int win, int32_t *__restrict__ doa,
           int32_t *__restrict__ doa_peak, const int32_t *__restrict__ rows_b = nullptr) {
    extern __shared__ __align__(16) long long S[];      // [G]
    __shared__ long long red_v[128];
    __shared__ int red_i[128];
    const long long b = blockIdx.x;
    if (rows_b && rows_b[b] == 0) return;               // (stream batches: a slot with no final rows; uniform per block)
    const int32_t *c = counts + b * (long long)G * F;
    for (int g = threadIdx.x; g < G; g += blockDim.x) {
        long long a = 0;
        for (int f = 0; f < F; ++f) a += c[(long long)f * G + g];
        S[g] = a;
    }
    __syncthreads();
    for (int pass = 0; pass < 2; ++pass) {
        if (pass == 1 && (!doa_peak || win < 1)) break;
        const int J = pass == 0 ? G : G + win - 1;
        long long best = -1; int besti = 0x7fffffff;
        for (int j = threadIdx.x; j < J; j += blockDim.x) {
            long long v;
            if (pass == 0) v = S[j];
            else {
                const int lo = max(0, j - win + 1), hi = min(j, G - 1);
                v = 0;
                for (int k = lo; k <= hi; ++k) v += S[k];
            }
            if (v > best) { best = v; besti = j; }      // ascending j: first maximum kept
        }
        red_v[threadIdx.x] = best; red_i[threadIdx.x] = besti;
        __syncthreads();
        for (int st = blockDim.x / 2; st > 0; st >>= 1) {
            if (threadIdx.x < st) {
                const long long ov = red_v[threadIdx.x + st]; const int oi = red_i[threadIdx.x + st];
                if (ov > red_v[threadIdx.x] || (ov == red_v[threadIdx.x] && oi < red_i[threadIdx.x])) {
                    red_v[threadIdx.x] = ov; red_i[threadIdx.x] = oi;
                }
            }
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            if (pass == 0) { if (doa) doa[b] = red_i[0]; }
            else {
                int idx = (red_i[0] - win / 2) % G;
                if (idx < 0) idx += G;
                doa_peak[b] = idx;
            }
        }
        __syncthreads();
    }
}

// signed raster [n][CI] -> Demo.spike_encoding's layout [n][N_in] in {0,1}; rows_b (nullable, stream batches): row r
// of clip r / T is only converted below rows_b[r / T]
__global__ void __launch_bounds__(256)
k_xylo_split(const int8_t *__restrict__ s, int8_t *__restrict__ out, long long rows, int CI, int bipolar,
             const int32_t *__restrict__ rows_b = nullptr, long long T = 1) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * CI) return;
    const long long r = i / CI;
    if (rows_b && r % T >= rows_b[r / T]) return;
    const int c = (int)(i % CI);
    const int v = s[i];
    if (bipolar) {
        out[r * 2 * CI + c] = v > 0;
        out[r * 2 * CI + CI + c] = v < 0;
    } else {
        out[r * CI + c] = (int8_t)v;
    }
}

}  // namespace micloc

using namespace micloc;

struct micloc_xylo {
    int device = 0;
    ChainParams p{};
    int F = 1, N = 0, G = 0, N_in = 0, CT = 0, nba = 0, max_spikes = 31;
    bool has_rec = false;
    bool sat_isyn = true;           // I_syn can reach the int16 limits: keep the clamps
    bool sat_v = true;              // V_mem can reach the int16 limits
    float *d_taps = nullptr;        // float32 compacted STHT taps (fast front end)
    float *d_band_sos = nullptr;    // [F][kMaxSections][5]
    double *d_h = nullptr;          // [K] float64 STHT kernel (exact front end)
    double *d_g = nullptr;          // [n_g] its non-zero taps, oldest sample first, when every other tap is exactly zero
    int n_g = 0;
    long long n_fallback = 0;       // clips the fast exact front end handed to the unbounded kernels so far
    double *d_ba_b = nullptr, *d_ba_a = nullptr;   // [F][nba]
    int16_t *d_w = nullptr;         // [N_in][N] input weights, shift applied
    int8_t *d_w8 = nullptr;         // [N_in][N] input weights as given (tensor-core input path)
    int w_shift = 0;
    bool lif_mma = false;           // k_xylo_lif_mma applies (N_in <= 32, weighted sums fit int16)
    int16_t *d_thr = nullptr, *d_bias = nullptr;
    int8_t *d_ds = nullptr, *d_dm = nullptr;
    DevBuf q, qd, zd, signed_spk, counts, flags;
    // float32 front end through the fused SNN kernel (one band, <= 8 microphones): its spike raster is
    // exactly Demo.spike_encoding's signed raster; the neuron / power tail runs on a dummy 1-column bf_mat
    bool use_fused = false;
    ChainParams pf{};
    double *d_Wd1 = nullptr;        // [2M][1] zeros
    unsigned int *d_sm_slots = nullptr;
    int sm_count = 148;
};
static constexpr size_t kXyloSlotWords = kSlotWords;

extern "C" int micloc_xylo_destroy(micloc_xylo *c) {
    if (!c) return MICLOC_OK;
    cudaSetDevice(c->device);
    cudaFree(c->d_taps); cudaFree(c->d_band_sos); cudaFree(c->d_h); cudaFree(c->d_g); cudaFree(c->d_ba_b); cudaFree(c->d_ba_a);
    cudaFree(c->d_w); cudaFree(c->d_w8); cudaFree(c->d_thr); cudaFree(c->d_bias); cudaFree(c->d_ds); cudaFree(c->d_dm);
    cudaFree(c->d_Wd1); cudaFree(c->d_sm_slots);
    c->q.release(); c->qd.release(); c->zd.release(); c->signed_spk.release(); c->counts.release(); c->flags.release();
    delete c;
    return MICLOC_OK;
}

template <typename T>
static int upload(T **dst, const T *src, size_t n) {
    MICLOC_CUDA(cudaMalloc((void **)dst, n * sizeof(T)));
    MICLOC_CUDA(cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice));
    return MICLOC_OK;
}

extern "C" int micloc_xylo_create(const micloc_xylo_config *cfg, int device, micloc_xylo **out) {
    if (!cfg || !out) return set_error(MICLOC_ERR_CONFIG, "null config");
    *out = nullptr;
    if (cfg->num_mic < 1 || cfg->num_mic > 128)
        return set_error(MICLOC_ERR_CONFIG, "num_mic %d out of range [1, 128]", cfg->num_mic);
    if (!cfg->stht_kernel || !cfg->sos || !cfg->w_in || !cfg->threshold || !cfg->dash_syn || !cfg->dash_mem)
        return set_error(MICLOC_ERR_CONFIG, "null array in config");
    if (cfg->num_bands < 1 || cfg->num_bands > 16) return set_error(MICLOC_ERR_CONFIG, "num_bands %d out of range [1, 16]", cfg->num_bands);
    if (cfg->robust_width < 1) return set_error(MICLOC_ERR_CONFIG, "`distance` must be greater or equal to 1");
    if (cfg->num_doa < 1 || cfg->num_hidden != cfg->num_doa * cfg->num_bands)
        return set_error(MICLOC_ERR_CONFIG, "num_hidden %d must equal num_doa %d x num_bands %d", cfg->num_hidden, cfg->num_doa, cfg->num_bands);
    if (cfg->n_ba < 0 || cfg->n_ba > kMaxBa || (cfg->n_ba > 0 && (!cfg->ba_b || !cfg->ba_a)))
        return set_error(MICLOC_ERR_CONFIG, "bad b/a filter description (n_ba %d, at most %d)", cfg->n_ba, kMaxBa);
    if (cfg->weight_shift_in < 0 || cfg->weight_shift_in > 7 || cfg->weight_shift_rec < 0 || cfg->weight_shift_rec > 7)
        return set_error(MICLOC_ERR_CONFIG, "weight shifts must be in [0, 7]");
    if (cfg->max_spikes < 1 || cfg->max_spikes > 255) return set_error(MICLOC_ERR_CONFIG, "max_spikes must be in [1, 255]");
    const int CT = 2 * cfg->num_mic * cfg->num_bands;
    const int N_in = CT * (cfg->bipolar ? 2 : 1);
    if (N_in > 128) return set_error(MICLOC_ERR_UNSUPPORTED, "at most 128 input channels (got %d)", N_in);
    const int N = cfg->num_hidden;
    bool has_rec = false;
    if (cfg->w_rec)
        for (size_t i = 0; i < (size_t)N * N && !has_rec; ++i) has_rec = cfg->w_rec[i] != 0;
    if (has_rec)
        return set_error(MICLOC_ERR_UNSUPPORTED, "non-zero quantised recurrent weights are not supported on the device "
                                                 "(the reference's w_rec = -0.1/N quantises to zero)");
    for (int n = 0; n < N; ++n) {
        if (cfg->threshold[n] < 1) return set_error(MICLOC_ERR_CONFIG, "threshold[%d] = %d must be >= 1", n, cfg->threshold[n]);
        if (cfg->dash_syn[n] < 0 || cfg->dash_syn[n] > 15 || cfg->dash_mem[n] < 0 || cfg->dash_mem[n] > 15)
            return set_error(MICLOC_ERR_CONFIG, "dash[%d] out of range [0, 15]", n);
    }
    MICLOC_CUDA(cudaSetDevice(device));
    micloc_xylo *c = new micloc_xylo();
    c->device = device;
    ChainParams &p = c->p;
    p.M = cfg->num_mic; p.C2 = 2 * cfg->num_mic;
    p.w = cfg->robust_width; p.bipolar = cfg->bipolar ? 1 : 0;
    p.nsec = cfg->n_sections;
    p.na = 0.5f; p.nc = 1.f; p.ncT = 0.f; p.nLf = 1.f; p.nL = 1; p.G = cfg->num_doa;
    c->F = cfg->num_bands; c->N = N; c->G = cfg->num_doa; c->N_in = N_in; c->CT = CT; c->nba = cfg->n_ba;
    c->max_spikes = cfg->max_spikes;
    int rc = setup_stht(p, cfg->stht_kernel, cfg->kernel_len, &c->d_taps);
    if (rc) { micloc_xylo_destroy(c); return rc; }
    std::vector<float> sosf((size_t)c->F * kMaxSections * 5);
    for (int f = 0; f < c->F && !rc; ++f)
        rc = sos_to_f32(cfg->sos + (size_t)f * cfg->n_sections * 6, cfg->n_sections, &sosf[(size_t)f * kMaxSections * 5]);
    if (!rc) { for (int k = 0; k < kMaxSections * 5; ++k) (&p.sos[0][0])[k] = sosf[k]; }
    if (!rc) rc = upload(&c->d_band_sos, sosf.data(), sosf.size());
    if (!rc) rc = upload(&c->d_h, cfg->stht_kernel, (size_t)cfg->kernel_len);
    if (!rc) {
        // Hilbert kernels (snn_beamformer.py:50-53) are exactly zero at every even index: the register-blocked
        // float64 FIR walks the K/2 other taps only
        const int K = cfg->kernel_len;
        bool sparse = K % 8 == 0 && K >= 8;
        for (int k = 0; k < K && sparse; k += 2) sparse = cfg->stht_kernel[k] == 0.0;
        if (sparse) {
            std::vector<double> g((size_t)K / 2);
            for (int i = 0; i < K / 2; ++i) g[i] = cfg->stht_kernel[K - 1 - 2 * i];
            c->n_g = K / 2;
            rc = upload(&c->d_g, g.data(), g.size());
        }
    }
    if (!rc && cfg->n_ba > 0) {
        rc = upload(&c->d_ba_b, cfg->ba_b, (size_t)c->F * cfg->n_ba);
        if (!rc) rc = upload(&c->d_ba_a, cfg->ba_a, (size_t)c->F * cfg->n_ba);
        for (int f = 0; f < c->F && !rc; ++f)
            if (cfg->ba_a[(size_t)f * cfg->n_ba] != 1.0) rc = set_error(MICLOC_ERR_CONFIG, "band filter %d: a[0] must be 1", f);
    }
    if (!rc) {
        std::vector<int16_t> w16((size_t)N_in * N);
        for (size_t i = 0; i < w16.size(); ++i) w16[i] = (int16_t)((int)cfg->w_in[i] << cfg->weight_shift_in);
        rc = upload(&c->d_w, w16.data(), w16.size());
        if (!rc) rc = upload(&c->d_w8, cfg->w_in, (size_t)N_in * N);
        c->w_shift = cfg->weight_shift_in;
        // tensor-core input path (k_xylo_lif_mma): 32 input columns per MMA, int16 hand-over of the weighted sum
        c->lif_mma = N_in <= 32 && cfg->weight_shift_in >= 0 && (((long long)N_in * 128) << cfg->weight_shift_in) <= 32767;
        // |I_syn| <= 2^dash_syn * (sum_i |w_i| + 1) by induction over the decay recurrence
        c->sat_isyn = false;
        for (int n = 0; n < N && !c->sat_isyn; ++n) {
            long long sabs = 1;
            for (int i = 0; i < N_in; ++i) sabs += w16[(size_t)i * N + n] < 0 ? -w16[(size_t)i * N + n] : w16[(size_t)i * N + n];
            if ((sabs << cfg->dash_syn[n]) > 32767) c->sat_isyn = true;
        }
        // |V_mem| <= 2^dash_mem * (I + |bias| + 1) with I the bound on |I_syn|: one decay step removes at least
        // |V| / 2^dash_mem - 1, the spikes only move a positive V towards zero
        c->sat_v = c->sat_isyn;
        for (int n = 0; n < N && !c->sat_v; ++n) {
            long long sabs = 1;
            for (int i = 0; i < N_in; ++i) sabs += w16[(size_t)i * N + n] < 0 ? -w16[(size_t)i * N + n] : w16[(size_t)i * N + n];
            const long long ib = sabs << cfg->dash_syn[n];
            const long long bb = cfg->bias ? (cfg->bias[n] < 0 ? -(long long)cfg->bias[n] : (long long)cfg->bias[n]) : 0;
            if (((ib + bb + 1) << cfg->dash_mem[n]) > 32767) c->sat_v = true;
        }
    }
    if (!rc) rc = upload(&c->d_thr, cfg->threshold, (size_t)N);
    if (!rc) rc = upload(&c->d_ds, cfg->dash_syn, (size_t)N);
    if (!rc) rc = upload(&c->d_dm, cfg->dash_mem, (size_t)N);
    if (!rc && cfg->bias) rc = upload(&c->d_bias, cfg->bias, (size_t)N);
    if (!rc) {
        c->pf = p;
        c->pf.G = 1;
        if (c->pf.nsec == 1) {      // identity second section: y = 1*x + 0 exactly
            c->pf.nsec = 2;
            c->pf.sos[1][0] = 1.f; c->pf.sos[1][1] = c->pf.sos[1][2] = c->pf.sos[1][3] = c->pf.sos[1][4] = 0.f;
        }
        c->use_fused = c->F == 1 && fused_supported(c->pf);
        if (c->use_fused) {
            std::vector<double> z((size_t)p.C2, 0.0);
            rc = upload(&c->d_Wd1, z.data(), z.size());
            if (!rc && (cudaMalloc(&c->d_sm_slots, kXyloSlotWords * sizeof(unsigned int)) != cudaSuccess ||
                        cudaMemset(c->d_sm_slots, 0, kXyloSlotWords * sizeof(unsigned int)) != cudaSuccess))
                rc = set_error(MICLOC_ERR_CUDA, "cudaMalloc(sm_slots) failed");
            cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
        }
    }
    if (rc) { micloc_xylo_destroy(c); return rc; }
    *out = c;
    return MICLOC_OK;
}

static int check_xylo_args(micloc_xylo *c, const void *in, int64_t B, int64_t T) {
    if (!c) return set_error(MICLOC_ERR_CONFIG, "null context");
    if (!in) return set_error(MICLOC_ERR_SHAPE, "null input pointer");
    if (B < 1 || T < 1) return set_error(MICLOC_ERR_SHAPE, "empty batch (B=%lld, T=%lld)", (long long)B, (long long)T);
    if (T > (1ll << 30) || B > 0x7fffffffll) return set_error(MICLOC_ERR_SHAPE, "batch too large");
    return MICLOC_OK;
}

// integer network on a spike raster already on the device (STATE: stream batches, see k_xylo_lif)
template <bool SIGNED_IN, bool STATE = false>
static int launch_lif(micloc_xylo *c, const int8_t *spikes, long long B, long long T, uint8_t *raster,
                      int32_t *counts, cudaStream_t st, const int32_t *rows_b = nullptr, int2 *nstate = nullptr) {
    const int N = c->N;
    const int nchunks = (N + 479) / 480;                       // <= 480 neurons (15 warps) per CTA
    const int npb = (N + nchunks - 1) / nchunks;
    const int threads = ((npb + 31) & ~31) + 32;             // neuron warps + the producer warp
    const int row_in = SIGNED_IN ? c->CT : c->N_in;
    if (c->lif_mma && row_in <= 32 && (row_in & 1) == 0 && ((uintptr_t)spikes & 1) == 0 && !getenv("MICLOC_XYLO_LIF_ADDS")) {
        const size_t smem_m = (size_t)2 * kMmaTile * 32 + (size_t)((threads - 32) / 32) * 32 * kTrPitch * 4 + 16;
        dim3 grid_m((unsigned)B, (unsigned)nchunks);
        void (*kern)(const int8_t *, int, int, int, const int8_t *, int, const int16_t *, const int8_t *, const int8_t *,
                     const int16_t *, int, int, int, long long, uint8_t *, int32_t *, const int32_t *, int2 *) = nullptr;
        const bool hb = c->d_bias != nullptr;
#define MICLOC_MMA_PICK(SI, SV, HB)                                                                          \
        kern = raster ? k_xylo_lif_mma<SIGNED_IN, SI, SV, HB, true, STATE> : k_xylo_lif_mma<SIGNED_IN, SI, SV, HB, false, STATE>
        if (c->sat_isyn) { if (hb) MICLOC_MMA_PICK(true, true, true); else MICLOC_MMA_PICK(true, true, false); }
        else if (c->sat_v) { if (hb) MICLOC_MMA_PICK(false, true, true); else MICLOC_MMA_PICK(false, true, false); }
        else { if (hb) MICLOC_MMA_PICK(false, false, true); else MICLOC_MMA_PICK(false, false, false); }
#undef MICLOC_MMA_PICK
        MICLOC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_m));
        kern<<<grid_m, threads, smem_m, st>>>(spikes, c->CT, c->p.bipolar, c->N_in, c->d_w8, c->w_shift, c->d_thr, c->d_ds, c->d_dm,
                                              c->d_bias, c->max_spikes, N, npb, T, raster, counts, rows_b, nstate);
        count_launch(1);
        MICLOC_CUDA(cudaGetLastError());
        return MICLOC_OK;
    }
    const int W = (c->N_in + 31) / 32;
    const int npb_pad = (npb + 7) & ~7;
    const int row = SIGNED_IN ? c->CT : c->N_in;
    const size_t smem = (((size_t)c->N_in * npb_pad * 2 + 15) & ~(size_t)15) + (size_t)2 * kLifTile * W * 4 + (size_t)kLifTile * row + 16;
    if (smem > 227 * 1024) return set_error(MICLOC_ERR_UNSUPPORTED, "LIF kernel needs %zu B of shared memory", smem);
    dim3 grid((unsigned)B, (unsigned)nchunks);
#define MICLOC_LIF_CASE(WW)                                                                                       \
    case WW: {                                                                                                    \
        auto kern = raster ? (c->sat_isyn ? k_xylo_lif<SIGNED_IN, WW, true, true, STATE> : k_xylo_lif<SIGNED_IN, WW, false, true, STATE>)   \
                           : (c->sat_isyn ? k_xylo_lif<SIGNED_IN, WW, true, false, STATE> : k_xylo_lif<SIGNED_IN, WW, false, false, STATE>); \
        MICLOC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));          \
        kern<<<grid, threads, smem, st>>>(spikes, c->CT, c->p.bipolar, c->N_in, c->d_w, c->d_thr, c->d_ds, c->d_dm, \
                                          c->d_bias, c->max_spikes, N, npb, T, raster, counts, rows_b, nstate);   \
    } break
    switch (W) {
        MICLOC_LIF_CASE(1);
        MICLOC_LIF_CASE(2);
        MICLOC_LIF_CASE(3);
        MICLOC_LIF_CASE(4);
        default: return set_error(MICLOC_ERR_UNSUPPORTED, "too many input channels");
    }
#undef MICLOC_LIF_CASE
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}

static int check_peak_win(const micloc_xylo *c, const int32_t *doa_peak, int win) {
    if (doa_peak && (win < 1 || (win & 1) == 0 || win > c->G / 2))
        return set_error(MICLOC_ERR_CONFIG, "averaging window size should be odd and at most half the DoA grid");  // utils.py:103-111
    return MICLOC_OK;
}

static int launch_doa(micloc_xylo *c, const int32_t *counts, long long B, int32_t *doa, int32_t *doa_peak, int win,
                      cudaStream_t st, const int32_t *rows_b = nullptr) {
    if (!doa && !doa_peak) return MICLOC_OK;
    if (doa_peak && (win < 1 || (win & 1) == 0 || win > c->G / 2))
        return set_error(MICLOC_ERR_CONFIG, "averaging window size should be odd and at most half the DoA grid");  // utils.py:103-111
    const size_t smem = (size_t)c->G * sizeof(long long);
    MICLOC_CUDA(cudaFuncSetAttribute(k_xylo_doa, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_xylo_doa<<<(unsigned)B, 128, smem, st>>>(counts, c->G, c->F, doa_peak ? win : 0, doa, doa_peak, rows_b);
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}

// exact float64 front end, staged (unbounded candidate clusters): STHT -> q, band filters -> z, RZCC -> signed spikes
static int exact_front_staged(micloc_xylo *c, const void *a, int dtype, long long nb, long long T, int8_t *sgn, cudaStream_t st) {
    const ChainParams &p = c->p;
    const int CT = c->CT;
    MICLOC_TRY(c->qd.reserve((size_t)nb * T * p.M * sizeof(double)));
    MICLOC_TRY(c->zd.reserve((size_t)nb * T * CT * sizeof(double)));
    const bool sparse = c->n_g > 0 && !getenv("MICLOC_XYLO_DENSE_F64");
    const int tile = sparse ? kSTile : kF64Tile;
    const int ntiles = (int)((T + tile - 1) / tile);
    const int mgmax = p.M < kF64MG ? p.M : kF64MG;
    const size_t smem = sparse ? ((size_t)c->n_g + (size_t)mgmax * ((f64_pad(kSTile + p.K - 1) + 9) & ~1)) * sizeof(double)
                               : ((size_t)p.K + (size_t)mgmax * (kF64Tile + p.K - 1)) * sizeof(double);
    if (smem > 227 * 1024) return set_error(MICLOC_ERR_UNSUPPORTED, "exact STHT tile needs %zu B of shared memory", smem);
    dim3 grid((unsigned)(nb * ntiles), (unsigned)((p.M + kF64MG - 1) / kF64MG));
    double *qd = (double *)c->qd.ptr;
    if (dtype == MICLOC_I16) {
        const int16_t *a16 = (const int16_t *)a;
        if (sparse) {
            MICLOC_CUDA(cudaFuncSetAttribute(k_stht_f64_sparse<int16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k_stht_f64_sparse<int16_t><<<grid, 256, smem, st>>>(a16, c->d_g, qd, p.M, p.K, c->n_g, T, ntiles);
        } else {
            MICLOC_CUDA(cudaFuncSetAttribute(k_stht_f64<int16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k_stht_f64<int16_t><<<grid, kF64Tile, smem, st>>>(a16, c->d_h, qd, p.M, p.K, T, ntiles);
        }
        launch_iir_f64(a16, qd, c->d_ba_b, c->d_ba_a, (double *)c->zd.ptr, p.M, p.half, c->nba, c->F, nb, T, st);
    } else {
        const float *a32 = (const float *)a;
        if (sparse) {
            MICLOC_CUDA(cudaFuncSetAttribute(k_stht_f64_sparse<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k_stht_f64_sparse<float><<<grid, 256, smem, st>>>(a32, c->d_g, qd, p.M, p.K, c->n_g, T, ntiles);
        } else {
            MICLOC_CUDA(cudaFuncSetAttribute(k_stht_f64<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k_stht_f64<float><<<grid, kF64Tile, smem, st>>>(a32, c->d_h, qd, p.M, p.K, T, ntiles);
        }
        launch_iir_f64(a32, qd, c->d_ba_b, c->d_ba_a, (double *)c->zd.ptr, p.M, p.half, c->nba, c->F, nb, T, st);
    }
    count_launch(2);
    MICLOC_CUDA(cudaGetLastError());
    return micloc_rzcc_encode_f64((const double *)c->zd.ptr, nb, T, CT, p.w, p.bipolar, sgn, c->device, st);
}

// exact float64 front end, fast form: register-blocked STHT (q in HBM) + one warp per clip for everything behind it;
// clips whose clusters overflow the streaming encoder are redone by the unbounded staged kernels
static bool chain_f64_geometry(const micloc_xylo *c) {
    return c->n_g > 0 && c->n_g % 4 == 0 && c->nba >= 1 && c->nba <= 5 && c->CT <= 64 && c->p.M <= 32;
}
static bool chain_f64_supported(const micloc_xylo *c) { return chain_f64_geometry(c) && !getenv("MICLOC_XYLO_STAGED_F64"); }

template <typename IN_T>
static int launch_front_f64(micloc_xylo *c, const IN_T *a, long long nb, long long T, int8_t *sgn, int32_t *flg, cudaStream_t st) {
    const ChainParams &p = c->p;
    MICLOC_TRY(c->qd.reserve((size_t)nb * T * p.M * sizeof(double)));
    double *qd = (double *)c->qd.ptr;
    {
        const int ntiles = (int)((T + kSTile - 1) / kSTile);
        const int mgmax = p.M < kF64MG ? p.M : kF64MG;
        const size_t smem = ((size_t)c->n_g + (size_t)mgmax * ((f64_pad(kSTile + p.K - 1) + 9) & ~1)) * sizeof(double);
        if (smem > 227 * 1024) return set_error(MICLOC_ERR_UNSUPPORTED, "exact STHT tile needs %zu B of shared memory", smem);
        dim3 grid((unsigned)(nb * ntiles), (unsigned)((p.M + kF64MG - 1) / kF64MG));
        MICLOC_CUDA(cudaFuncSetAttribute(k_stht_f64_sparse<IN_T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_stht_f64_sparse<IN_T><<<grid, 256, smem, st>>>(a, c->d_g, qd, p.M, p.K, c->n_g, T, ntiles);
    }
    MICLOC_CUDA(cudaMemsetAsync(sgn, 0, (size_t)nb * T * c->CT, st));
    const size_t smem = (size_t)kChainWarps * kChainTile * p.M * (sizeof(double) + sizeof(float));
    const unsigned grid = (unsigned)((nb + kChainWarps - 1) / kChainWarps);
    if (c->nba <= 3) {
        MICLOC_CUDA(cudaFuncSetAttribute(k_xylo_chain_f64<IN_T, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_xylo_chain_f64<IN_T, 3><<<grid, 32 * kChainWarps, smem, st>>>(a, qd, c->d_ba_b, c->d_ba_a, sgn, flg, p.M, p.half, c->nba,
                                                                     c->F, p.w, p.bipolar, nb, T);
    } else {
        MICLOC_CUDA(cudaFuncSetAttribute(k_xylo_chain_f64<IN_T, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_xylo_chain_f64<IN_T, 5><<<grid, 32 * kChainWarps, smem, st>>>(a, qd, c->d_ba_b, c->d_ba_a, sgn, flg, p.M, p.half, c->nba,
                                                                     c->F, p.w, p.bipolar, nb, T);
    }
    count_launch(2);
    MICLOC_CUDA(cudaGetLastError());
    // overflowed clips (rare: more than kF64Cluster candidates in one cluster) take the unbounded kernels
    std::vector<int32_t> hf((size_t)nb);
    MICLOC_CUDA(cudaMemcpyAsync(hf.data(), flg, (size_t)nb * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MICLOC_CUDA(cudaStreamSynchronize(st));
    for (long long i = 0; i < nb; ++i)
        if (hf[(size_t)i] & 1) {
            MICLOC_TRY(exact_front_staged(c, a + (size_t)i * T * p.M, sizeof(IN_T) == 2 ? MICLOC_I16 : MICLOC_F32, 1, T,
                                          sgn + (size_t)i * T * c->CT, st));
            MICLOC_CUDA(cudaMemsetAsync(flg + i, 0, sizeof(int32_t), st));
            c->n_fallback++;
        }
    return MICLOC_OK;
}

extern "C" int micloc_xylo_run(micloc_xylo *c, const void *audio, int dtype, int64_t B, int64_t T, int exact,
                               int8_t *spikes_in_dev, uint8_t *raster_dev, int32_t *counts_dev,
                               int32_t *doa_dev, int32_t *doa_peak_dev, int32_t peak_win,
                               int32_t *flags_dev, void *stream) {
    MICLOC_TRY(check_xylo_args(c, audio, B, T));
    if (dtype != MICLOC_F32 && dtype != MICLOC_I16) return set_error(MICLOC_ERR_SHAPE, "dtype must be MICLOC_F32 or MICLOC_I16");
    if (exact && c->nba < 1) return set_error(MICLOC_ERR_CONFIG, "the exact front end needs the band filters in b/a form (n_ba)");
    MICLOC_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    const ChainParams &p = c->p;
    const int CT = c->CT;
    int32_t *counts = counts_dev;
    if (!counts) { MICLOC_TRY(c->counts.reserve((size_t)B * c->N * sizeof(int32_t))); counts = (int32_t *)c->counts.ptr; }
    int32_t *flg = flags_dev;
    if (!flg) { MICLOC_TRY(c->flags.reserve((size_t)B * sizeof(int32_t))); flg = (int32_t *)c->flags.ptr; }
    MICLOC_CUDA(cudaMemsetAsync(flg, 0, (size_t)B * sizeof(int32_t), st));
    // the batch goes through in chunks that bound the scratch (float64 intermediates of the exact front end)
    const bool staged_f64 = exact && !chain_f64_supported(c);       // float64 q AND z in HBM (else q only)
    const size_t per_clip = (size_t)T * (staged_f64 ? (size_t)p.M * 8 + (size_t)CT * 8 * 2 + (size_t)CT * 3 : (size_t)p.M * (exact ? 8 : 4) + CT);
    // a quarter of the free HBM, at most 24 GB (B200: 180 GB), at least 2 GB: the one-warp-per-clip chain kernel of the
    // exact front end wants >= 24 clips per SM in flight
    size_t mem_free = 0, mem_total = 0;
    size_t budget = (size_t)6 << 30;
    if (cudaMemGetInfo(&mem_free, &mem_total) == cudaSuccess) {
        budget = mem_free / 4;
        if (budget > ((size_t)24 << 30)) budget = (size_t)24 << 30;
        if (budget < ((size_t)2 << 30)) budget = (size_t)2 << 30;
    }
    long long chunk = (long long)(budget / per_clip);
    if (chunk < 1) chunk = 1;
    if (chunk > B) chunk = B;
    MICLOC_TRY(c->signed_spk.reserve((size_t)chunk * T * CT));
    bool fused_front = !exact && c->use_fused && !getenv("MICLOC_XYLO_STAGED_FRONT");
    const size_t esz = dtype == MICLOC_I16 ? 2 : 4;
    for (long long b0 = 0; b0 < B; b0 += chunk) {
        const long long nb = B - b0 < chunk ? B - b0 : chunk;
        const char *a = (const char *)audio + (size_t)b0 * T * p.M * esz;
        int8_t *sgn = (int8_t *)c->signed_spk.ptr;
        if (exact) {
            if (chain_f64_supported(c)) {
                if (dtype == MICLOC_I16) MICLOC_TRY(launch_front_f64(c, (const int16_t *)a, nb, T, sgn, flg + b0, st));
                else MICLOC_TRY(launch_front_f64(c, (const float *)a, nb, T, sgn, flg + b0, st));
            } else {
                MICLOC_TRY(exact_front_staged(c, a, dtype, nb, T, sgn, st));
            }
        } else {
            bool done = false;
            if (fused_front) {
                const int rcf = launch_fused(c->pf, c->d_taps, c->d_Wd1, a, dtype, nb, T, sgn, nullptr, nullptr, flg + b0,
                                             c->d_sm_slots, c->sm_count, st);
                if (rcf == MICLOC_OK) done = true;
                else if (rcf != MICLOC_ERR_UNSUPPORTED) return rcf;
                else fused_front = c->use_fused = false;   // e.g. a robust_width beyond the fused kernel's spike ring
            }
            if (!done) {
                MICLOC_TRY(c->q.reserve((size_t)chunk * T * p.M * sizeof(float)));
                MICLOC_TRY(launch_stht_any(p, c->d_taps, a, dtype, (float *)c->q.ptr, nb, T, st));
                MICLOC_TRY(launch_chain_any(p, sequential_chain(T), a, dtype, (const float *)c->q.ptr, c->d_band_sos, c->F,
                                            nullptr, sgn, flg + b0, nb, T, st));
            }
        }
        if (spikes_in_dev) {
            const long long rows = nb * T;
            k_xylo_split<<<(unsigned)((rows * CT + 255) / 256), 256, 0, st>>>(sgn, spikes_in_dev + (size_t)b0 * T * c->N_in, rows, CT, p.bipolar);
            count_launch(1);
        }
        MICLOC_TRY(launch_lif<true>(c, sgn, nb, T, raster_dev ? raster_dev + (size_t)b0 * T * c->N : nullptr,
                                    counts + (size_t)b0 * c->N, st));
    }
    MICLOC_TRY(launch_doa(c, counts, B, doa_dev, doa_peak_dev, peak_win, st));
    return MICLOC_OK;
}

extern "C" int micloc_xylo_process(micloc_xylo *c, const int8_t *spikes_in_dev, int64_t B, int64_t T,
                                   uint8_t *raster_dev, int32_t *counts_dev, int32_t *doa_dev,
                                   int32_t *doa_peak_dev, int32_t peak_win, void *stream) {
    MICLOC_TRY(check_xylo_args(c, spikes_in_dev, B, T));
    MICLOC_CUDA(cudaSetDevice(c->device));
    cudaStream_t st = (cudaStream_t)stream;
    int32_t *counts = counts_dev;
    if (!counts) { MICLOC_TRY(c->counts.reserve((size_t)B * c->N * sizeof(int32_t))); counts = (int32_t *)c->counts.ptr; }
    MICLOC_TRY(launch_lif<false>(c, spikes_in_dev, B, T, raster_dev, counts, st));
    MICLOC_TRY(launch_doa(c, counts, B, doa_dev, doa_peak_dev, peak_win, st));
    return MICLOC_OK;
}

// ---------------------------------------------------------------------------
// Xylo stream batches: S continuous recordings through the exact front end and the integer network, one push per
// frame tick (see include/micloc_b200.h).  Positions, slot lists, frame checks, the host mirror and the frame assembly
// are the SlotBook's (micloc_stream.cuh, as for the float batches); the chain, network state and flags are this
// batch's.  Per push: k_stream_assemble (float64 rows) -> k_stht_f64_sparse over the frame rows only ->
// k_xylo_chain_f64<STREAM> -> k_xylo_lif(_mma)<STATE> -> [k_xylo_doa] -> [k_xylo_split].
// ---------------------------------------------------------------------------
namespace micloc {
// fresh chain state, LIF state, ring, position and flags of the selected slots (sel == nullptr: all); one thread per
// (slot, j < max(CT, N, ring bytes / 16))
__global__ void __launch_bounds__(256)
k_xylo_streams_reset(XyloChanState *__restrict__ state, int2 *__restrict__ nstate, int8_t *__restrict__ ring,
                     SlotPos *__restrict__ pos, int32_t *__restrict__ flags, const int32_t *__restrict__ sel, long long S,
                     int CT, int N, int ring16, int W) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S * W) return;
    const long long s = i / W;
    const int j = (int)(i % W);
    if (sel && !sel[s]) return;
    if (j < CT) {
        XyloChanState &g = state[s * CT + j];
        for (int k = 0; k < 5; ++k) g.zs[k] = 0.0;
        g.cs = 0.0; g.rise = g.fall = -1;
        rzcc_reset(g.rz);
    }
    if (j < N) nstate[s * N + j] = make_int2(0, 0);
    if (j < ring16) reinterpret_cast<uint4 *>(ring)[s * ring16 + j] = make_uint4(0u, 0u, 0u, 0u);
    if (j == 0) { pos[s] = SlotPos{0, 0, 1, 0}; flags[s] = 0; }
}
}  // namespace micloc

struct micloc_xylo_streams {
    micloc_xylo *c = nullptr;
    int device = 0;
    SlotBook book;
    int hist = 0;                   // K - 1
    int ring_len = 0;
    int chain_warps = kChainWarps;  // slots per CTA of the chain kernel (fewer when float64 tiles of many microphones)
    double *xbuf[2] = {nullptr, nullptr}, *q = nullptr;
    XyloChanState *state = nullptr;
    int2 *nstate = nullptr;
    int8_t *ring = nullptr, *sgn = nullptr;
    int32_t *flags = nullptr, *counts = nullptr;
};

extern "C" int micloc_xylo_streams_destroy(micloc_xylo_streams *xs) {
    if (!xs) return MICLOC_OK;
    cudaSetDevice(xs->device);
    xs->book.destroy();
    cudaFree(xs->xbuf[0]); cudaFree(xs->xbuf[1]); cudaFree(xs->q); cudaFree(xs->state); cudaFree(xs->nstate);
    cudaFree(xs->ring); cudaFree(xs->sgn); cudaFree(xs->flags); cudaFree(xs->counts);
    delete xs;
    return MICLOC_OK;
}

static size_t xylo_stht_smem(const micloc_xylo *c) {
    const int mgmax = c->p.M < kF64MG ? c->p.M : kF64MG;
    return ((size_t)c->n_g + (size_t)mgmax * ((f64_pad(kSTile + c->p.K - 1) + 9) & ~1)) * sizeof(double);
}

extern "C" int micloc_xylo_streams_reset(micloc_xylo_streams *xs, const int32_t *slots_host, int32_t n_slots, void *stream) {
    if (!xs) return set_error(MICLOC_ERR_CONFIG, "null stream batch");
    MICLOC_CUDA(cudaSetDevice(xs->device));
    cudaStream_t st = (cudaStream_t)stream;
    SlotBook &bk = xs->book;
    if (slots_host) MICLOC_TRY(bk.upload(slots_host, n_slots, st));
    const micloc_xylo *c = xs->c;
    const int ring16 = (int)((long long)xs->ring_len * c->CT / 16);
    const int W = std::max(std::max(c->CT, c->N), ring16);
    k_xylo_streams_reset<<<(unsigned)((bk.S * W + 255) / 256), 256, 0, st>>>(
        xs->state, xs->nstate, xs->ring, bk.pos[bk.pcur], xs->flags, slots_host ? bk.sel : nullptr, bk.S, c->CT, c->N,
        ring16, W);
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    return bk.reset_done(slots_host != nullptr, st);
}

extern "C" int micloc_xylo_streams_create(micloc_xylo *c, int32_t num_streams, int64_t max_frame_len, micloc_xylo_streams **out) {
    if (!c || !out) return set_error(MICLOC_ERR_CONFIG, "null argument");
    *out = nullptr;
    if (c->nba < 1) return set_error(MICLOC_ERR_CONFIG, "the exact front end needs the band filters in b/a form (n_ba)");
    if (!chain_f64_geometry(c))
        return set_error(MICLOC_ERR_UNSUPPORTED,
                         "Xylo stream batches need the fast exact front end: a Hilbert kernel with every other tap zero "
                         "(K a multiple of 8), len(b) <= 5, 2 M F <= 64 and M <= 32 (got K %d, len(b) %d, M %d, F %d)",
                         c->p.K, c->nba, c->p.M, c->F);
    if (xylo_stht_smem(c) > 227 * 1024) return set_error(MICLOC_ERR_UNSUPPORTED, "exact STHT tile needs too much shared memory");
    MICLOC_CUDA(cudaSetDevice(c->device));
    micloc_xylo_streams *xs = new micloc_xylo_streams();
    xs->c = c; xs->device = c->device;
    xs->hist = c->p.K - 1;
    const int w = c->p.w;
    SlotBook &bk = xs->book;
    bk.D = (kF64Cluster - 1) * (w - 1) + w + kChainTile + kF64FlatTop / 2;
    int rc = bk.create(num_streams, max_frame_len);
    if (rc) { micloc_xylo_streams_destroy(xs); return rc; }
    xs->ring_len = 64;
    while (xs->ring_len < max_frame_len + bk.D) xs->ring_len <<= 1;
    const size_t per_warp = (size_t)kChainTile * c->p.M * 2 * sizeof(double);
    xs->chain_warps = (int)std::min<size_t>(kChainWarps, (size_t)(227 * 1024) / per_warp);
    const size_t S = (size_t)num_streams, M = (size_t)c->p.M, CT = (size_t)c->CT;
    const size_t rows = (size_t)xs->hist + max_frame_len;
    const size_t fin = (size_t)max_frame_len + bk.D;
    bool ok = cudaMalloc(&xs->xbuf[0], S * rows * M * sizeof(double)) == cudaSuccess &&
              cudaMalloc(&xs->xbuf[1], S * rows * M * sizeof(double)) == cudaSuccess &&
              cudaMalloc(&xs->q, S * rows * M * sizeof(double)) == cudaSuccess &&
              cudaMalloc(&xs->state, S * CT * sizeof(XyloChanState)) == cudaSuccess &&
              cudaMalloc(&xs->nstate, S * c->N * sizeof(int2)) == cudaSuccess &&
              cudaMalloc(&xs->ring, S * CT * (size_t)xs->ring_len) == cudaSuccess &&
              cudaMalloc(&xs->sgn, S * fin * CT) == cudaSuccess &&
              cudaMalloc(&xs->flags, S * sizeof(int32_t)) == cudaSuccess &&
              cudaMalloc(&xs->counts, S * c->N * sizeof(int32_t)) == cudaSuccess;
    if (!ok) { micloc_xylo_streams_destroy(xs); return set_error(MICLOC_ERR_CUDA, "cudaMalloc(Xylo stream batch) failed"); }
    rc = micloc_xylo_streams_reset(xs, nullptr, 0, nullptr);
    if (rc) { micloc_xylo_streams_destroy(xs); return rc; }
    *out = xs;
    return MICLOC_OK;
}

extern "C" int micloc_xylo_streams_latency(micloc_xylo_streams *xs) { return xs ? xs->book.D : 0; }

// shared by push and flush: chain of the new samples (n = 0: flush of the slots in close_sel), then the integer
// network, DoA and the {0,1} input spikes over each slot's final rows (row stride `rows`)
template <int NBA>
static void launch_chain_stream(micloc_xylo_streams *xs, const int32_t *close_sel, long long n, long long rows, cudaStream_t st) {
    const micloc_xylo *c = xs->c;
    const ChainParams &p = c->p;
    const SlotBook &bk = xs->book;
    XyloChainStream sa;
    sa.state = xs->state; sa.pos_in = bk.pos[bk.pcur]; sa.pos_out = bk.pos[bk.pcur ^ 1]; sa.m_out = bk.m;
    sa.close_sel = close_sel; sa.ring = xs->ring; sa.ring_len = xs->ring_len; sa.hist = xs->hist; sa.rows = (int)rows;
    sa.D = bk.D;
    const int nw = xs->chain_warps;
    const size_t smem = (size_t)nw * kChainTile * p.M * 2 * sizeof(double);
    cudaFuncSetAttribute(k_xylo_chain_f64<double, NBA, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    k_xylo_chain_f64<double, NBA, true><<<(unsigned)((bk.S + nw - 1) / nw), 32 * nw, smem, st>>>(
        xs->xbuf[bk.xcur], xs->q, c->d_ba_b, c->d_ba_a, xs->sgn, xs->flags, p.M, p.half, c->nba, c->F, p.w, p.bipolar, bk.S,
        n, sa);
}

// the chain's positions are flipped by the caller (SlotBook::pushed / flushed)
static int xylo_streams_advance(micloc_xylo_streams *xs, const int32_t *close_sel, long long n, long long rows,
                                int8_t *spikes_in_dev, uint8_t *raster_dev, int32_t *counts_dev, int32_t *doa_dev,
                                int32_t *doa_peak_dev, int32_t peak_win, int32_t *flags_dev, cudaStream_t st) {
    micloc_xylo *c = xs->c;
    const SlotBook &bk = xs->book;
    if (c->nba <= 3) launch_chain_stream<3>(xs, close_sel, n, rows, st);
    else launch_chain_stream<5>(xs, close_sel, n, rows, st);
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    int32_t *counts = counts_dev ? counts_dev : xs->counts;
    MICLOC_TRY((launch_lif<true, true>(c, xs->sgn, bk.S, rows, raster_dev, counts, st, bk.m, xs->nstate)));
    MICLOC_TRY(launch_doa(c, counts, bk.S, doa_dev, doa_peak_dev, peak_win, st, bk.m));
    if (spikes_in_dev) {
        const long long r = bk.S * rows;
        k_xylo_split<<<(unsigned)((r * c->CT + 255) / 256), 256, 0, st>>>(xs->sgn, spikes_in_dev, r, c->CT, c->p.bipolar, bk.m, rows);
        count_launch(1);
        MICLOC_CUDA(cudaGetLastError());
    }
    if (flags_dev) MICLOC_CUDA(cudaMemcpyAsync(flags_dev, xs->flags, (size_t)bk.S * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    return MICLOC_OK;
}

extern "C" int micloc_xylo_streams_push(micloc_xylo_streams *xs, const void *frames_dev, int dtype, int64_t n, int32_t in_channels,
                                        int8_t *spikes_in_dev, uint8_t *raster_dev, int32_t *counts_dev, int32_t *doa_dev,
                                        int32_t *doa_peak_dev, int32_t peak_win, int32_t *flags_dev, int64_t *n_out_host,
                                        void *stream) {
    if (!xs || !n_out_host) return set_error(MICLOC_ERR_SHAPE, "null argument");
    if (!frames_dev) return set_error(MICLOC_ERR_SHAPE, "null frame pointer");
    micloc_xylo *c = xs->c;
    const ChainParams &p = c->p;
    SlotBook &bk = xs->book;
    MICLOC_TRY(bk.check_push(dtype, n, in_channels, p.M));
    MICLOC_TRY(check_peak_win(c, doa_peak_dev, peak_win));
    MICLOC_CUDA(cudaSetDevice(xs->device));
    cudaStream_t st = (cudaStream_t)stream;
    // [K-1 history rows | frame] in float64
    MICLOC_TRY(bk.assemble(xs->xbuf, frames_dev, dtype, n, in_channels, p.M, xs->hist, st));
    // STHT of the frame rows only (the history rows were the previous push's frame rows)
    {
        const long long rows_in = xs->hist + n;
        const int ntiles = (int)((n + kSTile - 1) / kSTile);
        const size_t smem = xylo_stht_smem(c);
        dim3 grid((unsigned)(bk.S * ntiles), (unsigned)((p.M + kF64MG - 1) / kF64MG));
        MICLOC_CUDA(cudaFuncSetAttribute(k_stht_f64_sparse<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_stht_f64_sparse<double><<<grid, 256, smem, st>>>(xs->xbuf[bk.xcur], c->d_g, xs->q, p.M, p.K, c->n_g, rows_in, ntiles,
                                                          (long long)xs->hist);
        count_launch(1);
        MICLOC_CUDA(cudaGetLastError());
    }
    MICLOC_TRY(xylo_streams_advance(xs, nullptr, n, n + bk.D, spikes_in_dev, raster_dev, counts_dev, doa_dev, doa_peak_dev,
                                    peak_win, flags_dev, st));
    bk.pushed(n, n_out_host);
    return MICLOC_OK;
}

extern "C" int micloc_xylo_streams_flush(micloc_xylo_streams *xs, const int32_t *slots_host, int32_t n_slots,
                                         int8_t *spikes_in_dev, uint8_t *raster_dev, int32_t *counts_dev, int32_t *doa_dev,
                                         int32_t *doa_peak_dev, int32_t peak_win, int32_t *flags_dev, int64_t *n_out_host,
                                         int32_t *flags_host, void *stream) {
    if (!xs || !n_out_host) return set_error(MICLOC_ERR_CONFIG, "null stream batch");
    MICLOC_TRY(check_peak_win(xs->c, doa_peak_dev, peak_win));
    MICLOC_CUDA(cudaSetDevice(xs->device));
    cudaStream_t st = (cudaStream_t)stream;
    SlotBook &bk = xs->book;
    MICLOC_TRY(bk.upload(slots_host, n_slots, st));
    MICLOC_TRY(xylo_streams_advance(xs, bk.sel, 0, bk.max_frame + bk.D, spikes_in_dev, raster_dev, counts_dev, doa_dev,
                                    doa_peak_dev, peak_win, flags_dev, st));
    bk.flushed(n_out_host);
    if (flags_host) {
        MICLOC_CUDA(cudaMemcpyAsync(flags_host, xs->flags, (size_t)bk.S * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        MICLOC_CUDA(cudaStreamSynchronize(st));
    }
    return MICLOC_OK;
}
