// micloc_stream.cu -- stateful frames of the float SNN chain (SURVEY.md 8f rank 3) + the Envelope tracker.
//
// Reference sites:
//   live frame loop             micloc/localization_demo_snn.py:125-193 (one recording = one frame; int32 `T x 8` wav
//                               frames, last channel dropped: micloc/record.py:54-75, localization_demo_snn.py:145)
//   chain                       micloc/snn_beamformer.py:283-370
//   Envelope                    micloc/utils.py:15-81; per-sample argmax tests/test_snn_hilbert_localization.py:284-293
//
// The reference restarts every filter from zero state at each frame.  A stream keeps the state instead, so that N
// pushed frames give exactly what ONE clip of their concatenation gives: the K-1 newest audio frames (STHT history and
// the K/2 in-phase delay), the band-pass biquad state, the running sum and the open candidate clusters of the RZCC
// encoder, the neuron recurrences and the envelope state all carry over.  Differences to a one-shot clip, by nature of
// a stream: the in-phase branch is the CAUSAL delay x[t - K/2] (zeros before the stream starts; np.roll's wrap-around
// needs the clip's end), and results lag the input by D = rzcc_lag(robust_width) samples -- a spike at p is only final
// once the distance rule has seen D more samples.  A push returns the n_out samples that became final; a flush closes
// the stream like a clip end and returns the rest.
//
// A STREAM BATCH carries S such recordings ("slots") at once; the single stream (micloc_snn_stream_*) is a batch of
// one.  Slots are independent (own position, reset and flush), but a push hands every slot one frame of the same
// length n, so that one launch per stage serves all of them.  A batch is a SlotBook (micloc_stream.cuh: positions,
// slot lists, frame checks, host mirror) plus one StreamBand (the chain's device state).  Per push, whatever S:
//   k_stream_assemble        [K-1 history rows | frame] of every slot (from the previous push's buffer: ping-pong)
//   STHT                     launch_stht_any over S clips of K-1+n rows
//   k_stream_blk             band-pass + RZCC of the new samples, then the neuron filter of the final ones
//   k_gram, k_power_argmax   power / DoA over each slot's final rows            (when power or doa is requested)
//   k_dense, k_envelope, k_argmax_rows                                      (when env or doa_t is requested)
//
// A MULTI-BAND STREAM BATCH (micloc_snn_mb_streams_*) is the live localiser of micloc/localization_demo_snn.py:125-193
// made continuous: a Butterworth filterbank on the raw frame, one chain per band, power summed over the bands.  It is
// one SlotBook plus F StreamBands; the book's latency D = max_f rzcc_lag(w_f) is common, so every band finalises the
// same samples in a push and every band's k_stream_blk writes the same positions and row counts.  One kernel runs the
// filterbank with its state carried across pushes and writes every band's [history | frame] rows
// (k_mb_stream_assemble).  Per push, whatever S:
//   k_mb_stream_assemble                                                    1
//   per band: STHT, k_stream_blk, k_gram, k_power_argmax (into band f's slice of [F][S][G])   4 F
//   k_power_fuse       sum over bands, argmax, periodic-ML estimators over each slot's final rows   1
#include <cuda_runtime.h>

#include <algorithm>
#include <vector>

#include "micloc_common.h"
#include "micloc_staged.cuh"
#include "micloc_stream.cuh"

namespace micloc {

struct ChanState {            // one per (slot, real channel): in-phase | quadrature
    BiquadState bq;
    RzccState rz;
    int cl_pos[2 * kClusterMax];
    float cl_h[2 * kClusterMax];
    NeuronState nr;
};

// SlotPos and k_stream_assemble (the [K-1 history rows | frame] buffer of every slot): micloc_stream.cuh

// Multi-band frame assembly: one thread per (slot, microphone) steps the F band-pass cascades of the filterbank
// (biquad_step with the float32 sections of k_filterbank, so band f's rows are micloc_filterbank's bits for the whole
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
                for (int f = 0; f < NF; ++f) row[f][(long long)t * M] = biquad_step(ap.fb.sos[f], ap.fb.nsec, st[f], x[u]);
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

// Band-pass + RZCC of the new samples [N, N + n) of every slot, then the neuron filter of the samples that became
// final, one thread per (slot, channel) with its state in global memory.  The chain is k_chain_blk's (32-sample blocks:
// branch-free band-pass and running sum, sign / flat-top masks, rzcc_segment_masks, the next block's inputs loaded
// meanwhile) with the blocks aligned to ABSOLUTE time: the head and tail of a frame that are no whole aligned block go
// through the same masks with nvalid < 32, and the clusters are closed exactly where the one-clip chain closes them
// (after every sample t with t % 32 == 31, and at the end), so the spikes are the one-shot clip's bits.  Spikes go to
// the thread's ring row (int8 [S][C2][R], R a power of two >= n + D + L + 64) at their absolute position; the neuron
// then reads the row at t and t - L.  Outputs: spikes / membrane rows [S][rows][C2], row i = sample F + i.
// close_sel != nullptr: flush -- no new samples, the selected slots close their clusters like a clip end, return the
// rest and stop.  pos_out / m_out: each slot's new position and its number of final rows (read by the later stages).
// Register budget and CTA size: the chains are latency-bound (one dependent recurrence per thread), so what counts is
// threads in flight.  152 registers (no spills) leave 13 warps per SM; one-warp CTAs use all 13 (larger CTAs round
// down), i.e. 61 568 threads on 148 SMs: 4096 slots of 7 microphones (57 344 chains) run in ONE wave.
constexpr int kStreamBlkThreads = 32;
template <int NSEC>          // biquads of the band-pass (0 = p.nsec at run time)
__global__ void __maxnreg__(152)
k_stream_blk(const float *__restrict__ xbuf, const float *__restrict__ q, ChanState *__restrict__ state,
             const SlotPos *__restrict__ pos_in, SlotPos *__restrict__ pos_out, int32_t *__restrict__ m_out,
             const int32_t *__restrict__ close_sel, int8_t *__restrict__ ring, int ring_len, int32_t *__restrict__ flags,
             int8_t *__restrict__ spikes_out, float *__restrict__ vmem, const __grid_constant__ ChainParams p,
             long long S, int n, int hist, int rows, int D) {
    __shared__ float cs_s[kSeg * kStreamBlkThreads];
    const int C2 = p.C2, M = p.M;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool in = idx < S * C2;                    // (no early return: keep the warp whole)
    const long long idc = in ? idx : 0;
    const int c = (int)(idc % C2);
    const long long s = idc / C2;
    const SlotPos ps = pos_in[s];
    const bool flush = close_sel != nullptr;
    const bool run = in && ps.active && (!flush || close_sel[s] != 0);
    const int N0 = ps.N, F0 = ps.F;
    const int t_end = run ? N0 + n : N0;
    const int F1 = !run ? F0 : (flush ? N0 : max(t_end - D, F0));
    if (in && c == 0) {
        pos_out[s] = SlotPos{t_end, F1, (run && flush) ? 0 : ps.active, 0};
        m_out[s] = F1 - F0;
    }
    constexpr int NS = NSEC ? NSEC : kMaxSections;
    const int nsec = NSEC ? NSEC : p.nsec;
    float sos[kMaxSections][5];
#pragma unroll
    for (int k = 0; k < kMaxSections; ++k)
#pragma unroll
        for (int e = 0; e < 5; ++e) sos[k][e] = p.sos[k][e];

    ChanState &st = state[idc];
    BiquadState bq = st.bq;
    RzccState rz = st.rz;
    NeuronState nr = st.nr;
    int cl_pos[2 * kClusterMax]; float cl_h[2 * kClusterMax];
#pragma unroll
    for (int i = 0; i < 2 * kClusterMax; ++i) { cl_pos[i] = st.cl_pos[i]; cl_h[i] = st.cl_h[i]; }
    const RzccStore store{cl_pos, cl_h, 1};
    int8_t *rr = ring + idc * (long long)ring_len;
    const int rmask = ring_len - 1;
    auto emit = [&](int pos, int sign) { rr[pos & rmask] = (int8_t)sign; };

    // in-phase: x[t - K/2] = row hist + i - K/2 of the slot's buffer; quadrature: q of row hist + i  (i = t - N0)
    const bool inphase = c < M;
    const long long base = s * ((long long)hist + n) * M;
    const float *src = inphase ? xbuf + base + (long long)(hist - p.half) * M + c : q + base + (long long)hist * M + (c - M);
    float x[kSeg];
    auto load_block = [&](int t0, int nv) {
        const float *pp = src + (long long)(t0 - N0) * M;
        if (nv == kSeg) {
#pragma unroll
            for (int i = 0; i < kSeg; ++i) { x[i] = *pp; pp += M; }
        } else {
#pragma unroll
            for (int i = 0; i < kSeg; ++i) x[i] = i < nv ? pp[(long long)i * M] : 0.f;
        }
    };
    float *cs = cs_s + threadIdx.x;
    int t = N0;
    if (t < t_end) load_block(t, min(kSeg - (t & (kSeg - 1)), t_end - t));
    while (t < t_end) {
        const int nvalid = min(kSeg - (t & (kSeg - 1)), t_end - t);
        // the ring bytes of this block: only spikes are stored
        if (nvalid == kSeg) {
            uint4 *r4 = reinterpret_cast<uint4 *>(rr + (t & rmask));
            r4[0] = make_uint4(0u, 0u, 0u, 0u);
            r4[1] = make_uint4(0u, 0u, 0u, 0u);
        } else {
            for (int i = 0; i < nvalid; ++i) rr[(t + i) & rmask] = 0;
        }
        // ---- band-pass + running sum of the block, branch-free ----
        const float carry = rz.csum;
        float csum = carry;
        unsigned neg = 0u, zero = 0u;
#pragma unroll
        for (int i = 0; i < kSeg; ++i) {
            if (i < nvalid) {
                float v = x[i];
#pragma unroll
                for (int k = 0; k < NS; ++k) {
                    if (k < nsec) {
                        const float y = fmaf(sos[k][0], v, bq.s1[k]);
                        bq.s1[k] = fmaf(sos[k][1], v, fmaf(-sos[k][3], y, bq.s2[k]));
                        bq.s2[k] = fmaf(sos[k][2], v, -sos[k][4] * y);
                        v = y;
                    }
                }
                const float cprev = csum;
                csum = cprev + v;
                neg |= (__float_as_uint(v) & 0x80000000u) >> i;
                zero |= rzcc_flat(v, cprev) ? (0x80000000u >> i) : 0u;
                cs[i * kStreamBlkThreads] = csum;
            }
        }
        const int tn = t + nvalid;
        // ---- the next block's inputs on their way while the candidates of this one are handled ----
        if (tn < t_end) load_block(tn, min(kSeg, t_end - tn));
        rzcc_segment_masks(rz, store, p.bipolar, p.w, t, nvalid, neg, zero, cs, kStreamBlkThreads, carry, emit);
        rz.csum = csum;
        if ((tn & (kSeg - 1)) == 0) rzcc_close(rz, store, p.w, tn - 1, false, emit);
        t = tn;
    }
    if (run && flush && N0 > 0) rzcc_close(rz, store, p.w, N0 - 1, true, emit);

    // ---- neuron filter of the final samples [F0, F1); the spike bytes of the next kNeuBlk steps are requested
    //      before the current ones are computed (k_neuron_seg) ----
    constexpr int kNeuBlk = 16;
    const int nL = p.nL;
    int nx_s[kNeuBlk], nx_d[kNeuBlk];
    auto request = [&](int t0) {
#pragma unroll
        for (int u = 0; u < kNeuBlk; ++u) {
            nx_s[u] = rr[(t0 + u) & rmask];
            nx_d[u] = rr[(t0 + u - nL) & rmask];
        }
    };
    int8_t *so = spikes_out ? spikes_out + s * (long long)rows * C2 + c : nullptr;
    float *vo = vmem + s * (long long)rows * C2 + c;
    if (F0 < F1) request(F0);
    for (int t0 = F0; t0 < F1; t0 += kNeuBlk) {
        int cur_s[kNeuBlk]; float cur_d[kNeuBlk];
#pragma unroll
        for (int u = 0; u < kNeuBlk; ++u) { cur_s[u] = nx_s[u]; cur_d[u] = t0 + u >= nL ? (float)nx_d[u] : 0.f; }
        if (t0 + kNeuBlk < F1) request(t0 + kNeuBlk);
#pragma unroll
        for (int u = 0; u < kNeuBlk; ++u) {
            if (t0 + u < F1) {
                const long long i = t0 + u - F0;
                if (so) so[i * C2] = (int8_t)cur_s[u];
                vo[i * C2] = neuron_step(p, nr, (float)cur_s[u], cur_d[u]);
            }
        }
    }
    if (run) {
        st.bq = bq;
        st.rz = rz;
        st.nr = nr;
#pragma unroll
        for (int i = 0; i < 2 * kClusterMax; ++i) { st.cl_pos[i] = cl_pos[i]; st.cl_h[i] = cl_h[i]; }
        if (rz.overflow) atomicOr(flags + s, 1);
    }
}

// fresh state for the selected slots (sel == nullptr: all): one thread per (slot, j < max(C2, G)); pos == nullptr:
// the positions are left alone (the bands of a multi-band batch share them: one band's reset writes them)
__global__ void __launch_bounds__(256)
k_stream_reset(ChanState *__restrict__ state, SlotPos *__restrict__ pos, int32_t *__restrict__ flags,
               float *__restrict__ env_state, int32_t *__restrict__ env_started, const int32_t *__restrict__ sel,
               long long S, int C2, int G) {
    const int W = C2 > G ? C2 : G;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S * W) return;
    const long long s = i / W;
    const int j = (int)(i % W);
    if (sel && !sel[s]) return;
    if (j < C2) {
        ChanState &c = state[s * C2 + j];
        biquad_reset(c.bq);
        rzcc_reset(c.rz);
        neuron_reset(c.nr);
        for (int k = 0; k < 2 * kClusterMax; ++k) { c.cl_pos[k] = 0; c.cl_h[k] = 0.f; }
    }
    if (j < G) { env_state[s * G + j] = 0.f; env_started[s * G + j] = 0; }
    if (j == 0) {
        if (pos) pos[s] = SlotPos{0, 0, 1, 0};
        flags[s] = 0;
    }
}

}  // namespace micloc

// Envelope.evolve (micloc/utils.py:49-81) over rows of |x|, one thread per (clip, channel), state carried between
// calls:  first row ever: state = |x[0]|, out[0] = state;  afterwards  rise = |x| >= state,  win = rise ?
// int(fs rise_time) : int(fs fall_time),  state = (1 - 1/win) state + (1/win) |x| rise,  out = state.
// x, env [B][T][C]; state, started [B][C]; rows_b (nullable): clip b takes its first rows_b[b] rows (T = row stride).
namespace micloc {
__global__ void __launch_bounds__(128)
k_envelope(const float *__restrict__ x, float *__restrict__ env, float *__restrict__ state, int32_t *__restrict__ started,
           const int32_t *__restrict__ rows_b, long long B, long long T, int C, float inv_fall, float inv_rise) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * C) return;
    const long long b = i / C;
    const int c = (int)(i % C);
    const long long Tn = rows_b ? rows_b[b] : T;
    const float *xb = x + b * T * C;
    float *eb = env + b * T * C;
    float s = state[i];
    long long t = 0;
    if (!started[i] && Tn > 0) { s = fabsf(xb[c]); eb[c] = s; t = 1; started[i] = 1; }
    for (; t < Tn; ++t) {
        const float a = fabsf(xb[t * C + c]);
        const bool rise = a >= s;
        const float iw = rise ? inv_rise : inv_fall;
        s = (1.f - iw) * s + (rise ? iw * a : 0.f);
        eb[t * C + c] = s;
    }
    state[i] = s;
}

// first argmax over the C channels of every row (np.argmax(env, axis=1)); one warp per row of env [B][T][C]
// (rows_b as in k_envelope: rows past a clip's count are not written)
__global__ void __launch_bounds__(256)
k_argmax_rows(const float *__restrict__ env, int32_t *__restrict__ idx, const int32_t *__restrict__ rows_b, long long B,
              long long T, int C) {
    const long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= B * T) return;
    if (rows_b && r % T >= rows_b[r / T]) return;
    float best = -1.f; int bi = 0x7fffffff;
    for (int c = lane; c < C; c += 32) {
        const float v = env[r * C + c];
        if (v > best) { best = v; bi = c; }
    }
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
    }
    if (lane == 0) idx[r] = bi;
}
}  // namespace micloc

using namespace micloc;

// one band's chain over the slots of a SlotBook: its [history | frame] buffers, STHT output, chain state, spike ring,
// membrane, flags, Gram and envelope
struct StreamBand {
    micloc_snn_params prm{};        // copy of what the kernels need from the band's context
    int hist = 0;                   // K - 1
    int ring_len = 0;
    float *xbuf[2] = {nullptr, nullptr}, *q = nullptr, *vmem = nullptr, *env_state = nullptr;
    int8_t *ring = nullptr;
    ChanState *state = nullptr;
    int32_t *flags = nullptr, *env_started = nullptr;
    double *gram = nullptr;
    DevBuf y, env;                  // envelope scratch: allocated on the first request, grow-only
    float rise_time = 10e-3f, fall_time = 100e-3f, fs = 48000.f;
};

struct micloc_stream_batch {
    int device = 0;
    SlotBook book;
    StreamBand band;
};

// the single stream: a batch of one slot
struct micloc_stream {
    micloc_stream_batch *sb = nullptr;
};

static void band_free(StreamBand &b) {
    cudaFree(b.xbuf[0]); cudaFree(b.xbuf[1]); cudaFree(b.q); cudaFree(b.vmem); cudaFree(b.env_state);
    cudaFree(b.ring); cudaFree(b.state); cudaFree(b.flags); cudaFree(b.env_started); cudaFree(b.gram);
    b.y.release(); b.env.release();
}

// the band's buffers for the book's slots, frame length and latency
static int band_alloc(StreamBand &b, const micloc_snn_params &prm, const SlotBook &bk) {
    b.prm = prm;
    const ChainParams &p = prm.chain;
    b.hist = p.K - 1;
    const long long need = bk.max_frame + bk.D + p.nL + 2 * kSeg;
    b.ring_len = 32;
    while (b.ring_len < need) b.ring_len <<= 1;
    const size_t S = (size_t)bk.S;
    const size_t rows = (size_t)b.hist + bk.max_frame;
    const size_t fin = (size_t)bk.max_frame + bk.D;                // most samples one call can finalise
    bool ok = cudaMalloc(&b.xbuf[0], S * rows * p.M * sizeof(float)) == cudaSuccess &&
              cudaMalloc(&b.xbuf[1], S * rows * p.M * sizeof(float)) == cudaSuccess &&
              cudaMalloc(&b.q, S * rows * p.M * sizeof(float)) == cudaSuccess &&
              cudaMalloc(&b.vmem, S * fin * p.C2 * sizeof(float)) == cudaSuccess &&
              cudaMalloc(&b.env_state, S * p.G * sizeof(float)) == cudaSuccess &&
              cudaMalloc(&b.env_started, S * p.G * sizeof(int32_t)) == cudaSuccess &&
              cudaMalloc(&b.ring, S * p.C2 * (size_t)b.ring_len) == cudaSuccess &&
              cudaMalloc(&b.state, S * p.C2 * sizeof(ChanState)) == cudaSuccess &&
              cudaMalloc(&b.flags, S * sizeof(int32_t)) == cudaSuccess &&
              cudaMalloc(&b.gram, S * p.C2 * p.C2 * sizeof(double)) == cudaSuccess;
    return ok ? MICLOC_OK : set_error(MICLOC_ERR_CUDA, "cudaMalloc(stream batch) failed");
}

// fresh state for the listed slots (slots_host NULL: every slot) of every band; band 0's launch writes the positions.
// Synchronises `st`.
static int reset_bands(SlotBook &bk, StreamBand *band, int F, const int32_t *slots_host, int32_t n_slots, cudaStream_t st) {
    if (slots_host) MICLOC_TRY(bk.upload(slots_host, n_slots, st));
    for (int f = 0; f < F; ++f) {
        StreamBand &b = band[f];
        const ChainParams &p = b.prm.chain;
        const long long W = p.C2 > p.G ? p.C2 : p.G;
        k_stream_reset<<<(unsigned)((bk.S * W + 255) / 256), 256, 0, st>>>(b.state, f == 0 ? bk.pos[bk.pcur] : nullptr, b.flags,
                                                                          b.env_state, b.env_started,
                                                                          slots_host ? bk.sel : nullptr, bk.S, p.C2, p.G);
        count_launch(1);
        MICLOC_CUDA(cudaGetLastError());
    }
    return bk.reset_done(slots_host != nullptr, st);
}

// envelope scratch for outputs of `rows` rows, taken before a push or flush launches anything: a failed allocation
// leaves every slot where it stood
static int reserve_env(StreamBand &b, long long S, long long rows, const float *env_dev, const int32_t *doa_t_dev) {
    if (!env_dev && !doa_t_dev) return MICLOC_OK;
    const size_t bytes = (size_t)S * rows * b.prm.chain.G * sizeof(float);
    MICLOC_TRY(b.y.reserve(bytes));
    return env_dev ? MICLOC_OK : b.env.reserve(bytes);
}

// One band's part of a push of n samples (close_sel == nullptr: STHT of the newest [history | frame] buffer first) or
// of a flush of the slots in close_sel (n = 0): band-pass + RZCC + neuron (k_stream_blk reads the book's positions and
// writes the next ones and the final row counts m), then power / DoA and envelope over each slot's final rows; outputs
// [S][rows][...].  The owner flips the book once every band has run.
static int band_step(StreamBand &b, const SlotBook &bk, const int32_t *close_sel, long long n, long long rows,
                     int8_t *spikes_dev, float *power_dev, int32_t *doa_dev, float *env_dev, int32_t *doa_t_dev,
                     cudaStream_t st) {
    const ChainParams &p = b.prm.chain;
    const long long S = bk.S;
    // STHT of the extended clips [history | frame]: rows >= hist see their whole window
    if (!close_sel)
        MICLOC_TRY(launch_stht_any(p, (const float *)b.prm.taps_dev, b.xbuf[bk.xcur], MICLOC_F32, b.q, S, b.hist + n, st));
    const unsigned grid = (unsigned)((S * p.C2 + kStreamBlkThreads - 1) / kStreamBlkThreads);
    auto kernel = p.nsec == 2 ? k_stream_blk<2> : k_stream_blk<0>;
    kernel<<<grid, kStreamBlkThreads, 0, st>>>(b.xbuf[bk.xcur], b.q, b.state, bk.pos[bk.pcur], bk.pos[bk.pcur ^ 1], bk.m,
                                              close_sel, b.ring, b.ring_len, b.flags, spikes_dev, b.vmem, p, S, (int)n,
                                              b.hist, (int)rows, bk.D);
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    if (power_dev || doa_dev) {
        dim3 gg((unsigned)S, (unsigned)((p.C2 * p.C2 + 255) / 256));
        k_gram<<<gg, 256, 0, st>>>(b.vmem, b.gram, p.C2, rows, 0, bk.m);
        count_launch(1);
        MICLOC_TRY(launch_power(b.gram, (const double *)b.prm.bf_f64_dev, power_dev, doa_dev, p.C2, p.G, S, 1.0, bk.m, 1,
                                nullptr, nullptr, st));
    }
    if (env_dev || doa_t_dev) {                         // scratch: reserve_env
        float *y = (float *)b.y.ptr;
        float *env = env_dev ? env_dev : (float *)b.env.ptr;
        const int slab = 256;
        dim3 grid((unsigned)((p.G + 127) / 128), (unsigned)((rows + slab - 1) / slab), (unsigned)S);
        if (p.C2 <= 16) k_dense<16><<<grid, 128, 0, st>>>(b.vmem, (const float *)b.prm.bf_f32_dev, y, p.C2, p.G, rows, slab);
        else k_dense<0><<<grid, 128, 0, st>>>(b.vmem, (const float *)b.prm.bf_f32_dev, y, p.C2, p.G, rows, slab);
        k_envelope<<<(unsigned)((S * p.G + 127) / 128), 128, 0, st>>>(y, env, b.env_state, b.env_started, bk.m, S, rows, p.G,
                                                                      1.f / (float)(int)(b.fs * b.fall_time),
                                                                      1.f / (float)(int)(b.fs * b.rise_time));
        count_launch(2);
        if (doa_t_dev) {
            k_argmax_rows<<<(unsigned)((S * rows * 32 + 255) / 256), 256, 0, st>>>(env, doa_t_dev, bk.m, S, rows, p.G);
            count_launch(1);
        }
    }
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}

// a push (close_sel == nullptr) or flush of every band, then the slots' new positions; band f's spikes and power go to
// spikes_dev + f S rows 2M and power_dev + f S G
static int step_bands(SlotBook &bk, StreamBand *band, int F, const int32_t *close_sel, long long n, long long rows,
                      int8_t *spikes_dev, float *power_dev, int32_t *doa_dev, float *env_dev, int32_t *doa_t_dev,
                      int64_t *n_out_host, cudaStream_t st) {
    for (int f = 0; f < F; ++f) {
        const ChainParams &p = band[f].prm.chain;
        MICLOC_TRY(band_step(band[f], bk, close_sel, n, rows, spikes_dev ? spikes_dev + f * bk.S * rows * p.C2 : nullptr,
                             power_dev ? power_dev + f * bk.S * p.G : nullptr, doa_dev, env_dev, doa_t_dev, st));
    }
    if (close_sel) bk.flushed(n_out_host);
    else bk.pushed(n, n_out_host);
    return MICLOC_OK;
}

// the listed slots (slots_host NULL: every slot) of every band close like a clip end; flags_host [S] (nullable, host):
// bit 0 = RZCC overflow in any band (the only bit k_stream_blk sets).  Synchronises `st`.
static int flush_bands(SlotBook &bk, StreamBand *band, int F, const int32_t *slots_host, int32_t n_slots,
                       int8_t *spikes_dev, float *power_dev, int32_t *doa_dev, float *env_dev, int32_t *doa_t_dev,
                       int64_t *n_out_host, int32_t *flags_host, cudaStream_t st) {
    MICLOC_TRY(bk.upload(slots_host, n_slots, st));
    MICLOC_TRY(step_bands(bk, band, F, bk.sel, 0, bk.max_frame + bk.D, spikes_dev, power_dev, doa_dev, env_dev, doa_t_dev,
                          n_out_host, st));
    if (!flags_host) return MICLOC_OK;
    const size_t S = (size_t)bk.S;
    std::vector<int32_t> h((size_t)F * S);
    for (int f = 0; f < F; ++f)
        MICLOC_CUDA(cudaMemcpyAsync(h.data() + f * S, band[f].flags, S * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MICLOC_CUDA(cudaStreamSynchronize(st));
    for (size_t s = 0; s < S; ++s) {
        flags_host[s] = 0;
        for (int f = 0; f < F; ++f) flags_host[s] |= h[f * S + s] & 1;
    }
    return MICLOC_OK;
}

extern "C" int micloc_snn_streams_destroy(micloc_stream_batch *sb) {
    if (!sb) return MICLOC_OK;
    cudaSetDevice(sb->device);
    sb->book.destroy();
    band_free(sb->band);
    delete sb;
    return MICLOC_OK;
}

extern "C" int micloc_snn_streams_reset(micloc_stream_batch *sb, const int32_t *slots_host, int32_t n_slots, void *stream) {
    if (!sb) return set_error(MICLOC_ERR_CONFIG, "null stream");
    MICLOC_CUDA(cudaSetDevice(sb->device));
    return reset_bands(sb->book, &sb->band, 1, slots_host, n_slots, (cudaStream_t)stream);
}

extern "C" int micloc_snn_streams_create(micloc_snn *ctx, int32_t num_streams, int64_t max_frame_len, double fs,
                                         double rise_time, double fall_time, micloc_stream_batch **out) {
    if (!ctx || !out) return set_error(MICLOC_ERR_CONFIG, "null argument");
    *out = nullptr;
    if (rise_time > fall_time)
        return set_error(MICLOC_ERR_CONFIG, "for proper functioning, an envelope estimator should have a larger fall time!");
    if ((int)(fs * rise_time) < 1 || (int)(fs * fall_time) < 1) return set_error(MICLOC_ERR_CONFIG, "envelope windows shorter than one sample");
    micloc_snn_params prm;
    MICLOC_TRY(micloc_snn_get_params(ctx, &prm));
    MICLOC_CUDA(cudaSetDevice(prm.device));
    micloc_stream_batch *sb = new micloc_stream_batch();
    sb->device = prm.device;
    sb->band.fs = (float)fs; sb->band.rise_time = (float)rise_time; sb->band.fall_time = (float)fall_time;
    sb->book.D = rzcc_lag(prm.chain.w);
    int rc = sb->book.create(num_streams, max_frame_len);
    if (!rc) rc = band_alloc(sb->band, prm, sb->book);
    if (!rc) rc = reset_bands(sb->book, &sb->band, 1, nullptr, 0, nullptr);
    if (rc) { micloc_snn_streams_destroy(sb); return rc; }
    *out = sb;
    return MICLOC_OK;
}

extern "C" int micloc_snn_streams_latency(micloc_stream_batch *sb) { return sb ? sb->book.D : 0; }

extern "C" int micloc_snn_streams_push(micloc_stream_batch *sb, const void *frames_dev, int dtype, int64_t n,
                                       int32_t in_channels, int8_t *spikes_dev, float *power_dev, int32_t *doa_dev,
                                       float *env_dev, int32_t *doa_t_dev, int64_t *n_out_host, void *stream) {
    if (!sb || !frames_dev || !n_out_host) return set_error(MICLOC_ERR_SHAPE, "null argument");
    SlotBook &bk = sb->book;
    StreamBand &b = sb->band;
    MICLOC_TRY(bk.check_push(dtype, n, in_channels, b.prm.chain.M));
    MICLOC_CUDA(cudaSetDevice(sb->device));
    cudaStream_t st = (cudaStream_t)stream;
    MICLOC_TRY(reserve_env(b, bk.S, n + bk.D, env_dev, doa_t_dev));
    MICLOC_TRY(bk.assemble(b.xbuf, frames_dev, dtype, n, in_channels, b.prm.chain.M, b.hist, st));
    return step_bands(bk, &b, 1, nullptr, n, n + bk.D, spikes_dev, power_dev, doa_dev, env_dev, doa_t_dev, n_out_host, st);
}

extern "C" int micloc_snn_streams_flush(micloc_stream_batch *sb, const int32_t *slots_host, int32_t n_slots,
                                        int8_t *spikes_dev, float *power_dev, int32_t *doa_dev, float *env_dev,
                                        int32_t *doa_t_dev, int64_t *n_out_host, int32_t *flags_host, void *stream) {
    if (!sb || !n_out_host) return set_error(MICLOC_ERR_CONFIG, "null stream");
    MICLOC_CUDA(cudaSetDevice(sb->device));
    MICLOC_TRY(reserve_env(sb->band, sb->book.S, sb->book.max_frame + sb->book.D, env_dev, doa_t_dev));
    return flush_bands(sb->book, &sb->band, 1, slots_host, n_slots, spikes_dev, power_dev, doa_dev, env_dev, doa_t_dev,
                       n_out_host, flags_host, (cudaStream_t)stream);
}

// ---- multi-band stream batches: F bands on one slot book, behind one filterbank ----
struct micloc_mb_streams {
    int F = 0, device = 0, M = 0, G = 0;
    SlotBook book;
    StreamBand band[8];
    FilterbankParams fb{};
    BiquadState *fb_state = nullptr;    // [F][S][M] filterbank state
    double *doa_list = nullptr;         // [G] on the device, null: no ML estimators
    float *power = nullptr;             // [F][S][G] per-band power when the caller passes no power_dev
};

extern "C" int micloc_snn_mb_streams_destroy(micloc_mb_streams *mb) {
    if (!mb) return MICLOC_OK;
    cudaSetDevice(mb->device);
    mb->book.destroy();
    for (int f = 0; f < mb->F; ++f) band_free(mb->band[f]);
    cudaFree(mb->fb_state); cudaFree(mb->doa_list); cudaFree(mb->power);
    delete mb;
    return MICLOC_OK;
}

extern "C" int micloc_snn_mb_streams_create(micloc_snn *const *ctxs, int32_t F, int32_t n_sections, const double *sos,
                                            const double *doa_list, int32_t num_streams, int64_t max_frame_len,
                                            micloc_mb_streams **out) {
    if (!ctxs || !sos || !out) return set_error(MICLOC_ERR_CONFIG, "null argument");
    *out = nullptr;
    if (F < 1 || F > 8) return set_error(MICLOC_ERR_CONFIG, "multi-band stream batch of %d bands (1..8 supported)", F);
    FilterbankParams fb;
    MICLOC_TRY(filterbank_params(F, n_sections, sos, &fb));
    micloc_snn_params prm[8];
    int D = 0;
    for (int f = 0; f < F; ++f) {
        if (!ctxs[f]) return set_error(MICLOC_ERR_CONFIG, "null context of band %d", f);
        MICLOC_TRY(micloc_snn_get_params(ctxs[f], &prm[f]));
        if (prm[f].device != prm[0].device)
            return set_error(MICLOC_ERR_CONFIG, "band %d's context is on device %d, band 0's on device %d", f, prm[f].device, prm[0].device);
        if (prm[f].chain.M != prm[0].chain.M || prm[f].chain.G != prm[0].chain.G)
            return set_error(MICLOC_ERR_SHAPE, "band %d's context has %d microphones and %d DoAs, band 0's %d and %d", f,
                             prm[f].chain.M, prm[f].chain.G, prm[0].chain.M, prm[0].chain.G);
        D = std::max(D, rzcc_lag(prm[f].chain.w));      // one latency: every band finalises the same samples
    }
    MICLOC_CUDA(cudaSetDevice(prm[0].device));
    micloc_mb_streams *mb = new micloc_mb_streams();
    mb->F = F; mb->device = prm[0].device; mb->M = prm[0].chain.M; mb->G = prm[0].chain.G; mb->fb = fb;
    mb->book.D = D;
    int rc = mb->book.create(num_streams, max_frame_len);
    for (int f = 0; f < F && !rc; ++f) rc = band_alloc(mb->band[f], prm[f], mb->book);
    const size_t S = (size_t)num_streams;
    if (!rc && !(cudaMalloc(&mb->fb_state, (size_t)F * S * mb->M * sizeof(BiquadState)) == cudaSuccess &&
                 cudaMalloc(&mb->power, (size_t)F * S * mb->G * sizeof(float)) == cudaSuccess &&
                 (!doa_list || cudaMalloc(&mb->doa_list, (size_t)mb->G * sizeof(double)) == cudaSuccess)))
        rc = set_error(MICLOC_ERR_CUDA, "cudaMalloc(multi-band stream batch) failed");
    if (!rc && ((doa_list && cudaMemcpy(mb->doa_list, doa_list, (size_t)mb->G * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess) ||
                cudaMemset(mb->fb_state, 0, (size_t)F * S * mb->M * sizeof(BiquadState)) != cudaSuccess))
        rc = set_error(MICLOC_ERR_CUDA, "multi-band stream batch set-up failed");
    if (!rc) rc = reset_bands(mb->book, mb->band, F, nullptr, 0, nullptr);
    if (rc) { micloc_snn_mb_streams_destroy(mb); return rc; }
    *out = mb;
    return MICLOC_OK;
}

extern "C" int micloc_snn_mb_streams_latency(micloc_mb_streams *mb) { return mb ? mb->book.D : 0; }

// the filterbank state of a reset slot is dropped by k_mb_stream_assemble (it restarts at N == 0)
extern "C" int micloc_snn_mb_streams_reset(micloc_mb_streams *mb, const int32_t *slots_host, int32_t n_slots, void *stream) {
    if (!mb) return set_error(MICLOC_ERR_CONFIG, "null stream");
    MICLOC_CUDA(cudaSetDevice(mb->device));
    return reset_bands(mb->book, mb->band, mb->F, slots_host, n_slots, (cudaStream_t)stream);
}

// sum over the bands + estimators over each slot's final rows
static int mb_fuse(micloc_mb_streams *mb, const float *power, float *power_grid_dev, int32_t *doa_dev, double *periodic_ml_dev,
                   double *trimmed_ml_dev, int32_t *flags_dev, cudaStream_t st) {
    const int32_t *band_flags[8];
    for (int f = 0; f < mb->F; ++f) band_flags[f] = mb->band[f].flags;
    return launch_power_fuse(power, mb->F, mb->book.S, mb->G, mb->doa_list, power_grid_dev, doa_dev, periodic_ml_dev,
                             trimmed_ml_dev, flags_dev, mb->book.m, band_flags, st);
}

extern "C" int micloc_snn_mb_streams_push(micloc_mb_streams *mb, const void *frames_dev, int dtype, int64_t n,
                                          int32_t in_channels, int8_t *spikes_dev, float *power_dev, float *power_grid_dev,
                                          int32_t *doa_dev, double *periodic_ml_dev, double *trimmed_ml_dev,
                                          double *sumsq_dev, int32_t *flags_dev, int64_t *n_out_host, void *stream) {
    if (!mb || !frames_dev || !n_out_host) return set_error(MICLOC_ERR_SHAPE, "null argument");
    SlotBook &bk = mb->book;
    MICLOC_TRY(bk.check_push(dtype, n, in_channels, mb->M));
    if ((periodic_ml_dev || trimmed_ml_dev) && !mb->doa_list) return set_error(MICLOC_ERR_SHAPE, "the ML estimators need doa_list");
    MICLOC_CUDA(cudaSetDevice(mb->device));
    cudaStream_t st = (cudaStream_t)stream;
    MbAssembleParams ap{};
    ap.fb = mb->fb;
    for (int f = 0; f < mb->F; ++f) {
        ap.prev[f] = mb->band[f].xbuf[bk.xcur];
        ap.cur[f] = mb->band[f].xbuf[bk.xcur ^ 1];
        ap.hist[f] = mb->band[f].hist;
    }
    if (sumsq_dev) MICLOC_CUDA(cudaMemsetAsync(sumsq_dev, 0, (size_t)bk.S * sizeof(double), st));
    const unsigned grid = (unsigned)((bk.S * mb->M + 127) / 128);
    auto launch = dtype == MICLOC_F32 ? launch_mb_assemble<float> : dtype == MICLOC_I16 ? launch_mb_assemble<int16_t>
                                                                                    : launch_mb_assemble<int32_t>;
    launch(mb->F, grid, st, frames_dev, mb->fb_state, sumsq_dev, bk.pos[bk.pcur], ap, bk.S, (int)n, (int)bk.n_prev,
           in_channels, mb->M);
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    bk.xcur ^= 1;
    bk.n_prev = n;
    const bool fuse = power_dev || power_grid_dev || doa_dev || periodic_ml_dev || trimmed_ml_dev || flags_dev;
    float *power = power_dev ? power_dev : mb->power;
    MICLOC_TRY(step_bands(bk, mb->band, mb->F, nullptr, n, n + bk.D, spikes_dev, fuse ? power : nullptr, nullptr, nullptr,
                          nullptr, n_out_host, st));
    if (!fuse) return MICLOC_OK;
    return mb_fuse(mb, power, power_grid_dev, doa_dev, periodic_ml_dev, trimmed_ml_dev, flags_dev, st);
}

extern "C" int micloc_snn_mb_streams_flush(micloc_mb_streams *mb, const int32_t *slots_host, int32_t n_slots,
                                           int8_t *spikes_dev, float *power_dev, float *power_grid_dev, int32_t *doa_dev,
                                           double *periodic_ml_dev, double *trimmed_ml_dev, int32_t *flags_dev,
                                           int64_t *n_out_host, int32_t *flags_host, void *stream) {
    if (!mb || !n_out_host) return set_error(MICLOC_ERR_CONFIG, "null stream");
    if ((periodic_ml_dev || trimmed_ml_dev) && !mb->doa_list) return set_error(MICLOC_ERR_SHAPE, "the ML estimators need doa_list");
    MICLOC_CUDA(cudaSetDevice(mb->device));
    cudaStream_t st = (cudaStream_t)stream;
    const bool fuse = power_dev || power_grid_dev || doa_dev || periodic_ml_dev || trimmed_ml_dev || flags_dev;
    float *power = power_dev ? power_dev : mb->power;
    MICLOC_TRY(flush_bands(mb->book, mb->band, mb->F, slots_host, n_slots, spikes_dev, fuse ? power : nullptr, nullptr,
                           nullptr, nullptr, n_out_host, flags_host, st));
    if (!fuse) return MICLOC_OK;
    return mb_fuse(mb, power, power_grid_dev, doa_dev, periodic_ml_dev, trimmed_ml_dev, flags_dev, st);
}

// ---- the single stream: slot 0 of a one-slot batch ----
extern "C" int micloc_snn_stream_create(micloc_snn *ctx, int64_t max_frame_len, double fs, double rise_time,
                                        double fall_time, micloc_stream **out) {
    if (!ctx || !out) return set_error(MICLOC_ERR_CONFIG, "null argument");
    *out = nullptr;
    micloc_stream_batch *sb = nullptr;
    MICLOC_TRY(micloc_snn_streams_create(ctx, 1, max_frame_len, fs, rise_time, fall_time, &sb));
    *out = new micloc_stream{sb};
    return MICLOC_OK;
}

extern "C" int micloc_snn_stream_destroy(micloc_stream *s) {
    if (!s) return MICLOC_OK;
    micloc_snn_streams_destroy(s->sb);
    delete s;
    return MICLOC_OK;
}

extern "C" int micloc_snn_stream_reset(micloc_stream *s, void *stream) {
    if (!s) return set_error(MICLOC_ERR_CONFIG, "null stream");
    return micloc_snn_streams_reset(s->sb, nullptr, 0, stream);
}

extern "C" int micloc_snn_stream_latency(micloc_stream *s) { return s ? s->sb->book.D : 0; }

extern "C" int micloc_snn_stream_push(micloc_stream *s, const void *frame_dev, int dtype, int64_t n, int32_t in_channels,
                                      int8_t *spikes_dev, float *power_dev, int32_t *doa_dev, float *env_dev,
                                      int32_t *doa_t_dev, int64_t *n_out, void *stream) {
    if (!s || !frame_dev) return set_error(MICLOC_ERR_SHAPE, "null argument");
    if (!s->sb->book.active[0]) return set_error(MICLOC_ERR_CONFIG, "stream was flushed: reset it before pushing again");
    int64_t m = 0;
    MICLOC_TRY(micloc_snn_streams_push(s->sb, frame_dev, dtype, n, in_channels, spikes_dev, power_dev, doa_dev, env_dev,
                                       doa_t_dev, &m, stream));
    if (n_out) *n_out = m;
    return MICLOC_OK;
}

extern "C" int micloc_snn_stream_flush(micloc_stream *s, int8_t *spikes_dev, float *power_dev, int32_t *doa_dev,
                                       float *env_dev, int32_t *doa_t_dev, int64_t *n_out, int32_t *flags_host,
                                       void *stream) {
    if (!s) return set_error(MICLOC_ERR_CONFIG, "null stream");
    int64_t m = 0;
    MICLOC_TRY(micloc_snn_streams_flush(s->sb, nullptr, 0, spikes_dev, power_dev, doa_dev, env_dev, doa_t_dev, &m,
                                        flags_host, stream));
    if (n_out) *n_out = m;
    return MICLOC_OK;
}

// Envelope.evolve on a whole device array [T][C] (fresh state) + optional per-row argmax
extern "C" int micloc_envelope(const float *x_dev, int64_t T, int32_t C, double fs, double rise_time, double fall_time,
                               float *env_dev, int32_t *argmax_dev, int device, void *stream) {
    if (!x_dev || !env_dev || T < 1 || C < 1) return set_error(MICLOC_ERR_SHAPE, "bad envelope arguments");
    if (rise_time > fall_time)
        return set_error(MICLOC_ERR_CONFIG, "for proper functioning, an envelope estimator should have a larger fall time!");
    const int wf = (int)(fs * fall_time), wr = (int)(fs * rise_time);
    if (wf < 1 || wr < 1) return set_error(MICLOC_ERR_CONFIG, "envelope windows shorter than one sample");
    MICLOC_CUDA(cudaSetDevice(device));
    cudaStream_t st = (cudaStream_t)stream;
    float *state = nullptr; int32_t *started = nullptr;
    MICLOC_CUDA(cudaMallocAsync(&state, (size_t)C * sizeof(float), st));
    MICLOC_CUDA(cudaMallocAsync(&started, (size_t)C * sizeof(int32_t), st));
    MICLOC_CUDA(cudaMemsetAsync(state, 0, (size_t)C * sizeof(float), st));
    MICLOC_CUDA(cudaMemsetAsync(started, 0, (size_t)C * sizeof(int32_t), st));
    k_envelope<<<(C + 127) / 128, 128, 0, st>>>(x_dev, env_dev, state, started, nullptr, 1, T, C, 1.f / (float)wf, 1.f / (float)wr);
    count_launch(1);
    if (argmax_dev) {
        k_argmax_rows<<<(unsigned)((T * 32 + 255) / 256), 256, 0, st>>>(env_dev, argmax_dev, nullptr, 1, T, C);
        count_launch(1);
    }
    MICLOC_CUDA(cudaGetLastError());
    MICLOC_CUDA(cudaFreeAsync(state, st));
    MICLOC_CUDA(cudaFreeAsync(started, st));
    return MICLOC_OK;
}
