// micloc_staged.cuh -- one kernel per stage of the float SNN chain, with every
// intermediate in global memory.  These are the debug-tap path of the C-ABI
// (micloc_snn_run_taps), the building blocks of Beamformer.apply_to_signal and of
// the Xylo front end, and the cross-check of the fused kernel.
#pragma once
#include "micloc_device.cuh"
#include <cuda_fp16.h>

namespace micloc {

// ---------------------------------------------------------------------------
// S1: STHT quadrature FIR   q[b][t][m] = sum_k h[k] * x[b][t-k][m]
//     (micloc/snn_beamformer.py:327, zero initial state)
// grid.x = B * ntiles, grid.y = mic groups of <= MG mics; dynamic smem:
//   taps[n_taps] | rows[MG][pitch]
// Each thread owns kFirR consecutive outputs of one mic and walks the kept taps
// in blocks of kFirJB with a register window: 128 FFMA per 8+2 LDS.128.
// ---------------------------------------------------------------------------
template <typename IN_T, int STRIDE>
__global__ void __launch_bounds__(256)
k_stht(const IN_T *__restrict__ audio, float *__restrict__ q, const float *__restrict__ taps,
       const __grid_constant__ ChainParams p, long long T, int TT, int ntiles, int MG) {
    extern __shared__ __align__(16) float smem[];
    float *taps_s = smem;
    const int pitch = fir_row_pitch(TT, p.span);
    float *rows = smem + ((p.n_taps + 3) & ~3);

    const long long b = blockIdx.x / ntiles;
    const long long t0 = (long long)(blockIdx.x % ntiles) * TT;
    const int m0 = blockIdx.y * MG;
    const int mg = min(MG, p.M - m0);
    const IN_T *clip = audio + b * T * p.M;

    for (int i = threadIdx.x; i < p.n_taps; i += blockDim.x) taps_s[i] = taps[i];
    fir_fill_rows<IN_T>(rows, pitch, clip, T, p.M, m0, mg, t0, p.span, TT + p.span + 8);
    __syncthreads();

    const int chunks = TT / kFirR;
    for (int item = threadIdx.x; item < mg * chunks; item += blockDim.x) {
        const int mm = item / chunks, chunk = item % chunks;
        float acc[kFirR];
        fir_accumulate<STRIDE>(rows + mm * pitch, taps_s, p.n_taps, p.span, p.tap_first, chunk, acc);
        float *dst = q + (b * T + t0 + (long long)chunk * kFirR) * p.M + m0 + mm;
#pragma unroll
        for (int i = 0; i < kFirR; ++i)
            if (t0 + chunk * kFirR + i < T) dst[(long long)i * p.M] = acc[i];
    }
}

// band-pass output of one clip -> input of the unbounded float64 encoder (heal_overflow).  Denormals become zeros:
// in digital silence the float32 filter never decays to 0 but cycles through denormals, whose sign changes are noise.
static __global__ void __launch_bounds__(256)
k_f32_to_f64(const float *__restrict__ x, double *__restrict__ y, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = fabsf(x[i]) < 1.17549435e-38f ? 0.0 : (double)x[i];
}

// ---------------------------------------------------------------------------
// S2: band-pass + RZCC, one thread per (clip, time segment, band, channel).
//   channel c < M : in-phase  = x[(t - K/2) mod T]   (np.roll, snn_beamformer.py:325)
//   channel c >= M: quadrature = q[t]
//   z = SOS cascade (snn_beamformer.py:330-335 / filterbank.py:40-44)
//   spikes = RZCC(z)          (spike_encoder.py:115-137)
// Output channel index is band*C2 + c (Demo.spike_encoding's hstack over bands,
// xylo_snn_localization.py:341-342); nb == 1 for the float SNN chain.
// `band_sos` [nb][kMaxSections][5]; sos of band 0 also sits in p.sos.
//
// TIME SEGMENTS, for few long clips (BASELINE config 5: one 10 s clip of 64 microphones is 128 sequential chains of
// 480 000 steps -- 128 threads).  Band-pass and alpha kernel forget their past geometrically and the RZCC decisions are
// local (a cluster ends at the first gap >= w), so segment s starts from zero state `warm` samples early, runs `tail`
// samples past its end and keeps only the spikes / membrane values of its own range: (clip, channel, segment) chains
// run in parallel.  What a segment cannot vouch for sets the clip's flag bit 0 and the clip is redone sequentially by
// the host code: a cluster still open at the segment start that began inside the settling half of the warm-up, or one
// that holds a spike of the segment and is still open at the end of the tail.  The running sum restarts at every
// warm-up: heights are only compared inside a cluster, where a common offset cancels (up to float32 rounding of the
// sum, i.e. within the path's tolerance, not bit for bit).  RZCC is scale-free: in digital silence the band-pass's
// decaying tail IS the signal and keeps spiking for tens of milliseconds, so "forgetting" only holds relative to a live
// input -- a block of kSeg exactly-zero input samples anywhere in a segment's span flags the clip as well.  One segment
// per chain (seg_len >= T, warm = tail = 0) is the sequential recurrence: only an overflowed cluster flags the clip.
//
// 32 samples at a time: a per-sample candidate test runs its divergent cluster path on almost every step, because with
// 32 channels in a warp SOME lane has a zero crossing (ncu: 144 warp instructions per sample).  Here a thread first
// runs the band-pass and the running sum over a block of kSeg samples without a branch (bandpass_block: sign /
// flat-top bit masks, the running sums of the block in shared memory), then hands the block to rzcc_segment_masks --
// the front end of the fused kernels, which visits only the sign changes -- and the next block's 32 inputs travel from
// HBM to registers meanwhile.  The spike raster must be ZEROED before the launch (launch_chain_any does): only spikes
// are stored.
// ---------------------------------------------------------------------------
constexpr int kChainBlkThreads = 128;

// The input of channel c of clip b from t_begin on: c < M the in-phase x[(t - K/2) mod T] of microphone c (np.roll,
// snn_beamformer.py:325), c >= M the quadrature q[t] of microphone c - M.  k_chain_blk and the Hilbert front end read
// their clips through it.
template <typename IN_T>
struct ClipChannelInput {
    const IN_T *xa;
    const float *xq;
    bool inphase;
    int src0, T, M, t_begin;

    __device__ __forceinline__ ClipChannelInput(const IN_T *audio, const float *q, const ChainParams &p, long long b,
                                                int c, int T_, int t_begin_)
        : inphase(c < p.M), T(T_), M(p.M), t_begin(t_begin_) {
        xa = audio + b * (long long)T * M + (inphase ? c : 0);
        xq = q + b * (long long)T * M + (inphase ? 0 : c - M);
        src0 = (int)(((long long)t_begin - p.half) % T + T) % T;     // (t - K/2) mod T at t = t_begin
    }
    // x[i] = input at ts + i for i < t_stop - ts, 0 beyond
    __device__ __forceinline__ void load(int ts, int t_stop, float (&x)[kSeg]) const {
        const int left = t_stop - ts;
        if (inphase) {
            int s0 = src0 + (ts - t_begin);
            if (s0 >= T) s0 -= T;
            const int wrap = T - s0;                       // the source index wraps after this many samples
            const IN_T *pp = xa + (long long)s0 * M;
            if (left >= kSeg && wrap >= kSeg) {            // (almost always: one pointer, one stride)
#pragma unroll
                for (int i = 0; i < kSeg; ++i) { x[i] = to_f32<IN_T>(*pp); pp += M; }
            } else {
#pragma unroll
                for (int i = 0; i < kSeg; ++i)
                    x[i] = i < left ? to_f32<IN_T>(pp[(long long)(i < wrap ? i : i - T) * M]) : 0.f;
            }
        } else {
            const float *pp = xq + (long long)ts * M;
            if (left >= kSeg) {
#pragma unroll
                for (int i = 0; i < kSeg; ++i) { x[i] = *pp; pp += M; }
            } else {
#pragma unroll
                for (int i = 0; i < kSeg; ++i) x[i] = i < left ? pp[(long long)i * M] : 0.f;
            }
        }
    }
};

template <typename IN_T, int NSEC>          // NSEC: biquads of the band-pass (kNsecRuntime: p.nsec)
__global__ void __launch_bounds__(kChainBlkThreads, 3)
k_chain_blk(const IN_T *__restrict__ audio, const float *__restrict__ q, const float *__restrict__ band_sos,
            float *__restrict__ z_out, int8_t *__restrict__ spikes, int32_t *__restrict__ flags,
            const __grid_constant__ ChainParams p, long long B, long long T64, int nb, int seg_len, int warm, int tail,
            int nseg) {
    __shared__ float cs_s[kSeg * kChainBlkThreads];
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int CT = p.C2 * nb;
    const bool live = idx < B * nseg * CT;           // (no early return: nothing below is a CTA barrier, but keep the warp whole)
    const long long idc = live ? idx : 0;
    const int cc = (int)(idc % CT);
    const int seg = (int)((idc / CT) % nseg);
    const long long b = idc / ((long long)CT * nseg);
    const int band = cc / p.C2, c = cc % p.C2;
    const int T = (int)T64;

    float sos[kMaxSections][5];
    load_sos(sos, band_sos + band * kMaxSections * 5);
    const int nsec = p.nsec;

    const int start = seg * seg_len;
    const int end = min(T, start + seg_len);
    const int t_begin = max(0, start - warm);                 // a multiple of kSeg (seg_len and warm are)
    const int t_stop = live ? min(T, end + tail) : t_begin;
    BiquadState bq; biquad_reset(bq);
    RzccState rz; rzcc_reset(rz);
    int cl_pos[2 * kClusterMax]; float cl_h[2 * kClusterMax];
    const RzccStore store{cl_pos, cl_h, 1};
    int8_t *sp = spikes + b * T64 * CT + cc;
    auto emit = [&](int pos, int sign) { if (pos >= start && pos < end) sp[(long long)pos * CT] = (int8_t)sign; };

    const ClipChannelInput<IN_T> src(audio, q, p, b, c, T, t_begin);
    float x[kSeg];
    bool unsynced = false;
    float *cs = cs_s + threadIdx.x;
    src.load(t_begin, t_stop, x);
    for (int ts = t_begin; ts < t_stop; ts += kSeg) {
        const int nvalid = min(kSeg, t_stop - ts);
        if (ts == start && seg > 0) {
            // decisions from here on are this segment's: every open cluster must have begun after the filters settled
            const int settled = t_begin + (warm >> 1);
            if ((rz.n1 > 0 && cl_pos[kClusterMax] < settled) || (rz.n0 > 0 && cl_pos[0] < settled)) unsynced = true;
        }
        // ---- band-pass + running sum of the block, branch-free (zeros past t_stop too: the loop ends with them) ----
        const float carry = rz.csum;
        float csum = carry;
        const bool keep_z = z_out != nullptr && ts >= start && ts < end;     // (start is a multiple of kSeg)
        float *zo = keep_z ? z_out + (b * T64 + ts) * CT + cc : nullptr;
        auto store_z = [&](int i, float v) { if (keep_z && ts + i < end) zo[(long long)i * CT] = v; };
        const BlockMasks m = bandpass_block<NSEC, false>(x, nvalid, sos, nsec, bq, csum, cs, kChainBlkThreads, store_z);
        // digital silence: a whole block of exactly-zero inputs (either sign)
        if ((m.any << 1) == 0u && nvalid == kSeg && nseg > 1) unsynced = true;
        // ---- the next block's inputs on their way while the candidates of this one are handled ----
        if (ts + kSeg < t_stop) src.load(ts + kSeg, t_stop, x);
        rzcc_segment_masks(rz, store, p.bipolar, p.w, ts, nvalid, m.neg, m.zero, cs, kChainBlkThreads, carry, emit);
        rz.csum = nvalid == kSeg ? csum : cs[(nvalid - 1) * kChainBlkThreads];
        const bool last = ts + nvalid == T;
        if (last || nvalid == kSeg) rzcc_close(rz, store, p.w, ts + nvalid - 1, last, emit);
    }
    // a cluster that is still open behind the tail and holds a candidate of this segment was not decided
    if (t_stop < T && ((rz.n1 > 0 && cl_pos[kClusterMax] < end) || (rz.n0 > 0 && cl_pos[0] < end))) unsynced = true;
    if (live && (rz.overflow || unsynced) && flags) atomicOr(flags + b, 1);
}

static __global__ void __launch_bounds__(128)
k_neuron_seg(const int8_t *__restrict__ spikes, float *__restrict__ vmem, const __grid_constant__ ChainParams p,
             long long B, long long T, int seg_len, int warm, int nseg) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= B * nseg * p.C2) return;
    const int c = (int)(idx % p.C2);
    const int seg = (int)((idx / p.C2) % nseg);
    const long long b = idx / ((long long)p.C2 * nseg);
    const int8_t *sp = spikes + b * T * p.C2 + c;
    float *vm = vmem + b * T * p.C2 + c;
    const long long start = (long long)seg * seg_len, end = min(T, start + seg_len);
    NeuronState n; neuron_reset(n);
    // (few threads per SM: a step that waits for its own two spike bytes runs at one memory latency per sample -- the
    //  bytes of the next kNeuBlk steps are requested before the current kNeuBlk steps are computed)
    constexpr int kNeuBlk = 16;
    const int C2 = p.C2, nL = p.nL;
    const int t_first = (int)max(0ll, start - warm), t_end = (int)end;
    const int last = t_end - 1;
    int nx_s[kNeuBlk], nx_d[kNeuBlk];
    auto request = [&](int t0) {
        // clamped addresses (always inside the clip); what lies outside [0, end) is masked when it is used
        const int8_t *ps = sp + (long long)min(t0, last) * C2;
        const int room = last - min(t0, last);
#pragma unroll
        for (int u = 0; u < kNeuBlk; ++u) nx_s[u] = ps[(long long)min(u, room) * C2];
        const int td = t0 - nL;
#pragma unroll
        for (int u = 0; u < kNeuBlk; ++u) nx_d[u] = sp[(long long)min(max(td + u, 0), last) * C2];
    };
    request(t_first);
    for (int t0 = t_first; t0 < t_end; t0 += kNeuBlk) {
        float cs[kNeuBlk], cd[kNeuBlk];
#pragma unroll
        for (int u = 0; u < kNeuBlk; ++u) {
            cs[u] = t0 + u < t_end ? (float)nx_s[u] : 0.f;
            cd[u] = (t0 + u < t_end && t0 + u >= nL) ? (float)nx_d[u] : 0.f;
        }
        request(t0 + kNeuBlk);
#pragma unroll
        for (int u = 0; u < kNeuBlk; ++u) {
            const int t = t0 + u;
            const float v = neuron_step(p, n, cs[u], cd[u]);
            if (t >= start && t < t_end) vm[(long long)t * C2] = v;
        }
    }
}

// ---------------------------------------------------------------------------
// S4a: Gram matrix of the membrane signals   C[b][i][j] = sum_t v[t][i] v[t][j]
//      mean_t (v[t] . w_g)^2 == w_g^T (C/T) w_g, so the per-DoA power of
//      snn_beamformer.py:368 + target_snn_localization.py:462 needs no T x G pass.
//      rows_b (nullable, stream batches): clip b sums its first rows_b[b] rows only (T stays the row stride), and a
//      clip with no rows is not written.
// ---------------------------------------------------------------------------
static __global__ void __launch_bounds__(256)
k_gram(const float *__restrict__ vmem, double *__restrict__ gram, int C2, long long T, long long t_start,
       const int32_t *__restrict__ rows_b = nullptr) {
    const long long b = blockIdx.x;
    const int pair = blockIdx.y * blockDim.x + threadIdx.x;
    if (pair >= C2 * C2) return;
    const int i = pair / C2, j = pair % C2;
    if (j < i) return;  // symmetric: upper triangle only
    const long long t_end = rows_b ? rows_b[b] : T;
    if (t_end == 0) return;
    const float *v = vmem + b * T * C2;
    double acc = 0.0;
    // the loads of 16 rows are issued before their FMAs (the sum is latency-bound otherwise; same order of FMAs)
    constexpr int kU = 16;
    long long t = t_start;
    for (; t + kU <= t_end; t += kU) {
        float a[kU], c[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) { a[u] = v[(t + u) * C2 + i]; c[u] = v[(t + u) * C2 + j]; }
#pragma unroll
        for (int u = 0; u < kU; ++u) acc = fma((double)a[u], (double)c[u], acc);
    }
    for (; t < t_end; ++t) acc = fma((double)v[t * C2 + i], (double)v[t * C2 + j], acc);
    gram[(b * C2 + i) * C2 + j] = acc;
    gram[(b * C2 + j) * C2 + i] = acc;
}

// the same sum cut into time slabs (few long clips): part[slab][b][i][j], added up in slab order by k_gram_reduce
// (a fixed order: the result does not depend on scheduling)
static __global__ void __launch_bounds__(256)
k_gram_slab(const float *__restrict__ vmem, double *__restrict__ part, int C2, long long B, long long T, long long t_start,
            long long slab_len) {
    const long long b = blockIdx.x;
    const int pair = blockIdx.y * blockDim.x + threadIdx.x;
    if (pair >= C2 * C2) return;
    const int i = pair / C2, j = pair % C2;
    if (j < i) return;
    const long long t0 = t_start + (long long)blockIdx.z * slab_len, t1 = min(T, t0 + slab_len);
    const float *v = vmem + b * T * C2;
    double acc = 0.0;
    for (long long t = t0; t < t1; ++t) acc = fma((double)v[t * C2 + i], (double)v[t * C2 + j], acc);
    part[((long long)blockIdx.z * B + b) * C2 * C2 + i * C2 + j] = acc;
}
// The same partial sums for WIDE arrays as a tiled float32 product (config 5: 128 channels, C = V^T V is a real GEMM,
// 7.9 G multiply-adds per 10 s clip; one thread per matrix element looping over time ran 14 ms).  A CTA owns one
// 128 x 128 block (bi <= bj) of the Gram matrix over its time slab: rows of the membrane tile go through shared
// memory 32 samples at a time, every thread keeps an 8 x 8 register tile (rows 4 ty.., 64 + 4 ty..; columns 4 tx..,
// 64 + 4 tx..: conflict-free 128-bit reads).  A slab is kGtFlush samples: the float32 rounding of a 1024-term sum is
// ~1e-6 relative, below the chain's own float32 error; the slabs are summed in float64 by k_gram_reduce.
constexpr int kGtTile = 128, kGtK = 32, kGtFlush = 1024;
static __global__ void __launch_bounds__(256, 1)
k_gram_tiled(const float *__restrict__ vmem, double *__restrict__ part, int C2, long long B, long long T, long long t_start,
             long long slab_len) {
    __shared__ __align__(16) float As[kGtK][kGtTile + 4];
    __shared__ __align__(16) float Bs[kGtK][kGtTile + 4];
    const long long b = blockIdx.x;
    const int nblk = (C2 + kGtTile - 1) / kGtTile;
    int y = blockIdx.y, bi = 0;
    while (y >= nblk - bi) { y -= nblk - bi; ++bi; }
    const int bj = bi + y;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    const long long t0 = t_start + (long long)blockIdx.z * slab_len, t1 = min(T, t0 + slab_len);
    const float *v = vmem + b * T * C2;
    const bool vec = (C2 & 3) == 0 && (reinterpret_cast<uintptr_t>(v) & 15) == 0;
    for (long long t = t0; t < t1; t += kGtK) {
        for (int e = threadIdx.x; e < kGtK * (kGtTile / 4); e += 256) {
            const int r = e / (kGtTile / 4), c4 = e % (kGtTile / 4);
            const long long tt = t + r;
#pragma unroll
            for (int side = 0; side < 2; ++side) {
                if (side == 1 && bj == bi) break;
                const int col = (side ? bj : bi) * kGtTile + 4 * c4;
                float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
                if (tt < t1) {
                    const float *src = v + tt * C2 + col;
                    if (vec && col + 3 < C2) val = *reinterpret_cast<const float4 *>(src);
                    else {
                        if (col < C2) val.x = src[0];
                        if (col + 1 < C2) val.y = src[1];
                        if (col + 2 < C2) val.z = src[2];
                        if (col + 3 < C2) val.w = src[3];
                    }
                }
                *reinterpret_cast<float4 *>(side ? &Bs[r][4 * c4] : &As[r][4 * c4]) = val;
            }
        }
        __syncthreads();
        const float (*Bp)[kGtTile + 4] = bj == bi ? As : Bs;
#pragma unroll 4
        for (int r = 0; r < kGtK; ++r) {
            const float4 a0 = *reinterpret_cast<const float4 *>(&As[r][4 * ty]), a1 = *reinterpret_cast<const float4 *>(&As[r][64 + 4 * ty]);
            const float4 b0 = *reinterpret_cast<const float4 *>(&Bp[r][4 * tx]), b1 = *reinterpret_cast<const float4 *>(&Bp[r][64 + 4 * tx]);
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int gi = bi * kGtTile + (i < 4 ? 4 * ty + i : 64 + 4 * ty + i - 4);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int gj = bj * kGtTile + (j < 4 ? 4 * tx + j : 64 + 4 * tx + j - 4);
            if (gi < C2 && gj < C2 && gi <= gj)
                part[(((long long)blockIdx.z * B + b) * C2 + gi) * C2 + gj] = (double)acc[i][j];
        }
    }
}
// The same 128 x 128 block on the TENSOR CORES: the membrane tile (x 2^12) is split into fp16 hi + lo (22 significant
// bits, as the fused kernel's Gram role does), staged [sample][channel] in shared memory, and both operands of
// C += V^T V are read from it with ldmatrix.trans (A[m][k] = V[k][m], B[k][n] = V[k][n]: the same transposed 8 x 8
// pieces).  Three mma.sync.m16n8k16 per tile and k step (hi.hi, hi.lo, lo.hi), float32 accumulators over the slab of
// kGtFlush samples, float64 across slabs (k_gram_reduce).  8 warps, warp tile 64 x 32; the next 32 samples travel from
// HBM to registers while the current ones are multiplied.
constexpr int kGcK = 32;                 // samples per stage: two k steps of 16
constexpr int kGcPitch = kGtTile + 8;    // halves per shared-memory row: 272 B, eight ldmatrix rows hit eight bank groups
constexpr float kGcScale = 4096.f;       // |v| x 2^12 < 65504: the host checks the neuron kernel's absolute sum (< 15)
__device__ __forceinline__ void ldsm_x4_trans(unsigned (&r)[4], const void *p) {
    const unsigned a = (unsigned)__cvta_generic_to_shared(p);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void mma_gram_k16(float (&d)[4], const unsigned (&a)[4], unsigned b0, unsigned b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
template <bool DIAG_ONLY>      // every block is a diagonal block (C2 <= 128): one staged operand, half the prefetch registers
static __global__ void __launch_bounds__(256, 2)
k_gram_tc(const float *__restrict__ vmem, double *__restrict__ part, int C2, long long B, long long T, long long t_start,
          long long slab_len) {
    __shared__ __align__(16) __half S[DIAG_ONLY ? 1 : 2][2][kGcK][kGcPitch];   // [row block | column block][hi | lo][sample][channel]
    const long long b = blockIdx.x;
    const int nblk = (C2 + kGtTile - 1) / kGtTile;
    int y = blockIdx.y, bi = 0;
    while (y >= nblk - bi) { y -= nblk - bi; ++bi; }
    const int bj = bi + y;
    const bool diag = DIAG_ONLY || bi == bj;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp & 1, wn = warp >> 1;
    float acc[4][4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[i][j][e] = 0.f;
    const long long t0 = t_start + (long long)blockIdx.z * slab_len, t1 = min(T, t0 + slab_len);
    const float *v = vmem + b * T * C2;
    const bool vec = (C2 & 3) == 0 && (reinterpret_cast<uintptr_t>(v) & 15) == 0;
    // staging: thread -> sample r = e / 32, channels 4 (e % 32) .. + 3, e = tid + 256 q
    constexpr int kSides = DIAG_ONLY ? 1 : 2;
    float4 pre[kSides][4];
    auto fetch = [&](long long t) {
#pragma unroll
        for (int side = 0; side < kSides; ++side) {
            if (side == 1 && diag) break;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int e = tid + 256 * q;
                const long long tt = t + (e >> 5);
                const int col = (side ? bj : bi) * kGtTile + 4 * (e & 31);
                float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
                if (tt < t1) {
                    const float *src = v + tt * C2 + col;
                    if (vec && col + 3 < C2) val = __ldg(reinterpret_cast<const float4 *>(src));
                    else {
                        if (col < C2) val.x = src[0];
                        if (col + 1 < C2) val.y = src[1];
                        if (col + 2 < C2) val.z = src[2];
                        if (col + 3 < C2) val.w = src[3];
                    }
                }
                pre[side][q] = val;
            }
        }
    };
    auto stash = [&]() {
#pragma unroll
        for (int side = 0; side < kSides; ++side) {
            if (side == 1 && diag) break;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int e = tid + 256 * q;
                const float4 val = pre[side][q];
                const float s0 = val.x * kGcScale, s1 = val.y * kGcScale, s2 = val.z * kGcScale, s3 = val.w * kGcScale;
                const __half2 h01 = __floats2half2_rn(s0, s1), h23 = __floats2half2_rn(s2, s3);
                const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
                const __half2 l01 = __floats2half2_rn(s0 - f01.x, s1 - f01.y), l23 = __floats2half2_rn(s2 - f23.x, s3 - f23.y);
                uint2 hv, lv;
                hv.x = *reinterpret_cast<const unsigned *>(&h01); hv.y = *reinterpret_cast<const unsigned *>(&h23);
                lv.x = *reinterpret_cast<const unsigned *>(&l01); lv.y = *reinterpret_cast<const unsigned *>(&l23);
                *reinterpret_cast<uint2 *>(&S[side][0][e >> 5][4 * (e & 31)]) = hv;
                *reinterpret_cast<uint2 *>(&S[side][1][e >> 5][4 * (e & 31)]) = lv;
            }
        }
    };
    const int sb = diag ? 0 : 1;
    // ldmatrix row of this lane: A pieces (samples +8 in matrices 2, 3; channels +8 in matrices 1, 3), B pieces
    // (samples +8 in matrices 1, 3; channels +8 in matrices 2, 3: two column blocks of 8 per load)
    const int a_row = (lane & 7) + 8 * (lane >> 4), a_col = wm * 64 + 8 * ((lane >> 3) & 1);
    const int b_row = (lane & 7) + 8 * ((lane >> 3) & 1), b_col = wn * 32 + 8 * (lane >> 4);
    fetch(t0);
    for (long long t = t0; t < t1; t += kGcK) {
        stash();
        __syncthreads();
        if (t + kGcK < t1) fetch(t + kGcK);
#pragma unroll
        for (int ks = 0; ks < kGcK / 16; ++ks) {
            const int k0 = 16 * ks;
            unsigned ah[4][4], bh[4][2], x[4];
#pragma unroll
            for (int mb = 0; mb < 4; ++mb) ldsm_x4_trans(ah[mb], &S[0][0][k0 + a_row][a_col + 16 * mb]);
#pragma unroll
            for (int n2 = 0; n2 < 2; ++n2) {
                ldsm_x4_trans(x, &S[sb][0][k0 + b_row][b_col + 16 * n2]);
                bh[2 * n2][0] = x[0]; bh[2 * n2][1] = x[1]; bh[2 * n2 + 1][0] = x[2]; bh[2 * n2 + 1][1] = x[3];
            }
#pragma unroll
            for (int mb = 0; mb < 4; ++mb)
#pragma unroll
                for (int nb = 0; nb < 4; ++nb) mma_gram_k16(acc[mb][nb], ah[mb], bh[nb][0], bh[nb][1]);
#pragma unroll
            for (int n2 = 0; n2 < 2; ++n2) {                              // hi . lo
                ldsm_x4_trans(x, &S[sb][1][k0 + b_row][b_col + 16 * n2]);
#pragma unroll
                for (int mb = 0; mb < 4; ++mb) {
                    mma_gram_k16(acc[mb][2 * n2], ah[mb], x[0], x[1]);
                    mma_gram_k16(acc[mb][2 * n2 + 1], ah[mb], x[2], x[3]);
                }
            }
#pragma unroll
            for (int mb = 0; mb < 4; ++mb) {                              // lo . hi
                ldsm_x4_trans(x, &S[0][1][k0 + a_row][a_col + 16 * mb]);
#pragma unroll
                for (int nb = 0; nb < 4; ++nb) mma_gram_k16(acc[mb][nb], x, bh[nb][0], bh[nb][1]);
            }
        }
        __syncthreads();
    }
    const int g = lane >> 2, tq = lane & 3;
    const double unscale = 1.0 / ((double)kGcScale * (double)kGcScale);
    double *out = part + ((long long)blockIdx.z * B + b) * C2 * C2;
#pragma unroll
    for (int mb = 0; mb < 4; ++mb)
#pragma unroll
        for (int nb = 0; nb < 4; ++nb)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int gi = bi * kGtTile + wm * 64 + mb * 16 + g + 8 * (e >> 1);
                const int gj = bj * kGtTile + wn * 32 + nb * 8 + 2 * tq + (e & 1);
                if (gi < C2 && gj < C2 && gi <= gj) out[(long long)gi * C2 + gj] = (double)acc[mb][nb][e] * unscale;
            }
}
// ---------------------------------------------------------------------------
// S1 on the TENSOR CORES, for wide arrays (M > 8: the fused kernels do not apply and k_stht's FP32 FIR is 27-50 % of a
// config-5 clip).  Polyphase: the Hilbert kernel keeps every other tap, so the outputs of one time parity are a DENSE
// n_taps-tap FIR of the input samples of one parity:  Q[2u + pi] = sum_j g[j] xs[u - j - c],  xs[v] = x[2v + rho].
// Per CTA: U = 16 MB outputs of each parity x 32 microphones.  D[a][n] = sum_e A[a][e] B[e][n] with B[e][n] = xs[vb + e]
// of microphone n (the staged window, fp16 hi + lo of x * 2^k, k from the window's largest magnitude; int16 input is
// exact) and A[a][e] = g[a - e + L] the Toeplitz matrix of the taps (x 2^14, fp16 hi + lo).  A is never stored: the
// mma.sync fragment of the 16 x 16 block (mb, ks) depends on mb - ks only, so ND = n_taps/16 + 1 fragments per split
// piece sit in shared memory (one LDS.128 per fragment and lane) and a warp that owns two consecutive row blocks gets
// the second block's fragment by keeping the first one's for one more k step.  B fragments come from the [sample][mic]
// tile by ldmatrix.trans (16-byte chunks XOR-swizzled by the row: stores and matrix loads both conflict-free).  Three
// products per tile (hi.hi, hi.lo, lo.hi), float32 accumulation: ~1e-6 relative against float64 (bar 1e-4).
// ---------------------------------------------------------------------------
constexpr int kStMB = 8;                    // row blocks of 16 outputs per parity and CTA (U = 128): two per warp
constexpr int kStThreads = 32 * kStMB;      // 2 parities x kStMB/2 pairs = kStMB warps
constexpr int kStMics = 32;                 // microphones per CTA
constexpr float kStTapScale = 16384.f;
__host__ __device__ inline int stht_tc_nd(int n_taps) { return (n_taps + 14) / 16 + 1; }
__host__ __device__ inline int stht_tc_window(int n_taps) { return 16 * (kStMB + stht_tc_nd(n_taps) - 1); }
__host__ __device__ inline size_t stht_tc_smem(int n_taps) {
    return (size_t)2 * 2 * stht_tc_window(n_taps) * 64 + (size_t)stht_tc_nd(n_taps) * 2 * 512 + 16;
}
template <typename IN_T>
__global__ void __launch_bounds__(kStThreads, 2)
k_stht_tc(const IN_T *__restrict__ audio, float *__restrict__ q, const float *__restrict__ taps,
          const __grid_constant__ ChainParams p, long long T64, int ntiles) {
    extern __shared__ __align__(16) unsigned char st_smem[];
    const int ND = stht_tc_nd(p.n_taps), W = stht_tc_window(p.n_taps), L = 16 * (ND - 1);
    unsigned char *Xs = st_smem;                                            // [rho][hi | lo][W][64 B]
    uint4 *Fs = reinterpret_cast<uint4 *>(st_smem + (size_t)4 * W * 64);      // [ND][hi | lo][32 lanes]
    unsigned int *amax_s = reinterpret_cast<unsigned int *>(st_smem + (size_t)4 * W * 64 + (size_t)ND * 1024);
    const int T = (int)T64, M = p.M;
    const long long b = blockIdx.x / ntiles;
    const int u0 = (int)(blockIdx.x % ntiles) * (16 * kStMB);
    const int m0 = blockIdx.y * kStMics;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const IN_T *clip = audio + b * T64 * M;
    // input parity rho serves output parity pi = (rho + tap_first) & 1; first staged stream sample vb = u0 - c - L
    const int tf = p.tap_first;
    auto vbase = [&](int rho) { const int pi = (rho + tf) & 1; return u0 - ((tf + rho - pi) >> 1) - L; };

    if (tid == 0) *amax_s = 0u;
    // ---- Toeplitz fragments of the taps ----
    for (int e = tid; e < ND * 32; e += kStThreads) {
        const int d = e >> 5, ln = e & 31, g = ln >> 2, tq = ln & 3;
        unsigned hv[4], lv[4];
#pragma unroll
        for (int qd = 0; qd < 4; ++qd) {
            const int r = g + 8 * (qd & 1), c0 = 2 * tq + 8 * (qd >> 1);
            unsigned short hh[2], ll[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int j = 16 * d + r - (c0 + u);
                const float gs = (j >= 0 && j < p.n_taps) ? taps[j] * kStTapScale : 0.f;
                const __half hi = __float2half_rn(gs);
                hh[u] = __half_as_ushort(hi);
                ll[u] = __half_as_ushort(__float2half_rn(gs - __half2float(hi)));
            }
            hv[qd] = (unsigned)hh[0] | ((unsigned)hh[1] << 16);
            lv[qd] = (unsigned)ll[0] | ((unsigned)ll[1] << 16);
        }
        Fs[(d * 2 + 0) * 32 + ln] = make_uint4(hv[0], hv[1], hv[2], hv[3]);
        Fs[(d * 2 + 1) * 32 + ln] = make_uint4(lv[0], lv[1], lv[2], lv[3]);
    }
    __syncthreads();
    // ---- window: four microphones of one sample row per thread (one 16-byte load); all of a thread's loads are in
    //      flight at once and stay in registers across the scan for the largest magnitude (float32 input) ----
    const int nvec = 2 * W * (kStMics / 4);
    const bool vec_ok = (M & 3) == 0 && (reinterpret_cast<uintptr_t>(clip) & 15) == 0;
    auto load4 = [&](int idx) -> float4 {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (idx < nvec) {
            const int row = idx >> 3, c4 = idx & 7;
            const int rho = row >= W ? 1 : 0, e = row - rho * W;
            const long long i = 2ll * (vbase(rho) + e) + rho;
            const int m = m0 + 4 * c4;
            if (i >= 0 && i < T && m < M) {
                const IN_T *src = clip + i * M + m;
                if (vec_ok) {                                   // (M % 4 == 0: the four microphones exist)
                    if (sizeof(IN_T) == 4) v = __ldg(reinterpret_cast<const float4 *>(src));
                    else {
                        const short4 s4 = __ldg(reinterpret_cast<const short4 *>(src));
                        v = make_float4((float)s4.x, (float)s4.y, (float)s4.z, (float)s4.w);
                    }
                } else {
                    v.x = to_f32<IN_T>(src[0]);
                    if (m + 1 < M) v.y = to_f32<IN_T>(src[1]);
                    if (m + 2 < M) v.z = to_f32<IN_T>(src[2]);
                    if (m + 3 < M) v.w = to_f32<IN_T>(src[3]);
                }
            }
        }
        return v;
    };
    auto amax4 = [](float mx, const float4 &v) {
        return fmaxf(fmaxf(mx, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
    };
    float scale = 1.f, unscale = 1.f / kStTapScale;
    auto set_scale = [&]() {
        if (sizeof(IN_T) == 4) {
            const unsigned am = *amax_s;
            int ex = (int)((am >> 23) & 0xffu) - 127;              // floor(log2(amax)); x * 2^(14 - ex) < 2^15
            if (am == 0u) ex = 14;
            ex = ex < -90 ? -90 : (ex > 100 ? 100 : ex);
            scale = __uint_as_float((unsigned)(127 + 14 - ex) << 23);
            unscale = __uint_as_float((unsigned)(127 + ex - 28) << 23);
        }
    };
    auto publish_amax = [&](float mx) {
        unsigned mb = __float_as_uint(mx);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { const unsigned ot = __shfl_xor_sync(0xffffffffu, mb, o); mb = ot > mb ? ot : mb; }
        if (lane == 0) atomicMax(amax_s, mb);
    };
    auto stash4 = [&](int idx, const float4 &v) {
        if (idx >= nvec) return;
        const int row = idx >> 3, c4 = idx & 7;
        const int rho = row >= W ? 1 : 0, e = row - rho * W;
        const float s0 = v.x * scale, s1 = v.y * scale, s2 = v.z * scale, s3 = v.w * scale;
        const __half2 h01 = __floats2half2_rn(s0, s1), h23 = __floats2half2_rn(s2, s3);
        const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
        const __half2 l01 = __floats2half2_rn(s0 - f01.x, s1 - f01.y), l23 = __floats2half2_rn(s2 - f23.x, s3 - f23.y);
        uint2 hv, lv;
        hv.x = *reinterpret_cast<const unsigned *>(&h01); hv.y = *reinterpret_cast<const unsigned *>(&h23);
        lv.x = *reinterpret_cast<const unsigned *>(&l01); lv.y = *reinterpret_cast<const unsigned *>(&l23);
        unsigned char *rowp = Xs + ((size_t)(rho * 2) * W + e) * 64 + 16 * ((c4 >> 1) ^ ((e >> 1) & 3)) + 8 * (c4 & 1);
        *reinterpret_cast<uint2 *>(rowp) = hv;
        *reinterpret_cast<uint2 *>(rowp + (size_t)W * 64) = lv;
    };
    constexpr int kStHold = 24;                                  // 16-byte pieces a thread keeps: W <= 384 (n_taps <= 264)
    if (nvec <= kStHold * kStThreads) {
        float4 hold[kStHold];
#pragma unroll
        for (int k = 0; k < kStHold; ++k) hold[k] = load4(tid + kStThreads * k);
        if (sizeof(IN_T) == 4) {
            float mx = 0.f;
#pragma unroll
            for (int k = 0; k < kStHold; ++k) mx = amax4(mx, hold[k]);
            publish_amax(mx);
            __syncthreads();
            set_scale();
        }
#pragma unroll
        for (int k = 0; k < kStHold; ++k) stash4(tid + kStThreads * k, hold[k]);
    } else {
        // long kernels: two passes over the window (the second one hits L2)
        if (sizeof(IN_T) == 4) {
            float mx = 0.f;
#pragma unroll 4
            for (int idx = tid; idx < nvec; idx += kStThreads) mx = amax4(mx, load4(idx));
            publish_amax(mx);
            __syncthreads();
            set_scale();
        }
#pragma unroll 4
        for (int idx = tid; idx < nvec; idx += kStThreads) stash4(idx, load4(idx));
    }
    __syncthreads();

    // ---- this warp: output parity pi, row blocks mb0 and mb0 + 1 ----
    const int pi = warp / (kStMB / 2), mb0 = 2 * (warp % (kStMB / 2));
    const int rho = (pi + tf) & 1;                       // (rho + tf) & 1 == pi
    const unsigned char *Xh = Xs + (size_t)(rho * 2) * W * 64, *Xl = Xh + (size_t)W * 64;
    const int mg = min(kStMics, M - m0), nblk = (mg + 7) >> 3;     // column blocks of 8 microphones in use
    float acc[2][4][4];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[i][j][e] = 0.f;
    unsigned fa_h[4] = {0u, 0u, 0u, 0u}, fa_l[4] = {0u, 0u, 0u, 0u}, fb_h[4], fb_l[4];
    const int b_row = (lane & 7) + 8 * ((lane >> 3) & 1), b_chunk = lane >> 4;
    for (int ks = mb0; ks <= mb0 + ND; ++ks) {
        const int dA = mb0 - ks + ND - 1;                // fragment of block mb0; block mb0 + 1 uses dA + 1 = last step's
#pragma unroll
        for (int i = 0; i < 4; ++i) { fb_h[i] = fa_h[i]; fb_l[i] = fa_l[i]; }
        const bool useA = dA >= 0, useB = ks > mb0;
        if (useA) {
            const uint4 h4 = Fs[(dA * 2 + 0) * 32 + lane], l4 = Fs[(dA * 2 + 1) * 32 + lane];
            fa_h[0] = h4.x; fa_h[1] = h4.y; fa_h[2] = h4.z; fa_h[3] = h4.w;
            fa_l[0] = l4.x; fa_l[1] = l4.y; fa_l[2] = l4.z; fa_l[3] = l4.w;
        }
        const int e = 16 * ks + b_row;
        const int sw = (e >> 1) & 3;
#pragma unroll
        for (int np = 0; np < 2; ++np) {
            if (2 * np >= nblk) break;
            unsigned bh[4], bl[4];
            const size_t off = (size_t)e * 64 + 16 * ((2 * np + b_chunk) ^ sw);
            ldsm_x4_trans(bh, Xh + off);
            ldsm_x4_trans(bl, Xl + off);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int nb = 2 * np + h;
                if (useA) {
                    mma_gram_k16(acc[0][nb], fa_h, bh[2 * h], bh[2 * h + 1]);
                    mma_gram_k16(acc[0][nb], fa_h, bl[2 * h], bl[2 * h + 1]);
                    mma_gram_k16(acc[0][nb], fa_l, bh[2 * h], bh[2 * h + 1]);
                }
                if (useB) {
                    mma_gram_k16(acc[1][nb], fb_h, bh[2 * h], bh[2 * h + 1]);
                    mma_gram_k16(acc[1][nb], fb_h, bl[2 * h], bl[2 * h + 1]);
                    mma_gram_k16(acc[1][nb], fb_l, bh[2 * h], bh[2 * h + 1]);
                }
            }
        }
    }
    // ---- out: row a of block mb -> time 2 (u0 + 16 mb + a) + pi, columns = microphones ----
    const int g = lane >> 2, tq = lane & 3;
    float *qc = q + b * T64 * M;
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int nb = 0; nb < 4; ++nb)
#pragma unroll
            for (int hr = 0; hr < 2; ++hr) {
                const long long t = 2ll * (u0 + 16 * (mb0 + i) + g + 8 * hr) + pi;
                const int m = m0 + 8 * nb + 2 * tq;
                if (t < T) {
                    if (m < M) qc[t * M + m] = acc[i][nb][2 * hr] * unscale;
                    if (m + 1 < M) qc[t * M + m + 1] = acc[i][nb][2 * hr + 1] * unscale;
                }
            }
}

// part[slab][b][i][j] (upper triangle) -> gram[b][i][j], both halves.  A block owns 32 consecutive elements; its eight
// warps add up interleaved slab groups (coalesced 256-byte rows of `part`), the eight partial sums are added in group
// order: a fixed order, so the result does not depend on scheduling.
static __global__ void __launch_bounds__(256)
k_gram_reduce(const double *__restrict__ part, double *__restrict__ gram, int C2, long long B, int nslab) {
    __shared__ double red[8][32];
    const int ex = threadIdx.x & 31, sg = threadIdx.x >> 5;
    const long long e = (long long)blockIdx.x * 32 + ex;
    const bool in = e < B * C2 * C2;
    const int j = (int)(e % C2), i = (int)((e / C2) % C2);
    const long long b = e / ((long long)C2 * C2);
    double acc = 0.0;
    if (in && i <= j)
        for (int s = sg; s < nslab; s += 8) acc += part[((long long)s * B + b) * C2 * C2 + i * C2 + j];
    red[sg][ex] = acc;
    __syncthreads();
    if (sg == 0 && in && i <= j) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += red[k][ex];
        gram[e] = t;
        gram[(b * C2 + j) * C2 + i] = t;
    }
}

// ---------------------------------------------------------------------------
// S4b: power[b][g] = w_g^T C_b w_g / T (float64), doa[b] = first argmax.
// One block per clip; dynamic smem: C2*C2 doubles (kSmemGram) + reduction scratch.  Without kSmemGram the Gram rows are
// read from global memory (C2 > 168: C2^2 doubles exceed the shared memory of a block; all threads read the same
// element, so each load is one broadcast from L1 / L2).
// rows_b (nullable, stream batches): clip b averages over rows_b[b] samples instead of 1/inv_T, and a clip with no
// rows is not written.
// ---------------------------------------------------------------------------
template <bool kSmemGram>
static __global__ void __launch_bounds__(256)
k_power_argmax(const double *__restrict__ gram, const double *__restrict__ Wd, float *__restrict__ power,
               int32_t *__restrict__ doa, int C2, int G, double inv_T, int nchunk, double *__restrict__ chunk_v,
               int *__restrict__ chunk_i, const int32_t *__restrict__ rows_b = nullptr) {
    extern __shared__ __align__(16) double sm_d[];
    const double *Cs = kSmemGram ? sm_d : gram + blockIdx.x * (long long)C2 * C2;
    __shared__ double red_v[256];
    __shared__ int red_i[256];
    const long long b = blockIdx.x;
    if (rows_b) {                            // (uniform across the block: before any barrier)
        if (rows_b[b] == 0) return;
        inv_T = 1.0 / (double)rows_b[b];
    }
    // few clips and a wide array (BASELINE config 5): blockIdx.y takes a slice of the DoA grid, k_argmax_chunks finishes
    const int gper = (G + nchunk - 1) / nchunk;
    const int g_lo = blockIdx.y * gper, g_hi = min(G, g_lo + gper);
    if (kSmemGram) {
        for (int e = threadIdx.x; e < C2 * C2; e += blockDim.x) sm_d[e] = gram[b * C2 * C2 + e];
        __syncthreads();
    }
    double best = -1.0; int besti = 0x7fffffff;
    for (int g = g_lo + threadIdx.x; g < g_hi; g += blockDim.x) {
        double acc = 0.0;
        for (int i = 0; i < C2; ++i) {
            double r = 0.0;
            for (int j = 0; j < C2; ++j) r = fma(Cs[i * C2 + j], Wd[(long long)j * G + g], r);
            acc = fma(Wd[(long long)i * G + g], r, acc);
        }
        acc *= inv_T;
        if (power) power[b * G + g] = (float)acc;
        if (acc > best) { best = acc; besti = g; }  // ascending g: first maximum kept
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
    if (threadIdx.x == 0) {
        if (nchunk == 1) { if (doa) doa[b] = red_i[0]; }
        else { chunk_v[b * nchunk + blockIdx.y] = red_v[0]; chunk_i[b * nchunk + blockIdx.y] = red_i[0]; }
    }
}
// The same for WIDE arrays (config 5: C2 = 128, G = 512, a handful of clips): one thread per DoA would leave 32 threads
// of a CTA running 16 384 dependent float64 FMAs each (0.5 ms).  Here a warp owns one slice of the Gram rows for 32
// DoAs (lane = DoA, 4 rows in flight = 4 independent sums), the steering weights of the 32 DoAs sit in shared memory,
// and the kPwSlices partial sums of a DoA are added in slice order (a fixed order: deterministic).
constexpr int kPwSlices = 8;
static __global__ void __launch_bounds__(32 * kPwSlices)
k_power_wide(const double *__restrict__ gram, const double *__restrict__ Wd, float *__restrict__ power,
             int32_t *__restrict__ doa, int C2, int G, double inv_T, int nchunk, double *__restrict__ chunk_v,
             int *__restrict__ chunk_i) {
    extern __shared__ __align__(16) double sm_d[];
    double *Cs = sm_d;                       // [C2][C2]
    double *Ws = Cs + (size_t)C2 * C2;       // [C2][32]
    double *Ps = Ws + (size_t)C2 * 32;       // [kPwSlices][32]
    const long long b = blockIdx.x;
    const int gper = (((G + nchunk - 1) / nchunk) + 31) & ~31;
    const int g_lo = blockIdx.y * gper, g_hi = min(G, g_lo + gper);
    const int gl = threadIdx.x & 31, sl = threadIdx.x >> 5;
    const int rows = (C2 + kPwSlices - 1) / kPwSlices;
    const int i0 = min(C2, sl * rows), i1 = min(C2, i0 + rows);
    for (int e = threadIdx.x; e < C2 * C2; e += blockDim.x) Cs[e] = gram[b * C2 * C2 + e];
    double best = -1.0; int besti = 0x7fffffff;
    for (int g0 = g_lo; g0 < g_hi; g0 += 32) {
        __syncthreads();                     // Cs loaded; the previous pass is done with Ws / Ps
        for (int e = threadIdx.x; e < C2 * 32; e += blockDim.x) {
            const int gg = g0 + (e & 31);
            Ws[e] = gg < g_hi ? Wd[(long long)(e >> 5) * G + gg] : 0.0;
        }
        __syncthreads();
        double part = 0.0;
        int i = i0;
        for (; i + 4 <= i1; i += 4) {
            const double *c0 = Cs + (size_t)i * C2;
            double r0 = 0.0, r1 = 0.0, r2 = 0.0, r3 = 0.0;
            for (int j = 0; j < C2; ++j) {
                const double w = Ws[j * 32 + gl];
                r0 = fma(c0[j], w, r0);
                r1 = fma(c0[C2 + j], w, r1);
                r2 = fma(c0[2 * C2 + j], w, r2);
                r3 = fma(c0[3 * C2 + j], w, r3);
            }
            part = fma(Ws[i * 32 + gl], r0, part);
            part = fma(Ws[(i + 1) * 32 + gl], r1, part);
            part = fma(Ws[(i + 2) * 32 + gl], r2, part);
            part = fma(Ws[(i + 3) * 32 + gl], r3, part);
        }
        for (; i < i1; ++i) {
            const double *c0 = Cs + (size_t)i * C2;
            double r = 0.0;
            for (int j = 0; j < C2; ++j) r = fma(c0[j], Ws[j * 32 + gl], r);
            part = fma(Ws[i * 32 + gl], r, part);
        }
        Ps[sl * 32 + gl] = part;
        __syncthreads();
        if (sl == 0 && g0 + gl < g_hi) {
            double acc = 0.0;
#pragma unroll
            for (int s = 0; s < kPwSlices; ++s) acc += Ps[s * 32 + gl];
            acc *= inv_T;
            if (power) power[b * G + g0 + gl] = (float)acc;
            if (acc > best) { best = acc; besti = g0 + gl; }     // ascending g per lane: first maximum kept
        }
    }
    if (sl == 0) {
        // first maximum over the 32 lanes: larger value wins, equal values keep the lower index
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) {
            const double ov = __shfl_down_sync(0xffffffffu, best, s);
            const int oi = __shfl_down_sync(0xffffffffu, besti, s);
            if (ov > best || (ov == best && oi < besti)) { best = ov; besti = oi; }
        }
        if (gl == 0) {
            if (nchunk == 1) { if (doa) doa[b] = besti; }
            else { chunk_v[b * nchunk + blockIdx.y] = best; chunk_i[b * nchunk + blockIdx.y] = besti; }
        }
    }
}
// first maximum over the DoA slices of k_power_argmax (ascending slices: a later slice only wins with a larger value)
static __global__ void __launch_bounds__(32)
k_argmax_chunks(const double *__restrict__ chunk_v, const int *__restrict__ chunk_i, int32_t *__restrict__ doa,
                long long B, int nchunk) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double best = -1.0; int besti = 0x7fffffff;
    for (int c = 0; c < nchunk; ++c) {
        const double v = chunk_v[b * nchunk + c]; const int i = chunk_i[b * nchunk + c];
        if (v > best || (v == best && i < besti)) { best = v; besti = i; }
    }
    doa[b] = besti;
}

// ---------------------------------------------------------------------------
// S5: dense beamformed signal  y[b][t][g] = sum_c vmem[b][t][c] * W[c][g]
//     (the value apply_to_signal returns, snn_beamformer.py:368); one thread per
//     DoA neuron looping over a slab of time steps, weights held in registers
//     when C2 <= 16.
// ---------------------------------------------------------------------------
template <int C2T>
__global__ void __launch_bounds__(128)
k_dense(const float *__restrict__ vmem, const float *__restrict__ W, float *__restrict__ y,
        int C2, int G, long long T, int slab) {
    const long long b = blockIdx.z;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const long long t0 = (long long)blockIdx.y * slab;
    const long long t1 = min(T, t0 + slab);
    const bool live = g < G;
    const float *v = vmem + b * T * C2;
    float *yo = y + b * T * G + g;
    if (C2T > 0) {
        float wr[C2T > 0 ? C2T : 1];
#pragma unroll
        for (int c = 0; c < C2T; ++c) wr[c] = (live && c < C2) ? W[(long long)c * G + g] : 0.f;
        for (long long t = t0; t < t1; ++t) {
            float acc = 0.f;
#pragma unroll
            for (int c = 0; c < C2T; ++c)
                if (c < C2) acc = fmaf(__ldg(v + t * C2 + c), wr[c], acc);
            if (live) yo[t * G] = acc;
        }
    } else {
        for (long long t = t0; t < t1; ++t) {
            float acc = 0.f;
            for (int c = 0; c < C2; ++c)
                acc = fmaf(__ldg(v + t * C2 + c), live ? __ldg(W + (long long)c * G + g) : 0.f, acc);
            if (live) yo[t * G] = acc;
        }
    }
}

// ---------------------------------------------------------------------------
// Beamformer.apply_to_signal tail (micloc/beamformer.py:290):
//   y[b][t][g] = sum_m (zr + i zi)[t][m] * conj(bf[m][g]),  z = [T][2M] (real | imag)
// ---------------------------------------------------------------------------
static __global__ void __launch_bounds__(128)
k_cproject(const float *__restrict__ z, const float *__restrict__ bfr, const float *__restrict__ bfi,
           float2 *__restrict__ y, int M, int G, long long T, int slab) {
    const long long b = blockIdx.z;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    const long long t0 = (long long)blockIdx.y * slab;
    const long long t1 = min(T, t0 + slab);
    const float *zz = z + b * T * 2 * M;
    for (long long t = t0; t < t1; ++t) {
        float ar = 0.f, ai = 0.f;
        for (int m = 0; m < M; ++m) {
            const float sr = __ldg(zz + t * 2 * M + m), si = __ldg(zz + t * 2 * M + M + m);
            const float wr = __ldg(bfr + (long long)m * G + g), wi = -__ldg(bfi + (long long)m * G + g);
            ar = fmaf(sr, wr, fmaf(-si, wi, ar));
            ai = fmaf(sr, wi, fmaf(si, wr, ai));
        }
        y[(b * T + t) * G + g] = make_float2(ar, ai);
    }
}

// power[b][g] = mean_t |y|^2 in float64 + argmax; one block per (clip), thread per g
static __global__ void __launch_bounds__(256)
k_cpower_argmax(const float2 *__restrict__ y, float *__restrict__ power, int32_t *__restrict__ doa,
                int G, long long T) {
    __shared__ double red_v[256];
    __shared__ int red_i[256];
    const long long b = blockIdx.x;
    double best = -1.0; int besti = 0x7fffffff;
    for (int g = threadIdx.x; g < G; g += blockDim.x) {
        double acc = 0.0;
        for (long long t = 0; t < T; ++t) {
            const float2 v = y[(b * T + t) * G + g];
            acc += (double)v.x * v.x + (double)v.y * v.y;
        }
        acc /= (double)T;
        if (power) power[b * G + g] = (float)acc;
        if (acc > best) { best = acc; besti = g; }
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

}  // namespace micloc
