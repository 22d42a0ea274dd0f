// micloc_fused.cu -- the fused hot-path kernel: raw audio in, spikes + per-DoA
// power + DoA index out; nothing else touches HBM.
//
// Reference sites: micloc/snn_beamformer.py:283-370 and the callers' power/argmax
// paper_plots/target_snn_localization.py:462-464.
//
// A clip-pair GROUP of eight warps owns kSlots = 2 clips at a time and walks them in time tiles
// of kTile = 64 samples.  The warps are specialised BY FUNCTION (every role serves both clips with
// all its lanes, so that the serial depth of each role per tile is short) and run as a software
// pipeline, one named barrier per tile (iteration k):
//
//   FIR warps x4 tile k+1   audio (HBM) -> mic-major ring in shared memory (two warps per clip, 32
//                           samples each)
//                tile k     STHT quadrature FIR, first half of the taps: every lane owns 16
//                           consecutive outputs of one microphone and walks 120 of the 240 non-zero
//                           Hilbert taps in blocks of 8 with a sliding register window; the
//                           multiply-adds are packed FFMA2 (fma.rn.f32x2)
//                tile k-1   second warp of the clip: continues the SAME running sums (handed over
//                           in shared memory) through the other 120 taps: the summation order is
//                           that of one warp walking all taps
//   band-pass    tile k-2   one lane per (clip, channel): SOS band-pass recurrence, running sum,
//                           sign bit masks of every 32-sample segment -> shared memory (exact zeros:
//                           the segment is redone sample by sample)
//   RZCC         tile k-3   one lane per (clip, channel): the masks are turned into RZCC
//                           candidates and resolved (find_peaks distance rule) into a bit-packed
//                           spike ring
//   neuron       tile k-d   (d = the latency of the exact find_peaks decision) one lane per (clip,
//                           channel): alpha-kernel neuron recurrences driven by the final spike
//                           bits -> membrane tiles (fp16 hi / lo pairs) + int8 spike tile in shared memory
//   Gram         tile k-d-1 C += V V^T of the membrane tile on the tensor cores (ldmatrix + fp16
//                           m16n8k16 MMAs on the hi / lo split), int8 spike raster of the tile -> HBM
//   clip end                power[g] = w_g^T C w_g / T (float64), DoA = first argmax.
//
// One CTA of sixteen warps per SM holds two such groups (own barrier, own shared memory, own clip pairs): one
// FIR warp of each group per SM sub-partition.  What bounds the kernel is the issue port of the sub-partitions:
// an FFMA2 with three register operands issues every ~2.6 cycles, and every instruction of a serial role displaces
// FIR work (a scheduler micro-benchmark, DESIGN.md 4.1).  micloc_fused_tc.cu (the default) runs the FIR on the tensor cores instead.
#include <cstdlib>

#include "micloc_fused_common.cuh"

namespace micloc {

constexpr int kRows = 8;       // most microphones per clip the lane maps cover
constexpr int kRingWords = 32; // spike-bit ring: 32 words of 32 samples per channel and polarity
constexpr int kFirWarps = 4;

struct FusedGeom {
    int ring_x;      // audio ring length in samples (multiple of 32)
    int pitch_x;     // floats per ring row; pitch_x / 4 is odd (conflict-free LDS.128 across microphones)
    int shift;       // ring coordinate of sample t is (t + shift) mod ring_x
    int nblk;        // FIR tap blocks of 8 (multiple of 6: two halves walked in groups of three)
    int dtile;       // the neuron warp runs dtile tiles behind the pipeline step (RZCC decision latency)
    int tiles_is;    // tiles whose in-phase input comes from the clip tail (t < K/2)
    int perm;        // serial roles of group 1 on sub-partitions 0..3, two bits each (see k_fused)
    int off_x, off_q, off_vm, off_is, off_cs, off_seg, off_clus, off_bits, off_stage, off_qa;   // byte offsets in dynamic smem
    int smem_bytes;
};

struct Chunk { unsigned long long p[8]; };   // 16 consecutive samples as 8 float pairs

__device__ __forceinline__ void load_chunk(Chunk &c, const float *row, int coord) {
    const ulonglong2 *src = reinterpret_cast<const ulonglong2 *>(row + coord);
#pragma unroll
    for (int v = 0; v < 4; ++v) {
        const ulonglong2 u = src[v];
        c.p[2 * v] = u.x; c.p[2 * v + 1] = u.y;
    }
}

// 8 taps x 16 outputs: acc[ip] += g[jj] * W[ip + 7 - jj], W = lo pairs 0..7 | hi pairs 0..6
struct Taps8 { float4 a, b; };
__device__ __forceinline__ void load_taps(Taps8 &t, const float *__restrict__ taps8) {
    t.a = *reinterpret_cast<const float4 *>(taps8);
    t.b = *reinterpret_cast<const float4 *>(taps8 + 4);
}
// Written window-major (the window pair is shared by consecutive multiply-adds).  ptxas schedules the 64 FFMA2 of a
// block in its own order whatever the source says (`volatile` does not pin it); the sequence it emits for this
// source measured fastest of five source forms (FIR warps alone 290 k clips/s; tap-major 278 k, accumulator-major
// 283 k, older chunk first 285-291 k; whole kernel 171.8-174.1 k).  A scheduler micro-benchmark of the FIR's operand
// patterns measured between 2.4 and 5.2 cycles per FFMA2 and sub-partition depending on the sequence.
__device__ __forceinline__ void ffma2_ordered(unsigned long long &acc, unsigned long long w, unsigned long long g2) {
    asm volatile("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(w), "l"(g2));
}
__device__ __forceinline__ void fir_block(unsigned long long (&acc)[8], const Chunk &lo, const Chunk &hi,
                                          const Taps8 &t) {
    const float g[8] = {t.a.x, t.a.y, t.a.z, t.a.w, t.b.x, t.b.y, t.b.z, t.b.w};
    unsigned long long g2[8];
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) g2[jj] = pack2(g[jj], g[jj]);
    // newest window pair first: every accumulator still meets its taps in ascending order (lfilter's summation order)
#pragma unroll
    for (int w = 14; w >= 0; --w) {
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
            const int ip = w - 7 + jj;
            if (ip >= 0 && ip < 8) ffma2_ordered(acc[ip], w < 8 ? lo.p[w] : hi.p[w - 8], g2[jj]);
        }
    }
}

struct FusedSmem {
    float *taps, *xs, *qs, *qa, *is_s, *cs;
    __half *vms;            // [2: hi, lo][2 tiles][kVmRows][kVmPitch] membrane tiles (x 2^14, fp16 split), channel-major
    unsigned int *seg;      // [2 tiles][kTile/kSeg][3: neg mask, zero mask, carry][32 lanes]: band-pass -> RZCC hand-over
    int *clus;
    unsigned int *bits;     // [2 polarities][kRingWords][32 lanes]
    int8_t *stage;          // [2 tiles][kSlots][kTile][C2]
    double *gram;           // [kSlots][16][16], clip epilogue only (reuses the audio rings)
    unsigned int *dbg;      // sm_slots (debug counters behind the first 256 entries)
    int bar_id;             // named barrier of this clip-pair group
    int bar_threads;        // threads meeting at it
    int k_first;            // first pipeline step of the serial roles (-1 here)
    int rec;                // index of this group's debug record (MICLOC_ROLE_TIMING builds)
};

// ======= FIR warp (one per clip slot): audio tile k+1 -> ring, STHT FIR of tile k =======

template <typename IN_T, int MM>
__device__ __forceinline__ void fir_role(const FusedSmem &sm, const ChainParams &p, const FusedGeom &g,
                                         const IN_T *__restrict__ audio, long long clip, bool clip_ok, long long T64,
                                         int slot, int half, int lane, int NT, int k_last) {
    const int M = MM ? MM : p.M;
    const int T = (int)T64;
    const int f_chunk = lane >> 3, f_mic = lane & 7;     // FIR lanes: lane = chunk * 8 + mic
    const bool work = clip_ok && f_mic < M;
    const float *row = sm.xs + (slot * M + f_mic) * g.pitch_x;
    const IN_T *src = audio + (clip_ok ? clip : 0) * T64 * M;
    float *rows_w = sm.xs + slot * M * g.pitch_x;
    const int nb2 = g.nblk / 2;                          // tap blocks of this warp: [half * nb2, (half + 1) * nb2)
    // this lane's sample of the tile being filled (tile 0 at k = -1): the warp fills samples [32*half, 32*half + 32)
    int fill_t = lane + 32 * half;
    const IN_T *fill_src = src + (fill_t < T ? fill_t * M : 0);
    int fill_c = (fill_t + g.shift) % g.ring_x;
    // ring coordinate of this lane's window of the warp's first tap block at tile 0, kept incrementally
    int c0 = ((16 * f_chunk - p.tap_first - 14 + g.shift - 16 * half * nb2) % g.ring_x + g.ring_x) % g.ring_x;
    ROLE_TIMER_DECL;

    for (int k = -1; k <= k_last; ++k) {
        // (a) audio tile k+1 -> mic-major ring: every lane moves one whole frame (all microphones of one
        //     sample); the loads are issued here and stored after the FIR so that their latency is hidden
        const int kf = k + 1;
        const bool filling = kf < NT && clip_ok;
        float v[kRows];
        if (filling) {
            const bool ok = fill_t < T;
#pragma unroll
            for (int m = 0; m < kRows; ++m) v[m] = (ok && m < M) ? to_f32<IN_T>(fill_src[m]) : 0.f;
        }
        // (b) this warp's half of the taps of the STHT quadrature FIR: half 0 starts the running sums of tile k,
        //     half 1 picks up those of tile k - 1 and finishes them
        const int kk = k - half;
        if (kk >= 0 && kk < NT) {
            if (work) {
                unsigned long long acc[8];
                float *part = sm.qa + (((kk & 1) * kSlots + slot) * M + f_mic) * kQPitch + 16 * f_chunk;
                if (half == 0) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) acc[i] = 0ull;
                } else {
#pragma unroll
                    for (int v4 = 0; v4 < 4; ++v4) {
                        const float4 o = reinterpret_cast<const float4 *>(part)[v4];
                        acc[2 * v4] = pack2(o.x, o.y);
                        acc[2 * v4 + 1] = pack2(o.z, o.w);
                    }
                }
                Chunk A, Bq, Cq;
                { int ch = c0 + 16; if (ch >= g.ring_x) ch -= g.ring_x; load_chunk(Bq, row, ch); }
                load_chunk(A, row, c0);
                int cn = c0 - 16; if (cn < 0) cn += g.ring_x;
                // window chunks and taps are fetched one block ahead of their use
                const float *tp = sm.taps + 8 * half * nb2;
                Taps8 t0, t1;
                load_taps(t0, tp);
#pragma unroll 1
                for (int jb = 0; jb < nb2; jb += 3) {
                    load_chunk(Cq, row, cn); cn -= 16; if (cn < 0) cn += g.ring_x;
                    load_taps(t1, tp + 8);
                    fir_block(acc, A, Bq, t0);
                    load_chunk(Bq, row, cn); cn -= 16; if (cn < 0) cn += g.ring_x;
                    load_taps(t0, tp + 16);
                    fir_block(acc, Cq, A, t1);
                    load_chunk(A, row, cn); cn -= 16; if (cn < 0) cn += g.ring_x;
                    load_taps(t1, tp + 24);             // first block of the next round (zero padding behind the last)
                    fir_block(acc, Bq, Cq, t0);
                    t0 = t1;
                    tp += 24;
                }
                float *dst = half == 0 ? part : sm.qs + (((kk & 1) * kSlots + slot) * M + f_mic) * kQPitch + 16 * f_chunk;
#pragma unroll
                for (int v4 = 0; v4 < 4; ++v4) {
                    float4 o;
                    unpack2(acc[2 * v4], o.x, o.y);
                    unpack2(acc[2 * v4 + 1], o.z, o.w);
                    reinterpret_cast<float4 *>(dst)[v4] = o;
                }
            }
            c0 += kTile; if (c0 >= g.ring_x) c0 -= g.ring_x;
        }
        // (the zero-padded first tap block of tile k reads one sample into tile k+1, times a zero tap: the window reads of
        //  every lane come before the stores below -- compute-sanitizer racecheck)
        __syncwarp();
        if (filling) {
#pragma unroll
            for (int m = 0; m < kRows; ++m)
                if (m < M) rows_w[m * g.pitch_x + fill_c] = v[m];
            // next tile: time, source frame and ring coordinate of this lane's sample
            fill_t += kTile;
            fill_src += (fill_t < T ? kTile * M : 0);
            fill_c += kTile; if (fill_c >= g.ring_x) fill_c -= g.ring_x;
        }
        ROLE_BARRIER();
    }
    ROLE_TIMER_FLUSH(2 * slot + half);
}

// ============ band-pass warp: SOS cascade + running sum + sign / zero masks, lane = slot*16 + channel ============
template <typename IN_T, int MM>
__device__ __forceinline__ void bandpass_role(const FusedSmem &sm, const ChainParams &p, const FusedGeom &g,
                                              const IN_T *__restrict__ audio, long long clip0, long long B,
                                              long long T64, int lane, int k_last) {
    const int M = MM ? MM : p.M, C2 = 2 * M;
    const int T = (int)T64;
    const int c_slot = lane >> 4, c_ch = lane & 15;
    const bool slot_ok = clip0 + c_slot < B;
    const bool c_valid = c_ch < C2 && slot_ok;
    const bool c_inphase = c_ch < M;
    const IN_T *clip_audio = audio + (slot_ok ? clip0 + c_slot : clip0) * T64 * M;
    Sos2 sos;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        sos.b0[k] = p.sos[k][0]; sos.b1[k] = p.sos[k][1]; sos.b2[k] = p.sos[k][2];
        sos.a1[k] = p.sos[k][3]; sos.a2[k] = p.sos[k][4];
    }
    BiquadState bq; biquad_reset(bq);
    float csum = 0.f;
    // ring coordinate of the in-phase sample x[ts - K/2] of the next segment (warp-uniform, kept incrementally)
    int cin_u = ((g.shift - p.half) % g.ring_x + g.ring_x) % g.ring_x;
    ROLE_TIMER_DECL;

    for (int k = -1; k <= k_last; ++k) {
        const int kc = k - 2;
        const int t0 = kc * kTile;
        if (kc >= 0 && t0 < T) {
            const bool from_is = kc < g.tiles_is;
            if (from_is) {
                // in-phase input of the first K/2 samples is the clip's tail (np.roll, snn_beamformer.py:325)
                if (slot_ok) {
                    float *dsti = sm.is_s + c_slot * kTile * M;
                    for (int e = c_ch; e < kTile * M; e += 16) {
                        const int t = t0 + e / M;
                        float v = 0.f;
                        if (t < T) {
                            int src = (t - p.half) % T;
                            if (src < 0) src += T;
                            v = to_f32<IN_T>(clip_audio[(long long)src * M + (e % M)]);
                        }
                        dsti[e] = v;
                    }
                }
                __syncwarp();
            }
#pragma unroll 1
            for (int sg = 0; sg < kSegsPerTile; ++sg) {
                const int ts = t0 + sg * kSeg;            // first sample of this segment
                float *cs = sm.cs + ((kc & 1) * kSegsPerTile + sg) * kSeg * 32 + lane;
                unsigned int *sgm = sm.seg + ((kc & 1) * kSegsPerTile + sg) * 3 * 32 + lane;
                const int cin = cin_u;                    // ring coordinate of x[ts - K/2]
                cin_u += kSeg; if (cin_u >= g.ring_x) cin_u -= g.ring_x;
                if (ts >= T || !c_valid) continue;
                const float *xp;
                int stride = 1, wrap_at = kSeg;
                if (!c_inphase) {
                    xp = sm.qs + (((kc & 1) * kSlots + c_slot) * M + (c_ch - M)) * kQPitch + sg * kSeg;
                } else if (from_is) {
                    xp = sm.is_s + c_slot * kTile * M + sg * kSeg * M + c_ch;
                    stride = M;
                } else {
                    xp = sm.xs + (c_slot * M + c_ch) * g.pitch_x + cin;
                    wrap_at = g.ring_x - cin;
                }
                // (warp-uniform) no lane wraps around the audio ring inside this segment
                const bool fast = !from_is && ts + kSeg <= T && cin + kSeg <= g.ring_x;
                const float carry = csum;
                unsigned int neg = 0u, zero = 0u;
                // sample by sample with explicit sign / zero masks (ragged segments, ring wrap, clip-tail input, exact zeros)
                auto slow_segment = [&](int nvalid) {
                    const float *xq = xp;
#pragma unroll 1
                    for (int i = 0; i < nvalid; ++i) {
                        if (i == wrap_at) xq -= g.ring_x;
                        const float z = biquad2_step(sos, bq, xq[i * stride]);
                        zero |= (rzcc_flat(z, csum) ? 1u : 0u) << (31 - i);      // (sum before this sample)
                        csum += z;
                        cs[i * 32] = csum;
                        neg |= (__float_as_uint(z) >> 31) << (31 - i);
                    }
                };
                if (fast) {
                    const BiquadState bq0 = bq;
                    float zmin = 1.f;                   // smallest |z| of the segment: exact zeros are rare (silence)
                    float xn[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) xn[i] = xp[i];
#pragma unroll 1
                    for (int o = 0; o < kSeg / 8; ++o) {
                        float xc[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) xc[i] = xn[i];
                        if (o + 1 < kSeg / 8) {         // inputs of the next group: their latency hides behind this one
#pragma unroll
                            for (int i = 0; i < 8; ++i) xn[i] = xp[8 * (o + 1) + i];
                        }
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const float z = biquad2_step(sos, bq, xc[i]);
                            csum += z;
                            cs[(8 * o + i) * 32] = csum;
                            neg = __funnelshift_l(__float_as_uint(z), neg, 1);
                            zmin = fminf(zmin, fabsf(z));
                        }
                    }
                    // a sample that does not move the reference's float64 running sum (exact zeros, the decaying tail in
                    // digital silence) counts as zero: redo this lane's segment for its zero mask (same arithmetic)
                    if (zmin <= kFlatTrigger * fmaxf(fabsf(carry), fabsf(csum))) {
                        bq = bq0; csum = carry; neg = 0u;
                        slow_segment(kSeg);
                    }
                } else {
                    slow_segment(T - ts < kSeg ? T - ts : kSeg);
                }
                sgm[0] = neg; sgm[32] = zero; sgm[64] = __float_as_uint(carry);
            }
        }
        ROLE_BARRIER();
    }
    ROLE_TIMER_FLUSH(kRoleBandpass);
}

// GROUPS = 1: a CTA is one clip-pair group of eight warps, two CTAs per SM, FIR roles placed per SM
//             sub-partition at run time (hardware warp slots of a second CTA are not known in advance).
// GROUPS = 2: ONE CTA of sixteen warps per SM holding two independent clip-pair groups (own named barrier,
//             own shared-memory region, own clip pairs).  The warp slots are then known: warps 0..7 are the
//             FIR warps (two per sub-partition, one of each group), warps 8..15 the serial roles.  The
//             scheduler of a sub-partition prefers the eligible warp with the highest warp id, so the
//             latency-bound serial roles (a chain of dependent instructions per sample) always win their few
//             issue slots and run at their dependency-chain pace, while the FIR warps fill every remaining
//             FMA-pipe cycle; with the FIR warps in front the serial roles starve behind a stream of
//             independent FFMA2s and FIR and serial phases alternate instead of overlapping.
template <typename IN_T, int MM, int GROUPS>
__global__ void __launch_bounds__(kThreads * GROUPS, GROUPS == 1 ? 2 : 1)
k_fused(const IN_T *__restrict__ audio, const float *__restrict__ taps, const double *__restrict__ Wd,
        int8_t *__restrict__ spikes, float *__restrict__ power, int32_t *__restrict__ doa,
        int32_t *__restrict__ flags, unsigned int *__restrict__ sm_slots,
        const __grid_constant__ ChainParams p, const __grid_constant__ FusedGeom g, long long B, long long T) {
    extern __shared__ __align__(16) unsigned char smem_all[];
    __shared__ int s_smsp[kWarps * GROUPS], s_role[kWarps * GROUPS];
    __shared__ long long s_pair[GROUPS];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int M = MM ? MM : p.M, C2 = 2 * M;
#ifdef MICLOC_ROLE_TIMING
    long long dbg_c0 = rt_clock();
    unsigned long long dbg_g0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_g0));
#endif

    // ---- which group and role this warp serves ----
    int group = 0, role;
    if (GROUPS == 1) {
        // A hardware warp slot w belongs to SM sub-partition w % 4, and the FMA pipe of a sub-partition is
        // what the FIR warps compete for: the four FIR roles go to the warps of this CTA whose sub-partition
        // holds the fewest FIR warps of the CTAs already resident on this SM (counters per SM in
        // sm_slots[4*smid + smsp], reset per launch); the other four roles follow in warp order, rotated by
        // two for every second CTA of an SM so that the band-pass / Gram warps (the ones with FMA work)
        // spread out.
        if (lane == 0) {
            unsigned int wid;
            asm volatile("mov.u32 %0, %%warpid;" : "=r"(wid));
            s_smsp[warp] = (int)(wid & 3u);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned int smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            unsigned int *fir_cnt = sm_slots + 4 * (smid & 255u);
            const unsigned int arrival = atomicAdd(sm_slots + kSlotPair + 1 + (smid & 255u) % 254u, 1u);
            bool taken[kWarps];
            for (int w = 0; w < kWarps; ++w) { taken[w] = false; s_role[w] = -1; }
            for (int r = 0; r < kFirWarps; ++r) {
                int best = -1; unsigned int bestc = 0xffffffffu;
                for (int w = 0; w < kWarps; ++w) {
                    if (taken[w]) continue;
                    const unsigned int c = *(volatile unsigned int *)(fir_cnt + s_smsp[w]);
                    if (c < bestc) { bestc = c; best = w; }
                }
                taken[best] = true;
                s_role[best] = r;
                atomicAdd(fir_cnt + s_smsp[best], 1u);
            }
            int next = (int)(2u * (arrival & 1u));
            for (int w = 0; w < kWarps; ++w)
                if (!taken[w]) { s_role[w] = kFirWarps + (next & 3); ++next; }
        }
        __syncthreads();
        role = s_role[warp];
    } else {
        // warps 0..3: FIR of group 0, 4..7: FIR of group 1 (one per sub-partition each); warps 8..11 / 12..15:
        // band-pass, RZCC, neuron, Gram of group 0 / 1; group 1's order (g.perm) decides which roles share a
        // sub-partition (band-pass + Gram, RZCC + neuron)
        if (warp < 2 * kFirWarps) {
            group = warp >> 2;
            role = warp & 3;
        } else {
            group = (warp - 2 * kFirWarps) >> 2;
            role = kFirWarps + (group == 0 ? (warp & 3) : (g.perm >> (2 * (warp & 3))) & 3);
        }
        if (lane == 0) {
            unsigned int wid;
            asm volatile("mov.u32 %0, %%warpid;" : "=r"(wid));
            s_smsp[warp] = (int)(wid & 3u);
            s_role[warp] = role;
        }
    }
    // 0..3: FIR (+ fill) of clip slot role >> 1, tap half role & 1; 4: band-pass; 5: RZCC; 6: neuron; 7: Gram
    const int tid = role * 32 + lane;       // thread index inside the group
    const int bar_id = 1 + group;
    auto group_sync = [&]() { tile_barrier(bar_id); };

    unsigned char *smem_raw = smem_all + (size_t)group * g.smem_bytes;
    FusedSmem sm;
    sm.taps = reinterpret_cast<float *>(smem_raw);
    sm.xs = reinterpret_cast<float *>(smem_raw + g.off_x);       // [kSlots*M][pitch_x]
    sm.qs = reinterpret_cast<float *>(smem_raw + g.off_q);       // [2 tiles][kSlots*M][kQPitch]: finished quadrature tiles
    sm.qa = reinterpret_cast<float *>(smem_raw + g.off_qa);      // [2 tiles][kSlots*M][kQPitch]: running sums after the first tap half
    sm.vms = reinterpret_cast<__half *>(smem_raw + g.off_vm);
    sm.is_s = reinterpret_cast<float *>(smem_raw + g.off_is);    // [kSlots][kTile][M]
    sm.cs = reinterpret_cast<float *>(smem_raw + g.off_cs);      // [2][kSegsPerTile][kSeg][32] running sums
    sm.seg = reinterpret_cast<unsigned int *>(smem_raw + g.off_seg);     // [2][kSegsPerTile][3][32]
    sm.clus = reinterpret_cast<int *>(smem_raw + g.off_clus);    // RZCC cluster buffers, interleaved over 32 lanes
    sm.bits = reinterpret_cast<unsigned int *>(smem_raw + g.off_bits);   // [2][kRingWords][32]
    sm.stage = reinterpret_cast<int8_t *>(smem_raw + g.off_stage);       // [2][kSlots][kTile][C2]
    sm.gram = reinterpret_cast<double *>(smem_raw + g.off_x);    // [kSlots][16][16], clip epilogue only
    sm.dbg = sm_slots;
    sm.bar_id = bar_id;
    sm.bar_threads = kThreads;
    sm.k_first = -1;
    sm.rec = GROUPS * (int)blockIdx.x + group;
    double *red_v = reinterpret_cast<double *>(smem_raw + g.off_cs);     // [kThreads], clip epilogue only (reuses the running sums)
    int *red_i = reinterpret_cast<int *>(smem_raw + g.off_cs + kThreads * sizeof(double));

    for (int i = tid; i < 8 * g.nblk + 8; i += kThreads) sm.taps[i] = i < p.n_taps ? taps[i] : 0.f;

    const int NT = (int)((T + kTile - 1) / kTile);
    const int k_last = NT + g.dtile;    // the Gram warp runs dtile + 1 tiles behind
    const long long npairs = (B + kSlots - 1) / kSlots;

    // Clip pairs are handed out dynamically: co-resident groups do not run at the same speed, so a static
    // split would wait for the slowest one.
    for (;;) {
        group_sync();
        if (tid == 0) s_pair[group] = (long long)atomicAdd(sm_slots + kSlotPair, 1u);
        group_sync();
        const long long pair = s_pair[group];
        if (pair >= npairs) break;
        const long long clip0 = pair * kSlots;
        {   // zero the audio rings: samples before the clip start are zeros (lfilter's zero state)
            float4 *x4 = reinterpret_cast<float4 *>(sm.xs);
            const int n4 = kSlots * M * g.pitch_x / 4;
            for (int i = tid; i < n4; i += kThreads) x4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            // no spikes before the clip start; membrane columns of unused lanes stay zero
            for (int i = tid; i < 2 * kRingWords * 32; i += kThreads) sm.bits[i] = 0u;
            for (int i = tid; i < 2 * 2 * kVmRows * kVmPitch / 2; i += kThreads) reinterpret_cast<unsigned int *>(sm.vms)[i] = 0u;
        }
        group_sync();

        if (role < kFirWarps)
            fir_role<IN_T, MM>(sm, p, g, audio, clip0 + (role >> 1), clip0 + (role >> 1) < B, T, role >> 1, role & 1, lane,
                               NT, k_last);
        else if (role == kRoleBandpass) bandpass_role<IN_T, MM>(sm, p, g, audio, clip0, B, T, lane, k_last);
        else if (role == kRoleRzcc) rzcc_role<FusedSmem, kRingWords>(sm, p, flags, clip0, B, T, M, lane, k_last);
        else if (role == kRoleNeuron) neuron_role<FusedSmem, FusedGeom, kRingWords>(sm, p, g, clip0, B, T, M, lane, k_last);
        else gram_role<FusedSmem, FusedGeom>(sm, g, spikes, clip0, B, T, M, lane, k_last);
        group_sync();
        // ---- clip epilogue: power[g] = w_g^T C w_g / T (float64), DoA = first argmax ----
        // one DoA column per thread and pass: its 2M weights are fetched first (independent loads, one
        // memory latency), then the quadratic form runs from registers and shared memory
        const double inv_T = 1.0 / (double)T;
        for (int s = 0; s < kSlots; ++s) {
            const long long clip = clip0 + s;
            if (clip >= B) break;
            const double *Cd = sm.gram + s * 256;
            double best = -1.0; int besti = 0x7fffffff;
            for (int gg = tid; gg < p.G; gg += kThreads) {
                double w[2 * kRows];
#pragma unroll
                for (int c = 0; c < 2 * kRows; ++c) w[c] = c < C2 ? Wd[(long long)c * p.G + gg] : 0.0;
                double accp = 0.0;
#pragma unroll 2
                for (int r = 0; r < C2; ++r) {
                    double rr = 0.0;
#pragma unroll
                    for (int c = 0; c < 2 * kRows; ++c)
                        if (c < C2) rr = fma(Cd[r * 16 + c], w[c], rr);
                    double wr = 0.0;
#pragma unroll
                    for (int c = 0; c < 2 * kRows; ++c) wr = c == r ? w[c] : wr;
                    accp = fma(wr, rr, accp);
                }
                accp *= inv_T;
                if (power) power[clip * p.G + gg] = (float)accp;
                if (accp > best) { best = accp; besti = gg; }
            }
            red_v[tid] = best; red_i[tid] = besti;
            group_sync();
            for (int st = kThreads / 2; st > 0; st >>= 1) {
                if (tid < st) {
                    const double ov = red_v[tid + st]; const int oi = red_i[tid + st];
                    if (ov > red_v[tid] || (ov == red_v[tid] && oi < red_i[tid])) { red_v[tid] = ov; red_i[tid] = oi; }
                }
                group_sync();
            }
            if (tid == 0 && doa) doa[clip] = red_i[0];
            group_sync();
        }
    }
#ifdef MICLOC_ROLE_TIMING
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        unsigned long long g1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
        unsigned long long *d = reinterpret_cast<unsigned long long *>(sm_slots + kSlotDbg);
        d[16] = (unsigned long long)(rt_clock() - dbg_c0);
        d[17] = g1 - dbg_g0;
    }
    if (tid == 0 && GROUPS * blockIdx.x + group < 512) {
        unsigned long long g1;
        unsigned int smid;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        unsigned long long *d = reinterpret_cast<unsigned long long *>(sm_slots + kSlotCta) + 16 * (GROUPS * blockIdx.x + group);
        unsigned long long map = 0;
        for (int w = 0; w < kWarps * GROUPS; ++w)
            if (GROUPS == 1 || ((w < 2 * kFirWarps ? w >> 2 : (w - 2 * kFirWarps) >> 2) == group)) {
                const int r = s_role[w] & 7;
                map |= (unsigned long long)(r | ((s_smsp[w] & 3) << 3)) << (8 * r);
            }
        d[0] = dbg_g0; d[1] = g1; d[2] = smid; d[3] = map;     // d[4..11]: busy cycles per role
    }
#endif
}

bool fused_supported(const ChainParams &p) {
    return p.tap_stride == 2 && p.M <= kRows && p.nsec == 2 && (p.n_taps % 8) == 0;
}

template <typename IN_T, int MM, int GROUPS>
static int launch_fused_t(const ChainParams &p, const FusedGeom &g, const float *d_taps, const double *d_Wd,
                          const IN_T *audio, long long B, long long T, int8_t *spikes, float *power, int32_t *doa,
                          int32_t *flags, unsigned int *sm_slots, int sm_count, cudaStream_t st) {
    auto kern = k_fused<IN_T, MM, GROUPS>;
    const int smem = GROUPS * g.smem_bytes;
    MICLOC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    // all of the SM's L1/shared array as shared memory: two clip-pair groups of ~100 KB must be resident together
    MICLOC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    int per_sm = 1;
    MICLOC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads * GROUPS, smem));
    if (per_sm > 2 / GROUPS) per_sm = 2 / GROUPS;     // two groups per SM: the role placement balances exactly two
    if (per_sm < 1) return set_error(MICLOC_ERR_UNSUPPORTED, "fused kernel does not fit (smem %d B)", smem);
    long long grid = (long long)sm_count * per_sm;
    const long long npairs = (B + kSlots - 1) / kSlots;
    const long long want = (npairs + GROUPS - 1) / GROUPS;
    if (grid > want) grid = want;
    MICLOC_CUDA(cudaMemsetAsync(sm_slots, 0, kSlotResetWords * sizeof(unsigned int), st));   // FIR placement counters + pair counter restart per launch
    kern<<<(unsigned)grid, kThreads * GROUPS, smem, st>>>(audio, d_taps, d_Wd, spikes, power, doa, flags, sm_slots, p, g, B, T);
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}

int launch_fused(const ChainParams &p, const float *d_taps, const double *d_Wd, const void *audio, int dtype,
                 long long B, long long T, int8_t *spikes, float *power, int32_t *doa, int32_t *flags,
                 unsigned int *sm_slots, int sm_count, cudaStream_t st) {
    // default: the tensor-core kernel (micloc_fused_tc.cu) wherever its geometry applies; this FFMA kernel covers
    // the rest (long STHT kernels that do not fit its rings) and stays selectable with MICLOC_FUSED_FIR=ffma
    {
        const char *e = getenv("MICLOC_FUSED_FIR");
        const bool want_ffma = e && e[0] == 'f';        // "ffma": force this kernel (A/B measurements)
        if (!want_ffma && tc::fused_supported(p)) {
            const int rc = tc::launch_fused(p, d_taps, d_Wd, audio, dtype, B, T, spikes, power, doa, flags, sm_slots, sm_count, st);
            if (rc != MICLOC_ERR_UNSUPPORTED) return rc;
        }
    }
    if (!fused_supported(p))
        return set_error(MICLOC_ERR_UNSUPPORTED,
                         "fused kernel covers Hilbert-type STHT kernels (every other tap zero), a 2-section band-pass "
                         "and up to %d microphones; use the staged path", kRows);
    FusedGeom g{};
    // group 0 runs band-pass, RZCC, neuron, Gram on sub-partitions 0..3; group 1's order decides which roles share one.
    // The reverse order (band-pass + Gram, RZCC + neuron) measured fastest of the three pairings.
    g.perm = 3 | 2 << 2 | 1 << 4 | 0 << 6;
    // FIR tap blocks of 8, two halves walked in groups of three (zero taps appended up to a multiple of 48)
    g.nblk = (p.n_taps / 8 + 5) / 6 * 6;
    const int lookback = p.tap_first + 14 + 16 * (g.nblk - 1);      // oldest sample a tile's FIR windows load
    g.ring_x = ((lookback + 3 * kTile) + 31) / 32 * 32;             // history + the two tiles in the FIR + tile being filled
    g.pitch_x = g.ring_x + 4;
    g.shift = ((p.tap_first + 14) % 16 + 16) % 16;
    // a spike at p is final once the RZCC warp passed p + rzcc_lag(w) - 1; the neuron warp works on
    // tile k - dtile while the RZCC warp has completed tile k - 4
    g.dtile = 4 + (rzcc_lag(p.w) - 1 + kTile - 1) / kTile;
    g.tiles_is = (p.half + kTile - 1) / kTile;
    int off = ((8 * g.nblk + 8) * (int)sizeof(float) + 15) & ~15;
    g.off_x = off; off += kSlots * p.M * g.pitch_x * (int)sizeof(float);
    g.off_q = off; off += 2 * kSlots * p.M * kQPitch * (int)sizeof(float);
    g.off_qa = off; off += 2 * kSlots * p.M * kQPitch * (int)sizeof(float);
    g.off_vm = off; off += 2 * 2 * kVmRows * kVmPitch * (int)sizeof(__half);
    g.off_is = off; off += kSlots * kTile * p.M * (int)sizeof(float);
    g.off_cs = off; off += 2 * kSegsPerTile * kSeg * 32 * (int)sizeof(float);
    g.off_seg = off; off += 2 * kSegsPerTile * 3 * 32 * (int)sizeof(int);
    g.off_clus = off; off += 4 * kClusterMax * 32 * (int)sizeof(int);
    g.off_bits = off; off += 2 * kRingWords * 32 * (int)sizeof(int);
    g.off_stage = off; off += (2 * kSlots * kTile * p.C2 + 15) & ~15;
    g.smem_bytes = (off + 15) & ~15;
    // the spike-bit ring must hold the back warp's oldest read and the front warp's newest write
    // (the neuron warp reads back to (k - dtile) * kTile - nL while the RZCC warp clears the words of tile k - 3)
    if (kTile * (g.dtile - 2) + p.nL + kSeg > kRingWords * 32)
        return set_error(MICLOC_ERR_UNSUPPORTED, "robust_width %d / neuron length %d exceed the fused kernel's spike ring; "
                         "use the staged path", p.w, p.nL);
    if (kSlots * 256 * (int)sizeof(double) > kSlots * p.M * g.pitch_x * (int)sizeof(float))
        return set_error(MICLOC_ERR_UNSUPPORTED, "shared-memory tiles too small for the epilogue");
    if (g.smem_bytes > 227 * 1024)
        return set_error(MICLOC_ERR_UNSUPPORTED, "fused kernel needs %d B of shared memory; use the staged path", g.smem_bytes);
    if (T + 16 * kTile >= (1ll << 31)) return set_error(MICLOC_ERR_SHAPE, "T too large for the fused kernel");
    // one CTA of two clip-pair groups per SM when both fit its shared memory (the usual case), else the
    // single-group CTA twice per SM
    const int groups = 2 * g.smem_bytes <= 227 * 1024 ? 2 : 1;
#define MICLOC_FUSED_CASE(IN, MMV)                                                                                \
    do {                                                                                                          \
        if (groups == 2)                                                                                          \
            return launch_fused_t<IN, MMV, 2>(p, g, d_taps, d_Wd, (const IN *)audio, B, T, spikes, power, doa,    \
                                              flags, sm_slots, sm_count, st);                                     \
        return launch_fused_t<IN, MMV, 1>(p, g, d_taps, d_Wd, (const IN *)audio, B, T, spikes, power, doa, flags, \
                                          sm_slots, sm_count, st);                                                \
    } while (0)
    const bool i16 = dtype == MICLOC_I16;
    if (p.M == 7) { if (i16) MICLOC_FUSED_CASE(int16_t, 7); else MICLOC_FUSED_CASE(float, 7); }
    if (i16) MICLOC_FUSED_CASE(int16_t, 0); else MICLOC_FUSED_CASE(float, 0);
#undef MICLOC_FUSED_CASE
}

}  // namespace micloc
