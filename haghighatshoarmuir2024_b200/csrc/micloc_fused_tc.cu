// micloc_fused_tc.cu -- the fused hot-path kernel with the STHT FIR on the 5th-generation tensor cores.
//
// Reference sites: micloc/snn_beamformer.py:283-370 (STHT :325-327) and the callers' power/argmax
// paper_plots/target_snn_localization.py:462-464.
//
// Same chain, same serial roles (band-pass, RZCC, neuron, Gram: micloc_fused_common.cuh) and the same pipeline of
// 64-sample steps as micloc_fused.cu, but the 240-tap quadrature FIR -- 84 % of the arithmetic -- no longer occupies
// issue slots of the SM sub-partitions: it runs as a Toeplitz GEMM on tcgen05.mma with the accumulators in tensor
// memory, issued by one thread.
//
//   polyphase   The Hilbert kernel has a tap at every other lag, so Q at odd times is a DENSE FIR of the even
//               samples E[n] = x[2n] and Q at even times the same FIR of the odd samples O[n] = x[2n-1]:
//               Q[2n+1] = sum_j g[j] E[n-j],  Q[2n] = sum_j g[j] O[n-j]   (g[j] = h[k0 + 2j], k0 odd).
//   GEMM        D[a][n] = sum_e A[a][e] B[n][e] per tile of 128 stream samples (256 frames) of the group's two clips:
//               A[a][e] = g[a + lag - e] is the constant Toeplitz matrix of the taps (128 output phases x window of
//               lag + 128 samples), resident in TENSOR MEMORY as two fp16 pieces (taps x 2^14 = hi + lo, written once
//               per CTA with tcgen05.st); B[n][e] = u_n[128 tile - lag + e] holds the window of stream n (2 clips x
//               microphones x parity = 28 columns, N = 32).  The streams live in shared memory in rings of 8-sample
//               chunks, the chunks of all streams interleaved -- exactly the canonical K-major core-matrix layout
//               of the B operand, so a descriptor with the right start address IS the sliding window (nothing is
//               copied) -- as two fp16 pieces u = hi + lo (22 significant bits; the clip is scaled by a power of two
//               so that it fits the fp16 range: band-pass and RZCC are scale invariant).  Three products per K step
//               (hi hi, hi lo, lo hi; the dropped lo lo is below 2^-22), float32 accumulation.  Shared-memory traffic
//               of an instruction: 1 KB.  (A first version had the samples as the A operand, a Hankel matrix read
//               through overlapping core matrices: correct, but 4.5 KB of shared-memory reads per instruction starved
//               the serial warps -- profiles/README.md.)
//   in          Front-end warp 0 streams 128-frame audio tiles with 1-D TMA bulk copies (cp.async.bulk + mbarrier)
//               into a staging buffer; the four front-end warps convert it into the hi/lo rings at the top of a step;
//               warp 3 issues the K steps of an MMA tile as their samples arrive, a quarter per step.
//   out         A step's 32 stream samples are one 32-lane quarter of the accumulator: the warp owning that quarter
//               moves them into the step's q rows (tcgen05.ld); all four warps rebuild the in-phase samples
//               x[t - K/2] (np.roll: the first K/2 come from the clip tail) from the rings.
//
// One CTA holds two independent clip-pair groups of eight warps: four serial roles (band-pass, RZCC, neuron, Gram) and
// four front-end warps (warp q owns tensor-memory lane quarter q; warp 0 also issues the TMA copies, warp 1 scans the
// next clip pair's largest magnitude, warp 3 issues the MMAs through one elected lane).  The same role of both groups
// sits on the same SM sub-partition (warp id mod 4): a sub-partition then runs ~20 KB of code (one serial role + the
// front end), which is what its instruction cache holds -- other pairings measured 3-7 % slower.

#include "micloc_fused_common.cuh"

namespace micloc {
namespace tc {

constexpr int kGWarps = 8;                // warps of a clip-pair group: four serial roles + four front-end warps
constexpr int kGThreads = kGWarps * 32;
constexpr int kRoleFront = 4;             // roles 0..3: band-pass, RZCC, neuron, Gram; 4 + q: front-end warp of lane quarter q
constexpr int kRingWords = 16;            // spike-bit ring: 16 words of 32 samples per channel and polarity
constexpr int kMac = 2 * kTile;           // frames per audio tile (TMA, conversion): 64 samples of every stream
constexpr int kBlk = 128;                 // stream samples per MMA tile = output phases = rows of A
constexpr int kQRow = kTile + 4;          // floats per channel row of a q sub-tile: [even times: 32][odd times: 32] + pad
constexpr int kRows = 8;                  // most microphones
constexpr float kTapScale = 16384.f;      // taps are stored x 2^14 as fp16 hi + lo
constexpr int kMmaN = 32;                 // columns of an MMA: the group's streams (2 clips x microphones x parity <= 32)
constexpr int kLead = 3;                  // steps the front end runs ahead of the serial roles

struct TcGeom {
    int RC;         // ring length in 8-sample chunks (even)
    int NSP;        // streams per chunk row: kSlots * 2M
    int piece_b;    // bytes of one ring piece: RC * NSP * 16
    int lag;        // the window of a tile starts `lag` samples before its first output (multiple of 16)
    int ksteps;     // MMA K steps of 16: (lag + 128) / 16
    int H;          // K/2 / 2: in-phase delay in stream samples
    int d0;         // leading zero taps of the polyphase filter
    int dtile;      // the neuron warp runs dtile steps behind (RZCC decision latency)
    int tiles_is;   // sub-tiles whose in-phase input comes from the clip tail
    int off_ring, off_stin, off_q, off_vm, off_cs, off_seg, off_clus, off_bits, off_stage, off_misc;
    int smem_group; // bytes of one group
    int smem_bytes; // bytes of the CTA
};

struct TcSmem {
    // what the shared roles use
    float *cs;
    unsigned int *seg;
    int *clus;
    unsigned int *bits;
    __half *vms;
    int8_t *stage;
    double *gram;
    unsigned int *dbg;
    int bar_id, bar_threads, rec, k_first;
    // tensor-core side
    unsigned char *ring;      // [2 pieces][RC chunks][NSP streams][8 halves]
    unsigned char *stin;      // TMA staging of one audio tile [kMac][M]
    float *q;                 // [2 sub-tiles][kSlots][2M][kQRow]
    float *scale;             // [kSlots] power-of-two clip scale
    unsigned int *amax;       // [kSlots]
    unsigned int *amax_next;  // [kSlots] of the clip pair this group takes next (scanned by the producer warp meanwhile)
    float *carry;             // [kSlots][2][8] last frame of the previous audio tile (first odd-stream sample of the next)
    unsigned long long *mbar; // [0..1] MMA done (accumulator buffer), [4] audio tile staged
};

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t a, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_inval(uint32_t a) { asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(a) : "memory"); }
// (a wait that never completes is a pipeline bug: trap after a few seconds instead of hanging the GPU)
#ifdef MICLOC_WAIT_DEBUG
__device__ unsigned long long g_wait_dbg[8];      // first wait that timed out: tag, block, thread, parity
#endif
__device__ __forceinline__ void mbar_wait(uint32_t a, uint32_t parity, int tag = 0) {
    uint32_t ok = 0, spins = 0;
    while (!ok) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(a), "r"(parity) : "memory");
#ifdef MICLOC_WAIT_DEBUG
        if (!ok && *(volatile unsigned long long *)&g_wait_dbg[0] != 0ull) return;      // somebody timed out: let the kernel drain
#endif
        if (!ok && ++spins > (1u << 21)) {
#ifdef MICLOC_WAIT_DEBUG
            if (atomicCAS(&g_wait_dbg[0], 0ull, (unsigned long long)(tag + 1)) == 0ull) {
                g_wait_dbg[1] = blockIdx.x; g_wait_dbg[2] = threadIdx.x; g_wait_dbg[3] = parity; g_wait_dbg[4] = a;
                unsigned long long w;
                asm volatile("ld.shared.b64 %0, [%1];" : "=l"(w) : "r"(a));
                g_wait_dbg[5] = w;
                // progress words of the group's MMA thread sit 16 and 24 bytes behind mbarrier 4 (misc + 48, + 56)
                const uint32_t base = a & ~127u;
                asm volatile("ld.shared.b64 %0, [%1];" : "=l"(w) : "r"(base + 48u));
                g_wait_dbg[6] = w;
                asm volatile("ld.shared.b64 %0, [%1];" : "=l"(w) : "r"(base + 56u));
                g_wait_dbg[7] = w;
            }
            return;
#else
            __trap();
#endif
        }
    }
}
__device__ __forceinline__ void mbar_arrive(uint32_t a) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(a) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t a, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(a), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// one lane of a converged warp, chosen by the hardware: ptxas then knows that the guarded code runs on a single thread
// and feeds tcgen05.mma's uniform-register operands with plain R2UR moves instead of an ELECT / BRA.U.ANY loop per MMA
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_mma_f16(uint32_t d, uint64_t ad, uint64_t bd, uint32_t idesc, uint32_t accum) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(d), "l"(ad), "l"(bd), "r"(idesc), "r"(accum) : "memory");
}
// A from tensor memory (lane = row, column c of a K step holds elements k = 2c (low half) and 2c + 1), B from shared memory
__device__ __forceinline__ void tc_mma_f16_ts(uint32_t d, uint32_t a_tmem, uint64_t bd, uint32_t idesc, uint32_t accum) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
                 ::"r"(d), "r"(a_tmem), "l"(bd), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void tc_st8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                 "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// K-major, no swizzle: 8-row x 16-byte core matrices; `lbo` = bytes between core matrices along K, `sbo` = bytes
// between 8-row groups along M / N (cute::UMMA::SmemDescriptor: start [0,14), LBO [16,30), SBO [32,46), version 1)
__device__ __forceinline__ uint64_t make_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((addr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// kind::f16, A and B fp16 K-major, D float32, M = 128, N = 16 (cute::UMMA::InstrDescriptor)
constexpr uint32_t kIdesc = (1u << 4) | ((uint32_t)(kMmaN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);

template <typename IN_T> __device__ __forceinline__ float clip_scale(unsigned int amax_bits);
template <> __device__ __forceinline__ float clip_scale<int16_t>(unsigned int) { return 1.f; }      // |x| <= 32768 fits fp16; hi + lo is exact
template <> __device__ __forceinline__ float clip_scale<float>(unsigned int amax_bits) {
    const float a = __uint_as_float(amax_bits);
    if (!(a > 0.f) || !(a < 3.0e38f)) return 1.f;
    int e = (int)((amax_bits >> 23) & 0xffu) - 127;      // floor(log2 a) for normal numbers
    int s = 13 - e;                                      // |x| 2^s < 2^14
    s = s > 120 ? 120 : (s < -120 ? -120 : s);
    return __uint_as_float((unsigned int)(s + 127) << 23);
}

// ======================= front-end warps (4 per group): audio in, STHT on the tensor cores, q rows out =======================
// The front end runs kLead steps ahead of the serial roles.  Step k handles audio tile `it` = k + kLead + 1:
// tile it is the 128-frame tile J = it / 2 of clip slot it & 1; the four tiles 4 Jb .. 4 Jb + 3 make up MMA tile Jb
// (256 frames of both clips).  Per step, all four warps:
//   (a) turn the staged audio tile into hi / lo ring chunks (a thread builds one 8-sample chunk of one stream),
//   (b) meet; warp 0 sends the next audio tile on its way (TMA) and, behind the fourth tile of an MMA tile, issues its
//       MMAs (one lane) and commits them to the accumulator buffer's mbarrier,
//   (c) move sub-tile k - 1 into the q rows the band-pass warp reads at the next step: the warp whose tensor-memory
//       lane quarter holds the sub-tile's 32 stream samples stores Q, every warp rebuilds the in-phase samples of one
//       (clip slot, parity) from the rings,
//   (d) warp 1 scans a slice of the NEXT clip pair for its largest magnitude (float32 input: fp16 clip scale).
__device__ __forceinline__ bool tile_of_step(int k, int NJ, bool ok1, int &it, int &slot, int &J) {
    it = k + kLead + 1;
    slot = it & 1;
    J = it >> 1;
    return J < NJ && (slot == 0 || ok1);
}

// Rare paths of the front end, kept out of line (the loop below runs once per step and is instruction-fetch bound):
// an audio tile that is ragged or not 16-byte aligned goes to the staging buffer with plain loads, zero-filled
// behind the clip end
template <typename IN_T>
__device__ __noinline__ void stage_tile_plain(IN_T *stin, const IN_T *s, int nvalid, int total, int lane) {
    for (int e = lane; e < total; e += 32) stin[e] = e < nvalid ? s[e] : (IN_T)0;
}
// in-phase samples of the first K/2 frames come from the clip's tail (np.roll, snn_beamformer.py:325)
template <typename IN_T>
__device__ __noinline__ void inphase_from_tail(float *dst, const IN_T *clip, int t0, int T, int half, int M, int mic, float sc) {
    for (int i = 0; i < 8; ++i) {
        const int t = t0 + 2 * i;
        float x = 0.f;
        if (t < T) {
            int srci = (t - half) % T;
            if (srci < 0) srci += T;
            x = to_f32<IN_T>(clip[(long long)srci * M + mic]) * sc;
        }
        dst[i] = x;
    }
}
// in-phase samples from the rings when K/2 is not a multiple of 16 (the 8 samples start anywhere in a chunk)
__device__ __noinline__ void inphase_from_ring_any(float *dst, const unsigned char *r0, const unsigned char *r1, int piece_b, int b0) {
    for (int i = 0; i < 8; ++i) {
        const int e = b0 + i;
        const unsigned char *r = (e < 8 ? r0 : r1) + 2 * (e & 7);
        dst[i] = __half2float(*reinterpret_cast<const __half *>(r)) + __half2float(*reinterpret_cast<const __half *>(r + piece_b));
    }
}

template <typename IN_T, int MM>
__device__ __forceinline__ void front_role(const TcSmem &sm, const ChainParams &p, const TcGeom &g,
                                           const IN_T *__restrict__ audio, long long clip0, long long B,
                                           long long T64, int quarter, int lane, int NT, int NJ, int k_last,
                                           uint32_t tmem_a, uint32_t tmem_d, uint32_t &tma_phase, uint32_t (&mma_base)[2],
                                           int front_bar, long long next_clip0) {
    const int M = MM ? MM : p.M, C2 = 2 * M;
    const int T = (int)T64;
    const bool ok1 = clip0 + 1 < B;
    const IN_T *src[kSlots] = {audio + clip0 * T64 * M, audio + (ok1 ? clip0 + 1 : clip0) * T64 * M};
    const bool al[kSlots] = {(reinterpret_cast<uintptr_t>(src[0]) & 15) == 0, (reinterpret_cast<uintptr_t>(src[1]) & 15) == 0};
    const uint32_t tile_bytes = (uint32_t)(kMac * M * sizeof(IN_T));
    const uint32_t bar_tma = smem_u32(sm.mbar + 4);
    const uint32_t stin_a = smem_u32(sm.stin);
    IN_T *stin = reinterpret_cast<IN_T *>(sm.stin);
    const int NJb = (NJ + 1) >> 1;            // MMA tiles of 256 frames
    const int t128 = quarter * 32 + lane;
    const float sx[kSlots] = {sm.scale[0], sm.scale[1]};
    auto front_sync = [&]() { asm volatile(MICLOC_BAR_SYNC " %0, 128;" ::"r"(front_bar) : "memory"); };
    ROLE_TIMER_DECL;
    PH_DECL;

    // audio tile J of clip slot `slot` -> staging (warp 0): one 1-D TMA bulk copy when the tile is whole and 16-byte
    // aligned, else plain loads with zero fill behind the clip end; either way its arrival completes a phase of bar_tma
    auto issue_load = [&](int slot, int J) {
        const int f0 = kMac * J;
        const IN_T *s = src[slot] + (long long)f0 * M;
        if (al[slot] && f0 + kMac <= T) {
            if (elect_one()) {
                fence_proxy_async();
                mbar_expect_tx(bar_tma, tile_bytes);
                tma_bulk_g2s(stin_a, s, tile_bytes, bar_tma);
            }
        } else {
            stage_tile_plain<IN_T>(stin, s, (T - f0 < kMac ? T - f0 : kMac) * M, kMac * M, lane);
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_tma);
        }
        __syncwarp();
    };

    // (d) state of the scan of the next pair (warp 1)
    const bool scan = quarter == 1 && sizeof(IN_T) == 4 && next_clip0 >= 0 && ((T64 * M) & 3) == 0 &&
                      (reinterpret_cast<uintptr_t>(audio + next_clip0 * T64 * M) & 15) == 0 &&
                      ((T64 * M) >> 2) <= 128ll * (k_last + kLead + 1);
    const long long n4 = (T64 * M) >> 2;
    constexpr int kScanLd = 4;                 // float4 loads per lane, clip and step
    float4 sv[kSlots][kScanLd];
#pragma unroll
    for (int c = 0; c < kSlots; ++c)
#pragma unroll
        for (int u = 0; u < kScanLd; ++u) sv[c][u] = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 *scan_src[kSlots] = {reinterpret_cast<const float4 *>(audio + (next_clip0 < 0 ? 0 : next_clip0) * T64 * M),
                                      reinterpret_cast<const float4 *>(audio + (next_clip0 < 0 ? 0 : next_clip0 + 1) * T64 * M)};
    const bool scan_ok1 = next_clip0 + 1 < B;
    float mx[kSlots] = {0.f, 0.f};
    long long scan_i = 0;

    // ring coordinates kept incrementally (a runtime modulo costs ~25 instructions and this loop is instruction-fetch bound)
    int cbase[kSlots] = {0, 0};               // ring chunk of the next audio tile's first sample, per clip slot
    int cwin = -(g.lag / 8) % g.RC;           // ring chunk of the first window sample of the MMA tile being issued
    if (cwin < 0) cwin += g.RC;
    int ibase = ((4 * (sm.k_first - 2) - g.H / 8) % g.RC + g.RC) % g.RC;     // chunk of stream sample 32 s - H of the step before the first (s = k - 1)

    if (quarter == 0) issue_load(0, 0);
    for (int k = sm.k_first; k <= k_last; ++k) {
        int it, slot, J;
        const bool valid = tile_of_step(k, NJ, ok1, it, slot, J);
        PH_START();
        // ---- (a) staging -> rings.  The chunks overwritten lie in the window of MMA tile Jb - 1 (second half of tile
        //      Jb) or Jb - 2 (first half): issued 3 or more steps ago, observed here ----
        if (valid) {
            const int Jw = (it >> 2) - ((it & 2) ? 1 : 2);
            if (Jw >= 0) mbar_wait(smem_u32(sm.mbar + (Jw & 1)), (mma_base[Jw & 1] + (uint32_t)(Jw >> 1)) & 1u, 100000 + (k + 8));
            mbar_wait(bar_tma, tma_phase, 200000 + (k + 8));
            tma_phase ^= 1u;
            PH_END(0);
            const int f0 = kMac * J;
            const int cb = slot ? cbase[1] : cbase[0];      // ring chunk of the tile's first stream position
            if (slot) { cbase[1] += 8; if (cbase[1] >= g.RC) cbase[1] -= g.RC; }
            else { cbase[0] += 8; if (cbase[0] >= g.RC) cbase[0] -= g.RC; }
            const float s_x = sx[slot];
            // thread (j, parity, mic) builds chunk j of its stream: samples 8 j .. 8 j + 7 = frames
            // 16 j - parity + 2 i (O[n] = x[2n-1]: the odd stream's first sample is the previous tile's last frame)
            if (t128 < 8 * C2) {
                const int j = t128 / C2, sidx = t128 - j * C2;
                const int par = sidx >= M ? 1 : 0, mic = sidx - par * M;
                const IN_T *sp = stin + (16 * j - par) * M + mic;
                float u[8];
                // frames f = 16 j - par + 2 i of the tile; those behind the clip end (f >= T - f0, last tile only) are
                // zeros: the first nv of the 8 are inside.  f = -1 (j = 0, odd stream) is the carry below.
                const int left = T - f0 - (16 * j - par);
                const int nv = left >= 16 ? 8 : (left > 0 ? (left + 1) >> 1 : 0);
#pragma unroll
                for (int i = 1; i < 8; ++i) u[i] = i < nv ? to_f32<IN_T>(sp[2 * i * M]) * s_x : 0.f;
                u[0] = (nv > 0 && 16 * j - par >= 0) ? to_f32<IN_T>(sp[0]) * s_x : 0.f;
                if (j == 0 && par == 1) u[0] = J > 0 ? sm.carry[(slot * 2 + ((J + 1) & 1)) * 8 + mic] : 0.f;   // x[128 J - 1]
                uint4 h4, l4;
                unsigned int *hp = &h4.x, *lp = &l4.x;
#pragma unroll
                for (int i2 = 0; i2 < 4; ++i2) {
                    const __half2 hh = __floats2half2_rn(u[2 * i2], u[2 * i2 + 1]);
                    const float2 hf = __half22float2(hh);
                    const __half2 ll = __floats2half2_rn(u[2 * i2] - hf.x, u[2 * i2 + 1] - hf.y);
                    hp[i2] = *reinterpret_cast<const unsigned int *>(&hh);
                    lp[i2] = *reinterpret_cast<const unsigned int *>(&ll);
                }
                int ch = cb + j;
                if (ch >= g.RC) ch -= g.RC;
                const int off = (ch * g.NSP + slot * C2 + 2 * mic + par) * 16;
                *reinterpret_cast<uint4 *>(sm.ring + off) = h4;
                *reinterpret_cast<uint4 *>(sm.ring + g.piece_b + off) = l4;
            }
            if (t128 < M) sm.carry[(slot * 2 + (J & 1)) * 8 + t128] = (f0 + kMac - 1 < T) ? to_f32<IN_T>(stin[(kMac - 1) * M + t128]) * s_x : 0.f;
            fence_proxy_async();
        }
        PH_END(1);
        front_sync();
        // ---- (b) next audio tile on its way (warp 0) ----
        if (quarter == 0 && valid) {
            int i2, s2, J2;
            bool have = tile_of_step(k + 1, NJ, ok1, i2, s2, J2);
            if (!have) have = tile_of_step(k + 2, NJ, ok1, i2, s2, J2);
            if (have) issue_load(s2, J2);
        }
        PH_END(2);
        // ---- (c) sub-tile s = k - 1 -> q rows ----
        const int s = k - 1;
        ibase += 4;
        if (ibase >= g.RC) ibase -= g.RC;
        if (s >= 0 && s < NT) {
            // Q: accumulator row a = stream sample a of MMA tile Jb, column n = stream; the 32 samples of this
            // sub-tile are lanes 32 (s & 3) ..: the warp that owns them stores column after column
            if ((s & 3) == quarter) {
                const int Jb = s >> 2;
                mbar_wait(smem_u32(sm.mbar + (Jb & 1)), (mma_base[Jb & 1] + (uint32_t)(Jb >> 1)) & 1u, 300000 + (k + 8));
                tc_fence_after();
                uint32_t r[32];
                tc_ld32(tmem_d + (uint32_t)((Jb & 1) * kMmaN) + ((uint32_t)(32 * quarter) << 16), r);
                tc_fence_before();
                float *qb = sm.q + (s & 1) * kSlots * C2 * kQRow + lane;
#pragma unroll
                for (int n = 0; n < 2 * kRows * kSlots; ++n) {
                    // stream n = slot * 2M + 2 mic + parity: even stream -> Q at odd times, odd stream -> Q at even times
                    if (n < kSlots * C2) {
                        const int slot2 = n / C2, rem = n - slot2 * C2;
                        if (clip0 + slot2 < B)
                            qb[(slot2 * C2 + M + (rem >> 1)) * kQRow + ((rem & 1) ? 0 : 32)] = __uint_as_float(r[n]);
                    }
                }
            }
            PH_END(3);
            // I[t] = x[(t - K/2) mod T] (scaled like the ring samples; the band-pass warp applies the 2^14 of the
            // taps): warp quarter = (clip slot, parity); a lane rebuilds 8 consecutive samples of one microphone
            const int islot = quarter >> 1, ipar = quarter & 1;
            if (lane < 4 * M && clip0 + islot < B) {
                const int mic = lane >> 2, chunk = lane & 3;
                float *dst = sm.q + (((s & 1) * kSlots + islot) * C2 + mic) * kQRow + ipar * 32 + 8 * chunk;
                if (s < g.tiles_is) {
                    inphase_from_tail<IN_T>(dst, src[islot], kTile * s + 16 * chunk + ipar, T, p.half, M, mic, sx[islot]);
                } else {
                    // I[2n] = E[n - H], I[2n+1] = O[n - H + 1]: 8 samples from ring position q0 on
                    const int q0 = (kTile / 2) * s + 8 * chunk - g.H + ipar;
                    const int n = islot * C2 + 2 * mic + ipar;
                    const int b0 = q0 & 7;
                    int c0 = (g.H & 7) == 0 ? ibase + chunk : (q0 >> 3) % g.RC;
                    if (c0 >= g.RC) c0 -= g.RC;
                    const int c1 = c0 + 1 == g.RC ? 0 : c0 + 1;
                    const unsigned char *r0 = sm.ring + (c0 * g.NSP + n) * 16, *r1 = sm.ring + (c1 * g.NSP + n) * 16;
                    if (b0 <= 1) {      // (warp-uniform) K/2 a multiple of 16: the 8 samples start at half 0 or 1 of a chunk
                        const uint4 h4 = *reinterpret_cast<const uint4 *>(r0), l4 = *reinterpret_cast<const uint4 *>(r0 + g.piece_b);
                        const unsigned int hw[4] = {h4.x, h4.y, h4.z, h4.w}, lw[4] = {l4.x, l4.y, l4.z, l4.w};
                        float a[9];
#pragma unroll
                        for (int w2 = 0; w2 < 4; ++w2) {
                            const float2 hf = __half22float2(*reinterpret_cast<const __half2 *>(&hw[w2]));
                            const float2 lf = __half22float2(*reinterpret_cast<const __half2 *>(&lw[w2]));
                            a[2 * w2] = hf.x + lf.x; a[2 * w2 + 1] = hf.y + lf.y;
                        }
                        a[8] = 0.f;
                        if (b0 == 1)
                            a[8] = __half2float(*reinterpret_cast<const __half *>(r1)) + __half2float(*reinterpret_cast<const __half *>(r1 + g.piece_b));
                        reinterpret_cast<float4 *>(dst)[0] = b0 ? make_float4(a[1], a[2], a[3], a[4]) : make_float4(a[0], a[1], a[2], a[3]);
                        reinterpret_cast<float4 *>(dst)[1] = b0 ? make_float4(a[5], a[6], a[7], a[8]) : make_float4(a[4], a[5], a[6], a[7]);
                    } else {
                        inphase_from_ring_any(dst, r0, r1, g.piece_b, b0);
                    }
                }
            }
        }
        PH_END(4);
        // ---- (b') MMAs (warp 3, one lane), last in the step: tcgen05.mma blocks its warp while the tensor core's queue
        //      is full.  The K steps of MMA tile Jb are issued as their samples arrive, a quarter per step: behind the
        //      tile's 1st and 2nd audio tile the steps over the history (warp 3 itself has just read the last quarter
        //      of the accumulator buffer's previous tile), behind the 3rd those up to the first 64 new samples,
        //      behind the 4th the rest + commit ----
        if (quarter == 3) {
            const int Jb = it >> 2, part = it & 3;
            if (Jb < NJb) {
                const int hist = g.lag / 16;              // K steps over samples before the tile
                const int e0 = (hist * 2) / 5, e1 = (hist * 4) / 5, e2 = hist + 4;
                const int ks0 = part == 0 ? 0 : (part == 1 ? e0 : (part == 2 ? e1 : e2));
                const int ks1 = part == 0 ? e0 : (part == 1 ? e1 : (part == 2 ? e2 : g.ksteps));
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t d = tmem_d + (uint32_t)((Jb & 1) * kMmaN);
                    int c = cwin + 2 * ks0;          // chunk of K step ks0
                    if (c >= g.RC) c -= g.RC;
                    const uint32_t rb_hi = smem_u32(sm.ring), rb_lo = rb_hi + (uint32_t)g.piece_b;
                    const uint32_t chunk_b = (uint32_t)g.NSP * 16u;
                    // B: K-major, no swizzle: 8 streams x 16 bytes per core matrix, next 8 streams 128 bytes on,
                    // next chunk (K) NSP * 16 bytes on
                    const uint64_t b_fix = make_desc(0u, chunk_b, 128u);
                    const uint32_t a_lo = tmem_a + 8u * (uint32_t)g.ksteps;
#pragma unroll 1
                    for (int ks = ks0; ks < ks1; ++ks) {
                        const uint32_t off = ((uint32_t)c * chunk_b) >> 4;
                        const uint64_t b_hi = b_fix | (uint64_t)(((rb_hi >> 4) + off) & 0x3FFFu);
                        const uint64_t b_lo = b_fix | (uint64_t)(((rb_lo >> 4) + off) & 0x3FFFu);
                        tc_mma_f16_ts(d, tmem_a + 8u * (uint32_t)ks, b_hi, kIdesc, ks ? 1u : 0u);
                        tc_mma_f16_ts(d, tmem_a + 8u * (uint32_t)ks, b_lo, kIdesc, 1u);
                        tc_mma_f16_ts(d, a_lo + 8u * (uint32_t)ks, b_hi, kIdesc, 1u);
                        c += 2;
                        if (c >= g.RC) c -= g.RC;
                    }
                    if (part == 3) tc_commit(smem_u32(sm.mbar + (Jb & 1)));
#ifdef MICLOC_WAIT_DEBUG
                    sm.mbar[6] = ((unsigned long long)(unsigned)it << 32) | (unsigned)(ks1 - ks0);     // last part issued
                    if (part == 3) sm.mbar[7] = sm.mbar[7] + 1ull;                                 // commits so far
#endif
                }
                __syncwarp();
            }
            if (part == 3) { cwin += 16; if (cwin >= g.RC) cwin -= g.RC; }
        }
        // ---- (d) amax scan of the next pair: the slice loaded at the previous step is folded in now, this step's
        //      slice is requested and not waited for ----
        if (scan) {
#pragma unroll
            for (int c = 0; c < kSlots; ++c)
#pragma unroll
                for (int u = 0; u < kScanLd; ++u)
                    mx[c] = fmaxf(fmaxf(mx[c], fmaxf(fabsf(sv[c][u].x), fabsf(sv[c][u].y))), fmaxf(fabsf(sv[c][u].z), fabsf(sv[c][u].w)));
#pragma unroll
            for (int c = 0; c < kSlots; ++c)
#pragma unroll
                for (int u = 0; u < kScanLd; ++u) {
                    const long long i = scan_i + 32 * u + lane;
                    sv[c][u] = (i < n4 && (c == 0 || scan_ok1)) ? __ldg(scan_src[c] + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            scan_i += 32 * kScanLd;
        }
        ROLE_BARRIER();
    }
    if (quarter == 1) {
        // amax of the next pair (bit pattern order = magnitude order); ~0 = "not scanned"
#pragma unroll
        for (int c = 0; c < kSlots; ++c) {
#pragma unroll
            for (int u = 0; u < kScanLd; ++u)
                mx[c] = fmaxf(fmaxf(mx[c], fmaxf(fabsf(sv[c][u].x), fabsf(sv[c][u].y))), fmaxf(fabsf(sv[c][u].z), fabsf(sv[c][u].w)));
            unsigned int mb = __float_as_uint(mx[c]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { const unsigned int ot = __shfl_xor_sync(0xffffffffu, mb, o); mb = ot > mb ? ot : mb; }
            if (lane == 0) sm.amax_next[c] = scan ? mb : 0xffffffffu;
        }
    }
    // the MMA barriers are never re-initialised: tile Jb of a pair is completion mma_base[Jb & 1] + Jb / 2 of its barrier
    mma_base[0] += (uint32_t)((NJb + 1) >> 1);
    mma_base[1] += (uint32_t)(NJb >> 1);
    ROLE_TIMER_FLUSH(quarter);
    if (quarter == 0) PH_FLUSH(sm.dbg, 0, 5);
}

// ============ band-pass warp: SOS cascade + running sum + sign / zero masks, lane = slot*16 + channel ============
// Inputs of sub-tile k-2 come from its q rows (even-time samples, then odd-time samples), in-phase and quadrature alike.
template <int MM>
__device__ __forceinline__ void bandpass_role(const TcSmem &sm, const ChainParams &p, long long clip0, long long B,
                                              long long T64, int lane, int k_last) {
    const int M = MM ? MM : p.M, C2 = 2 * M;
    const int T = (int)T64;
    const int c_slot = lane >> 4, c_ch = lane & 15;
    const bool c_valid = c_ch < C2 && clip0 + c_slot < B;
    Sos2 sos;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        sos.b0[k] = p.sos[k][0]; sos.b1[k] = p.sos[k][1]; sos.b2[k] = p.sos[k][2];
        sos.a1[k] = p.sos[k][3]; sos.a2[k] = p.sos[k][4];
    }
    if (c_ch < M) {     // in-phase rows of q are plain ring samples, quadrature rows carry the 2^14 of the tap matrix:
        sos.b0[0] *= kTapScale; sos.b1[0] *= kTapScale; sos.b2[0] *= kTapScale;      // exact (power of two)
    }
    BiquadState bq; biquad_reset(bq);
    float csum = 0.f;
    ROLE_TIMER_DECL;

    for (int k = sm.k_first; k <= k_last; ++k) {
        const int kc = k - 2;
        const int t0 = kc * kTile;
        if (kc >= 0 && t0 < T && c_valid) {
#pragma unroll 1
            for (int sg = 0; sg < kSegsPerTile; ++sg) {
                const int ts = t0 + sg * kSeg;            // first sample of this segment
                if (ts >= T) break;
                float *cs = sm.cs + ((kc & 1) * kSegsPerTile + sg) * kSeg * 32 + lane;
                unsigned int *sgm = sm.seg + ((kc & 1) * kSegsPerTile + sg) * 3 * 32 + lane;
                const float *xe = sm.q + (((kc & 1) * kSlots + c_slot) * C2 + c_ch) * kQRow + (kSeg / 2) * sg;
                const float *xo = xe + kTile / 2;
                const float carry = csum;
                unsigned int neg = 0u, zero = 0u;
                // sample by sample with explicit sign / zero masks (ragged segments, zeros)
                auto slow_segment = [&](int nvalid) {
#pragma unroll 1
                    for (int i = 0; i < nvalid; ++i) {
                        const float z = biquad2_step(sos, bq, (i & 1) ? xo[i >> 1] : xe[i >> 1]);
                        zero |= (rzcc_flat(z, csum) ? 1u : 0u) << (31 - i);      // (sum before this sample)
                        csum += z;
                        cs[i * 32] = csum;
                        neg |= (__float_as_uint(z) >> 31) << (31 - i);
                    }
                };
                if (ts + kSeg <= T) {
                    const BiquadState bq0 = bq;
                    float zmin = 1.f;                   // smallest |z| of the segment: exact zeros are rare (silence)
                    float4 en = *reinterpret_cast<const float4 *>(xe), on = *reinterpret_cast<const float4 *>(xo);
#pragma unroll 1
                    for (int o = 0; o < kSeg / 8; ++o) {
                        const float xc[8] = {en.x, on.x, en.y, on.y, en.z, on.z, en.w, on.w};
                        if (o + 1 < kSeg / 8) {         // inputs of the next group: their latency hides behind this one
                            en = *reinterpret_cast<const float4 *>(xe + 4 * (o + 1));
                            on = *reinterpret_cast<const float4 *>(xo + 4 * (o + 1));
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
                    slow_segment(T - ts);
                }
                sgm[0] = neg; sgm[32] = zero; sgm[64] = __float_as_uint(carry);
            }
        }
        ROLE_BARRIER();
    }
    ROLE_TIMER_FLUSH(kRoleBandpass);
}

// GROUPS = 2: warps 0..3 / 4..7 are the serial roles of group 0 / 1 (warp id mod 4 = role = tensor-memory lane
// quarter), warps 4..7 / 12..15 its front-end warps.
template <typename IN_T, int MM, int GROUPS>
__global__ void __launch_bounds__(kGThreads * GROUPS, 1)
k_fused_tc(const IN_T *__restrict__ audio, const float *__restrict__ taps, const double *__restrict__ Wd,
           int8_t *__restrict__ spikes, float *__restrict__ power, int32_t *__restrict__ doa,
           int32_t *__restrict__ flags, unsigned int *__restrict__ sm_slots,
           const __grid_constant__ ChainParams p, const __grid_constant__ TcGeom g, long long B, long long T) {
    extern __shared__ __align__(128) unsigned char smem_all[];
    __shared__ long long s_pair[GROUPS];
    __shared__ uint32_t s_tmem;

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int M = MM ? MM : p.M, C2 = 2 * M;
    // group = warps 8 group .. + 7: four serial-role warps, then four front-end warps
    const int group = warp >> 3;
    const int quarter = warp & 3;           // tensor-memory lanes 32 quarter .. + 31 are this warp's
    // the same role of both groups runs on the same SM sub-partition (warp id mod 4): the two warps share the lines of the
    // sub-partition's instruction cache -- instruction fetch is what the warps of this kernel stall on first
    const int role = (warp & 4) ? kRoleFront + quarter : quarter;
    const int tid = (warp & 7) * 32 + lane;       // thread index inside the group
    const int bar_id = 1 + group;
    auto group_sync = [&]() { tile_barrier(bar_id, kGThreads); };

    unsigned char *smem_raw = smem_all + (size_t)group * g.smem_group;
    TcSmem sm;
    sm.ring = smem_raw + g.off_ring;
    sm.stin = smem_raw + g.off_stin;
    sm.q = reinterpret_cast<float *>(smem_raw + g.off_q);
    sm.vms = reinterpret_cast<__half *>(smem_raw + g.off_vm);
    sm.cs = reinterpret_cast<float *>(smem_raw + g.off_cs);
    sm.seg = reinterpret_cast<unsigned int *>(smem_raw + g.off_seg);
    sm.clus = reinterpret_cast<int *>(smem_raw + g.off_clus);
    sm.bits = reinterpret_cast<unsigned int *>(smem_raw + g.off_bits);
    sm.stage = reinterpret_cast<int8_t *>(smem_raw + g.off_stage);
    sm.mbar = reinterpret_cast<unsigned long long *>(smem_raw + g.off_misc);
    sm.scale = reinterpret_cast<float *>(smem_raw + g.off_misc + 64);
    sm.amax = reinterpret_cast<unsigned int *>(smem_raw + g.off_misc + 72);
    sm.amax_next = reinterpret_cast<unsigned int *>(smem_raw + g.off_misc + 80);
    sm.carry = reinterpret_cast<float *>(smem_raw + g.off_misc + 128);
    sm.gram = reinterpret_cast<double *>(smem_raw + g.off_ring);     // [kSlots][16][16], clip epilogue only (the rings are dead then)
    sm.dbg = sm_slots;
    sm.bar_id = bar_id;
    sm.bar_threads = kGThreads;
    sm.rec = GROUPS * (int)blockIdx.x + group;
    double *red_v = reinterpret_cast<double *>(smem_raw + g.off_cs);         // [kGThreads], clip epilogue only
    int *red_i = reinterpret_cast<int *>(smem_raw + g.off_cs + kGThreads * sizeof(double));

    // ---- once per CTA: barriers, tensor memory, the Toeplitz tap matrix into tensor memory ----
    {
        if (tid == 0) {
            mbar_init(smem_u32(sm.mbar + 4), 1);
            for (int i = 0; i < 2; ++i) mbar_init(smem_u32(sm.mbar + i), 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        if (warp == 0) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&s_tmem)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
        // A[a][e] = g'[a + lag - e] x 2^14 (g'[d0 + j] = taps[j]) as fp16 hi (columns 8 ks + c) and lo (columns
        // 8 (ksteps + ks) + c): lane a, column c of K step ks holds e = 16 ks + 2 c (low half) and e + 1
        if (warp < 4) {       // (warp w writes tensor-memory lanes 32 (w % 4) ..)
            const int a = 32 * warp + lane;
            for (int ks = 0; ks < g.ksteps; ++ks) {
                uint32_t rh[8], rl[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    unsigned short hh[2], ll[2];
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        const int j = a + g.lag - (16 * ks + 2 * c + u) - g.d0;
                        const float gs = (j >= 0 && j < p.n_taps) ? taps[j] * kTapScale : 0.f;
                        const __half hi = __float2half_rn(gs);
                        hh[u] = __half_as_ushort(hi);
                        ll[u] = __half_as_ushort(__float2half_rn(gs - __half2float(hi)));
                    }
                    rh[c] = (uint32_t)hh[0] | ((uint32_t)hh[1] << 16);
                    rl[c] = (uint32_t)ll[0] | ((uint32_t)ll[1] << 16);
                }
                tc_st8(s_tmem + 8u * (uint32_t)ks + ((uint32_t)(32 * warp) << 16), rh);
                tc_st8(s_tmem + 8u * (uint32_t)(g.ksteps + ks) + ((uint32_t)(32 * warp) << 16), rl);
            }
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        }
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
    }
    const uint32_t tmem_a = s_tmem;
    const uint32_t tmem_d = s_tmem + 16u * (uint32_t)g.ksteps + (uint32_t)(group * 2 * kMmaN);
    uint32_t tma_phase = 0, mma_base[2] = {0u, 0u};

    const int NT = (int)((T + kTile - 1) / kTile);
    const int NJ = (int)((T + kMac - 1) / kMac);
    const int k_last = NT + g.dtile;    // the Gram warp runs dtile + 1 steps behind
    sm.k_first = -1 - kLead;            // the producer side starts kLead steps ahead
    const long long npairs = (B + kSlots - 1) / kSlots;
    const int ring_words = 2 * g.piece_b / 4;

    // Clip pairs are handed out dynamically, one ahead: while a group works on a pair its producer warp scans the
    // next one for its largest magnitude (the fp16 scale of float32 clips)
    if (tid == 0) s_pair[group] = (long long)atomicAdd(sm_slots + kSlotPair, 1u);
    if (tid < kSlots) sm.amax_next[tid] = 0xffffffffu;
    group_sync();
    long long pair = s_pair[group];
    while (pair < npairs) {
        group_sync();
        if (tid == 0) s_pair[group] = (long long)atomicAdd(sm_slots + kSlotPair, 1u);
        if (tid < kSlots) sm.amax[tid] = 0u;
        group_sync();
        const long long next_pair = s_pair[group];
        const long long clip0 = pair * kSlots;
        {   // zero the rings (samples before the clip start are zeros: lfilter's zero state), the spike bits
            // and the membrane tiles (columns of unused lanes stay zero)
            unsigned int *r4 = reinterpret_cast<unsigned int *>(sm.ring);
            for (int i = tid; i < ring_words; i += kGThreads) r4[i] = 0u;
            for (int i = tid; i < 2 * kRingWords * 32; i += kGThreads) sm.bits[i] = 0u;
            for (int i = tid; i < 2 * 2 * kVmRows * kVmPitch / 2; i += kGThreads) reinterpret_cast<unsigned int *>(sm.vms)[i] = 0u;
#ifdef MICLOC_WAIT_DEBUG
            if (tid == 0) { sm.mbar[6] = 0ull; sm.mbar[7] = 0ull; }
#endif
        }
        const bool scanned = sm.amax_next[0] != 0xffffffffu;        // (written before the barriers above)
        if (sizeof(IN_T) == 4 && !scanned) {
            // first pair of this group (or an unaligned batch): largest magnitude of each clip, all threads
            for (int s = 0; s < kSlots; ++s) {
                if (clip0 + s >= B) break;
                const float *c = reinterpret_cast<const float *>(audio) + (clip0 + s) * T * M;
                const long long n = T * M;
                float mx = 0.f;
                long long i0 = 0;
                if ((reinterpret_cast<uintptr_t>(c) & 15) == 0) {
                    const float4 *c4 = reinterpret_cast<const float4 *>(c);
                    const long long n4 = n >> 2;
#pragma unroll 8
                    for (long long i = tid; i < n4; i += kGThreads) {
                        const float4 v = __ldg(c4 + i);
                        mx = fmaxf(fmaxf(mx, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
                    }
                    i0 = n4 << 2;
                }
                for (long long i = i0 + tid; i < n; i += kGThreads) mx = fmaxf(mx, fabsf(c[i]));
                unsigned int mb = __float_as_uint(mx);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) { const unsigned int ot = __shfl_xor_sync(0xffffffffu, mb, o); mb = ot > mb ? ot : mb; }
                if (lane == 0) atomicMax(sm.amax + s, mb);
            }
        }
        fence_proxy_async();
        group_sync();
        if (tid < kSlots) sm.scale[tid] = clip_scale<IN_T>(scanned ? sm.amax_next[tid] : sm.amax[tid]);
        group_sync();

        if (role >= kRoleFront)
            front_role<IN_T, MM>(sm, p, g, audio, clip0, B, T, quarter, lane, NT, NJ, k_last, tmem_a, tmem_d, tma_phase,
                                 mma_base, 3 + group, next_pair < npairs ? next_pair * kSlots : -1);
        else if (role == 0) bandpass_role<MM>(sm, p, clip0, B, T, lane, k_last);
        else if (role == 1) rzcc_role<TcSmem, kRingWords>(sm, p, flags, clip0, B, T, M, lane, k_last);
        else if (role == 2) neuron_role<TcSmem, TcGeom, kRingWords>(sm, p, g, clip0, B, T, M, lane, k_last);
        else gram_role<TcSmem, TcGeom>(sm, g, spikes, clip0, B, T, M, lane, k_last);
        group_sync();
        // ---- clip epilogue: power[g] = w_g^T C w_g / T (float64), DoA = first argmax ----
        const double inv_T = 1.0 / (double)T;
        for (int s = 0; s < kSlots; ++s) {
            const long long clip = clip0 + s;
            if (clip >= B) break;
            const double *Cd = sm.gram + s * 256;
            double best = -1.0; int besti = 0x7fffffff;
            for (int gg = tid; gg < p.G; gg += kGThreads) {
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
            if (tid < 32) {
                for (int i = tid + 32; i < kGThreads; i += 32) {
                    const double ov = red_v[i]; const int oi = red_i[i];
                    if (ov > best || (ov == best && oi < besti)) { best = ov; besti = oi; }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ov = __shfl_xor_sync(0xffffffffu, best, o);
                    const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
                    if (ov > best || (ov == best && oi < besti)) { best = ov; besti = oi; }
                }
                if (tid == 0 && doa) doa[clip] = besti;
            }
            group_sync();
        }
        pair = next_pair;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(s_tmem) : "memory");
}

static bool make_geom(const ChainParams &p, int dtype, int groups, TcGeom &g) {
    g = TcGeom{};
    g.d0 = (p.tap_first - 1) / 2;
    g.H = p.half / 2;
    const int ntd = g.d0 + p.n_taps;                    // dense polyphase taps incl. leading zeros
    g.lag = (ntd - 1 + 15) / 16 * 16;
    g.ksteps = (g.lag + kBlk) / 16;
    // a window (lag + 128 samples) plus the audio tile being converted; the in-phase read-back needs less
    g.RC = (g.lag + kBlk) / 8 + kTile / 8;
    if (g.RC * 8 < g.H + 3 * kTile) g.RC = (g.H + 3 * kTile + 7) / 8;
    g.RC = (g.RC + 1) & ~1;
    g.NSP = kSlots * p.C2;
    g.piece_b = g.RC * g.NSP * 16;
    g.dtile = 4 + (rzcc_lag(p.w) - 1 + kTile - 1) / kTile;
    g.tiles_is = (p.half + kTile - 1) / kTile;
    const int esz = dtype == MICLOC_I16 ? 2 : 4;
    int off = 0;
    g.off_ring = off; off += 2 * g.piece_b + 128;       // (the last stream group of the last chunk reads a few bytes on)
    off = (off + 127) & ~127;
    g.off_stin = off; off += kMac * p.M * esz;
    off = (off + 15) & ~15;
    g.off_q = off; off += 2 * kSlots * p.C2 * kQRow * (int)sizeof(float);
    g.off_vm = off; off += 2 * 2 * kVmRows * kVmPitch * (int)sizeof(__half);
    g.off_cs = off; off += 2 * kSegsPerTile * kSeg * 32 * (int)sizeof(float);
    g.off_seg = off; off += 2 * kSegsPerTile * 3 * 32 * (int)sizeof(int);
    g.off_clus = off; off += 4 * kClusterMax * 32 * (int)sizeof(int);
    g.off_bits = off; off += 2 * kRingWords * 32 * (int)sizeof(int);
    g.off_stage = off; off += (2 * kSlots * kTile * p.C2 + 15) & ~15;
    off = (off + 127) & ~127;
    g.off_misc = off; off += 256;
    g.smem_group = (off + 127) & ~127;
    g.smem_bytes = groups * g.smem_group;
    return true;
}

bool fused_supported(const ChainParams &p) {
    // Hilbert-type kernel (every other tap zero) whose taps sit at odd lags and whose in-phase delay K/2 is even,
    // 2-section band-pass, up to 8 microphones
    return p.tap_stride == 2 && (p.tap_first & 1) == 1 && (p.half & 1) == 0 && p.M <= kRows && p.nsec == 2 &&
           (p.n_taps % 8) == 0;
}

template <typename IN_T, int MM, int GROUPS>
static int launch_t(const ChainParams &p, const TcGeom &g, const float *d_taps, const double *d_Wd, const IN_T *audio,
                    long long B, long long T, int8_t *spikes, float *power, int32_t *doa, int32_t *flags,
                    unsigned int *sm_slots, int sm_count, cudaStream_t st) {
    auto kern = k_fused_tc<IN_T, MM, GROUPS>;
    MICLOC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem_bytes));
    MICLOC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    long long grid = sm_count;
    const long long npairs = (B + kSlots - 1) / kSlots;
    const long long want = (npairs + GROUPS - 1) / GROUPS;
    if (grid > want) grid = want;
    MICLOC_CUDA(cudaMemsetAsync(sm_slots, 0, kSlotResetWords * sizeof(unsigned int), st));   // clip-pair counter restarts per launch
    kern<<<(unsigned)grid, kGThreads * GROUPS, g.smem_bytes, st>>>(audio, d_taps, d_Wd, spikes, power, doa, flags, sm_slots, p, g, B, T);
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}

int launch_fused(const ChainParams &p, const float *d_taps, const double *d_Wd, const void *audio, int dtype,
                 long long B, long long T, int8_t *spikes, float *power, int32_t *doa, int32_t *flags,
                 unsigned int *sm_slots, int sm_count, cudaStream_t st) {
    if (!tc::fused_supported(p)) return set_error(MICLOC_ERR_UNSUPPORTED, "tensor-core fused kernel: unsupported chain geometry");
    TcGeom g;
    int groups = 2;
    make_geom(p, dtype, groups, g);
    if (groups == 2 && g.smem_bytes > 227 * 1024) { groups = 1; make_geom(p, dtype, groups, g); }
    if (g.smem_bytes > 227 * 1024)
        return set_error(MICLOC_ERR_UNSUPPORTED, "tensor-core fused kernel needs %d B of shared memory", g.smem_bytes);
    // the spike-bit ring must hold the back warp's oldest read and the front warp's newest write
    if (kTile * (g.dtile - 2) + p.nL + kSeg > kRingWords * 32)
        return set_error(MICLOC_ERR_UNSUPPORTED, "robust_width %d / neuron length %d exceed the tensor-core kernel's spike ring", p.w, p.nL);
    if (kSlots * 256 * (int)sizeof(double) > 2 * g.piece_b)
        return set_error(MICLOC_ERR_UNSUPPORTED, "shared-memory rings too small for the epilogue");
    // tensor memory: the tap matrix (two pieces of 8 columns per K step) + two accumulator buffers per group
    if (16 * g.ksteps + groups * 2 * kMmaN > 512)
        return set_error(MICLOC_ERR_UNSUPPORTED, "STHT kernel of %d taps does not fit the tensor memory", p.n_taps);
    if (T + 16 * kTile >= (1ll << 31)) return set_error(MICLOC_ERR_SHAPE, "T too large for the fused kernel");
#define MICLOC_TC_CASE(IN, MMV)                                                                                   \
    do {                                                                                                          \
        if (groups == 2)                                                                                          \
            return launch_t<IN, MMV, 2>(p, g, d_taps, d_Wd, (const IN *)audio, B, T, spikes, power, doa, flags,   \
                                        sm_slots, sm_count, st);                                                  \
        return launch_t<IN, MMV, 1>(p, g, d_taps, d_Wd, (const IN *)audio, B, T, spikes, power, doa, flags,       \
                                    sm_slots, sm_count, st);                                                      \
    } while (0)
    const bool i16 = dtype == MICLOC_I16;
    if (p.M == 7) { if (i16) MICLOC_TC_CASE(int16_t, 7); else MICLOC_TC_CASE(float, 7); }
    if (i16) MICLOC_TC_CASE(int16_t, 0); else MICLOC_TC_CASE(float, 0);
#undef MICLOC_TC_CASE
}

}  // namespace tc
}  // namespace micloc

#ifdef MICLOC_WAIT_DEBUG
extern "C" int micloc_debug_wait(unsigned long long out[8]) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, micloc::tc::g_wait_dbg, 8 * sizeof(unsigned long long));
    unsigned long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    cudaMemcpyToSymbol(micloc::tc::g_wait_dbg, z, sizeof z);
    return 0;
}
#endif
