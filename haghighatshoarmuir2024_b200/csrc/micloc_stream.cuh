// micloc_stream.cuh -- the slot book and frame assembly shared by the stream batches: the float SNN chain's stream and
// multi-band batches (micloc_stream.cu) and the Xylo integer chain's (micloc_xylo.cu).  The rule of where a slot stands
// and what a push, flush or reset does to it lives here once; each batch keeps its chain state and flags next to it.
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

    // k_stream_assemble of the frames into xbuf[xcur ^ 1], which becomes the newest buffer
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
        xcur = nxt;
        n_prev = n;
        return MICLOC_OK;
    }

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

}  // namespace micloc
