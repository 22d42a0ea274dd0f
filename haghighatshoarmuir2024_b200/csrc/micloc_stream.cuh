// micloc_stream.cuh -- slot bookkeeping and frame assembly shared by the stream batches of the float SNN chain
// (micloc_stream.cu) and of the Xylo integer chain (micloc_xylo.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

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

}  // namespace micloc
