// micloc_design.cu -- design_from_template on the device: delayed templates and the batched float64 eigen-solver.
//
// k_design_templates   clips[g][t][m] = np.interp(time[t] - d_m(doa_g), time, sig) rounded once to float32, with
//                      d_m = -r_m cos(theta_m - doa) / speed - min_m(...) (float64), td clamped below at time[0]:
//                      SNNBeamformer._delayed_template and the Hilbert design loop, restated operation for operation
//                      (no FMA contraction: numpy computes slope * (x - xp_j) + fp_j with a rounded product).
// k_design_eig         one CTA per real symmetric n x n matrix (n = 2M <= 128): cyclic Jacobi, parallel (round-robin)
//                      pair order, all eigenpairs, then the mode's output column.
// k_design_csum        mode 3: C_sum = sum_g C_g in g order (the host's running sum).
// k_design_pencil      mode 3: per g, Cholesky L L^T = E(C_sum + diag - C_g) and K = L^-1 E(C_g) L^-T, in global
//                      scratch (L2-resident).
//
// Complex Hermitian problems (modes 1-3) go through the real symmetric embedding E(H) = [[Re H, -Im H], [Im H, Re H]]:
// every eigenvalue of E(H) is doubled, and any vector [a; b] of the top eigenspace gives the complex u = a + i b.
//
// Storage (n = 128): A as a packed upper triangle (66 KB) next to the eigenvector matrix V (128 KB), both in shared
// memory (206 KB per CTA in all).  A full A next to V would take 256 KB; V in global memory would put the whole n x n
// rotation update of every round behind L2 latency.  A Jacobi round rotates n/2 disjoint pairs; with A packed, each
// 2 x 2 block A[{p1,q1},{p2,q2}] of two pairs is owned by one thread and updated as J1^T B J2 in one step, so
// symmetric storage needs no row phase and column phase.
#include <cuda_runtime.h>

#include <cmath>

#include "micloc_common.h"

namespace micloc {

constexpr int kEigMaxN = 2 * kDesignMaxMic;
constexpr int kEigMaxSweeps = 40;
constexpr int kBisectMaxIter = 400;

// ---------------------------------------------------------------------------
// delayed templates
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_design_templates(const DesignGeom geo, const double *__restrict__ time, const double *__restrict__ sig, long long T,
                   const double *__restrict__ doa, float *__restrict__ clips) {
    __shared__ double d[kDesignMaxMic];
    const long long g = blockIdx.y;
    const int M = geo.M;
    if (threadIdx.x < M) {
        const int m = threadIdx.x;
        d[m] = __ddiv_rn(__dmul_rn(-geo.r[m], cos(__dsub_rn(geo.theta[m], doa[g]))), geo.speed);
    }
    __syncthreads();
    double dmin = d[0];
    for (int m = 1; m < M; ++m) dmin = d[m] < dmin ? d[m] : dmin;
    const double t0 = time[0], tl = time[T - 1];
    const double inv_dt = 1.0 / (time[1] - time[0]);
    float *out = clips + g * T * M;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < T * M; e += (long long)gridDim.x * blockDim.x) {
        const long long t = e / M;
        const int m = (int)(e % M);
        double x = __dsub_rn(time[t], __dsub_rn(d[m], dmin));
        if (x < t0) x = t0;
        double r;
        if (x >= tl) {
            r = sig[T - 1];
        } else {
            // the j with time[j] <= x < time[j + 1]: guessed from the grid step, then moved onto the array's own values
            long long j = (long long)((x - t0) * inv_dt);
            j = j < 0 ? 0 : (j > T - 2 ? T - 2 : j);
            while (j > 0 && time[j] > x) --j;
            while (j < T - 2 && time[j + 1] <= x) ++j;
            const double slope = __ddiv_rn(__dsub_rn(sig[j + 1], sig[j]), __dsub_rn(time[j + 1], time[j]));
            r = __dadd_rn(__dmul_rn(slope, __dsub_rn(x, time[j])), sig[j]);
        }
        out[t * M + m] = __double2float_rn(r);
    }
}

int launch_design_templates(const DesignGeom &geo, const double *time, const double *sig, long long T,
                            const double *doa, long long G, float *clips, cudaStream_t st) {
    const long long per = (T * geo.M + 2047) / 2048;        // ~8 samples per thread
    const unsigned gx = (unsigned)(per < 1 ? 1 : (per > 4096 ? 4096 : per));
    for (long long g0 = 0; g0 < G; g0 += 65535) {
        const long long nb = G - g0 < 65535 ? G - g0 : 65535;
        k_design_templates<<<dim3(gx, (unsigned)nb), 256, 0, st>>>(geo, time, sig, T, doa + g0, clips + g0 * T * geo.M);
        count_launch(1);
    }
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}

// x /= d (recip = 0: a true division, numpy's real array / int) or x *= 1 / d (recip = 1: numpy's complex / int)
__global__ void __launch_bounds__(256) k_design_scale(double *__restrict__ x, long long n, double d, int recip) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    x[i] = recip ? x[i] * (1.0 / d) : x[i] / d;
}

int launch_design_scale(double *x, long long n, double d, bool recip, cudaStream_t st) {
    k_design_scale<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, n, d, recip ? 1 : 0);
    count_launch(1);
    MICLOC_CUDA(cudaGetLastError());
    return MICLOC_OK;
}

// ---------------------------------------------------------------------------
// mode 3 preparation
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_design_csum(const double *__restrict__ cov, long long G, int M, double *__restrict__ csum) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    const int ne = M * M * 2;
    if (e >= ne) return;
    double s = 0.0;
    for (long long g = 0; g < G; ++g) s += cov[g * ne + e];
    csum[e] = s;
}

// E(H)[i][j] of a complex M x M matrix h [M][M][2]
__device__ __forceinline__ double embed(const double *h, int M, int i, int j) {
    const int a = i < M ? i : i - M, b = j < M ? j : j - M;
    const double *z = h + ((long long)a * M + b) * 2;
    if ((i < M) == (j < M)) return z[0];
    return i < M ? -z[1] : z[1];
}

__global__ void __launch_bounds__(256)
k_design_pencil(const double *__restrict__ cov, const double *__restrict__ csum, int M, double *__restrict__ Lb,
                double *__restrict__ Kb) {
    const long long g = blockIdx.x;
    const int n = 2 * M, tid = threadIdx.x, nt = blockDim.x;
    const double *Cg = cov + g * M * M * 2;
    double *L = Lb + g * n * n, *K = Kb + g * n * n;
    // np.diag(np.mean(np.diag(C_sum)) * ones) / 10 added to C_sum (the diagonal is real)
    double mean = 0.0;
    for (int m = 0; m < M; ++m) mean += csum[((long long)m * M + m) * 2];
    const double ridge = mean / M / 10.0;
    for (int e = tid; e < n * n; e += nt) {
        const int i = e / n, j = e % n;
        double b = embed(csum, M, i, j);
        if (i == j) b = __dadd_rn(b, ridge);
        L[e] = __dsub_rn(b, embed(Cg, M, i, j));
        K[e] = embed(Cg, M, i, j);
    }
    __syncthreads();
    // right-looking Cholesky, lower triangle in place
    for (int k = 0; k < n; ++k) {
        if (tid == 0) L[k * n + k] = sqrt(L[k * n + k]);
        __syncthreads();
        const double lkk = L[k * n + k];
        for (int i = k + 1 + tid; i < n; i += nt) L[i * n + k] /= lkk;
        __syncthreads();
        const int w = n - k - 1;
        for (int e = tid; e < w * w; e += nt) {
            const int i = k + 1 + e / w, j = k + 1 + e % w;
            if (j <= i) L[i * n + j] -= L[i * n + k] * L[j * n + k];
        }
        __syncthreads();
    }
    // X = L^-1 E(C_g), one column per thread
    for (int j = tid; j < n; j += nt)
        for (int i = 0; i < n; ++i) {
            double s = K[i * n + j];
            for (int k = 0; k < i; ++k) s -= L[i * n + k] * K[k * n + j];
            K[i * n + j] = s / L[i * n + i];
        }
    __syncthreads();
    // K = X L^-T, one row per thread
    for (int i = tid; i < n; i += nt)
        for (int j = 0; j < n; ++j) {
            double s = K[i * n + j];
            for (int k = 0; k < j; ++k) s -= L[j * n + k] * K[i * n + k];
            K[i * n + j] = s / L[j * n + j];
        }
}

// ---------------------------------------------------------------------------
// the eigen-solver
// ---------------------------------------------------------------------------
struct EigSmem {
    size_t a, v, cs, vec, red, rowoff, pairs, blk, total;
};
__host__ __device__ inline EigSmem eig_smem(int n) {
    const int h = n / 2, nb = h * (h - 1) / 2;
    EigSmem s;
    s.a = 0;
    s.v = s.a + (size_t)n * (n + 1) / 2 * sizeof(double);
    s.cs = s.v + (size_t)n * n * sizeof(double);
    s.vec = s.cs + (size_t)2 * h * sizeof(double);
    s.red = s.vec + (size_t)3 * n * sizeof(double);
    s.rowoff = s.red + 64 * sizeof(double);
    s.pairs = s.rowoff + (size_t)n * sizeof(int);
    s.blk = s.pairs + (size_t)2 * h * sizeof(int);
    s.total = s.blk + (size_t)(nb > 0 ? nb : 1) * sizeof(unsigned short);
    s.total = (s.total + 15) & ~(size_t)15;
    return s;
}

__device__ __forceinline__ double block_sum(double v, double *red) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int warp = threadIdx.x / 32, nw = blockDim.x / 32;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[warp] = v;
    __syncthreads();
    double s = 0.0;
    for (int w = 0; w < nw; ++w) s += red[w];
    return s;
}

// in: mode 0 / 1: C [G][n][n] real; mode 2: cov [G][M][M][2]; mode 3: K [G][n][n] (k_design_pencil), L alongside.
__global__ void __launch_bounds__(512)
k_design_eig(int mode, const double *__restrict__ in, const double *__restrict__ Lb, int M, long long G,
             double *__restrict__ bf, double *__restrict__ value) {
    extern __shared__ __align__(16) unsigned char eig_sm[];
    const int n = 2 * M, h = M, tid = threadIdx.x, nt = blockDim.x;
    const int nblk = h * (h - 1) / 2;
    const EigSmem L = eig_smem(n);
    double *A = (double *)(eig_sm + L.a);
    double *V = (double *)(eig_sm + L.v);
    double *cs = (double *)(eig_sm + L.cs);
    double *vec = (double *)(eig_sm + L.vec);
    double *red = (double *)(eig_sm + L.red);
    int *rowoff = (int *)(eig_sm + L.rowoff);
    int *pp = (int *)(eig_sm + L.pairs), *qq = pp + h;
    unsigned short *blk = (unsigned short *)(eig_sm + L.blk);
    __shared__ int s_rot;
    const long long g = blockIdx.x;

    for (int i = tid; i < n; i += nt) rowoff[i] = i * n - i * (i - 1) / 2 - i;     // A(i, j) = A[rowoff[i] + j], i <= j
    for (int b = tid; b < nblk; b += nt) {
        int k1 = 0, e = b;
        while (e >= h - 1 - k1) { e -= h - 1 - k1; ++k1; }
        blk[b] = (unsigned short)(k1 * 64 + k1 + 1 + e);
    }
    if (tid == 0) s_rot = 0;
    __syncthreads();
    auto at = [&](int i, int j) -> double & { return i <= j ? A[rowoff[i] + j] : A[rowoff[j] + i]; };

    // ---- load the real symmetric matrix (upper triangle)
    if (mode == 0) {
        const double *C = in + g * n * n;
        for (int e = tid; e < n * n; e += nt) {
            const int i = e / n, j = e % n;
            if (j >= i) A[rowoff[i] + j] = C[e];
        }
    } else if (mode == 2) {
        const double *H = in + g * M * M * 2;
        for (int e = tid; e < n * n; e += nt) {
            const int i = e / n, j = e % n;
            if (j >= i) A[rowoff[i] + j] = embed(H, M, i, j);
        }
    } else if (mode == 3) {
        const double *K = in + g * n * n;
        for (int e = tid; e < n * n; e += nt) {
            const int i = e / n, j = e % n;
            if (j >= i) A[rowoff[i] + j] = 0.5 * (K[e] + K[j * n + i]);
        }
    } else {
        // A = (C11 + C22)/2 + i (C12 + C21^T)/2 staged in V's space, then E(A A^H)
        const double *C = in + g * n * n;
        double *Ac = V;
        for (int e = tid; e < M * M; e += nt) {
            const int i = e / M, j = e % M;
            Ac[2 * e] = (C[i * n + j] + C[(M + i) * n + M + j]) / 2;
            Ac[2 * e + 1] = (C[i * n + M + j] + C[(M + j) * n + i]) / 2;
        }
        __syncthreads();
        for (int e = tid; e < M * M; e += nt) {
            const int i = e / M, j = e % M;
            if (j < i) continue;
            double re = 0.0, im = 0.0;
            for (int k = 0; k < M; ++k) {
                const double ar = Ac[2 * (i * M + k)], ai = Ac[2 * (i * M + k) + 1];
                const double br = Ac[2 * (j * M + k)], bi = Ac[2 * (j * M + k) + 1];
                re += ar * br + ai * bi;
                im += ai * br - ar * bi;
            }
            A[rowoff[i] + j] = re;                     // Re H block, upper
            A[rowoff[M + i] + M + j] = re;
            A[rowoff[i] + M + j] = -im;                // -Im H[i][j]
            if (i != j) A[rowoff[j] + M + i] = im;     // -Im H[j][i] = Im H[i][j]
        }
        __syncthreads();
    }
    __syncthreads();
    for (int e = tid; e < n * n; e += nt) V[e] = (e / n == e % n) ? 1.0 : 0.0;
    __syncthreads();

    // ---- cyclic Jacobi, round-robin pairs: round r pairs (r, n-1) and ((r+k) mod (n-1), (r-k) mod (n-1))
    for (int sweep = 0; sweep < kEigMaxSweeps; ++sweep) {
        for (int r = 0; r < n - 1; ++r) {
            if (tid < h) {
                const int k = tid;
                const int p = k == 0 ? r : (r + k) % (n - 1);
                const int q = k == 0 ? n - 1 : (r - k + n - 1) % (n - 1);
                pp[k] = p; qq[k] = q;
                double &apq = at(p, q);
                const double app = at(p, p), aqq = at(q, q), a = apq;
                const double gg = 100.0 * fabs(a);
                double c = 1.0, s = 0.0;
                if (a != 0.0 && !(fabs(app) + gg == fabs(app) && fabs(aqq) + gg == fabs(aqq))) {
                    const double hh = aqq - app;
                    double t;
                    if (fabs(hh) + gg == fabs(hh)) {
                        t = a / hh;
                    } else {
                        const double theta = 0.5 * hh / a;
                        t = 1.0 / (fabs(theta) + sqrt(1.0 + theta * theta));
                        if (theta < 0.0) t = -t;
                    }
                    c = 1.0 / sqrt(t * t + 1.0);
                    s = t * c;
                    at(p, p) = app - t * a;
                    at(q, q) = aqq + t * a;
                    s_rot = 1;
                }
                apq = 0.0;
                cs[k] = c; cs[h + k] = s;
            }
            __syncthreads();
            for (int b = tid; b < nblk; b += nt) {
                const int k1 = blk[b] / 64, k2 = blk[b] % 64;
                const double c1 = cs[k1], s1 = cs[h + k1], c2 = cs[k2], s2 = cs[h + k2];
                if (s1 == 0.0 && s2 == 0.0) continue;
                const int p1 = pp[k1], q1 = qq[k1], p2 = pp[k2], q2 = qq[k2];
                double &b00 = at(p1, p2), &b01 = at(p1, q2), &b10 = at(q1, p2), &b11 = at(q1, q2);
                const double t00 = c2 * b00 - s2 * b01, t01 = s2 * b00 + c2 * b01;
                const double t10 = c2 * b10 - s2 * b11, t11 = s2 * b10 + c2 * b11;
                b00 = c1 * t00 - s1 * t10; b10 = s1 * t00 + c1 * t10;
                b01 = c1 * t01 - s1 * t11; b11 = s1 * t01 + c1 * t11;
            }
            for (int w = tid; w < n * h; w += nt) {
                const int i = w / h, k = w % h;
                const double c = cs[k], s = cs[h + k];
                if (s == 0.0) continue;
                double *row = V + i * n;
                const double vp = row[pp[k]], vq = row[qq[k]];
                row[pp[k]] = c * vp - s * vq;
                row[qq[k]] = s * vp + c * vq;
            }
            __syncthreads();
        }
        const bool done = s_rot == 0;
        __syncthreads();
        if (done) break;
        if (tid == 0) s_rot = 0;
        __syncthreads();
    }

    double *dd = vec, *th = vec + n, *wk = vec + 2 * n;
    if (mode == 0) {
        // _find_dc_removed_sing_vec: singular values |lambda|, theta = U^T 1, bisection between the two largest
        for (int k = tid; k < n; k += nt) {
            dd[k] = fabs(A[rowoff[k] + k]);
            double s = 0.0;
            for (int i = 0; i < n; ++i) s += V[i * n + k];
            th[k] = s;
        }
        __syncthreads();
        if (tid < 32) {
            double d0 = -1.0, d1 = -1.0;
            for (int k = 0; k < n; ++k) {
                const double x = dd[k];
                if (x > d0) { d1 = d0; d0 = x; } else if (x > d1) d1 = x;
            }
            double lo = d1, hi = d0;
            for (int it = 0; it < kBisectMaxIter && (hi - lo) / lo >= 1e-8; ++it) {
                const double mid = (lo + hi) / 2;
                double f = 0.0;
                for (int k = tid; k < n; k += 32) f += th[k] * th[k] / (dd[k] - mid);
                for (int o = 16; o > 0; o >>= 1) f += __shfl_xor_sync(0xffffffffu, f, o);
                if (f < 0.0) lo = mid; else hi = mid;
            }
            const double root = (lo + hi) / 2.0;
            for (int k = tid; k < n; k += 32) wk[k] = th[k] / (dd[k] - root);
            if (tid == 0) red[32] = root;
        }
        __syncthreads();
        const double root = red[32];
        double part = 0.0;
        double x = 0.0;
        if (tid < n) {
            for (int k = 0; k < n; ++k) x += V[tid * n + k] * wk[k];
            part = x * x;
        }
        const double nrm = sqrt(block_sum(part, red));
        if (tid < n) bf[(long long)tid * G + g] = x / nrm;
        if (value && tid == 0) value[g] = root;
        return;
    }

    // modes 1-3: the top eigenvector (first index of the largest eigenvalue)
    __syncthreads();
    if (tid == 0) {
        int km = 0;
        double lm = A[rowoff[0]];
        for (int k = 1; k < n; ++k)
            if (A[rowoff[k] + k] > lm) { lm = A[rowoff[k] + k]; km = k; }
        red[32] = lm;
        red[33] = (double)km;
    }
    __syncthreads();
    const double lmax = red[32];
    const int km = (int)red[33];
    for (int i = tid; i < n; i += nt) wk[i] = V[i * n + km];
    __syncthreads();
    if (mode == 3) {
        // x = L^-T y: back substitution on the Cholesky factor of the pencil
        const double *Lg = Lb + g * n * n;
        for (int i = n - 1; i >= 0; --i) {
            if (tid == 0) wk[i] = wk[i] / Lg[i * n + i];
            __syncthreads();
            const double xi = wk[i];
            for (int j = tid; j < i; j += nt) wk[j] -= Lg[i * n + j] * xi;
            __syncthreads();
        }
    }
    const double nrm = sqrt(block_sum(tid < n ? wk[tid] * wk[tid] : 0.0, red));
    // phase rule: the entry of largest modulus (first such index) real and positive
    if (tid == 0) {
        int mm = 0;
        double best = -1.0;
        for (int m = 0; m < M; ++m) {
            const double a2 = wk[m] * wk[m] + wk[M + m] * wk[M + m];
            if (a2 > best) { best = a2; mm = m; }
        }
        const double mag = sqrt(best);
        red[34] = mag > 0.0 ? wk[mm] / mag : 1.0;        // conj(u_mm) / |u_mm| = (ur - i ui) / mag
        red[35] = mag > 0.0 ? -wk[M + mm] / mag : 0.0;
        red[36] = (double)mm;
        red[37] = mag;
    }
    __syncthreads();
    const double pr = red[34], pi = red[35];
    const int mm = (int)red[36];
    for (int m = tid; m < M; m += nt) {
        const double ur = wk[m], ui = wk[M + m];
        double vr = (ur * pr - ui * pi) / nrm, vi = (ur * pi + ui * pr) / nrm;
        if (m == mm) { vr = red[37] / nrm; vi = 0.0; }
        if (mode == 1) {
            bf[(long long)m * G + g] = vr;
            bf[(long long)(M + m) * G + g] = vi;
        } else {
            bf[((long long)m * G + g) * 2] = vr;
            bf[((long long)m * G + g) * 2 + 1] = vi;
        }
    }
    if (value && tid == 0) value[g] = mode == 1 ? sqrt(lmax > 0.0 ? lmax : 0.0) : lmax;
}

int design_vectors(int mode, const double *cov, int M, long long G, double *bf, double *value, cudaStream_t st) {
    const int n = 2 * M;
    const EigSmem sm = eig_smem(n);
    const int threads = n >= 96 ? 512 : (n >= 32 ? 256 : 128);
    MICLOC_CUDA(cudaFuncSetAttribute(k_design_eig, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm.total));
    if (mode != 3) {
        k_design_eig<<<(unsigned)G, threads, sm.total, st>>>(mode, cov, nullptr, M, G, bf, value);
        count_launch(1);
        MICLOC_CUDA(cudaGetLastError());
        return MICLOC_OK;
    }
    double *scratch = nullptr;
    const size_t nn = (size_t)n * n;
    MICLOC_CUDA(cudaMallocAsync((void **)&scratch, ((size_t)M * M * 2 + 2 * (size_t)G * nn) * sizeof(double), st));
    double *csum = scratch, *Lb = csum + (size_t)M * M * 2, *Kb = Lb + (size_t)G * nn;
    k_design_csum<<<(unsigned)((M * M * 2 + 255) / 256), 256, 0, st>>>(cov, G, M, csum);
    k_design_pencil<<<(unsigned)G, 256, 0, st>>>(cov, csum, M, Lb, Kb);
    k_design_eig<<<(unsigned)G, threads, sm.total, st>>>(3, Kb, Lb, M, G, bf, value);
    count_launch(3);
    const cudaError_t e = cudaGetLastError();
    MICLOC_CUDA(cudaFreeAsync(scratch, st));
    MICLOC_CUDA(e);
    return MICLOC_OK;
}

}  // namespace micloc
