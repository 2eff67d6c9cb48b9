// Block-cooperative small dense linear algebra on shared memory (fp64).
// One CTA owns one world's matrices; all routines are called by every thread of the CTA
// unless named warp_* (then: by all lanes of ONE warp).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace dsdf {

#define DSDF_FULL 0xffffffffu

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per size increase of a kernel, not once per launch
// (*granted: a per-kernel static of the calling translation unit; one process drives one GPU).
template <class K> static inline cudaError_t ensure_smem(K kernel, size_t smem, size_t* granted) {
    if (smem <= *granted) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) *granted = smem;
    return e;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(DSDF_FULL, v, o);
    return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(DSDF_FULL, v, o));
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(DSDF_FULL, v, o));
    return v;
}

// two minima and two maxima over the warp, the four butterflies interleaved (independent shuffles per level)
__device__ __forceinline__ void warp_minmax2(double& mn0, double& mn1, double& mx0, double& mx1) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double a = __shfl_xor_sync(DSDF_FULL, mn0, o), b = __shfl_xor_sync(DSDF_FULL, mn1, o);
        const double c = __shfl_xor_sync(DSDF_FULL, mx0, o), d = __shfl_xor_sync(DSDF_FULL, mx1, o);
        mn0 = fmin(mn0, a); mn1 = fmin(mn1, b); mx0 = fmax(mx0, c); mx1 = fmax(mx1, d);
    }
}

// a / b given r = 1 / b (correctly rounded): q = RN(a r) corrected by one exact-remainder step, fma(fma(-q, b, a), r, q),
// is the correctly rounded quotient RN(a / b) (Markstein's theorem), i.e. the bits of a / b, as long as nothing over- or
// underflows.  Operands outside [2^-500, 2^500] in magnitude (zeros, non-finite values included) take the plain
// division, so the reciprocal of a divisor that repeats replaces the dependent divisions without changing a bit.
__device__ __forceinline__ bool div_rcp_ok(double x) { const double ax = fabs(x); return ax > 0x1p-500 && ax < 0x1p500; }
__device__ __forceinline__ double div_rcp(double a, double b, double r) {
    if (!(div_rcp_ok(a) && div_rcp_ok(b))) return a / b;
    const double q = __dmul_rn(a, r);
    return fma(fma(-q, b, a), r, q);
}

// Deterministic block reductions; `red` is >= 33 doubles of shared memory. Result broadcast to all threads.
enum { RED_SUM = 0, RED_MIN = 1, RED_MAX = 2 };
template <int OP>
__device__ __forceinline__ double block_reduce(double v, double* red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = OP == RED_SUM ? warp_sum(v) : (OP == RED_MIN ? warp_min(v) : warp_max(v));
    __syncthreads();                       // protect `red` from the previous use
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (warp == 0) {
        double id = OP == RED_SUM ? 0.0 : (OP == RED_MIN ? INFINITY : -INFINITY);
        double t = lane < nw ? red[lane] : id;
        t = OP == RED_SUM ? warp_sum(t) : (OP == RED_MIN ? warp_min(t) : warp_max(t));
        if (lane == 0) red[32] = t;
    }
    __syncthreads();
    return red[32];
}

// In-place LU with partial (row) pivoting, A is n x n row-major with leading dimension ld.
// perm[i] = original row now at row i.  *fail set to 1 on a zero / NaN pivot column.
__device__ inline void block_lu(double* A, int ld, int n, int* perm, int* s_piv, int* fail) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
    for (int i = tid; i < n; i += nt) perm[i] = i;
    __syncthreads();
    for (int k = 0; k < n; ++k) {
        if (warp == 0) {
            double best = -1.0;
            int bi = k;
            for (int i = k + lane; i < n; i += 32) {
                double a = fabs(A[i * ld + k]);
                if (a > best) { best = a; bi = i; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                double ob = __shfl_xor_sync(DSDF_FULL, best, o);
                int oi = __shfl_xor_sync(DSDF_FULL, bi, o);
                if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
            }
            if (lane == 0) {
                *s_piv = bi;
                if (!(best > 0.0)) *fail = 1;
            }
        }
        __syncthreads();
        const int r = *s_piv;
        if (r != k) {
            for (int j = tid; j < n; j += nt) {
                double t = A[k * ld + j];
                A[k * ld + j] = A[r * ld + j];
                A[r * ld + j] = t;
            }
            if (tid == 0) { int t = perm[k]; perm[k] = perm[r]; perm[r] = t; }
        }
        __syncthreads();
        const double piv = A[k * ld + k];
        for (int i = k + 1 + tid; i < n; i += nt) A[i * ld + k] /= piv;
        __syncthreads();
        for (int i = k + 1 + warp; i < n; i += nw) {
            const double l = A[i * ld + k];
            for (int j = k + 1 + lane; j < n; j += 32) A[i * ld + j] -= l * A[k * ld + j];
        }
        __syncthreads();
    }
}

// x <- L^-1 x (unit lower triangle of LU), one warp, x in shared memory.
__device__ inline void warp_trsv_lower_unit(const double* LU, int ld, int n, double* x) {
    const int lane = threadIdx.x & 31;
    for (int c0 = 0; c0 < n; c0 += 32) {
        const int w = min(32, n - c0), r = c0 + lane;
        const bool act = lane < w;
        double v = act ? x[r] : 0.0;
        for (int kk = 0; kk < w; ++kk) {
            double xk = __shfl_sync(DSDF_FULL, v, kk);
            if (act && lane > kk) v -= LU[r * ld + c0 + kk] * xk;
        }
        if (act) x[r] = v;
        __syncwarp();
        for (int r2 = c0 + 32 + lane; r2 < n; r2 += 32) {
            double acc = x[r2];
            for (int kk = 0; kk < w; ++kk) acc -= LU[r2 * ld + c0 + kk] * x[c0 + kk];
            x[r2] = acc;
        }
        __syncwarp();
    }
}

// x <- U^-1 x (upper triangle incl. diagonal of LU), one warp.
__device__ inline void warp_trsv_upper(const double* LU, int ld, int n, double* x) {
    const int lane = threadIdx.x & 31;
    for (int cb = (n + 31) / 32 - 1; cb >= 0; --cb) {
        const int c0 = cb * 32, w = min(32, n - c0), r = c0 + lane;
        const bool act = lane < w;
        double v = act ? x[r] : 0.0;
        const double dg = act ? LU[r * ld + r] : 1.0;
        const double rdg = 1.0 / dg;           // every lane its own diagonal at once, off the dependent chain below
        for (int kk = w - 1; kk >= 0; --kk) {
            if (lane == kk) v = div_rcp(v, dg, rdg);
            double xk = __shfl_sync(DSDF_FULL, v, kk);
            if (act && lane < kk) v -= LU[r * ld + c0 + kk] * xk;
        }
        if (act) x[r] = v;
        __syncwarp();
        for (int r2 = lane; r2 < c0; r2 += 32) {
            double acc = x[r2];
            for (int kk = w - 1; kk >= 0; --kk) acc -= LU[r2 * ld + c0 + kk] * x[c0 + kk];
            x[r2] = acc;
        }
        __syncwarp();
    }
}

// x <- (P L U)^-1 b.  b and x in shared memory, may NOT alias. Called by all threads; warp 0 works.
__device__ inline void block_lu_solve(const double* LU, int ld, int n, const int* perm, const double* b, double* x) {
    if (threadIdx.x < 32) {
        for (int i = threadIdx.x; i < n; i += 32) x[i] = b[perm[i]];
        __syncwarp();
        warp_trsv_lower_unit(LU, ld, n, x);
        warp_trsv_upper(LU, ld, n, x);
    }
    __syncthreads();
}

// In-place LU with partial (row) pivoting by one warp, same contract as block_lu; returns 1 on a zero / NaN pivot column.
__device__ inline int warp_lu(double* A, int ld, int n, int* perm) {
    const int lane = threadIdx.x & 31;
    int fail = 0;
    for (int i = lane; i < n; i += 32) perm[i] = i;
    __syncwarp();
    for (int k = 0; k < n; ++k) {
        // pivot search over the m = n - k remaining rows by the lowest g lanes, g = 8, 16 or 32 the smallest >= min(m, 32);
        // lanes L and L + g, L + 2g, ... read the same rows, so every lane holds the result after log2(g) butterfly levels.
        // The combine keeps the largest |a| and the lowest index on ties (NaN entries never win), an order-free
        // selection: the same pivot as the full-warp search.
        const int m = n - k, g = m <= 8 ? 8 : (m <= 16 ? 16 : 32);
        double best = -1.0; int bi = k;
        for (int i = k + (lane & (g - 1)); i < n; i += g) { double v = fabs(A[i * ld + k]); if (v > best) { best = v; bi = i; } }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            if (o >= g) continue;                  // warp-uniform
            double ob = __shfl_xor_sync(DSDF_FULL, best, o); int oi = __shfl_xor_sync(DSDF_FULL, bi, o);
            if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
        }
        if (!(best > 0.0)) fail = 1;
        if (bi != k) {
            for (int j = lane; j < n; j += 32) { double t = A[k * ld + j]; A[k * ld + j] = A[bi * ld + j]; A[bi * ld + j] = t; }
            if (lane == 0) { int t = perm[k]; perm[k] = perm[bi]; perm[bi] = t; }
        }
        __syncwarp();
        const double piv = A[k * ld + k];
        for (int i = k + 1 + lane; i < n; i += 32) {
            const double l = A[i * ld + k] / piv;
            A[i * ld + k] = l;
            for (int j = k + 1; j < n; ++j) A[i * ld + j] -= l * A[k * ld + j];
        }
        __syncwarp();
    }
    return fail;
}

// x <- (P L U)^-1 b by one warp.  b and x in shared memory, may NOT alias.
__device__ inline void warp_lu_solve(const double* LU, int ld, int n, const int* perm, const double* b, double* x) {
    const int lane = threadIdx.x & 31;
    for (int i = lane; i < n; i += 32) x[i] = b[perm[i]];
    __syncwarp();
    warp_trsv_lower_unit(LU, ld, n, x);
    warp_trsv_upper(LU, ld, n, x);
    __syncwarp();
}

// Per-thread solve of one right-hand side with a SMALL factorisation (used for many-RHS solves):
// src read with stride ss, result written with stride ds; `n` small (nz / neq).
__device__ inline void thread_lu_solve(const double* LU, int ld, int n, const int* perm,
                                       const double* src, int ss, double* dst, int ds) {
    for (int i = 0; i < n; ++i) {
        double acc = src[perm[i] * ss];
        for (int k = 0; k < i; ++k) acc -= LU[i * ld + k] * dst[k * ds];
        dst[i * ds] = acc;
    }
    for (int i = n - 1; i >= 0; --i) {
        double acc = dst[i * ds];
        for (int k = i + 1; k < n; ++k) acc -= LU[i * ld + k] * dst[k * ds];
        dst[i * ds] = acc / LU[i * ld + i];
    }
}

}  // namespace dsdf
