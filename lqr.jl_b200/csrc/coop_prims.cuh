// coop_prims.cuh — cooperative dense primitives: G threads of a group (a warp, or a whole CTA) work on one small
// matrix in shared or global memory.  Stand-ins for the BLAS / LAPACK calls the reference makes (gemm, potrf, trsm).
// Used by the general KKT kernel (kkt_coop.cu) and the condensed least-squares path (lsq.cu).
#pragma once
#include "riccati_kernels.cuh"  // group_sync

// ------------------------------------------------------------------ cooperative primitives ----
// All matrices column-major with explicit leading dimension; every primitive ends with a group sync.
template <int G>
__device__ __forceinline__ void co_gemm(int ta, int tb, int M, int Nn, int K, double alpha,
                                        const double *A, int lda, const double *B, int ldb, double beta,
                                        double *C, int ldc, int t) {
    for (int e = t; e < M * Nn; e += G) {
        const int i = e % M, j = e / M;
        double s = 0.0;
        for (int l = 0; l < K; ++l) {
            const double a = ta ? A[l + i * lda] : A[i + l * lda];
            const double b = tb ? B[j + l * ldb] : B[l + j * ldb];
            s = fma(a, b, s);
        }
        C[i + j * ldc] = (beta == 0.0) ? alpha * s : fma(alpha, s, beta * C[i + j * ldc]);
    }
    group_sync<G>();
}

// in-place upper Cholesky (right-looking); strict lower untouched.  info: 1-based bad pivot or 0.
template <int G>
__device__ __forceinline__ int co_chol(double *A, int k, int lda, int t) {
    int info = 0;
    for (int j = 0; j < k; ++j) {
        const double djj = A[j + j * lda];
        if (!(djj > 0.0) && info == 0) info = j + 1;
        const double d = sqrt(djj);
        group_sync<G>();
        for (int i = j + t; i < k; i += G) A[j + i * lda] = (i == j) ? d : A[j + i * lda] / d;
        group_sync<G>();
        const int rem = k - j - 1;
        for (int e = t; e < rem * rem; e += G) {
            const int a = j + 1 + e % rem, b = j + 1 + e / rem;
            if (a <= b) A[a + b * lda] = fma(-A[j + a * lda], A[j + b * lda], A[a + b * lda]);
        }
        group_sync<G>();
    }
    return info;
}

// B <- U^-T B  (one thread per right-hand-side column)
template <int G>
__device__ __forceinline__ void co_trsm_ut(const double *U, int k, int ldu, double *B, int nrhs, int ldb,
                                           int t) {
    for (int c = t; c < nrhs; c += G) {
        double *x = B + (size_t)c * ldb;
        for (int i = 0; i < k; ++i) {
            double s = x[i];
            for (int l = 0; l < i; ++l) s = fma(-U[l + i * ldu], x[l], s);
            x[i] = s / U[i + i * ldu];
        }
    }
    group_sync<G>();
}

// B <- U^-1 B
template <int G>
__device__ __forceinline__ void co_trsm_un(const double *U, int k, int ldu, double *B, int nrhs, int ldb,
                                           int t) {
    for (int c = t; c < nrhs; c += G) {
        double *x = B + (size_t)c * ldb;
        for (int i = k - 1; i >= 0; --i) {
            double s = x[i];
            for (int l = i + 1; l < k; ++l) s = fma(-U[i + l * ldu], x[l], s);
            x[i] = s / U[i + i * ldu];
        }
    }
    group_sync<G>();
}

// Sum of v over the G threads, returned to every thread.  A fixed xor-butterfly inside each warp, then (G > 32) the
// warp totals summed in warp order by every thread: the result is the same bits on every run.  `red` holds G/32
// doubles of shared memory.
template <int G>
__device__ __forceinline__ double co_sum(double v, double *red, int t) {
    constexpr int W = G < 32 ? G : 32;
    for (int o = W / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o, W);
    if constexpr (G <= 32) {
        return v;
    } else {
        if ((t & 31) == 0) red[t >> 5] = v;
        group_sync<G>();
        double s = 0.0;
        for (int w = 0; w < G / 32; ++w) s += red[w];
        group_sync<G>();
        return s;
    }
}

// In-place LU with row pivoting (getrf): P A = L U, L unit lower below the diagonal, U on and above it.  Whole rows
// are swapped, as LAPACK does.  The pivot of column j is the first row of largest |a_ij|, i >= j, found by a group
// reduction.  piv[j] = the row swapped with row j.  `red` holds 2 G/32 doubles.  Returns 0, or the 1-based column
// of the first zero pivot (the factorisation then stops).
template <int G>
__device__ __forceinline__ int co_lu(double *A, int k, int lda, int *piv, double *red, int t) {
    constexpr int W = G < 32 ? G : 32;
    for (int j = 0; j < k; ++j) {
        double best = -1.0;
        int bi = k;
        for (int i = j + t; i < k; i += G) {
            const double a = fabs(A[i + j * lda]);
            if (a > best) best = a, bi = i;  // rows ascend per thread: the first of equal values stays
        }
        for (int o = W / 2; o > 0; o >>= 1) {
            const double ob = __shfl_xor_sync(0xffffffffu, best, o, W);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o, W);
            if (ob > best || (ob == best && oi < bi)) best = ob, bi = oi;
        }
        if constexpr (G > 32) {
            if ((t & 31) == 0) red[2 * (t >> 5)] = best, red[2 * (t >> 5) + 1] = (double)bi;
            group_sync<G>();
            best = -1.0, bi = k;
            for (int w = 0; w < G / 32; ++w) {
                const double ob = red[2 * w];
                const int oi = (int)red[2 * w + 1];
                if (ob > best || (ob == best && oi < bi)) best = ob, bi = oi;
            }
        }
        if (!(best > 0.0)) {  // zero column (or NaN throughout): singular
            group_sync<G>();
            return j + 1;
        }
        if (t == 0) piv[j] = bi;
        if (bi != j)
            for (int c = t; c < k; c += G) {
                const double x = A[j + c * lda];
                A[j + c * lda] = A[bi + c * lda];
                A[bi + c * lda] = x;
            }
        group_sync<G>();
        const double d = A[j + j * lda];
        for (int i = j + 1 + t; i < k; i += G) A[i + j * lda] /= d;
        group_sync<G>();
        const int rem = k - j - 1;
        for (int e = t; e < rem * rem; e += G) {
            const int a = j + 1 + e % rem, b = j + 1 + e / rem;
            A[a + b * lda] = fma(-A[a + j * lda], A[j + b * lda], A[a + b * lda]);
        }
        group_sync<G>();
    }
    return 0;
}

// B <- A^-1 B with the factors of co_lu (getrs, one thread per right-hand-side column)
template <int G>
__device__ __forceinline__ void co_lu_solve(const double *LU, int k, int lda, const int *piv, double *B, int nrhs,
                                            int ldb, int t) {
    for (int c = t; c < nrhs; c += G) {
        double *x = B + (size_t)c * ldb;
        for (int j = 0; j < k; ++j) {
            const int p = piv[j];
            if (p != j) {
                const double v = x[j];
                x[j] = x[p];
                x[p] = v;
            }
        }
        for (int i = 1; i < k; ++i) {
            double s = x[i];
            for (int l = 0; l < i; ++l) s = fma(-LU[i + l * lda], x[l], s);
            x[i] = s;
        }
        for (int i = k - 1; i >= 0; --i) {
            double s = x[i];
            for (int l = i + 1; l < k; ++l) s = fma(-LU[i + l * lda], x[l], s);
            x[i] = s / LU[i + i * lda];
        }
    }
    group_sync<G>();
}

