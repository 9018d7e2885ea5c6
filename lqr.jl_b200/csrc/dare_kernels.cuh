// dare_kernels.cuh — batched discrete algebraic Riccati equation (DESIGN §4.11).
//
//   dare_kernel<G>       P = Q + A'PA - A'PB (R + B'PB)^-1 B'PA by the structured doubling algorithm, then
//                        K = (R + B'PB)^-1 B'PA (u = -K x, the sign of lqrb_riccati_f64).
//   dare_grad_kernel<G>  the gradient of l(P, K) through it: one Stein equation Y = Acl Y Acl' + S, solved by Smith
//                        doubling, then closed-form products.
//
// G threads own one instance (32: a warp, four instances per 128-thread block; 256: a CTA), every operand lives in
// shared memory, the instance-major column-major caller arrays are read and written directly.  Every sum runs in a
// fixed order (co_gemm's per-element loops, co_sum's fixed butterfly), so the results are bitwise reproducible.
#pragma once
#include "coop_prims.cuh"

// Relative size of the last doubling increment at which both iterations stop: ||dH||_F <= eps ||H||_F.  The
// increments go to zero (A_k -> 0 as Acl^(2^k)), they are not a rounding-noise difference, so the test is met in one
// more step once the iteration converges quadratically; at eps = 2^-52 a further step would change H below its last
// bit in norm.
#define DARE_EPS 2.220446049250313e-16
#define DARE_MAX_STEPS 64

// info codes of lqrb_dare_f64 / lqrb_dare_grad_f64 (include/lqrb200.h)
#define DARE_NOT_CONVERGED 1
#define DARE_R_NOT_PD 1000
#define DARE_W_SINGULAR 2000
#define DARE_GAIN_NOT_PD 3000

// shared memory doubles per instance: A_k | G_k | H_k | W | W^-1 [A_k G_k] | pivots | reductions
__host__ __device__ inline size_t dare_smem_doubles(int n) { return (size_t)6 * n * n + n + 16; }
// P | PA | M | T | Y (n x n) | B | PB | BG (later K Y) (n x m) | K | Yk (m x n) | E | Gbar (m x m) | reductions
__host__ __device__ inline size_t dare_grad_smem_doubles(int n, int m) {
    return (size_t)5 * n * n + 5 * n * m + 2 * m * m + 16;
}

// count of non-finite values among a[0..cnt), summed over the group (0 on every thread when all are finite)
template <int G>
__device__ __forceinline__ double co_nonfinite(const double *a, int cnt, double *red, int t) {
    double c = 0.0;
    for (int e = t; e < cnt; e += G) c += isfinite(a[e]) ? 0.0 : 1.0;
    return co_sum<G>(c, red, t);
}

// E <- R (upper triangle read, both written) and the Cholesky factor of R + B'PB in place; K <- E^-1 B'PA.
// PB, PA, B as in the callers.  Returns 0 or the 1-based bad pivot.
template <int G>
__device__ __forceinline__ int co_dare_gain(const double *R, const double *B, const double *PB, const double *PA,
                                            double *E, double *K, int n, int m, int t) {
    for (int e = t; e < m * m; e += G) {
        const int i = e % m, j = e / m;
        E[e] = R[i <= j ? i + j * m : j + i * m];
    }
    group_sync<G>();
    co_gemm<G>(1, 0, m, m, n, 1.0, B, n, PB, n, 1.0, E, m, t);  // E = R + B'PB
    co_gemm<G>(1, 0, m, n, n, 1.0, B, n, PA, n, 0.0, K, m, t);  // K = B'PA
    const int bad = co_chol<G>(E, m, m, t);
    if (bad) return bad;
    co_trsm_ut<G>(E, m, m, K, n, m, t);
    co_trsm_un<G>(E, m, m, K, n, m, t);
    return 0;
}

template <int G, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
    dare_kernel(const double *__restrict__ Ag, const double *__restrict__ Bg, const double *__restrict__ Qg,
                const double *__restrict__ Rg, double *__restrict__ Pg, double *__restrict__ Kg,
                int32_t *__restrict__ iters, int32_t *__restrict__ info, int n, int m, int64_t batch) {
    extern __shared__ double smem[];
    constexpr int IPC = THREADS / G;
    const int g = threadIdx.x / G, t = threadIdx.x % G;
    const int64_t inst_raw = (int64_t)blockIdx.x * IPC + g;
    const bool active = inst_raw < batch;
    const int64_t inst = active ? inst_raw : batch - 1;  // idle groups shadow a valid instance
    const int nn = n * n;
    double *s = smem + (size_t)g * dare_smem_doubles(n);
    double *Ak = s, *Gk = Ak + nn, *Hk = Gk + nn, *W = Hk + nn, *X = W + nn, *X2 = X + nn;
    int *piv = (int *)(X2 + nn);
    double *red = X2 + nn + n;  // 16 doubles: 2 G/32 for co_lu, G/32 for co_sum
    const double *A = Ag + inst * nn, *B = Bg + inst * (int64_t)n * m, *Q = Qg + inst * nn,
                 *R = Rg + inst * (int64_t)m * m;

    // A_0 = A, H_0 = Q (upper triangle), G_0 = B R^-1 B' = (U^-T B')' (U^-T B') with R = U'U
    double *Y = W, *E = X;  // B' (m x n, ld m) and the factor of R
    for (int e = t; e < nn; e += G) {
        const int i = e % n, j = e / n;
        Ak[e] = A[e];
        Hk[e] = Q[i <= j ? e : j + i * n];
    }
    for (int e = t; e < n * m; e += G) {
        const int i = e % m, j = e / m;
        Y[e] = B[j + i * n];
    }
    for (int e = t; e < m * m; e += G) {
        const int i = e % m, j = e / m;
        E[e] = R[i <= j ? e : j + i * m];
    }
    group_sync<G>();
    int code = 0, steps = 0;
    if (co_nonfinite<G>(Ak, nn, red, t) + co_nonfinite<G>(Hk, nn, red, t) + co_nonfinite<G>(Y, n * m, red, t) +
            co_nonfinite<G>(E, m * m, red, t) > 0.0)
        code = DARE_NOT_CONVERGED;
    if (!code) {
        const int bad = co_chol<G>(E, m, m, t);
        if (bad) code = DARE_R_NOT_PD + bad;
    }
    if (!code) {
        co_trsm_ut<G>(E, m, m, Y, n, m, t);
        co_gemm<G>(1, 0, n, n, m, 1.0, Y, m, Y, m, 0.0, Gk, n, t);
        code = DARE_NOT_CONVERGED;
        for (int k = 1; k <= DARE_MAX_STEPS; ++k) {
            steps = k;
            // W = I + G_k H_k ; X = [A_k | G_k]
            for (int e = t; e < nn; e += G) {
                W[e] = (e % n == e / n) ? 1.0 : 0.0;
                X[e] = Ak[e];
                X2[e] = Gk[e];
            }
            group_sync<G>();
            co_gemm<G>(0, 0, n, n, n, 1.0, Gk, n, Hk, n, 1.0, W, n, t);
            const int bad = co_lu<G>(W, n, n, piv, red, t);
            if (bad) {
                code = DARE_W_SINGULAR + bad;
                break;
            }
            co_lu_solve<G>(W, n, n, piv, X, 2 * n, n, t);  // X = W^-1 A_k | W^-1 G_k
            // H_{k+1} = H_k + A_k' H_k W^-1 A_k, with ||dH|| and ||H_{k+1}|| for the stopping rule
            co_gemm<G>(0, 0, n, n, n, 1.0, Hk, n, X, n, 0.0, W, n, t);
            double dd = 0.0, hh = 0.0;
            for (int e = t; e < nn; e += G) {
                const int i = e % n, j = e / n;
                double d = 0.0;
                for (int l = 0; l < n; ++l) d = fma(Ak[l + i * n], W[l + j * n], d);
                const double h = Hk[e] + d;
                Hk[e] = h;
                dd = fma(d, d, dd);
                hh = fma(h, h, hh);
            }
            group_sync<G>();
            dd = co_sum<G>(dd, red, t);
            hh = co_sum<G>(hh, red, t);
            // G_{k+1} = G_k + A_k W^-1 G_k A_k' ; A_{k+1} = A_k W^-1 A_k (into X2, then back to A_k)
            co_gemm<G>(0, 0, n, n, n, 1.0, Ak, n, X2, n, 0.0, W, n, t);
            co_gemm<G>(0, 1, n, n, n, 1.0, W, n, Ak, n, 1.0, Gk, n, t);
            co_gemm<G>(0, 0, n, n, n, 1.0, Ak, n, X, n, 0.0, X2, n, t);
            // symmetrise G and H (one thread per pair), A_k <- A_{k+1}
            for (int e = t; e < nn; e += G) {
                const int i = e % n, j = e / n;
                Ak[e] = X2[e];
                if (i < j) {
                    const double g2 = 0.5 * (Gk[e] + Gk[j + i * n]), h2 = 0.5 * (Hk[e] + Hk[j + i * n]);
                    Gk[e] = Gk[j + i * n] = g2;
                    Hk[e] = Hk[j + i * n] = h2;
                }
            }
            group_sync<G>();
            if (!isfinite(hh) || !isfinite(dd)) break;  // diverged: no stabilising solution (or overflow)
            if (dd <= DARE_EPS * DARE_EPS * hh) {
                code = 0;
                break;
            }
        }
    }
    // K = (R + B'PB)^-1 B'PA with P = H_k.  Free slots: B | A, then K once PA is formed | PA | PB | E
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    double *K = W;
    if (!code && Kg) {
        double *Bs = Ak, *As = W, *PA = X, *PB = X2, *E2 = Gk;
        for (int e = t; e < nn; e += G) As[e] = A[e];
        for (int e = t; e < n * m; e += G) Bs[e] = B[e];
        group_sync<G>();
        co_gemm<G>(0, 0, n, m, n, 1.0, Hk, n, Bs, n, 0.0, PB, n, t);
        co_gemm<G>(0, 0, n, n, n, 1.0, Hk, n, As, n, 0.0, PA, n, t);
        const int bad = co_dare_gain<G>(R, Bs, PB, PA, E2, K, n, m, t);
        if (bad) code = DARE_GAIN_NOT_PD + bad;
    }
    if (active) {
        // a failed instance's P and K are NaN: nothing downstream can take them for a solution
        if (Kg)
            for (int e = t; e < m * n; e += G) Kg[inst * (int64_t)m * n + e] = code ? nan : K[e];
        if (Pg)
            for (int e = t; e < nn; e += G) Pg[inst * nn + e] = code ? nan : Hk[e];
        if (t == 0) {
            if (iters) iters[inst] = steps;
            if (info) info[inst] = code;
        }
    }
}

// Gradient of l(P, K) (DESIGN §4.11): with Gc = R + B'PB, Acl = A - BK, sym(X) = (X + X')/2,
//   Yk = Gc^-1 dK, Gbar = -sym(Yk K'), S = sym(dP) + B Gbar B' + sym(B Yk A'), Y = Acl Y Acl' + S,
//   gQ = Y, gR = K Y K' + Gbar, gA = 2 P Acl Y + P B Yk, gB = -2 P Acl Y K' + P A Yk' + 2 P B Gbar.
template <int G, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
    dare_grad_kernel(const double *__restrict__ Ag, const double *__restrict__ Bg, const double *__restrict__ Rg,
                     const double *__restrict__ Pg, const double *__restrict__ dPg, const double *__restrict__ dKg,
                     double *__restrict__ gA, double *__restrict__ gB, double *__restrict__ gQ,
                     double *__restrict__ gR, int32_t *__restrict__ info, int n, int m, int64_t batch) {
    extern __shared__ double smem[];
    constexpr int IPC = THREADS / G;
    const int g = threadIdx.x / G, t = threadIdx.x % G;
    const int64_t inst_raw = (int64_t)blockIdx.x * IPC + g;
    const bool active = inst_raw < batch;
    const int64_t inst = active ? inst_raw : batch - 1;
    const int nn = n * n, nm = n * m, mm = m * m;
    double *s = smem + (size_t)g * dare_grad_smem_doubles(n, m);
    double *P = s, *PA = P + nn, *M = PA + nn, *T = M + nn, *Y = T + nn, *B = Y + nn, *PB = B + nm, *BG = PB + nm,
           *K = BG + nm, *Yk = K + nm, *E = Yk + nm, *Gb = E + mm, *red = Gb + mm;
    const double *A = Ag + inst * nn, *R = Rg + inst * (int64_t)mm;
    const double *dP = dPg ? dPg + inst * nn : nullptr, *dK = dKg ? dKg + inst * (int64_t)nm : nullptr;

    double *As = T;  // A, until the Stein doubling needs T
    for (int e = t; e < nn; e += G) {
        const int i = e % n, j = e / n;
        As[e] = A[e];
        P[e] = Pg[inst * nn + (i <= j ? e : j + i * n)];
    }
    for (int e = t; e < nm; e += G) B[e] = Bg[inst * (int64_t)nm + e];
    group_sync<G>();
    co_gemm<G>(0, 0, n, m, n, 1.0, P, n, B, n, 0.0, PB, n, t);
    co_gemm<G>(0, 0, n, n, n, 1.0, P, n, As, n, 0.0, PA, n, t);
    int code = co_dare_gain<G>(R, B, PB, PA, E, K, n, m, t);
    if (code) code += DARE_GAIN_NOT_PD;
    if (!code) {
        // Yk = Gc^-1 dK ; Gbar = -sym(Yk K')
        for (int e = t; e < nm; e += G) Yk[e] = dK ? dK[e] : 0.0;
        group_sync<G>();
        co_trsm_ut<G>(E, m, m, Yk, n, m, t);
        co_trsm_un<G>(E, m, m, Yk, n, m, t);
        for (int e = t; e < mm; e += G) {
            const int i = e % m, j = e / m;
            double a = 0.0, b = 0.0;
            for (int l = 0; l < n; ++l) {
                a = fma(Yk[i + l * m], K[j + l * m], a);
                b = fma(Yk[j + l * m], K[i + l * m], b);
            }
            Gb[e] = -0.5 * (a + b);
        }
        group_sync<G>();
        // BG = B Gbar ; M = B Yk (temporarily)
        co_gemm<G>(0, 0, n, m, m, 1.0, B, n, Gb, m, 0.0, BG, n, t);
        co_gemm<G>(0, 0, n, n, m, 1.0, B, n, Yk, m, 0.0, M, n, t);
        // S = sym(dP) + BG B' + sym(M A'), into Y
        for (int e = t; e < nn; e += G) {
            const int i = e % n, j = e / n;
            double v = dP ? 0.5 * (dP[e] + dP[j + i * n]) : 0.0;
            double a = 0.0, b = 0.0;
            for (int l = 0; l < m; ++l) v = fma(BG[i + l * n], B[j + l * n], v);
            for (int l = 0; l < n; ++l) {
                a = fma(M[i + l * n], As[j + l * n], a);
                b = fma(M[j + l * n], As[i + l * n], b);
            }
            Y[e] = v + 0.5 * (a + b);
        }
        group_sync<G>();
        // M = Acl = A - B K
        for (int e = t; e < nn; e += G) {
            const int i = e % n, j = e / n;
            double v = As[e];
            for (int l = 0; l < m; ++l) v = fma(-B[i + l * n], K[l + j * m], v);
            M[e] = v;
        }
        group_sync<G>();
        // Smith doubling: Y <- Y + M Y M', M <- M M, from Y = S, M = Acl
        code = DARE_NOT_CONVERGED;
        for (int k = 1; k <= DARE_MAX_STEPS; ++k) {
            co_gemm<G>(0, 0, n, n, n, 1.0, M, n, Y, n, 0.0, T, n, t);
            double dd = 0.0, yy = 0.0;
            for (int e = t; e < nn; e += G) {
                const int i = e % n, j = e / n;
                double d = 0.0;
                for (int l = 0; l < n; ++l) d = fma(T[i + l * n], M[j + l * n], d);
                const double y = Y[e] + d;
                Y[e] = y;
                dd = fma(d, d, dd);
                yy = fma(y, y, yy);
            }
            group_sync<G>();
            dd = co_sum<G>(dd, red, t);
            yy = co_sum<G>(yy, red, t);
            for (int e = t; e < nn; e += G) {
                const int i = e % n, j = e / n;
                if (i < j) {
                    const double y2 = 0.5 * (Y[e] + Y[j + i * n]);
                    Y[e] = Y[j + i * n] = y2;
                }
            }
            if (!isfinite(yy) || !isfinite(dd)) break;
            if (dd <= DARE_EPS * DARE_EPS * yy) {
                code = 0;
                break;
            }
            co_gemm<G>(0, 0, n, n, n, 1.0, M, n, M, n, 0.0, T, n, t);  // (its final sync orders the symmetrisation)
            double *sw = M;
            M = T;
            T = sw;
        }
        group_sync<G>();
    }
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    if (!code) {
        // M = P Acl = PA - PB K ; T = M Y ; BG = K Y (m x n)
        for (int e = t; e < nn; e += G) {
            const int i = e % n, j = e / n;
            double v = PA[e];
            for (int l = 0; l < m; ++l) v = fma(-PB[i + l * n], K[l + j * m], v);
            M[e] = v;
        }
        group_sync<G>();
        co_gemm<G>(0, 0, n, n, n, 1.0, M, n, Y, n, 0.0, T, n, t);
        co_gemm<G>(0, 0, m, n, n, 1.0, K, m, Y, n, 0.0, BG, m, t);
    }
    if (!active) return;
    if (gQ)
        for (int e = t; e < nn; e += G) gQ[inst * nn + e] = code ? nan : Y[e];
    if (gR)
        for (int e = t; e < mm; e += G) {
            const int i = e % m, j = e / m;
            double a = 0.0, b = 0.0;
            if (!code)
                for (int l = 0; l < n; ++l) {
                    a = fma(BG[i + l * m], K[j + l * m], a);
                    b = fma(BG[j + l * m], K[i + l * m], b);
                }
            gR[inst * (int64_t)mm + e] = code ? nan : 0.5 * (a + b) + Gb[e];
        }
    if (gA)
        for (int e = t; e < nn; e += G) {
            const int i = e % n, j = e / n;
            double v = 2.0 * T[e];
            if (!code)
                for (int l = 0; l < m; ++l) v = fma(PB[i + l * n], Yk[l + j * m], v);
            gA[inst * nn + e] = code ? nan : v;
        }
    if (gB)
        for (int e = t; e < nm; e += G) {
            const int i = e % n, j = e / n;
            double v = 0.0, w = 0.0;
            if (!code) {
                for (int l = 0; l < n; ++l) v = fma(T[i + l * n], K[j + l * m], v);
                for (int l = 0; l < n; ++l) w = fma(PA[i + l * n], Yk[j + l * m], w);
                for (int l = 0; l < m; ++l) w = fma(2.0 * PB[i + l * n], Gb[l + j * m], w);
            }
            gB[inst * (int64_t)nm + e] = code ? nan : w - 2.0 * v;
        }
    if (info && t == 0) info[inst] = code;
}
