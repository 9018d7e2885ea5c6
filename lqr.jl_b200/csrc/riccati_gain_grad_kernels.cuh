// riccati_gain_grad_kernels.cuh — the gains part of lqrb_riccati_grad_gains_f64: gradients of a loss of the feedback
// gains K_k and feedforward terms kff_k through the Riccati recursion, one lane group per instance (DESIGN §4.10).
#pragma once
#include "common.cuh"

struct RiccatiGainGradArgs {
    const double *A, *B, *Q, *R, *q, *r, *Qf, *qf;  // q, r, qf may be NULL (zero)
    const double *dK, *dkff;                          // cotangents of K[m,n,N-1], kff[m,N-1]; either may be NULL
    double *tape;                                     // gain_grad_tape_doubles(n, m) per knot per instance slot
    double *gA, *gB, *gQ, *gR, *gq, *gr, *gQf, *gqf;  // each may be NULL; accumulated into (+=)
    int32_t *info;                                    // may be NULL
};

// One knot of the tape: P_{k+1} (full n x n, column-major: the owner of row i reads row i as one contiguous piece
// across the group) | p_{k+1} | K_k (m x n, the layout of the forward call's K) | kff_k | the lower Cholesky factor
// of G_k (m x m column-major, upper part unused).
__host__ __device__ constexpr int64_t gain_grad_tape_doubles(int n, int m) {
    return (int64_t)n * n + n + (int64_t)m * n + m + (int64_t)m * m;
}

// Shared memory of one group: three n x n operands, three n x m ones, one (n+1) x m, one m x m and seven vectors.
__host__ __device__ constexpr int64_t gain_grad_smem_doubles(int n, int m) {
    return 3 * (int64_t)n * n + 3 * (int64_t)n * m + (int64_t)(n + 1) * m + (int64_t)m * m + 6 * n + m;
}

__device__ __forceinline__ double gg_sym(const double *__restrict__ M, int i, int j, int n) {
    return i <= j ? M[i + j * n] : M[j + i * n];
}

// Solves x G = b in place for one row b of the column-major buffer X (leading dimension ld), G = L Lᵀ with L lower
// column-major m x m: X[row, :] <- X[row, :] G⁻¹.
__device__ __forceinline__ void gg_chol_solve_row(double *X, int ld, int row, const double *L, int m) {
    for (int c = 0; c < m; ++c) {
        double s = X[row + c * ld];
        for (int d = 0; d < c; ++d) s = fma(-L[c + d * m], X[row + d * ld], s);
        X[row + c * ld] = s / L[c + c * m];
    }
    for (int c = m - 1; c >= 0; --c) {
        double s = X[row + c * ld];
        for (int d = c + 1; d < m; ++d) s = fma(-L[d + c * m], X[row + d * ld], s);
        X[row + c * ld] = s / L[c + c * m];
    }
}

// G lanes per instance (G >= n, or G = 32 with R = ceil(n / 32) rows per lane); lane l owns rows l, l + G, ... of every
// n-row operand and of every m-row one.  Groups of one warp synchronise with __syncwarp (the launch makes every warp
// whole).  Phase 1 runs the recursion backward and writes the tape; phase 2 runs the adjoint forward, k = 0 … N-2, and
// adds each knot's gradients into the lane's own rows of the outputs, so no atomics are needed and the order of every
// sum is fixed.  Groups past the batch compute on the last instance, write their own tape slot and no output.
template <int G, int R, bool LTI>
__global__ void __launch_bounds__(128)
    riccati_gain_grad_kernel(const RiccatiGainGradArgs a, int n, int m, int N, int64_t batch) {
    extern __shared__ double gg_smem[];
    const int lane = threadIdx.x % G, grp = threadIdx.x / G;
    const int64_t inst = (int64_t)blockIdx.x * (blockDim.x / G) + grp;
    const bool on = inst < batch;
    const int64_t ii = on ? inst : batch - 1;
    const int Kn = LTI ? 1 : N - 1, ld = n + 1;
    const int64_t nn = (int64_t)n * n, nm = (int64_t)n * m, mm = (int64_t)m * m, TR = gain_grad_tape_doubles(n, m);
    double *s = gg_smem + (int64_t)grp * gain_grad_smem_doubles(n, m);
    double *M0 = s, *M1 = M0 + nn, *M2 = M1 + nn, *N0 = M2 + nn, *N2 = N0 + nm, *N3 = N2 + nm, *X = N3 + nm,
           *Gm = X + (int64_t)ld * m, *V0 = Gm + mm, *V1 = V0 + n, *V2 = V1 + n, *V3 = V2 + n, *V4 = V3 + n,
           *V5 = V4 + n, *W0 = V5 + n;
    const double *A = a.A + ii * Kn * nn, *B = a.B + ii * Kn * nm, *Q = a.Q + ii * Kn * nn, *Rm = a.R + ii * Kn * mm;
    const double *q = a.q ? a.q + ii * Kn * n : nullptr, *r = a.r ? a.r + ii * Kn * m : nullptr;
    const double *Qf = a.Qf + ii * nn, *qf = a.qf ? a.qf + ii * n : nullptr;
    double *tape = a.tape + inst * (int64_t)(N - 1) * TR;
#define GG_ROWS(i, lim) \
    _Pragma("unroll") for (int r_ = 0, i = lane; r_ < R; ++r_, i += G) if (i < (lim))

    // ---------------------------------------------------------------- phase 1: backward sweep, tape
    GG_ROWS(i, n) {
        for (int j = 0; j < n; ++j) M0[i + j * n] = gg_sym(Qf, i, j, n);
        V0[i] = qf ? qf[i] : 0.0;
    }
    __syncwarp();
    int st = 0;
    for (int k = N - 2; k >= 0; --k) {
        const int kk = LTI ? 0 : k;
        const double *Ak = A + kk * nn, *Bk = B + kk * nm, *Qk = Q + kk * nn, *Rk = Rm + kk * mm;
        double *T = tape + (int64_t)k * TR, *Tp = T + nn, *TK = Tp + n, *Tkff = TK + nm, *TL = Tkff + m;
        // P′ = M0, p′ = V0 to the tape; P′B -> N0, P′A -> M1
        GG_ROWS(i, n) {
            for (int j = 0; j < n; ++j) T[i + j * n] = M0[i + j * n];
            Tp[i] = V0[i];
            for (int c = 0; c < m; ++c) {
                double t = 0.0;
                for (int l = 0; l < n; ++l) t = fma(M0[i + l * n], Bk[l + c * n], t);
                N0[i + c * n] = t;
            }
            for (int j = 0; j < n; ++j) {
                double t = 0.0;
                for (int l = 0; l < n; ++l) t = fma(M0[i + l * n], Ak[l + j * n], t);
                M1[i + j * n] = t;
            }
        }
        __syncwarp();
        // G = R + BᵀP′B -> Gm, h = r + Bᵀp′ -> W0 and row n of X, Hᵀ = AᵀP′B -> N2 and rows 0..n-1 of X
        GG_ROWS(c, m) {
            for (int d = 0; d < m; ++d) {
                double t = gg_sym(Rk, c, d, m);
                for (int l = 0; l < n; ++l) t = fma(Bk[l + c * n], N0[l + d * n], t);
                Gm[c + d * m] = t;
            }
            double t = r ? r[kk * m + c] : 0.0;
            for (int l = 0; l < n; ++l) t = fma(Bk[l + c * n], V0[l], t);
            W0[c] = t;
            X[n + c * ld] = t;
        }
        GG_ROWS(j, n) for (int c = 0; c < m; ++c) {
            double t = 0.0;
            for (int l = 0; l < n; ++l) t = fma(Ak[l + j * n], N0[l + c * n], t);
            N2[j + c * n] = t;
            X[j + c * ld] = t;
        }
        __syncwarp();
        // G = L Lᵀ in place (lower), column by column; a pivot that is not > 0 gives the forward solve's info code
        for (int j = 0; j < m; ++j) {
            const double d = Gm[j + j * m];
            if (!(d > 0.0) && st == 0) st = (k + 1) * 1000 + j + 1;
            const double dj = sqrt(d);
            __syncwarp();
            GG_ROWS(c, m) {
                if (c == j) Gm[j + j * m] = dj;
                else if (c > j) Gm[c + j * m] /= dj;
            }
            __syncwarp();
            GG_ROWS(c, m) if (c > j) for (int e = j + 1; e <= c; ++e) Gm[c + e * m] = fma(-Gm[c + j * m], Gm[e + j * m], Gm[c + e * m]);
            __syncwarp();
        }
        // rows of X times G⁻¹: Kᵀ (rows 0..n-1) and kffᵀ (row n, lane 0)
        GG_ROWS(j, n) {
            gg_chol_solve_row(X, ld, j, Gm, m);
            for (int c = 0; c < m; ++c) TK[c + j * m] = X[j + c * ld];
        }
        if (lane == 0) gg_chol_solve_row(X, ld, n, Gm, m);
        GG_ROWS(c, m) for (int d = 0; d <= c; ++d) TL[c + d * m] = Gm[c + d * m];
        __syncwarp();
        GG_ROWS(c, m) Tkff[c] = X[n + c * ld];
        // P = Q + AᵀP′A − HᵀK -> M2, p = q + Aᵀp′ − Kᵀh -> V1
        GG_ROWS(i, n) {
            for (int j = 0; j < n; ++j) {
                double t = gg_sym(Qk, i, j, n);
                for (int l = 0; l < n; ++l) t = fma(Ak[l + i * n], M1[l + j * n], t);
                for (int c = 0; c < m; ++c) t = fma(-N2[i + c * n], X[j + c * ld], t);
                M2[i + j * n] = t;
            }
            double t = q ? q[kk * n + i] : 0.0;
            for (int l = 0; l < n; ++l) t = fma(Ak[l + i * n], V0[l], t);
            for (int c = 0; c < m; ++c) t = fma(-X[i + c * ld], W0[c], t);
            V1[i] = t;
        }
        __syncwarp();
        GG_ROWS(i, n) {
            for (int j = 0; j < n; ++j) M0[i + j * n] = 0.5 * (M2[i + j * n] + M2[j + i * n]);
            V0[i] = V1[i];
        }
        __syncwarp();
    }
    if (on && a.info && st != 0 && lane == 0 && a.info[ii] == 0) a.info[ii] = st;

    // ---------------------------------------------------------------- phase 2: forward adjoint sweep
    // M0 = P̄, V0 = p̄ (zero: P_0, p_0 feed nothing)
    GG_ROWS(i, n) {
        for (int j = 0; j < n; ++j) M0[i + j * n] = 0.0;
        V0[i] = 0.0;
    }
    __syncwarp();
    for (int k = 0; k < N - 1; ++k) {
        const int kk = LTI ? 0 : k;
        const double *Ak = A + kk * nn, *Bk = B + kk * nm;
        const double *T = tape + (int64_t)k * TR, *Tp = T + nn, *TK = Tp + n, *Tkff = TK + nm, *TL = Tkff + m;
        const double *dK = a.dK ? a.dK + (ii * (N - 1) + k) * nm : nullptr;
        const double *dkff = a.dkff ? a.dkff + (ii * (N - 1) + k) * m : nullptr;
        double *gA = (on && a.gA) ? a.gA + (ii * Kn + kk) * nn : nullptr;
        double *gB = (on && a.gB) ? a.gB + (ii * Kn + kk) * nm : nullptr;
        double *gQ = (on && a.gQ) ? a.gQ + (ii * Kn + kk) * nn : nullptr;
        double *gR = (on && a.gR) ? a.gR + (ii * Kn + kk) * mm : nullptr;
        double *gq = (on && a.gq) ? a.gq + (ii * Kn + kk) * n : nullptr;
        double *gr = (on && a.gr) ? a.gr + (ii * Kn + kk) * m : nullptr;
        // A_cl = A − BK -> M1; Yᵀ = K̄ᵀG⁻¹ (rows 0..n-1) and yᵀ = k̄ᵀG⁻¹ (row n) -> X; Kp̄ -> W0; B kff -> V2
        GG_ROWS(i, n) {
            for (int j = 0; j < n; ++j) {
                double t = Ak[i + j * n];
                for (int c = 0; c < m; ++c) t = fma(-Bk[i + c * n], TK[c + j * m], t);
                M1[i + j * n] = t;
            }
            for (int c = 0; c < m; ++c) X[i + c * ld] = dK ? dK[c + i * m] : 0.0;
            gg_chol_solve_row(X, ld, i, TL, m);
            double t = 0.0;
            for (int c = 0; c < m; ++c) t = fma(Bk[i + c * n], Tkff[c], t);
            V2[i] = t;
        }
        if (lane == 0) {
            for (int c = 0; c < m; ++c) X[n + c * ld] = dkff ? dkff[c] : 0.0;
            gg_chol_solve_row(X, ld, n, TL, m);
        }
        GG_ROWS(c, m) {
            double t = 0.0;
            for (int j = 0; j < n; ++j) t = fma(TK[c + j * m], V0[j], t);
            W0[c] = t;
        }
        __syncwarp();
        // S = A_cl P̄ -> M2, P̄Kᵀ -> N2, A_cl p̄ -> V3, v = p′ − P′B kff -> V4, P′B -> N0, A Yᵀ -> N3,
        // Ḡ = −sym(Y Kᵀ + y kffᵀ) -> Gm
        GG_ROWS(i, n) {
            for (int j = 0; j < n; ++j) {
                double t = 0.0;
                for (int l = 0; l < n; ++l) t = fma(M1[i + l * n], M0[l + j * n], t);
                M2[i + j * n] = t;
            }
            for (int c = 0; c < m; ++c) {
                double t = 0.0, u = 0.0, w = 0.0;
                for (int j = 0; j < n; ++j) {
                    t = fma(M0[i + j * n], TK[c + j * m], t);
                    u = fma(T[i + j * n], Bk[j + c * n], u);
                    w = fma(Ak[i + j * n], X[j + c * ld], w);
                }
                N2[i + c * n] = t;
                N0[i + c * n] = u;
                N3[i + c * n] = w;
            }
            double t = 0.0, u = Tp[i];
            for (int j = 0; j < n; ++j) {
                t = fma(M1[i + j * n], V0[j], t);
                u = fma(-T[i + j * n], V2[j], u);
            }
            V3[i] = t;
            V4[i] = u;
        }
        GG_ROWS(c, m) for (int d = 0; d < m; ++d) {
            double t = fma(X[n + c * ld], Tkff[d], X[n + d * ld] * Tkff[c]);
            for (int j = 0; j < n; ++j) t = fma(X[j + c * ld], TK[d + j * m], fma(X[j + d * ld], TK[c + j * m], t));
            Gm[c + d * m] = -0.5 * t;
        }
        __syncwarp();
        // Q̄ += P̄, q̄ += p̄, R̄ += K P̄ Kᵀ + sym((K p̄) kffᵀ) + Ḡ, r̄ += −K p̄ + y; P′ A_cl p̄ -> V5
        GG_ROWS(i, n) {
            if (gQ)
                for (int j = 0; j < n; ++j) gQ[i + j * n] += M0[i + j * n];
            if (gq) gq[i] += V0[i];
            double t = 0.0;
            for (int l = 0; l < n; ++l) t = fma(T[i + l * n], V3[l], t);
            V5[i] = t;
        }
        GG_ROWS(c, m) {
            if (gR)
                for (int d = 0; d < m; ++d) {
                    double t = Gm[c + d * m] + 0.5 * fma(W0[c], Tkff[d], W0[d] * Tkff[c]);
                    for (int j = 0; j < n; ++j) t = fma(TK[c + j * m], N2[j + d * n], t);
                    gR[c + d * m] += t;
                }
            if (gr) gr[c] += X[n + c * ld] - W0[c];
        }
        __syncwarp();
        // W = P′ S -> M0 (P̄ is no longer read), B Ḡ -> N2
        GG_ROWS(i, n) {
            for (int j = 0; j < n; ++j) {
                double t = 0.0;
                for (int l = 0; l < n; ++l) t = fma(T[i + l * n], M2[l + j * n], t);
                M0[i + j * n] = t;
            }
            for (int c = 0; c < m; ++c) {
                double t = 0.0;
                for (int d = 0; d < m; ++d) t = fma(Bk[i + d * n], Gm[d + c * m], t);
                N2[i + c * n] = t;
            }
        }
        __syncwarp();
        // Ā += 2W + v p̄ᵀ + P′B Y;  B̄ += −2W Kᵀ − (P′A_cl p̄) kffᵀ − v (K p̄)ᵀ + P′A Yᵀ + 2P′B Ḡ + p′ yᵀ;
        // p̄′ = A_cl p̄ + B y -> V1
        GG_ROWS(i, n) {
            if (gA)
                for (int j = 0; j < n; ++j) {
                    double t = fma(2.0, M0[i + j * n], V4[i] * V0[j]);
                    for (int c = 0; c < m; ++c) t = fma(N0[i + c * n], X[j + c * ld], t);
                    gA[i + j * n] += t;
                }
            if (gB)
                for (int c = 0; c < m; ++c) {
                    double w = 0.0, t = 0.0, u = 0.0;
                    for (int j = 0; j < n; ++j) {
                        w = fma(M0[i + j * n], TK[c + j * m], w);
                        t = fma(T[i + j * n], N3[j + c * n], t);
                    }
                    for (int d = 0; d < m; ++d) u = fma(N0[i + d * n], Gm[d + c * m], u);
                    t = fma(-2.0, w, t);
                    t = fma(2.0, u, t);
                    t = fma(-V5[i], Tkff[c], t);
                    t = fma(-V4[i], W0[c], t);
                    t = fma(Tp[i], X[n + c * ld], t);
                    gB[i + c * n] += t;
                }
            double t = V3[i];
            for (int c = 0; c < m; ++c) t = fma(Bk[i + c * n], X[n + c * ld], t);
            V1[i] = t;
        }
        __syncwarp();
        // P̄′ = A_cl P̄ A_clᵀ − sym((A_cl p̄)(B kff)ᵀ) + B Ḡ Bᵀ + sym(B Y Aᵀ) -> M0
        GG_ROWS(i, n) {
            for (int j = 0; j < n; ++j) {
                double t = -0.5 * fma(V3[i], V2[j], V2[i] * V3[j]), u = 0.0;
                for (int l = 0; l < n; ++l) t = fma(M2[i + l * n], M1[j + l * n], t);
                for (int c = 0; c < m; ++c) {
                    t = fma(N2[i + c * n], Bk[j + c * n], t);
                    u = fma(Bk[i + c * n], N3[j + c * n], fma(Bk[j + c * n], N3[i + c * n], u));
                }
                M0[i + j * n] = fma(0.5, u, t);
            }
            V0[i] = V1[i];
        }
        __syncwarp();
    }
    // Q̄f = P̄, q̄f = p̄
    GG_ROWS(i, n) {
        if (on && a.gQf)
            for (int j = 0; j < n; ++j) a.gQf[ii * nn + i + j * n] += M0[i + j * n];
        if (on && a.gqf) a.gqf[ii * n + i] += V0[i];
    }
#undef GG_ROWS
}
