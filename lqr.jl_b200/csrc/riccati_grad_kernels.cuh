// riccati_grad_kernels.cuh — the backward sweep of lqrb_riccati_grad_f64: costates of the forward and the adjoint
// problem, and the gradients of every input, one pass over the instance-major arrays per instance (DESIGN §4.8).
#pragma once
#include "common.cuh"

struct RiccatiGradArgs {
    const double *A, *Q, *q, *Qf, *qf, *Z, *Zh, *dZ;  // q, qf may be NULL (zero); Zh = the adjoint solution
    double *gA, *gB, *gQ, *gR, *gq, *gr, *gQf, *gqf, *gx0;  // each may be NULL
};

// element (i, j) of the symmetric matrix whose upper triangle is stored in the column-major n x n block M (the solve
// reads nothing else)
__device__ __forceinline__ double grad_sym(const double *__restrict__ M, int i, int j, int n) {
    return i <= j ? M[i + j * n] : M[j + i * n];
}

// G lanes per instance (G >= n, or G = 32 with R = ceil(n / 32) rows per lane); lane l owns rows l, l + G, ....
// Every gradient element (i, j) is written by the owner of row i, so each store of a column j is one contiguous
// piece.  Aᵀλ and Q x read A_k and Q_k by column: the owner of row i walks column i of A_k (contiguous), and element
// (i, j) of Q_k from its upper triangle, i.e. column j above the diagonal (contiguous across lanes) and column i
// below it.  Each lane thus walks whole 32-byte sectors of the knot's contiguous blocks over consecutive iterations,
// so that L1 can serve the repeats (an intent: no sector counter has measured it).
// LTI: the matrix gradients are sums over the knots.  Each group accumulates them in its slice of shared memory
// (2n² + nm + m² doubles; every n the solve accepts fits) and writes them once at the end.  A lane only ever touches
// the elements of its own rows, so no barrier is needed.  gq and gr accumulate in registers.
template <int G, int R, bool LTI>
__global__ void __launch_bounds__(128)
    riccati_grad_kernel(const RiccatiGradArgs a, int n, int m, int N, int64_t batch) {
    extern __shared__ double grad_smem[];
    const int lane = threadIdx.x % G, grp = threadIdx.x / G;
    const int64_t inst = (int64_t)blockIdx.x * (blockDim.x / G) + grp;
    const bool on = inst < batch;
    const int64_t ii = on ? inst : batch - 1;  // idle groups read a valid instance and write nothing
    const int Kn = LTI ? 1 : N - 1;
    const int64_t nn = (int64_t)n * n, NN = (int64_t)N * n + (int64_t)(N - 1) * m;
    const double *A = a.A + ii * Kn * nn, *Q = a.Q + ii * Kn * nn, *Qf = a.Qf + ii * nn;
    const double *q = a.q ? a.q + ii * Kn * n : nullptr, *qf = a.qf ? a.qf + ii * n : nullptr;
    const double *Z = a.Z + ii * NN, *Zh = a.Zh + ii * NN, *dZ = a.dZ + ii * NN;

    int row[R];
    bool own[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        row[r] = lane + r * G;
        own[r] = row[r] < n;
    }

    // terminal knot: λ_{N-2} = Qf x_{N-1} + qf, λ̂_{N-2} = Qf x̂_{N-1} + dZ[x_{N-1}]
    double x[R], xh[R], lam[R], lamh[R];
    const int64_t zt = (int64_t)(N - 1) * (n + m);
#pragma unroll
    for (int r = 0; r < R; ++r) {
        x[r] = own[r] ? Z[zt + row[r]] : 0.0;
        xh[r] = own[r] ? Zh[zt + row[r]] : 0.0;
        lam[r] = lamh[r] = 0.0;
    }
    double *gQf = (on && a.gQf) ? a.gQf + ii * nn : nullptr;
#pragma unroll
    for (int rj = 0; rj < R; ++rj)
        for (int jl = 0; jl < G; ++jl) {
            const int j = rj * G + jl;
            if (j >= n) break;
            const double xj = __shfl_sync(0xffffffffu, x[rj], jl, G), xhj = __shfl_sync(0xffffffffu, xh[rj], jl, G);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                if (!own[r]) continue;
                const double qv = grad_sym(Qf, row[r], j, n);
                lam[r] = fma(qv, xj, lam[r]);
                lamh[r] = fma(qv, xhj, lamh[r]);
                if (gQf) gQf[row[r] + j * n] = 0.5 * (xh[r] * xj + x[r] * xhj);
            }
        }
#pragma unroll
    for (int r = 0; r < R; ++r) {
        if (!own[r]) continue;
        lam[r] += qf ? qf[row[r]] : 0.0;
        lamh[r] += dZ[zt + row[r]];
        if (on && a.gqf) a.gqf[ii * n + row[r]] = xh[r];
    }

    // where the matrix gradients go: LTV the knot's block of the output, LTI an accumulator (see above)
    double *gA = (on && a.gA) ? a.gA + ii * Kn * nn : nullptr, *gQ = (on && a.gQ) ? a.gQ + ii * Kn * nn : nullptr;
    double *gB = (on && a.gB) ? a.gB + ii * Kn * n * m : nullptr;
    double *gR = (on && a.gR) ? a.gR + ii * Kn * m * m : nullptr;
    double *accA = gA, *accQ = gQ, *accB = gB, *accR = gR;
    double gqa[R], gra[R];
    if (LTI) {
        double *s = grad_smem + (int64_t)grp * (2 * nn + (int64_t)n * m + (int64_t)m * m);
        accA = gA ? s : nullptr;
        accQ = gQ ? s + nn : nullptr;
        accB = gB ? s + 2 * nn : nullptr;
        accR = gR ? s + 2 * nn + n * m : nullptr;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            gqa[r] = gra[r] = 0.0;
            if (!own[r]) continue;
            for (int j = 0; j < n; ++j) {
                if (accA) accA[row[r] + j * n] = 0.0;
                if (accQ) accQ[row[r] + j * n] = 0.0;
            }
            for (int j = 0; j < m; ++j) {
                if (accB) accB[row[r] + j * n] = 0.0;
                if (accR && row[r] < m) accR[row[r] + j * m] = 0.0;
            }
        }
    }

    for (int k = N - 2; k >= 0; --k) {
        const int kk = LTI ? 0 : k;
        const double *Ak = A + kk * nn, *Qk = Q + kk * nn;
        const int64_t zo = (int64_t)k * (n + m);
        double u[R], uh[R], s[R], sh[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            x[r] = own[r] ? Z[zo + row[r]] : 0.0;
            xh[r] = own[r] ? Zh[zo + row[r]] : 0.0;
            u[r] = row[r] < m ? Z[zo + n + row[r]] : 0.0;
            uh[r] = row[r] < m ? Zh[zo + n + row[r]] : 0.0;
            s[r] = sh[r] = 0.0;
        }
        double *pA = LTI ? accA : (accA ? accA + k * nn : nullptr), *pQ = LTI ? accQ : (accQ ? accQ + k * nn : nullptr);
        double *pB = LTI ? accB : (accB ? accB + (int64_t)k * n * m : nullptr);
        double *pR = LTI ? accR : (accR ? accR + (int64_t)k * m * m : nullptr);
        // λ_{k-1} = Q_k x_k + q_k + A_kᵀ λ_k (and the same for the adjoint); ∂A_k = λ_k x̂_kᵀ + λ̂_k x_kᵀ,
        // ∂Q_k = ½(x̂_k x_kᵀ + x_k x̂_kᵀ)
#pragma unroll
        for (int rj = 0; rj < R; ++rj)
            for (int jl = 0; jl < G; ++jl) {
                const int j = rj * G + jl;
                if (j >= n) break;
                const double xj = __shfl_sync(0xffffffffu, x[rj], jl, G), xhj = __shfl_sync(0xffffffffu, xh[rj], jl, G);
                const double lj = __shfl_sync(0xffffffffu, lam[rj], jl, G);
                const double lhj = __shfl_sync(0xffffffffu, lamh[rj], jl, G);
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    if (!own[r]) continue;
                    const double av = Ak[j + row[r] * n], qv = grad_sym(Qk, row[r], j, n);
                    s[r] = fma(qv, xj, fma(av, lj, s[r]));
                    sh[r] = fma(qv, xhj, fma(av, lhj, sh[r]));
                    const double ga = fma(lam[r], xhj, lamh[r] * xj), gqv = 0.5 * fma(xh[r], xj, x[r] * xhj);
                    if (pA) pA[row[r] + j * n] = LTI ? pA[row[r] + j * n] + ga : ga;
                    if (pQ) pQ[row[r] + j * n] = LTI ? pQ[row[r] + j * n] + gqv : gqv;
                }
            }
        // ∂B_k = λ_k û_kᵀ + λ̂_k u_kᵀ, ∂R_k = ½(û_k u_kᵀ + u_k û_kᵀ)
        if (a.gB || a.gR) {  // uniform over the warp: idle groups take part in the shuffles
#pragma unroll
            for (int rj = 0; rj < R; ++rj)
                for (int jl = 0; jl < G; ++jl) {
                    const int j = rj * G + jl;
                    if (j >= m) break;
                    const double uj = __shfl_sync(0xffffffffu, u[rj], jl, G);
                    const double uhj = __shfl_sync(0xffffffffu, uh[rj], jl, G);
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        if (!own[r]) continue;
                        const double gb = fma(lam[r], uhj, lamh[r] * uj), gr = 0.5 * fma(uh[r], uj, u[r] * uhj);
                        if (pB) pB[row[r] + j * n] = LTI ? pB[row[r] + j * n] + gb : gb;
                        if (pR && row[r] < m) pR[row[r] + j * m] = LTI ? pR[row[r] + j * m] + gr : gr;
                    }
                }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            if (!own[r]) continue;
            if (LTI) {
                gqa[r] += xh[r];
                gra[r] += uh[r];
            } else {
                if (on && a.gq) a.gq[(ii * (N - 1) + k) * n + row[r]] = xh[r];
                if (on && a.gr && row[r] < m) a.gr[(ii * (N - 1) + k) * m + row[r]] = uh[r];
            }
            lam[r] = s[r] + (q ? q[kk * n + row[r]] : 0.0);
            lamh[r] = sh[r] + dZ[zo + row[r]];
        }
    }

#pragma unroll
    for (int r = 0; r < R; ++r) {
        if (!own[r] || !on) continue;
        if (a.gx0) a.gx0[ii * n + row[r]] = lamh[r];  // ∂x0 = λ̂_{-1}
        if (LTI) {
            if (a.gq) a.gq[ii * n + row[r]] = gqa[r];
            if (a.gr && row[r] < m) a.gr[ii * m + row[r]] = gra[r];
            for (int j = 0; j < n; ++j) {
                if (gA) gA[row[r] + j * n] = accA[row[r] + j * n];
                if (gQ) gQ[row[r] + j * n] = accQ[row[r] + j * n];
            }
            for (int j = 0; j < m; ++j) {
                if (gB) gB[row[r] + j * n] = accB[row[r] + j * n];
                if (gR && row[r] < m) gR[row[r] + j * m] = accR[row[r] + j * m];
            }
        }
    }
}
