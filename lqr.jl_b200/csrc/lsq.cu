// lsq.cu — the reference's condensed least-squares solve of the unconstrained LTI problem on the device.
//
// Replaces solve!(sol, ::LeastSquaresSolver, prob) : src/least_squares.jl:158-190 (build_toeplitz :136-156,
// build_least_squares! :106-134, buildAb! :61-104): with x_{i+2} = A^{i+1} x0 + sum_{j<=i} A^{i-j} B u_j  (T block
// Toeplitz, L the powers of A), the controls minimise |Hx (T U + L x0)|^2 + U' Hu U, i.e. solve the dense SPD system
//     (T' Qbar T + Rbar) U = -T' Qbar L x0,        Qbar = blkdiag(Q, ..., Q, Qf),  Rbar = blkdiag(R, ..., R)
// by Cholesky (LAPACK.potrf! / potrs!, :176-178), then rollout! (:195-202).  O((N m)^3) per instance and (N m)^2
// doubles of workspace: the alternative for short horizons (SURVEY §8f-4) and an independent cross-check of the
// Riccati path (test/least_squares.jl:38).  One CTA per instance, runtime sizes, workspace in global memory.
// (The reference leaves Hu = 0 in its default :Ab build mode, src/least_squares.jl:61-104 never fills it; this is the
// :lsq form, where Hu = Rbar, :117.)
#include "coop_prims.cuh"
#include "common.cuh"

static __host__ __device__ inline size_t lsq_ws_doubles(int n, int m, int N) {
    const size_t K = N - 1, Km = K * m;
    return 3 * K * n * m + K * n + Km * Km + Km + 2 * (size_t)n * n + 2 * (size_t)n;
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS)
    lsq_solve_kernel(const double *__restrict__ A, const double *__restrict__ B, const double *__restrict__ Q,
                     const double *__restrict__ R, const double *__restrict__ Qf, const double *__restrict__ x0,
                     double *__restrict__ Z, int32_t *__restrict__ info, double *__restrict__ ws, int n, int m, int N,
                     int64_t batch) {
    const int t = threadIdx.x;
    const int K = N - 1, Km = K * m;
    for (int64_t inst = blockIdx.x; inst < batch; inst += gridDim.x) {
        const double *Ai = A + inst * n * n, *Bi = B + inst * n * m, *Qi = Q + inst * n * n, *Ri = R + inst * m * m,
                     *Qfi = Qf + inst * n * n, *xi = x0 + inst * n;
        double *w = ws + (size_t)blockIdx.x * lsq_ws_doubles(n, m, N);
        double *P = w, *QP = P + (size_t)K * n * m, *QfP = QP + (size_t)K * n * m, *S = QfP + (size_t)K * n * m,
               *G = S + (size_t)K * n, *y = G + (size_t)Km * Km, *An = y + Km, *At = An + n * n, *xa = At + n * n,
               *xb = xa + n;
        // ---- P[k] = A^k B (the first block column of T), s_i = Q_{i+2} A^{i+1} x0 (Qbar L x0)
        for (int e = t; e < n * m; e += THREADS) P[e] = Bi[e];
        for (int e = t; e < n; e += THREADS) xa[e] = xi[e];
        __syncthreads();
        for (int k = 0; k < K; ++k) {
            const double *Pk = P + (size_t)k * n * m;
            const double *Qk = (k == K - 1) ? Qfi : Qi;
            if (k + 1 < K) co_gemm<THREADS>(0, 0, n, m, n, 1.0, Ai, n, Pk, n, 0.0, P + (size_t)(k + 1) * n * m, n, t);
            co_gemm<THREADS>(0, 0, n, m, n, 1.0, Qi, n, Pk, n, 0.0, QP + (size_t)k * n * m, n, t);
            co_gemm<THREADS>(0, 0, n, m, n, 1.0, Qfi, n, Pk, n, 0.0, QfP + (size_t)k * n * m, n, t);
            co_gemm<THREADS>(0, 0, n, 1, n, 1.0, Ai, n, xa, n, 0.0, xb, n, t);       // A^{k+1} x0
            co_gemm<THREADS>(0, 0, n, 1, n, 1.0, Qk, n, xb, n, 0.0, S + (size_t)k * n, n, t);
            for (int e = t; e < n; e += THREADS) xa[e] = xb[e];
            __syncthreads();
        }
        // ---- G = T' Qbar T + Rbar (upper triangle), y = T' Qbar L x0
        for (int64_t e = t; e < (int64_t)Km * Km; e += THREADS) {
            const int a = (int)(e % Km), b = (int)(e / Km);
            if (a > b) continue;
            const int j = a / m, al = a % m, jp = b / m, be = b % m;  // j <= jp
            double s = (j == jp) ? Ri[al + be * m] : 0.0;
            for (int i = jp; i < K; ++i) {
                const double *pa = P + (size_t)(i - j) * n * m + al * n;
                const double *qb = ((i == K - 1) ? QfP : QP) + (size_t)(i - jp) * n * m + be * n;
                for (int r = 0; r < n; ++r) s = fma(pa[r], qb[r], s);
            }
            G[a + (size_t)b * Km] = s;
        }
        for (int a = t; a < Km; a += THREADS) {
            const int j = a / m, al = a % m;
            double s = 0.0;
            for (int i = j; i < K; ++i) {
                const double *pa = P + (size_t)(i - j) * n * m + al * n, *si = S + (size_t)i * n;
                for (int r = 0; r < n; ++r) s = fma(pa[r], si[r], s);
            }
            y[a] = -s;
        }
        __syncthreads();
        // ---- U = G^-1 y  (potrf! + potrs!)
        const int st = co_chol<THREADS>(G, Km, Km, t);
        co_trsm_ut<THREADS>(G, Km, Km, y, 1, Km, t);
        co_trsm_un<THREADS>(G, Km, Km, y, 1, Km, t);
        if (info && t == 0) info[inst] = st;
        // ---- rollout!: Z = [x1; u1; ...; xN]
        double *zi = Z + inst * ((int64_t)N * n + (int64_t)K * m);
        for (int e = t; e < n; e += THREADS) {
            xa[e] = xi[e];
            zi[e] = xi[e];
        }
        __syncthreads();
        for (int k = 0; k < K; ++k) {
            for (int e = t; e < m; e += THREADS) zi[(int64_t)k * (n + m) + n + e] = y[k * m + e];
            co_gemm<THREADS>(0, 0, n, 1, n, 1.0, Ai, n, xa, n, 0.0, xb, n, t);
            co_gemm<THREADS>(0, 0, n, 1, m, 1.0, Bi, n, y + k * m, m, 1.0, xb, n, t);
            for (int e = t; e < n; e += THREADS) {
                xa[e] = xb[e];
                zi[(int64_t)(k + 1) * (n + m) + e] = xb[e];
            }
            __syncthreads();
        }
    }
}

extern "C" int32_t lqrb_lsq_solve_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, int64_t batch, const double *A,
                                      const double *B, const double *Q, const double *R, const double *Qf,
                                      const double *x0, double *Z, int32_t *info) {
    if (!h) return -1;
    if (n < 1 || n > 128) return lqrb_fail(h, -2, "n out of range [1,128]");
    if (m < 1 || m > n) return lqrb_fail(h, -3, "m out of range [1,n]");
    if (N < 2 || (int64_t)(N - 1) * m > 4096) return lqrb_fail(h, -4, "N out of range (the condensed system has (N-1) m <= 4096 unknowns)");
    if (batch < 0) return lqrb_fail(h, -5, "batch must be >= 0");
    if (!A || !B || !Q || !R || !Qf || !x0) return lqrb_fail(h, -6, "an input array is NULL");
    if (!Z) return lqrb_fail(h, -12, "Z is NULL");
    if (batch == 0) return 0;
    LQRB_CUDA(h, cudaSetDevice(h->device));
    const int64_t NN = lqrb_num_vars(n, m, N);
    const int64_t nn = (int64_t)n * n * 8, nm = (int64_t)n * m * 8, mm = (int64_t)m * m * 8;
    return lqrb_for_chunks(
        h, batch, batch, {{A, nn}, {B, nm}, {Q, nn}, {R, mm}, {Qf, nn}, {x0, (int64_t)n * 8}}, {{Z, NN * 8}, {info, 4}},
        [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
            constexpr int THREADS = 256;
            const unsigned grid = (unsigned)std::min<int64_t>(cb, (int64_t)h->sm_count * 2);
            double *ws = (double *)lqrb_scratch(h, SCR_MISC, (size_t)grid * lsq_ws_doubles(n, m, N) * 8, lane.index);
            if (!ws) return 1000 + (int)cudaErrorMemoryAllocation;
            const double *const *a = (const double *const *)in;
            lsq_solve_kernel<THREADS><<<grid, THREADS, 0, lane.stream>>>(a[0], a[1], a[2], a[3], a[4], a[5],
                                                                         (double *)out[0], (int32_t *)out[1], ws, n, m, N,
                                                                         cb);
            h->kernel_name = "lsq_solve(condensed least squares)";
            LQRB_LAUNCH_CHECK(h, "lsq_solve_kernel");
            return 0;
        });
}
