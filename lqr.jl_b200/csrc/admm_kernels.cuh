// admm_kernels.cuh — box-constrained LTI MPC by ADMM on the cached infinite-horizon Riccati factor (DESIGN §4.12).
//
//   admm_shift_kernel     Qt = Q + rho I, Rt = R + rho I (the rho-augmented costs the DARE is solved for).
//   admm_cache_kernel<G>  from Pt = DARE(A, B, Qt, Rt) and its K: the cache record [A | B | Q | R | Qf | K | C1 | C2 |
//                         rho] with Qf = Pt - rho I, C1 = (Rt + B'Pt B)^-1, C2 = (A - BK)'.
//   admm_kernel<G>        the ADMM iterations of one instance, every iteration inside the kernel: G lanes (4, 8, 16 or
//                         32, the least >= n) own an instance, lane i owns row i of the n-row (and, i < m, of the m-row)
//                         operands; vectors travel between lanes by group shuffles.  Every per-knot array lives in shared
//                         memory for all iterations, a lane reads and writes only its own rows of them, so the group
//                         needs no barrier after the set-up.  No atomics: results are bitwise reproducible.
#pragma once
#include "dare_kernels.cuh"  // coop_prims, DARE_GAIN_NOT_PD

// info codes of lqrb_admm_solve_f64 (include/lqrb200.h)
#define ADMM_MAX_ITER 1
#define ADMM_NAN 2
#define ADMM_EMPTY_BOX 3

// Cache record of one instance (column-major blocks): A n*n | B n*m | Q n*n | R m*m | Qf n*n | K m*n | C1 m*m | C2 n*n |
// rho, 4 n^2 + 2 n m + 2 m^2 + 1 doubles.
__host__ __device__ inline int64_t admm_cache_doubles(int n, int m) {
    return (int64_t)4 * n * n + 2 * n * m + 2 * m * m + 1;
}
struct AdmmCacheOffsets {
    int64_t A, B, Q, R, Qf, K, C1, C2, rho;
    __host__ __device__ AdmmCacheOffsets(int n, int m) {
        A = 0;
        B = A + n * n;
        Q = B + n * m;
        R = Q + n * n;
        Qf = R + m * m;
        K = Qf + n * n;
        C1 = K + m * n;
        C2 = C1 + m * m;
        rho = C2 + n * n;
    }
};

// Shared memory of one instance of admm_kernel: A | B | K | C1 | C2, then per knot (N - 1 rows each) q ref (knots
// 2..N-1, then -Qf xref_N at knot N) | xmin | xmax | v | g | x (knots 2..N) (n each) and r ref | umin | umax | z | y | d,
// later u (m each).
__host__ __device__ inline size_t admm_smem_doubles(int n, int m, int N) {
    return (size_t)2 * n * n + 2 * n * m + m * m + (size_t)(N - 1) * (6 * n + 6 * m);
}

// lanes per instance: the least of 4, 8, 16, 32 that is >= n
__host__ __device__ inline int admm_group(int n) { return n <= 4 ? 4 : n <= 8 ? 8 : n <= 16 ? 16 : 32; }

static __global__ void admm_shift_kernel(const double *__restrict__ Q, const double *__restrict__ R, double rho,
                                  double *__restrict__ Qt, double *__restrict__ Rt, int n, int m, int64_t batch) {
    const int64_t nn = (int64_t)n * n, mm = (int64_t)m * m, total = batch * (nn + mm);
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        if (e < batch * nn) {
            const int r = (int)(e % nn);
            Qt[e] = (r % n == r / n) ? Q[e] + rho : Q[e];
        } else {
            const int64_t f = e - batch * nn;
            const int r = (int)(f % mm);
            Rt[f] = (r % m == r / m) ? R[f] + rho : R[f];
        }
    }
}

// One instance per G threads; P, K, dinfo: the output of dare_kernel on (A, B, Qt, Rt), instance-major; Q and R are
// stored from their upper triangles.  A failed
// instance (DARE info != 0, or Rt + B'PB not positive definite: 3000 + j) writes a record of NaN.
template <int G, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
    admm_cache_kernel(const double *__restrict__ Ag, const double *__restrict__ Bg, const double *__restrict__ Qg,
                      const double *__restrict__ Rg, const double *__restrict__ Rtg, const double *__restrict__ Pg, const double *__restrict__ Kg,
                      const int32_t *__restrict__ dinfo, double rho, double *__restrict__ cache,
                      int32_t *__restrict__ info, int n, int m, int64_t batch) {
    extern __shared__ double smem[];
    constexpr int IPC = THREADS / G;
    const int g = threadIdx.x / G, t = threadIdx.x % G;
    const int64_t inst_raw = (int64_t)blockIdx.x * IPC + g;
    const bool active = inst_raw < batch;
    const int64_t inst = active ? inst_raw : batch - 1;  // idle groups shadow a valid instance
    const int nn = n * n, nm = n * m, mm = m * m;
    double *P = smem + (size_t)g * ((size_t)nn + 2 * nm + 2 * mm), *B = P + nn, *PB = B + nm, *E = PB + nm,
           *C1 = E + mm;
    const double *A = Ag + inst * nn, *Bi = Bg + inst * (int64_t)nm, *Q = Qg + inst * nn,
                 *R = Rg + inst * (int64_t)mm, *Rt = Rtg + inst * (int64_t)mm, *K = Kg + inst * (int64_t)nm;
    for (int e = t; e < nn; e += G) P[e] = Pg[inst * nn + e];
    for (int e = t; e < nm; e += G) B[e] = Bi[e];
    for (int e = t; e < mm; e += G) {
        const int i = e % m, j = e / m;
        E[e] = Rt[i <= j ? e : j + i * m];
        C1[e] = i == j ? 1.0 : 0.0;
    }
    group_sync<G>();
    int code = dinfo[inst];
    if (!code) {
        co_gemm<G>(0, 0, n, m, n, 1.0, P, n, B, n, 0.0, PB, n, t);   // PB = P B
        co_gemm<G>(1, 0, m, m, n, 1.0, B, n, PB, n, 1.0, E, m, t);   // E = Rt + B'PB
        const int bad = co_chol<G>(E, m, m, t);
        if (bad) code = DARE_GAIN_NOT_PD + bad;
    }
    if (!code) {
        co_trsm_ut<G>(E, m, m, C1, m, m, t);  // C1 = U^-T
        co_trsm_un<G>(E, m, m, C1, m, m, t);  // C1 = U^-1 U^-T = E^-1
    }
    if (!active) return;
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    const AdmmCacheOffsets o(n, m);
    double *c = cache + inst * admm_cache_doubles(n, m);
    for (int e = t; e < nn; e += G) {
        const int i = e % n, j = e / n;
        double acl = A[j + i * n];  // C2 = (A - B K)'
        for (int l = 0; l < m; ++l) acl = fma(-B[j + l * n], K[l + i * m], acl);
        c[o.A + e] = code ? nan : A[e];
        c[o.Q + e] = code ? nan : Q[i <= j ? e : j + i * n];
        c[o.Qf + e] = code ? nan : (i == j ? P[e] - rho : P[e]);
        c[o.C2 + e] = code ? nan : acl;
    }
    for (int e = t; e < nm; e += G) {
        c[o.B + e] = code ? nan : B[e];
        c[o.K + e] = code ? nan : K[e];
    }
    for (int e = t; e < mm; e += G) {
        const int i = e % m, j = e / m;
        c[o.R + e] = code ? nan : R[i <= j ? e : j + i * m];
        c[o.C1 + e] = code ? nan : 0.5 * (C1[e] + C1[j + i * m]);
    }
    if (t == 0) {
        c[o.rho] = code ? nan : rho;
        if (info) info[inst] = code;
    }
}

// max that propagates NaN (an iterate gone NaN must not look converged)
__device__ __forceinline__ double admm_max(double a, double b) { return (b > a || b != b) ? b : a; }

// clamp that propagates NaN, = numpy.clip for lo <= hi
__device__ __forceinline__ double admm_clamp(double a, double lo, double hi) { return a < lo ? lo : (a > hi ? hi : a); }

template <int G>
__device__ __forceinline__ double admm_group_max(double v, unsigned mask) {
    for (int o = G / 2; o > 0; o >>= 1) v = admm_max(v, __shfl_xor_sync(mask, v, o, G));
    return v;
}

// One instance per G lanes, `ipb` instances per block of ipb * G <= 32 threads (one warp: the groups of a warp run
// their own iteration counts, their shuffles carry the group's own mask).  Caller arrays instance-major as in
// include/lqrb200.h; state in/out [z; y; v; g], read when `warm`.
template <int G>
__global__ void __launch_bounds__(32)
    admm_kernel(const double *__restrict__ cache, const double *__restrict__ x0g, const double *__restrict__ xrefg,
                const double *__restrict__ urefg, const double *__restrict__ uming, const double *__restrict__ umaxg,
                const double *__restrict__ xming, const double *__restrict__ xmaxg, double *__restrict__ state,
                int warm, double *__restrict__ Zg, int32_t *__restrict__ iters, double *__restrict__ res,
                int32_t *__restrict__ info, int n, int m, int N, int max_iter, double eps_pri, double eps_dual,
                int64_t batch, int ipb) {
    extern __shared__ double smem[];
    const int g = threadIdx.x / G, t = threadIdx.x % G;
    const int64_t inst = (int64_t)blockIdx.x * ipb + g;
    if (inst >= batch) return;  // the whole group leaves
    const unsigned mask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << ((threadIdx.x & 31) & ~(G - 1)));
    const int Kn = N - 1, nn = n * n, nm = n * m;
    const bool rx = t < n, ru = t < m;
    double *sA = smem + (size_t)g * admm_smem_doubles(n, m, N), *sB = sA + nn, *sK = sB + nm, *sC1 = sK + nm,
           *sC2 = sC1 + m * m;
    double *qr = sC2 + nn, *xlo = qr + Kn * n, *xhi = xlo + Kn * n, *v = xhi + Kn * n, *gd = v + Kn * n,
           *xs = gd + Kn * n;
    double *rr = xs + Kn * n, *ulo = rr + Kn * m, *uhi = ulo + Kn * m, *z = uhi + Kn * m, *y = z + Kn * m,
           *du = y + Kn * m;
    const AdmmCacheOffsets o(n, m);
    const double *c = cache + inst * admm_cache_doubles(n, m);
    const double inf = __longlong_as_double(0x7ff0000000000000LL), nan = __longlong_as_double(0x7ff8000000000000LL);

    // ---- set-up: the cache's operators, the reference terms, the bounds and the state, all on chip
    bool bad = false, empty = false;
    for (int e = t; e < nn; e += G) {
        sA[e] = c[o.A + e];
        sC2[e] = c[o.C2 + e];
        bad |= isnan(sA[e]) || isnan(sC2[e]);
    }
    for (int e = t; e < nm; e += G) {
        sB[e] = c[o.B + e];
        sK[e] = c[o.K + e];
        bad |= isnan(sB[e]) || isnan(sK[e]);
    }
    for (int e = t; e < m * m; e += G) {
        sC1[e] = c[o.C1 + e];
        bad |= isnan(sC1[e]);
    }
    const double rho = c[o.rho];
    bad |= isnan(rho);
    double x0 = 0.0;
    if (rx) {
        x0 = x0g[inst * n + t];
        bad |= isnan(x0);
        const double *xr = xrefg ? xrefg + inst * (int64_t)n * N : nullptr;
        for (int k = 0; k < Kn; ++k) {  // row k: knot k + 2
            double s = 0.0;
            if (xr) {
                const double *M = (k < Kn - 1) ? c + o.Q : c + o.Qf;
                for (int l = 0; l < n; ++l) s = fma(M[t + l * n], xr[(k + 1) * n + l], s);
            }
            const int64_t gi = inst * (int64_t)Kn * n + k * n + t;
            const int e = k * n + t;
            qr[e] = -s;
            xlo[e] = xming ? xming[gi] : -inf;
            xhi[e] = xmaxg ? xmaxg[gi] : inf;
            bad |= isnan(qr[e]) || isnan(xlo[e]) || isnan(xhi[e]);
            empty |= xlo[e] > xhi[e];
            v[e] = warm ? state[inst * 2 * (int64_t)Kn * (n + m) + 2 * Kn * m + e] : 0.0;
            gd[e] = warm ? state[inst * 2 * (int64_t)Kn * (n + m) + 2 * Kn * m + Kn * n + e] : 0.0;
            bad |= isnan(v[e]) || isnan(gd[e]);
        }
    }
    if (ru) {
        const double *ur = urefg ? urefg + inst * (int64_t)Kn * m : nullptr;
        for (int k = 0; k < Kn; ++k) {  // row k: knot k + 1
            double s = 0.0;
            if (ur)
                for (int l = 0; l < m; ++l) s = fma(c[o.R + t + l * m], ur[k * m + l], s);
            const int64_t gi = inst * (int64_t)Kn * m + k * m + t;
            const int e = k * m + t;
            rr[e] = -s;
            ulo[e] = uming ? uming[gi] : -inf;
            uhi[e] = umaxg ? umaxg[gi] : inf;
            bad |= isnan(rr[e]) || isnan(ulo[e]) || isnan(uhi[e]);
            empty |= ulo[e] > uhi[e];
            z[e] = warm ? state[inst * 2 * (int64_t)Kn * (n + m) + e] : 0.0;
            y[e] = warm ? state[inst * 2 * (int64_t)Kn * (n + m) + Kn * m + e] : 0.0;
            bad |= isnan(z[e]) || isnan(y[e]);
        }
    }
    __syncwarp(mask);
    int code = __any_sync(mask, bad) ? ADMM_NAN : __any_sync(mask, empty) ? ADMM_EMPTY_BOX : 0;

    // ---- iterations (DESIGN §4.12; oracle/admm.py is the same loop in numpy)
    double r_pri = inf, r_dual = inf;
    int it = 0;
    bool converged = false;
    while (!code && it < max_iter) {
        ++it;
        // backward pass: p_N = -Qf xref_N - rho (v_N - g_N); for k = N-1..1:
        //   d_k = C1 (B' p_{k+1} + rt_k),  p_k = qt_k + C2 p_{k+1} - K' rt_k
        double p = rx ? qr[(Kn - 1) * n + t] - rho * (v[(Kn - 1) * n + t] - gd[(Kn - 1) * n + t]) : 0.0;
        for (int k = Kn - 1; k >= 0; --k) {
            const double rt = ru ? rr[k * m + t] - rho * (z[k * m + t] - y[k * m + t]) : 0.0;
            double bp = 0.0, c2p = 0.0;
            for (int l = 0; l < n; ++l) {
                const double pl = __shfl_sync(mask, p, l, G);
                if (ru) bp = fma(sB[l + t * n], pl, bp);
                if (rx) c2p = fma(sC2[t + l * n], pl, c2p);
            }
            const double sj = bp + rt;
            double dj = 0.0, ktr = 0.0;
            for (int l = 0; l < m; ++l) {
                const double sl = __shfl_sync(mask, sj, l, G), rl = __shfl_sync(mask, rt, l, G);
                if (ru) dj = fma(sC1[t + l * m], sl, dj);
                if (rx) ktr = fma(sK[l + t * m], rl, ktr);
            }
            if (ru) du[k * m + t] = dj;
            if (k > 0 && rx)
                p = (qr[(k - 1) * n + t] - rho * (v[(k - 1) * n + t] - gd[(k - 1) * n + t])) + c2p - ktr;
        }
        // forward pass u_k = -K x_k - d_k, x_{k+1} = A x_k + B u_k, with each knot's slack, dual and residual terms
        double x = x0, rp = 0.0, rd = 0.0;
        for (int k = 0; k < Kn; ++k) {
            double kx = 0.0, ax = 0.0;
            for (int l = 0; l < n; ++l) {
                const double xl = __shfl_sync(mask, x, l, G);
                if (ru) kx = fma(sK[t + l * m], xl, kx);
                if (rx) ax = fma(sA[t + l * n], xl, ax);
            }
            const double u = ru ? -kx - du[k * m + t] : 0.0;
            double bu = 0.0;
            for (int l = 0; l < m; ++l) {
                const double ul = __shfl_sync(mask, u, l, G);
                if (rx) bu = fma(sB[t + l * n], ul, bu);
            }
            if (ru) {
                const int e = k * m + t;
                const double zo = z[e], zn = admm_clamp(u + y[e], ulo[e], uhi[e]);
                du[e] = u;
                z[e] = zn;
                y[e] = y[e] + u - zn;
                rp = admm_max(rp, fabs(u - zn));
                rd = admm_max(rd, fabs(zn - zo));
            }
            x = ax + bu;
            if (rx) {
                const int e = k * n + t;
                const double vo = v[e], vn = admm_clamp(x + gd[e], xlo[e], xhi[e]);
                xs[e] = x;
                v[e] = vn;
                gd[e] = gd[e] + x - vn;
                rp = admm_max(rp, fabs(x - vn));
                rd = admm_max(rd, fabs(vn - vo));
            }
        }
        r_pri = admm_group_max<G>(rp, mask);
        r_dual = rho * admm_group_max<G>(rd, mask);
        if (isnan(r_pri) || isnan(r_dual)) {
            code = ADMM_NAN;
            break;
        }
        if (r_pri <= eps_pri && r_dual <= eps_dual) {
            converged = true;
            break;
        }
    }
    if (!code && !converged) code = ADMM_MAX_ITER;

    // ---- outputs: a NaN instance or an empty box writes NaN
    const bool fail = code == ADMM_NAN || code == ADMM_EMPTY_BOX;
    double *Z = Zg + inst * ((int64_t)N * n + (int64_t)Kn * m);
    if (rx) {
        Z[t] = fail ? nan : x0;
        for (int k = 0; k < Kn; ++k) Z[(k + 1) * (n + m) + t] = fail ? nan : xs[k * n + t];
    }
    if (ru)
        for (int k = 0; k < Kn; ++k) Z[k * (n + m) + n + t] = fail ? nan : du[k * m + t];
    if (state) {
        double *s = state + inst * 2 * (int64_t)Kn * (n + m);
        if (ru)
            for (int e = t; e < Kn * m; e += m) {
                s[e] = fail ? nan : z[e];
                s[Kn * m + e] = fail ? nan : y[e];
            }
        if (rx)
            for (int e = t; e < Kn * n; e += n) {
                s[2 * Kn * m + e] = fail ? nan : v[e];
                s[2 * Kn * m + Kn * n + e] = fail ? nan : gd[e];
            }
    }
    if (t == 0) {
        if (iters) iters[inst] = it;
        if (res) {
            res[2 * inst] = fail ? nan : r_pri;
            res[2 * inst + 1] = fail ? nan : r_dual;
        }
        if (info) info[inst] = code;
    }
}
