// kkt_grad_kernels.cuh — the gradient step of lqrb_kkt_grad_f64: every requested gradient as outer products of the
// forward solution (z, mult) and the adjoint solution (ẑ, ν̂), one thread per output element (DESIGN §4.9).
#pragma once
#include "common.cuh"

// Division by a runtime divisor d >= 1 as a multiply-high and a shift, exact for numerators below 2^31 (the
// round-up method, Granlund & Montgomery 1994).  A plain 32-bit division costs about 20 instructions; the kernel
// decodes up to three per element and would be instruction-bound with them.
struct KktGradDiv {
    uint32_t d, mul, shift;
};
static inline KktGradDiv kkt_grad_div(uint32_t d) {
    uint32_t s = 0;
    while ((1ull << s) < d) ++s;
    return {d, (uint32_t)(((1ull << 32) * ((1ull << s) - d)) / d + 1), s};
}
__device__ __forceinline__ uint32_t div_of(uint32_t x, const KktGradDiv &v) {
    return (uint32_t)(((uint64_t)__umulhi(x, v.mul) + x) >> v.shift);
}

// The outputs, in the order of the C ABI.
enum KktGradOut { KG_Q, KG_R, KG_HUX, KG_q, KG_r, KG_A, KG_B, KG_d, KG_D2, KG_C, KG_c, KG_COUNT };

// Per-knot offsets of the ragged arrays, N + 1 entries each (entry N = the total), built on the host from p:
// mu, lam: multiplier offsets of mu_k, lam_k | C, c: offset of knot k's block in the concatenated C, c | D2: offset of
// the block that couples lam_{k-1} with z_k (entries 0 and 1 are 0).
struct KktGradTables {
    const int32_t *mu, *lam, *C, *c, *D2;
};

struct KktGradArgs {
    const double *z, *mult, *zh, *multh;  // forward / adjoint solutions, instance-major [NN] / [P] records
    KktGradTables t;
    int nout;                  // requested outputs, listed first in the arrays below
    int kind[KG_COUNT];        // which output
    double *out[KG_COUNT];
    KktGradDiv per[KG_COUNT];  // elements per instance
    int64_t first_block[KG_COUNT + 1];  // blocks [first_block[o], first_block[o+1]) write output o
    KktGradDiv n, m, nn, mm, nm;
    int32_t NN, P;
    int diag;                  // LQRB_HESS_DIAG: Q, R gradients only on the diagonal
};

#define KKT_GRAD_THREADS 256
#define KKT_GRAD_PER_THREAD 4

// largest k in [lo, hi) with T[k] <= x (T non-decreasing, T[lo] <= x): the knot whose ragged block holds element x (an
// empty block repeats the next block's offset and is skipped)
__device__ __forceinline__ int kkt_grad_knot(const int32_t *__restrict__ T, int lo, int hi, int32_t x) {
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(T + mid) <= x) lo = mid; else hi = mid;
    }
    return lo;
}

// Consecutive threads write consecutive elements of one instance-major output, whatever n: the stores of a warp are
// 256 contiguous bytes.  Each thread decodes (instance, knot, i, j) of its element and reads the four vector entries
// that form it; those small per-instance vectors (NN + P doubles, twice) are re-read by every element of the instance
// and stay in L1 / L2, so the bytes that reach DRAM are the gradients written and the vectors read once.
__global__ void __launch_bounds__(KKT_GRAD_THREADS) kkt_grad_kernel(const KktGradArgs a, int n, int m, int N,
                                                                    int64_t batch) {
    int o = 0;
    while (o + 1 < a.nout && (int64_t)blockIdx.x >= a.first_block[o + 1]) ++o;
    const int kind = a.kind[o];
    double *__restrict__ out = a.out[o];
    const KktGradDiv per = a.per[o];
    const int64_t total = batch * (int64_t)per.d;
    const int64_t e0 = ((int64_t)blockIdx.x - a.first_block[o]) * (KKT_GRAD_THREADS * KKT_GRAD_PER_THREAD);
    const int64_t inst0 = e0 / per.d;
    const uint32_t l0 = (uint32_t)(e0 - inst0 * per.d);  // < per: every l below stays under 2^31
#pragma unroll
    for (int r = 0; r < KKT_GRAD_PER_THREAD; ++r) {
        const uint32_t lr = l0 + threadIdx.x + r * KKT_GRAD_THREADS;
        const uint32_t di = div_of(lr, per);
        const int64_t inst = inst0 + di;
        if (e0 + threadIdx.x + r * KKT_GRAD_THREADS >= total) break;
        const int32_t l = (int32_t)(lr - di * per.d);
        const double *z = a.z + inst * a.NN, *zh = a.zh + inst * a.NN;
        const double *mu = a.mult + inst * a.P, *muh = a.multh + inst * a.P;
        double v;
        switch (kind) {
        case KG_Q: {  // ½(x̂ x' + x x̂') at knot k; DIAG: the diagonal only
            const int k = (int)div_of(l, a.nn), e = l - k * (int)a.nn.d, j = (int)div_of(e, a.n), i = e - j * n;
            const int zo = k * (n + m);
            v = (a.diag && i != j) ? 0.0 : 0.5 * fma(zh[zo + i], z[zo + j], z[zo + i] * zh[zo + j]);
            break;
        }
        case KG_R: {
            const int k = (int)div_of(l, a.mm), e = l - k * (int)a.mm.d, j = (int)div_of(e, a.m), i = e - j * m;
            const int zo = k * (n + m) + n;
            v = (a.diag && i != j) ? 0.0 : 0.5 * fma(zh[zo + i], z[zo + j], z[zo + i] * zh[zo + j]);
            break;
        }
        case KG_HUX: {  // û x' + u x̂' (m x n)
            const int k = (int)div_of(l, a.nm), e = l - k * (int)a.nm.d, j = (int)div_of(e, a.m), i = e - j * m;
            const int zo = k * (n + m);
            v = fma(zh[zo + n + i], z[zo + j], z[zo + n + i] * zh[zo + j]);
            break;
        }
        case KG_q: {
            const int k = (int)div_of(l, a.n);
            v = zh[k * (n + m) + l - k * n];
            break;
        }
        case KG_r: {
            const int k = (int)div_of(l, a.m);
            v = zh[k * (n + m) + n + l - k * m];
            break;
        }
        case KG_A:
        case KG_B: {  // λ̂ x' + λ x̂' | λ̂ u' + λ û'
            const KktGradDiv &blk = kind == KG_A ? a.nn : a.nm;
            const int k = (int)div_of(l, blk), e = l - k * (int)blk.d, j = (int)div_of(e, a.n), i = e - j * n;
            const int zo = k * (n + m) + (kind == KG_A ? 0 : n), lo = __ldg(a.t.lam + k);
            v = fma(muh[lo + i], z[zo + j], mu[lo + i] * zh[zo + j]);
            break;
        }
        case KG_d: {
            const int k = (int)div_of(l, a.n);
            v = muh[__ldg(a.t.lam + k) + l - k * n];
            break;
        }
        case KG_D2: {  // λ̂_{k-1} z_k' + λ_{k-1} ẑ_k' (n x w_k)
            const int k = kkt_grad_knot(a.t.D2, 1, N, l), e = l - __ldg(a.t.D2 + k), j = (int)div_of(e, a.n), i = e - j * n;
            const int lo = __ldg(a.t.lam + k - 1), zo = k * (n + m);
            v = fma(muh[lo + i], z[zo + j], mu[lo + i] * zh[zo + j]);
            break;
        }
        case KG_C: {  // μ̂_k z_k' + μ_k ẑ_k' (p_k x w_k)
            const int k = kkt_grad_knot(a.t.C, 0, N, l), pk = __ldg(a.t.c + k + 1) - __ldg(a.t.c + k);
            const int e = l - __ldg(a.t.C + k), j = e / pk, i = e - j * pk;
            const int mo = __ldg(a.t.mu + k), zo = k * (n + m);
            v = fma(muh[mo + i], z[zo + j], mu[mo + i] * zh[zo + j]);
            break;
        }
        default: {  // KG_c
            const int k = kkt_grad_knot(a.t.c, 0, N, l);
            v = muh[__ldg(a.t.mu + k) + l - __ldg(a.t.c + k)];
            break;
        }
        }
        out[inst * per.d + l] = v;
    }
}
