// kkt_hw_kernels.cuh — constrained KKT solve for the "quadrotor-sized" class (n + m <= 16): half a warp
// per instance.
//
// Replaces _solve!(::CholeskySolver) : src/cholesky_solver.jl:166-182 for the stage pattern of the
// reference's own fixtures (test/problems.jl:58-88: initial condition + dynamics + goal constraint, i.e.
// p = [n, 0, ..., 0, n], D2 = [-I 0], block-diagonal cost Hessian):
//   calculate_shur_factors!  src/jacobian_blocks.jl:220-286   S = D H^-1 D', h = D H^-1 g - d
//   cholesky!(chol, shur)    src/cholesky_solve.jl:28-67
//   forward_substitution!    :93-117        backward_substitution! :119-143   (Lambda = -S^-1 h)
//   calculate_primals!       src/cholesky_solver.jl:185-236   res = D'Lambda + g,  dz = -H^-1 res
// S is block tridiagonal in the order [mu_1, lam_1, ..., lam_{N-1}, mu_N].  The reference factors it as
// U'U block by block (two potrf + three trsm per knot, all n x n, strictly sequential in k).  Here the same
// elimination is carried in block-LDL' form with explicit inverses so that everything of order n^3 is a
// product:  with  Hi = H_k^-1 (a fully parallel pre-pass, one thread per knot),  W = Qi A',  F_k = -W,
//   Sigma_{k-1} = Cp + Qi_k            (pending Schur complement of row k-1, A_k = C_{k-1} aliasing :165-167)
//   Si = Sigma^-1 (Gauss-Jordan),  U = Si F_k,  v = Si y_{k-1}                            -> record (U, v)
//   Cp <- A W + B Ri B' - F_k' U,      dp <- (D1 Hi g - d) - F_k' v
// and the backward sweep is  x_{k-1} = v_k - U_k x_k,  Lambda = -x,  res_k, dz_k = -Hi res_k.
// The first knot (general C_1: B = C Hi C', E = C Hi D1') and the last knot (C_N, no controls) run the same
// step with other operands.  Two instances share a warp (the lane layout of a half-warp is described at
// kkt_hw2_kernel).  Knot data and Hi are staged by cp.async.bulk + mbarrier, re-issued as soon as their last
// reader in the current knot is done.
#pragma once
#include "riccati_dmma_kernels.cuh"

namespace khw {
using rdmma::bulk_g2s;
using rdmma::fast_rcp;
using rdmma::mbar_expect_tx;
using rdmma::mbar_init;
using rdmma::mbar_wait;

template <int n, int m, int HESS = LQRB_HESS_BLOCKDIAG>
struct Lay {
    static constexpr int w = n + m;
    static_assert(w <= 16 && n % 2 == 0 && m % 2 == 0, "half-warp layout: n + m <= 16, even sizes");
    static_assert(HESS == LQRB_HESS_BLOCKDIAG || HESS == LQRB_HESS_DIAG, "block-diagonal or diagonal cost Hessian");
    static constexpr int HQ = HESS == LQRB_HESS_DIAG ? n : tri(n), HR = HESS == LQRB_HESS_DIAG ? m : tri(m);
    // core of a knot record (same place in every knot with controls): H | g | D1 = [A B] | d
    static constexpr int oQ = 0, oR = HQ, og = oR + HR, oD1 = og + w, od = oD1 + n * w, CORE = od + n;
    static constexpr int oC0 = CORE, FIRST = CORE + n * w + n;  // first knot: + C_1 (n x w) | c_1
    static constexpr int MID = CORE;
    static constexpr int oCl = HQ + n, LAST = oCl + n * n + n;  // last knot: Q | g | C_N (n x n) | c_N
    static constexpr int HI = n * n + m * m;                        // Qi (full) | Ri (full)
    static constexpr int REC = n * n + n;                           // U (column-major) | v
    static_assert(HQ % 2 == 0 && HR % 2 == 0 && CORE % 2 == 0 && FIRST % 2 == 0 && LAST % 2 == 0 && HI % 2 == 0,
                  "bulk copies need 16-byte pieces");
    __host__ __device__ static constexpr int64_t data_rows(int N) { return FIRST + (int64_t)(N - 2) * MID + LAST; }
    __host__ __device__ static constexpr int64_t knot_off(int k) { return k == 0 ? 0 : FIRST + (int64_t)(k - 1) * MID; }
    __host__ __device__ static constexpr int64_t mult_rows(int N) { return 2 * n + (int64_t)(N - 1) * n; }
    __host__ __device__ static constexpr int64_t z_rows(int N) { return (int64_t)N * n + (int64_t)(N - 1) * m; }
    // shared memory per instance (doubles): g | D1 | d of the knot (H is only read by the pre-pass), Hi, three
    // n x n operand buffers, 64 doubles of vectors.  7,008 bytes per instance for n = 12, m = 4: eight 2-warp
    // CTAs = 16 warps per SM (the kernel is bound by the latency of its serial chains: warps are throughput).
    static constexpr int sCore2 = CORE - og, sHi2 = sCore2, s2A = sHi2 + HI, s2B = s2A + n * n, s2C = s2B + n * n,
                         sVec2 = s2C + n * n, INST2 = sVec2 + 64;
    static_assert(INST2 % 2 == 0 && og % 2 == 0, "16-byte alignment of the per-instance buffers");
    static_assert(2 * n * n >= n * w, "first knot stages C Hi (n x w) in WC|SI");
};

// In-place inverse of an SPD matrix from its packed upper Cholesky factor (LAPACK potri = trtri + lauum):
// u holds U (A = U'U) with dinv[j] = 1/U(j,j) on entry and the upper triangle of A^-1 on exit.
template <int k>
__device__ __forceinline__ void potri_packed(double *u, const double *dinv) {
    SM_UNROLL
    for (int j = 0; j < k; ++j) {  // V = U^-1, column by column
        double x[k];
        SM_UNROLL
        for (int i = 0; i < j; ++i) {
            double s = 0.0;
            SM_UNROLL
            for (int l = i; l < j; ++l) s = fma(u[tri_idx(i, l)], u[tri_idx(l, j)], s);
            x[i] = s;
        }
        SM_UNROLL
        for (int i = 0; i < j; ++i) u[tri_idx(i, j)] = -dinv[j] * x[i];
        u[tri_idx(j, j)] = dinv[j];
    }
    SM_UNROLL
    for (int c = 0; c < k; ++c) {  // A^-1 = V V', column by column (columns > c are still V)
        SM_UNROLL
        for (int r = 0; r < c; ++r) {
            double s = u[tri_idx(r, c)] * u[tri_idx(c, c)];
            SM_UNROLL
            for (int l = c + 1; l < k; ++l) s = fma(u[tri_idx(r, l)], u[tri_idx(c, l)], s);
            u[tri_idx(r, c)] = s;
        }
        double d = 0.0;
        SM_UNROLL
        for (int l = c; l < k; ++l) d = fma(u[tri_idx(c, l)], u[tri_idx(c, l)], d);
        u[tri_idx(c, c)] = d;
    }
}

// 256-bit global accesses (sm_100: LDG/STG.256), streaming; addresses must be 32-byte aligned
__device__ __forceinline__ void ld256_cs(const double *p, double &a, double &b, double &c, double &d) {
    asm volatile("ld.global.cs.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(a), "=d"(b), "=d"(c), "=d"(d) : "l"(p));
}
__device__ __forceinline__ void st256_cs(double *p, double a, double b, double c, double d) {
    asm volatile("st.global.cs.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}

// ------------------------------------------------------------------ pre-pass: H_k^-1 for every knot ---
// BlockCholesky block-diagonal mode (src/block_cholesky.jl:69-77, ldiv! :93-96) applied to the identity.
// soc != 0: H = I (second_order_correction!, src/cholesky_solver.jl:254-273).
template <int n, int m, int HESS>
__global__ void __launch_bounds__(128)
    kkt_hinv_kernel(const double *__restrict__ data, double *__restrict__ hinv, int32_t *__restrict__ hinfo,
                    int N, int64_t batch, int soc) {
    using L = Lay<n, m, HESS>;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= batch * N) return;
    const int64_t inst = idx / N;
    const int k = (int)(idx % N);
    const double *kp = data + inst * L::data_rows(N) + L::knot_off(k);
    double *out = hinv + idx * L::HI;
    int st = 0;
    if (HESS == LQRB_HESS_DIAG || soc) {  // stores the inverse (src/block_cholesky.jl:82-91), or the identity
        SM_UNROLL
        for (int j = 0; j < n; ++j) {
            const double q = soc ? 1.0 : kp[j];
            if (!(q > 0.0) && st == 0) st = j + 1;
            SM_UNROLL
            for (int i = 0; i < n; i += 2)
                __stcs(reinterpret_cast<double2 *>(out + n * j + i), make_double2(i == j ? 1.0 / q : 0.0, i + 1 == j ? 1.0 / q : 0.0));
        }
        if (k < N - 1) {
            SM_UNROLL
            for (int j = 0; j < m; ++j) {
                const double r = soc ? 1.0 : kp[L::oR + j];
                if (!(r > 0.0) && st == 0) st = n + j + 1;
                SM_UNROLL
                for (int i = 0; i < m; i += 2)
                    __stcs(reinterpret_cast<double2 *>(out + n * n + m * j + i), make_double2(i == j ? 1.0 / r : 0.0, i + 1 == j ? 1.0 / r : 0.0));
            }
        }
        if (st != 0) atomicMin(hinfo + inst, (k + 1) * 1000 + st);
        return;
    }
    // The H part of a record (HQ + HR doubles, 16-byte aligned) is read straight through with 256-bit loads
    // (a 16-byte head when the record starts on an odd 16-byte slot); the inverse goes out with 256-bit
    // stores, one full 32-byte sector per request (16-byte pieces from 32 different knots per request cost a
    // whole L2 sector transaction each).
    constexpr int HH = L::HQ + L::HR;
    double h[HH];
    auto ld128 = [&](int e) {
        const double2 v = __ldcs(reinterpret_cast<const double2 *>(kp + e));
        h[e] = v.x;
        h[e + 1] = v.y;
    };
    if ((reinterpret_cast<uintptr_t>(kp) & 31) == 0) {
        SM_UNROLL
        for (int e = 0; e + 4 <= HH; e += 4) ld256_cs(kp + e, h[e], h[e + 1], h[e + 2], h[e + 3]);
        if constexpr (HH % 4 == 2) ld128(HH - 2);
    } else {
        ld128(0);
        SM_UNROLL
        for (int e = 2; e + 4 <= HH; e += 4) ld256_cs(kp + e, h[e], h[e + 1], h[e + 2], h[e + 3]);
        if constexpr (HH % 4 == 0) ld128(HH - 2);
    }
    {
        double u[tri(n)], dinv[n];
        SM_UNROLL
        for (int e = 0; e < tri(n); ++e) u[e] = h[e];
        st = chol_packed<n>(u, dinv);
        potri_packed<n>(u, dinv);
        SM_UNROLL
        for (int j = 0; j < n; ++j) {
            if constexpr (n % 4 == 0) {
                SM_UNROLL
                for (int i = 0; i < n; i += 4)
                    st256_cs(out + n * j + i, u[sym_idx(i, j)], u[sym_idx(i + 1, j)], u[sym_idx(i + 2, j)], u[sym_idx(i + 3, j)]);
            } else {
                SM_UNROLL
                for (int i = 0; i < n; i += 2)
                    __stcs(reinterpret_cast<double2 *>(out + n * j + i), make_double2(u[sym_idx(i, j)], u[sym_idx(i + 1, j)]));
            }
        }
    }
    if (k < N - 1) {
        double u[tri(m)], dinv[m];
        SM_UNROLL
        for (int e = 0; e < tri(m); ++e) u[e] = h[tri(n) + e];
        const int s2 = chol_packed<m>(u, dinv);
        if (st == 0 && s2 != 0) st = n + s2;
        potri_packed<m>(u, dinv);
        SM_UNROLL
        for (int j = 0; j < m; ++j) {
            if constexpr (n % 4 == 0 && m % 4 == 0) {
                SM_UNROLL
                for (int i = 0; i < m; i += 4)
                    st256_cs(out + n * n + m * j + i, u[sym_idx(i, j)], u[sym_idx(i + 1, j)], u[sym_idx(i + 2, j)], u[sym_idx(i + 3, j)]);
            } else {
                SM_UNROLL
                for (int i = 0; i < m; i += 2)
                    __stcs(reinterpret_cast<double2 *>(out + n * n + m * j + i), make_double2(u[sym_idx(i, j)], u[sym_idx(i + 1, j)]));
            }
        }
    }
    if (st != 0) atomicMin(hinfo + inst, (k + 1) * 1000 + st);
}

// ------------------------------------------------------------------ half-warp primitives -------------
// out[i] += sum_l M[i + n*l] * coef[l]   (M column-major in shared memory, every lane reads the same column)
template <int n, int K>
__device__ __forceinline__ void acc_cols(double (&out)[n], const double *M, const double (&coef)[K], double sign) {
    SM_UNROLL
    for (int l = 0; l < K; ++l) {
        const double c = sign * coef[l];
        SM_UNROLL
        for (int i = 0; i < n; i += 2) {
            const double2 v = *reinterpret_cast<const double2 *>(M + n * l + i);
            out[i] = fma(v.x, c, out[i]);
            out[i + 1] = fma(v.y, c, out[i + 1]);
        }
    }
}
// dot(M[:, i], x) for one column i of a shared matrix
template <int n>
__device__ __forceinline__ double dot_col(const double *col, const double (&x)[n]) {
    double s0 = 0.0, s1 = 0.0;
    SM_UNROLL
    for (int l = 0; l < n; l += 2) {
        const double2 v = *reinterpret_cast<const double2 *>(col + l);
        s0 = fma(v.x, x[l], s0);
        s1 = fma(v.y, x[l + 1], s1);
    }
    return s0 + s1;
}
// dot(x (registers), y (shared vector))
template <int n>
__device__ __forceinline__ double dot_vec(const double (&x)[n], const double *y) {
    return dot_col<n>(y, x);
}
template <int n>
__device__ __forceinline__ void store_col(double *dst, const double (&a)[n]) {
    SM_UNROLL
    for (int i = 0; i < n; i += 2) *reinterpret_cast<double2 *>(dst + i) = make_double2(a[i], a[i + 1]);
}

// In-place inverse of the SPD matrix whose column hl (< n) this lane holds (Gauss-Jordan, no pivoting; the
// pivots are the squared Cholesky pivots, so the sign test is potrf's).  colb: 2*n doubles of this instance.
template <int n>
__device__ __forceinline__ int gj_inverse(double (&a)[n], double *colb, int hl) {
    int bad = 0;
    SM_UNROLL
    for (int kk = 0; kk < n; ++kk) {
        double *cb = colb + (kk & 1) * n;
        if (hl == kk) store_col<n>(cb, a);
        __syncwarp();
        double c[n];
        SM_UNROLL
        for (int i = 0; i < n; i += 2) {
            const double2 v = *reinterpret_cast<const double2 *>(cb + i);
            c[i] = v.x;
            c[i + 1] = v.y;
        }
        if (!(c[kk] > 0.0) && bad == 0) bad = kk + 1;
        const double p = fast_rcp(c[kk]);
        const bool piv = hl == kk;
        const double f = piv ? -p : a[kk] * p;
        SM_UNROLL
        for (int i = 0; i < n; ++i) {
            if (i == kk) a[i] = piv ? p : f;
            else a[i] = piv ? c[i] * f : fma(-c[i], f, a[i]);
        }
    }
    return bad;
}

// ------------------------------------------------------------------ block layout ----------------------
// Every n x n block is spread over the 16 lanes of the half-warp as a 4 x 4 grid of (n/4) x (n/4) register blocks.
// A product C = X Y' then needs only the lane's n/4 rows of X and n/4 rows of Y from shared memory (2 n^2 / 4
// doubles per lane instead of n^2 broadcast to every lane with one column per lane, which halves the shared-memory
// wavefronts); Gauss-Jordan exchanges the pivot row / column with 7 shuffles per pivot and the exact symmetrisation
// is a block transpose by shuffle.  Vectors stay one entry per lane.
template <int n, int bs>
__device__ __forceinline__ void gemm_rr(double (&acc)[bs][bs], const double *X, const double *Y, double sign) {
    // acc[r][c] += sign * sum_l X[r*n + l] * Y[c*n + l]
    SM_UNROLL
    for (int l = 0; l < n; l += 2) {
        double2 xv[bs], yv[bs];
        SM_UNROLL
        for (int r = 0; r < bs; ++r) xv[r] = *reinterpret_cast<const double2 *>(X + r * n + l);
        SM_UNROLL
        for (int c = 0; c < bs; ++c) yv[c] = *reinterpret_cast<const double2 *>(Y + c * n + l);
        SM_UNROLL
        for (int r = 0; r < bs; ++r)
            SM_UNROLL
            for (int c = 0; c < bs; ++c) {
                acc[r][c] = fma(sign * xv[r].x, yv[c].x, acc[r][c]);
                acc[r][c] = fma(sign * xv[r].y, yv[c].y, acc[r][c]);
            }
    }
}

// Two products that share the Y operand: acc1 += s1 * X1 Y', acc2 += s2 * X2 Y' (the Y rows are loaded once).
template <int n, int bs>
__device__ __forceinline__ void gemm_rr2(double (&acc1)[bs][bs], double (&acc2)[bs][bs], const double *X1, const double *X2,
                                         const double *Y, double s1, double s2) {
    SM_UNROLL
    for (int l = 0; l < n; l += 2) {
        double2 x1[bs], x2[bs], yv[bs];
        SM_UNROLL
        for (int r = 0; r < bs; ++r) x1[r] = *reinterpret_cast<const double2 *>(X1 + r * n + l);
        SM_UNROLL
        for (int r = 0; r < bs; ++r) x2[r] = *reinterpret_cast<const double2 *>(X2 + r * n + l);
        SM_UNROLL
        for (int c = 0; c < bs; ++c) yv[c] = *reinterpret_cast<const double2 *>(Y + c * n + l);
        SM_UNROLL
        for (int r = 0; r < bs; ++r)
            SM_UNROLL
            for (int c = 0; c < bs; ++c) {
                acc1[r][c] = fma(s1 * x1[r].x, yv[c].x, acc1[r][c]);
                acc1[r][c] = fma(s1 * x1[r].y, yv[c].y, acc1[r][c]);
                acc2[r][c] = fma(s2 * x2[r].x, yv[c].x, acc2[r][c]);
                acc2[r][c] = fma(s2 * x2[r].y, yv[c].y, acc2[r][c]);
            }
    }
}

// In-place Gauss-Jordan inverse of the SPD matrix held as register blocks: lane (bi, bj) of the half-warp
// owns rows bs*bi.., columns bs*bj...  Returns the 1-based index of the first non-positive pivot or 0.
// `spread` collects the largest (max - min) of the pivots' high words met so far: positive doubles order like their
// high words, so spread >> 20 is log2 of the pivot ratio — the conditioning estimate of the explicit inverse (integer
// pipe only, nothing on the FP64 chain).
template <int n, int bs>
__device__ __forceinline__ int gj_block(double (&a)[bs][bs], int bi, int bj, int &spread) {
    int bad = 0, lo = 0x7fffffff, hi = 0;
    SM_UNROLL
    for (int k = 0; k < n; ++k) {
        const int kb = k / bs, kr = k % bs;
        double prow[bs], pcol[bs];
        SM_UNROLL
        for (int c = 0; c < bs; ++c) prow[c] = __shfl_sync(0xffffffffu, a[kr][c], (kb << 2) | bj, 16);  // A[k][cols]
        SM_UNROLL
        for (int r = 0; r < bs; ++r) pcol[r] = __shfl_sync(0xffffffffu, a[r][kr], (bi << 2) | kb, 16);  // A[rows][k]
        const double piv = __shfl_sync(0xffffffffu, a[kr][kr], (kb << 2) | kb, 16);
        if (!(piv > 0.0) && bad == 0) bad = k + 1;
        lo = min(lo, __double2hiint(piv));
        hi = max(hi, __double2hiint(piv));
        const double p = fast_rcp(piv);
        const bool rowk = bi == kb, colk = bj == kb;
        SM_UNROLL
        for (int r = 0; r < bs; ++r) {
            const double f = pcol[r] * p;
            SM_UNROLL
            for (int c = 0; c < bs; ++c) {
                const bool pr = rowk && r == kr, pc = colk && c == kr;
                const double upd = fma(-f, prow[c], a[r][c]);
                a[r][c] = pr ? (pc ? p : prow[c] * p) : (pc ? -f : upd);
            }
        }
    }
    if (lo > 0 && hi >= lo) spread = max(spread, hi - lo);
    return bad;
}

template <int n, int m, int HESS, int WARPS, int MINB>
__global__ void __launch_bounds__(WARPS * 32, MINB)
    kkt_hw2_kernel(const double *__restrict__ data, const double *__restrict__ hinv, const int32_t *__restrict__ hinfo,
                   double *__restrict__ recs, double *__restrict__ dz, double *__restrict__ mult,
                   double *__restrict__ res, int32_t *__restrict__ info, int32_t *__restrict__ cinfo, int N,
                   int64_t batch, int soc) {
    using L = Lay<n, m, HESS>;
    static_assert(n % 4 == 0, "4 x 4 lane grid");
    constexpr int bs = n / 4;
    const double gsc = soc ? 0.0 : 1.0;  // second-order correction: g = 0
    constexpr int w = L::w;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, hh = lane >> 4, hl = lane & 15;
    const int bi = hl >> 2, bj = hl & 3, r0 = bs * bi, c0 = bs * bj;
    const int64_t inst_raw = ((int64_t)blockIdx.x * WARPS + warp) * 2 + hh;
    if (((int64_t)blockIdx.x * WARPS + warp) * 2 >= batch) return;  // whole warp leaves
    const bool active = inst_raw < batch;
    const int64_t inst = active ? inst_raw : batch - 1;  // an odd tail shadows the last instance (no stores)

    double *wb = reinterpret_cast<double *>(smem_raw) + (size_t)warp * (2 * L::INST2 + 4);
    double *S = wb + hh * L::INST2;
    // AT: X row-major (A_k or C_N), later U column-major; WC: W (or E0) column-major; SI: Sigma^-1
    // `core` keeps the offsets of a knot record; its H part (offsets < og) is not backed by shared memory
    double *core = S - L::og, *hi = S + L::sHi2, *AT = S + L::s2A, *WC = S + L::s2B, *SI = S + L::s2C, *vec = S + L::sVec2;
    double *UC = AT;
    double *ys = vec, *vs = vec + 16, *hgs = vec + 32, *xs = vec + 32 /* backward sweep only */, *rs_ = vec + 48;
    uint64_t *bars = reinterpret_cast<uint64_t *>(wb + 2 * L::INST2);  // [0] core, [1] Hi
    if (lane == 0) {
        mbar_init(bars, 1);
        mbar_init(bars + 1, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    uint32_t phC = 0, phH = 0;

    const double *db = data + inst * L::data_rows(N);
    const double *hb = hinv + inst * (int64_t)N * L::HI;
    double *rb = recs + inst * (int64_t)N * L::REC;
    double *zb = dz + inst * L::z_rows(N);
    double *mb = mult + inst * L::mult_rows(N);
    double *resb = res ? res + inst * L::z_rows(N) : nullptr;

    auto issue_core = [&](int k) {
        // only g | D1 | d of a record is read here (H went through the pre-pass)
        if (lane == 0) mbar_expect_tx(bars, 2u * (uint32_t)((k < N - 1 ? L::CORE - L::og : n + n * n + n) * 8));
        __syncwarp();
        if (hl == 0) {
            const double *src = db + L::knot_off(k);
            if (k < N - 1) {
                bulk_g2s(core + L::og, src + L::og, (L::CORE - L::og) * 8, bars);
            } else {
                bulk_g2s(core + L::og, src + L::HQ, n * 8, bars);
                bulk_g2s(core + L::oD1, src + L::oCl, n * n * 8, bars);
                bulk_g2s(core + L::od, src + L::oCl + n * n, n * 8, bars);
            }
        }
    };
    auto issue_hi = [&](int k) {
        if (lane == 0) mbar_expect_tx(bars + 1, 2u * (uint32_t)(L::HI * 8));
        __syncwarp();
        if (hl == 0) bulk_g2s(hi, hb + (int64_t)k * L::HI, L::HI * 8, bars + 1);
    };
    issue_hi(0);
    issue_core(0);

    int st_all = 0, spread = 0;
    double Cp[bs][bs], dp = 0.0;  // pending Schur complement (this lane's block) and right-hand side (entry hl)
    SM_UNROLL
    for (int r = 0; r < bs; ++r)
        SM_UNROLL
        for (int c = 0; c < bs; ++c) Cp[r][c] = 0.0;

    // ---------------- forward sweep: k = 0 .. N-1
    for (int k = 0; k < N; ++k) {
        const bool first = k == 0, last = k == N - 1;
        const int mk = last ? 0 : m;
        mbar_wait(bars + 1, phH);
        phH ^= 1;
        mbar_wait(bars, phC);
        phC ^= 1;
        const double *Xs = core + L::oD1;          // A_k, or C_N at the last knot (n x n, column-major)
        const double *Bs = core + L::oD1 + n * n;  // B_k
        // hg = Hi g  (one entry per lane)
        double hgj = 0.0;
        if (hl < n) {
            double gq[n];
            SM_UNROLL
            for (int l = 0; l < n; l += 2) {
                const double2 v = *reinterpret_cast<const double2 *>(core + L::og + l);
                gq[l] = gsc * v.x;
                gq[l + 1] = gsc * v.y;
            }
            hgj = dot_col<n>(hi + n * hl, gq);
        } else if (hl < n + mk) {
            SM_UNROLL
            for (int s = 0; s < m; ++s) hgj = fma(hi[n * n + m * (hl - n) + s], gsc * core[L::og + n + s], hgj);
        }
        hgs[hl] = hgj;
        // X row hl -> AT (row-major copy of the column-major knot block)
        double xrow[n];
        SM_UNROLL
        for (int l = 0; l < n; ++l) xrow[l] = hl < n ? Xs[hl + n * l] : 0.0;
        if (hl < n) store_col<n>(AT + n * hl, xrow);
        __syncwarp();
        // rho = X hg_x + B hg_u - d
        double rho = 0.0;
        if (hl < n) {
            rho = -core[L::od + hl];
            SM_UNROLL
            for (int l = 0; l < n; ++l) rho = fma(xrow[l], hgs[l], rho);
            if (!last) {
                SM_UNROLL
                for (int t = 0; t < m; ++t) rho = fma(Bs[hl + n * t], hgs[n + t], rho);
            }
        }
        // W = Qi X'  (block), published column-major
        double Wb[bs][bs];
        SM_UNROLL
        for (int r = 0; r < bs; ++r)
            SM_UNROLL
            for (int c = 0; c < bs; ++c) Wb[r][c] = 0.0;
        gemm_rr<n, bs>(Wb, hi + n * r0, AT + n * c0, 1.0);
        SM_UNROLL
        for (int c = 0; c < bs; ++c)
            SM_UNROLL
            for (int r = 0; r < bs; ++r) WC[(c0 + c) * n + r0 + r] = Wb[r][c];
        // Sigma block (middle / last knots) and right-hand side
        double Sb[bs][bs], y = dp - hgj;  // d += next.r_[1]
        SM_UNROLL
        for (int r = 0; r < bs; ++r)
            SM_UNROLL
            for (int c = 0; c < bs; ++c) Sb[r][c] = Cp[r][c] + hi[(r0 + r) * n + c0 + c];  // res.A .+= YYt[ip1,ip1]
        // V = Ri B[cols]' for the B Ri B' part of G22
        double Vb[m][bs];
        if (!last) {
            SM_UNROLL
            for (int c = 0; c < bs; ++c) {
                double brow[m];
                SM_UNROLL
                for (int s = 0; s < m; ++s) brow[s] = Bs[c0 + c + n * s];
                SM_UNROLL
                for (int t = 0; t < m; ++t) {
                    double v = 0.0;
                    SM_UNROLL
                    for (int s = 0; s < m; ++s) v = fma(hi[n * n + t + m * s], brow[s], v);
                    Vb[t][c] = v;
                }
            }
        }
        __syncwarp();  // WC is published
        // G22 = X W + B V
        double Gb[bs][bs];
        SM_UNROLL
        for (int r = 0; r < bs; ++r)
            SM_UNROLL
            for (int c = 0; c < bs; ++c) Gb[r][c] = 0.0;
        if (first) gemm_rr<n, bs>(Gb, AT + n * r0, WC + n * c0, 1.0);  // k >= 1: with U below (same W operand)
        if (!last) {
            SM_UNROLL
            for (int r = 0; r < bs; ++r)
                SM_UNROLL
                for (int t = 0; t < m; ++t) {
                    const double b = Bs[r0 + r + n * t];
                    SM_UNROLL
                    for (int c = 0; c < bs; ++c) Gb[r][c] = fma(b, Vb[t][c], Gb[r][c]);
                }
        }
        double sF = -1.0;  // F = sF * (matrix in WC): middle knots F = -W
        if (first) {
            // first knot: T0 = C Hi (n x w) staged in WC|SI, then B0 = T0 C', E0 = T0 D1', y0 = C hg - c
            __syncwarp();  // every lane is done reading W from WC
            const double *C0 = db + L::oC0;
            double t0[n];
            SM_UNROLL
            for (int i = 0; i < n; ++i) t0[i] = 0.0;
            if (hl < n) {
                SM_UNROLL
                for (int l = 0; l < n; ++l) {
                    const double c = hi[n * hl + l];
                    SM_UNROLL
                    for (int i = 0; i < n; ++i) t0[i] = fma(C0[i + n * l], c, t0[i]);
                }
            } else if (hl < w) {
                SM_UNROLL
                for (int s = 0; s < m; ++s) {
                    const double c = hi[n * n + m * (hl - n) + s];
                    SM_UNROLL
                    for (int i = 0; i < n; ++i) t0[i] = fma(C0[i + n * (n + s)], c, t0[i]);
                }
            }
            if (hl < w) store_col<n>(WC + n * hl, t0);
            __syncwarp();
            double a[n], Fc[n];
            SM_UNROLL
            for (int i = 0; i < n; ++i) a[i] = Fc[i] = 0.0;
            double yy = 0.0;
            if (hl < n) {
                double crow[w], drow[w];
                SM_UNROLL
                for (int j = 0; j < w; ++j) {
                    crow[j] = C0[hl + n * j];
                    drow[j] = core[L::oD1 + hl + n * j];
                    yy = fma(crow[j], hgs[j], yy);
                }
                acc_cols<n, w>(a, WC, crow, 1.0);
                acc_cols<n, w>(Fc, WC, drow, 1.0);
                yy -= C0[n * w + hl];
            }
            y = yy;
            __syncwarp();  // T0 is consumed
            if (hl < n) {
                store_col<n>(WC + n * hl, Fc);  // E0, column-major
                store_col<n>(SI + n * hl, a);   // B0 (symmetric)
            }
            __syncwarp();
            SM_UNROLL
            for (int r = 0; r < bs; ++r)
                SM_UNROLL
                for (int c = 0; c < bs; ++c) Sb[r][c] = SI[(r0 + r) * n + c0 + c];
            sF = 1.0;
        }
        __syncwarp();  // knot data, Hi and AT are no longer read
        if (k + 1 < N) {
            issue_hi(k + 1);
            issue_core(k + 1);
        }
        {
            const int bad = gj_block<n, bs>(Sb, bi, bj, spread);
            if (bad != 0 && st_all == 0) st_all = first ? 1000 + 100 + bad : k * 1000 + 200 + bad;
        }
        SM_UNROLL
        for (int r = 0; r < bs; ++r)
            SM_UNROLL
            for (int c = 0; c < bs; ++c) SI[(r0 + r) * n + c0 + c] = Sb[r][c];
        ys[hl] = y;
        __syncwarp();
        // v = Si y
        double v = 0.0;
        if (hl < n) {
            double yv[n];
            SM_UNROLL
            for (int l = 0; l < n; l += 2) {
                const double2 t = *reinterpret_cast<const double2 *>(ys + l);
                yv[l] = t.x;
                yv[l + 1] = t.y;
            }
            v = dot_col<n>(SI + n * hl, yv);
        }
        vs[hl] = v;
        // U = Si F  (block), published column-major in the AT buffer
        double Ub[bs][bs];
        SM_UNROLL
        for (int r = 0; r < bs; ++r)
            SM_UNROLL
            for (int c = 0; c < bs; ++c) Ub[r][c] = 0.0;
        if (first) {
            gemm_rr<n, bs>(Ub, SI + n * r0, WC + n * c0, sF);
        } else {
            gemm_rr2<n, bs>(Gb, Ub, AT + n * r0, SI + n * r0, WC + n * c0, 1.0, sF);
            __syncwarp();  // AT (the X rows) is consumed: U goes into the same buffer
        }
        SM_UNROLL
        for (int c = 0; c < bs; ++c)
            SM_UNROLL
            for (int r = 0; r < bs; ++r) UC[(c0 + c) * n + r0 + r] = Ub[r][c];
        __syncwarp();
        if (active && hl < n) {  // record (U column-major, v)
            double *rk = rb + (int64_t)k * L::REC;
            SM_UNROLL
            for (int i = 0; i < n; i += 2)
                *reinterpret_cast<double2 *>(rk + n * hl + i) = *reinterpret_cast<const double2 *>(UC + n * hl + i);
            rk[n * n + hl] = v;
        }
        // Cp' = G22 - F'U ; dp' = rho - F'v
        gemm_rr<n, bs>(Gb, WC + n * r0, UC + n * c0, -sF);
        if (hl < n) {
            double vv[n];
            SM_UNROLL
            for (int l = 0; l < n; l += 2) {
                const double2 t = *reinterpret_cast<const double2 *>(vs + l);
                vv[l] = t.x;
                vv[l + 1] = t.y;
            }
            dp = rho - sF * dot_col<n>(WC + n * hl, vv);
        } else {
            dp = 0.0;
        }
        // exact symmetrisation: block transpose by shuffle (an antisymmetric residue is amplified by |A|^2 per knot)
        SM_UNROLL
        for (int r = 0; r < bs; ++r)
            SM_UNROLL
            for (int c = 0; c < bs; ++c) {
                const double t = __shfl_sync(0xffffffffu, Gb[c][r], (bj << 2) | bi, 16);
                Cp[r][c] = 0.5 * (Gb[r][c] + t);
            }
        __syncwarp();
    }
    // ---------------- last block: mu_N' = Bl'^-1 y_mu  (Cp, dp hold Bl' and y_mu)
    double xcur = 0.0;
    {
        const int bad = gj_block<n, bs>(Cp, bi, bj, spread);
        if (bad != 0 && st_all == 0) st_all = N * 1000 + 100 + bad;
        SM_UNROLL
        for (int r = 0; r < bs; ++r)
            SM_UNROLL
            for (int c = 0; c < bs; ++c) SI[(r0 + r) * n + c0 + c] = Cp[r][c];
        ys[hl] = dp;
        __syncwarp();
        if (hl < n) {
            double yv[n];
            SM_UNROLL
            for (int l = 0; l < n; l += 2) {
                const double2 t = *reinterpret_cast<const double2 *>(ys + l);
                yv[l] = t.x;
                yv[l + 1] = t.y;
            }
            xcur = dot_col<n>(SI + n * hl, yv);
        }
        __syncwarp();
    }
    if (info && active && hl == 0) {
        const int hcode = hinfo[inst];
        info[inst] = hcode != 0x7f7f7f7f ? hcode : st_all;
    }
    if (active && hl == 0) cinfo[inst] = spread >> 20;  // log2 of the worst pivot ratio of any Sigma_k
    if (active && hl < n) __stcs(mb + L::mult_rows(N) - n + hl, -xcur);  // mu_N

    // ---------------- backward sweep: k = N-1 .. 0     x_{k-1} = v_k - U_k x_k,  Lambda = -x
    issue_hi(N - 1);
    issue_core(N - 1);
    for (int k = N - 1; k >= 0; --k) {
        const bool first = k == 0, last = k == N - 1;
        const int mk = last ? 0 : m, wk = n + mk;
        const double *rk = rb + (int64_t)k * L::REC;
        // record loads (written by this half-warp in the forward sweep)
        double ucol[n];  // row hl of U_k: U[hl][j] = rk[n*j + hl]
        SM_UNROLL
        for (int j = 0; j < n; ++j) ucol[j] = hl < n ? rk[n * j + hl] : 0.0;
        const double vk = hl < n ? rk[n * n + hl] : 0.0;
        xs[hl] = xcur;  // x of the block after this record: mu_N' (k = N-1) or lam_k'
        __syncwarp();
        double xprev = vk - dot_vec<n>(ucol, xs);  // k >= 1: lam_{k-1}' ; k = 0: mu_1'
        mbar_wait(bars + 1, phH);
        phH ^= 1;
        mbar_wait(bars, phC);
        phC ^= 1;
        // res_k = D1' lam_k + C' mu_k + D2' lam_{k-1} + g_k  with Lambda = -x   (calc_residual! :201-236)
        double r = 0.0;
        if (hl < wk) {
            r = gsc * core[L::og + hl];
            if (!last) {  // D1' lam_k : column hl of [A B] dotted with lam_k = -x_k
                double xv[n];
                SM_UNROLL
                for (int l = 0; l < n; l += 2) {
                    const double2 t = *reinterpret_cast<const double2 *>(xs + l);
                    xv[l] = t.x;
                    xv[l + 1] = t.y;
                }
                r -= dot_col<n>(core + L::oD1 + n * hl, xv);
            } else {  // C_N' mu_N
                double xv[n];
                SM_UNROLL
                for (int l = 0; l < n; l += 2) {
                    const double2 t = *reinterpret_cast<const double2 *>(xs + l);
                    xv[l] = t.x;
                    xv[l + 1] = t.y;
                }
                r -= dot_col<n>(core + L::oD1 + n * hl, xv);
            }
            if (!first && hl < n) r += xprev;  // D2' lam_{k-1} = -lam_{k-1} = +x_{k-1}
        }
        if (first) {  // C_1' mu_1 with mu_1 = -xprev
            ys[hl] = xprev;
            __syncwarp();
            if (hl < wk) {
                const double *C0 = db + L::oC0;
                double s = 0.0;
                SM_UNROLL
                for (int i = 0; i < n; ++i) s = fma(C0[i + n * hl], ys[i], s);
                r -= s;
            }
        }
        rs_[hl] = r;
        __syncwarp();
        // dz_k = -Hi res_k   (calc_primals! :195-199)
        double z = 0.0;
        if (hl < n) {
            double rv[n];
            SM_UNROLL
            for (int l = 0; l < n; l += 2) {
                const double2 t = *reinterpret_cast<const double2 *>(rs_ + l);
                rv[l] = t.x;
                rv[l + 1] = t.y;
            }
            z = -dot_col<n>(hi + n * hl, rv);
        } else if (hl < wk) {
            SM_UNROLL
            for (int s = 0; s < m; ++s) z = fma(-hi[n * n + m * (hl - n) + s], rs_[n + s], z);
        }
        if (active && hl < wk) {
            __stcs(zb + (int64_t)k * w + hl, z);
            if (resb) __stcs(resb + (int64_t)k * w + hl, r);
        }
        if (active && hl < n) {
            // multipliers: [mu_1 (n); lam_1 (n); ...; lam_{N-1}; mu_N]; this knot produces lam_{k-1} (k>=1) or mu_1
            __stcs(mb + (int64_t)k * n + hl, -xprev);
        }
        __syncwarp();  // knot data, Hi, xs, ys, rs_ are free
        if (k > 0) {
            issue_hi(k - 1);
            issue_core(k - 1);
        }
        xcur = xprev;
    }
}


}  // namespace khw
