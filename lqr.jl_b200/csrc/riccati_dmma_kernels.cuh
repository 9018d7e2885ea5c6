// riccati_dmma_kernels.cuh — warp-per-instance Riccati recursion on the FP64 tensor cores.
//
// Replaces solve!(sol, ::DPSolver, prob) : src/dynamic_programming.jl:54-72 for the "quadrotor-sized"
// class (n = 8 or 12 states, m <= 4 controls), where the per-knot work really is dense contractions:
//   compute_gain! :37-43  PB = P*B, PA = P*A, E = R + B'PB, K = E^-1 B'PA
//   compute_ctg!  :48-52  P_ = Q + A'PA - (A'PB) K
// written as one symmetric form (SURVEY Appendix A):   F = [A B]  (n x w, w = n + m)
//   T = F' * P^            (w x 16)      P^ = [P p; p' 0] embedded in a 16 x 16 "physical" tile space
//   M = T * F + blkdiag(Q, R)            (w x w)   = [Qxx Qxu; Qux Quu]
//   K = Quu^-1 [Qux | gu],  P^_ = Mxx^ - [Qxu | gu]' K     (Schur complement of the control block)
// One warp owns one instance for the whole horizon.  P^ lives in mma.sync m8n8k4 accumulator
// registers across all knots:
//   * P^ is symmetric, so its accumulator (C) fragment IS a valid B fragment of the next T = F'P^
//     (lane (g,q) of tile (rt,ct) holds P^[8rt+g][8ct+2q+e] = P^[k][col] with k = 8ct+2q+e) once the
//     contraction index is permuted — and the same permutation makes the T accumulators valid A
//     fragments of M = T*F.  No shared-memory round trip, no shuffles for the two GEMMs.
//   * the 6 (n=12) F fragments a lane loads are used as A fragments of T and B fragments of M: every
//     entry of A_k, B_k is read from shared memory exactly once per knot.
//   * physical positions: tile 0 = x0..x7; tile 1 = [x8 u0 x9 u1 x10 u2 x11 u3].  The control columns
//     of M land in register e=1 of tile column 1, one control per quad lane, which is what the Schur
//     MMA (k = 4 = one DMMA per tile) wants.  In P^ space position 9 (u0's slot) carries the affine
//     column p, so kff / p_ come out of the same MMAs.
// Knot records (tile width 1 layout: A | B | Q | R | q | r contiguous per knot) are streamed HBM ->
// shared memory with cp.async.bulk + mbarrier, STAGES-1 knots ahead, by the owning warp itself.
#pragma once
#include "smallmat.cuh"

namespace rdmma {

__device__ __forceinline__ void mma884(double &d0, double &d1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(d0), "+d"(d1)
        : "d"(a), "d"(b));
}

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok = 0;
    const uint32_t a = smem_u32(bar);
    do {
        asm volatile(
            "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
            : "=r"(ok)
            : "r"(a), "r"(parity)
            : "memory");
    } while (!ok);
}
// 1-D TMA bulk copy global -> shared (16-byte aligned addresses and size), completes on `bar`
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

template <int n, int m>
struct Map {
    static_assert(n == 8 || n == 12, "state tile map is written for n = 8, 12");
    static_assert(m >= 1 && m <= 4, "one control per quad lane");
    static constexpr int w = n + m;
    static constexpr int KS = n / 4;  // contraction steps over the state index
    static constexpr int oQ = n * w, oR = oQ + tri(n), oq = oR + tri(m), orr = oq + n;
    static constexpr int F = lqrb_riccati_knot_rows(n, m);  // doubles per knot record (orr + m, padded to even)
    static constexpr int TR = tri(n) + 2 * n;
    static constexpr int GR = m * n + m;
    static_assert(F % 2 == 0, "bulk copies need 16-byte records");
    // physical position -> index into z = [x; u] (M space); -1 = unused slot
    __host__ __device__ static constexpr int zmap(int pos) {
        if (pos < 8) return pos;
        const int j = pos - 8;
        if ((j & 1) == 0) return (8 + j / 2 < n) ? 8 + j / 2 : -1;
        return ((j - 1) / 2 < m) ? n + (j - 1) / 2 : -1;
    }
    // physical position -> state index (P^ space); -1 = unused, -2 = the affine ("1") slot
    __host__ __device__ static constexpr int xmap(int pos) {
        if (pos < 8) return pos;
        if (pos == 9) return -2;
        const int j = pos - 8;
        if ((j & 1) == 0) return (8 + j / 2 < n) ? 8 + j / 2 : -1;
        return -1;
    }
    // contraction step s, quad lane q -> state index k (the permutation that lets C fragments be
    // reused as operands): s = 0: tile-0 even columns, 1: tile-0 odd columns, 2: tile-1 even columns
    __host__ __device__ static constexpr int kperm(int s, int q) { return s == 0 ? 2 * q : s == 1 ? 2 * q + 1 : 8 + q; }
};

// per-warp shared memory: STAGES knot records | 184 doubles of staging (backward: control block, the
// lanes' right-hand sides and a zero row, laid out below; forward: [x;u] double buffer + one knot of gains)
// | STAGES mbarriers.  The backward layout keeps row stride 8: Qd uses 4 of its 8 rows and gud 4 of its 8
// entries.  Packing it tighter would save 40 doubles per warp and change nothing else: registers, not
// shared memory, limit the CTAs per SM.
#define RDMMA_AUX 184
__host__ __device__ inline size_t riccati_dmma_warp_smem(int F, int stages) {
    return ((size_t)stages * F * 8 + RDMMA_AUX * 8 + (size_t)stages * 8 + 15) / 16 * 16;
}

// 1/x from the hardware seed and two Newton steps (inputs here are O(1) pivots; no special cases)
__device__ __forceinline__ double fast_rcp(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    e = fma(-x, r, 1.0);
    return fma(r, e, r);
}

// The same seed (20 bits, measured: tools/ubench/rcp_test.cu) with ONE third-order step r (1 + e + e^2),
// e = 1 - x r: three dependent FMAs instead of four, within one ulp of the correctly rounded quotient.  For the
// serial 8 x 8 pivot chains of the CTA kernels, where the reciprocal is on the critical path of the whole CTA
// (5b-K: -2 %), and for the m dependent pivots of riccati_dmma's control block (5a-R: about 1 % against
// fast_rcp).  The other warp-level kernels keep fast_rcp: no gain there, or a small loss.
__device__ __forceinline__ double fast_rcp3(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    const double e = fma(-x, r, 1.0);
    const double t = fma(e, e, e);
    return fma(r, t, r);
}

// Row q of the inverse of the SPD m x m control block a (upper triangle read), factored as L D L' in the
// natural pivot order: L y = e_q, then L' x = D^-1 y.  Every quad lane factors the same block in the same
// order, so the m rows the quad applies to [Mux | gu] belong to one factorisation.  That is what keeps the
// gains within a small factor of the reference's chol_solve! when two cheap actuators act almost alike:
// the right-hand sides then lie along the large eigenvectors of Muu, and only rows of one factorisation
// cancel the huge entries of its inverse.  The former form (each lane's row by 2 x 2 adjugate/determinant
// blocks of the block cyclically shifted by its own control) reached relative errors of 17 where the
// reference order's error is 3e-9 (n = 12, m = 4, tests/test_gpu_riccati_conditioning.py).
// Pivots d_j are potrf's squared Cholesky pivots; only their reciprocals (fast_rcp3) enter the result.
// info: index of the first non-positive pivot (potrf semantics), the same in every lane.
template <int m>
__device__ __forceinline__ int spd_inv_row(double (&a)[4][4], int q, double (&mi)[4]) {
    int info = 0;
    double l[4][4], r[4];  // l[i][j] = a(j)[j][i] / d_j for i > j: the multipliers of pivot j; r[j] = 1 / d_j
    SM_UNROLL
    for (int j = 0; j < m; ++j) {
        if (info == 0 && !(a[j][j] > 0.0)) info = j + 1;
        r[j] = fast_rcp3(a[j][j]);
        SM_UNROLL
        for (int i = j + 1; i < m; ++i) l[i][j] = a[j][i] * r[j];
        SM_UNROLL
        for (int i = j + 1; i < m; ++i)
            SM_UNROLL
            for (int k = i; k < m; ++k) a[i][k] = fma(-l[i][j], a[j][k], a[i][k]);
    }
    SM_UNROLL
    for (int i = 0; i < m; ++i) {  // L y = e_q
        double s = q == i ? 1.0 : 0.0;
        SM_UNROLL
        for (int j = 0; j < i; ++j) s = fma(-l[i][j], mi[j], s);
        mi[i] = s;
    }
    SM_UNROLL
    for (int i = m - 1; i >= 0; --i) {  // L' x = D^-1 y
        double s = mi[i] * r[i];
        SM_UNROLL
        for (int j = i + 1; j < m; ++j) s = fma(-l[j][i], mi[j], s);
        mi[i] = s;
    }
    return info;
}

template <int n, int m, int STAGES, int WARPS, int MINB>
__global__ void __launch_bounds__(WARPS * 32, MINB)
    riccati_dmma_kernel(const double *__restrict__ knots, const double *__restrict__ term,
                        double *__restrict__ Z, double *__restrict__ gains, int32_t *__restrict__ info,
                        int N, int lti, int64_t batch) {
    using L = Map<n, m>;
    constexpr int F = L::F, KS = L::KS, w = L::w, GR = L::GR;
    constexpr bool HAS_X1 = n > 8;  // states live at the even positions of tile 1
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, q = lane & 3;
    const int64_t inst = (int64_t)blockIdx.x * WARPS + warp;
    if (inst >= batch) return;  // whole warp leaves; no CTA-wide barrier is used below

    unsigned char *wbase = smem_raw + (size_t)warp * riccati_dmma_warp_smem(F, STAGES);
    double *buf = reinterpret_cast<double *>(wbase);             // STAGES records
    double *aux = buf + (size_t)STAGES * F;                      // RDMMA_AUX doubles
    uint64_t *full = reinterpret_cast<uint64_t *>(aux + RDMMA_AUX);  // STAGES mbarriers
    // backward-pass staging (doubles): V0d[8][8] | Qd[8][8] (4 rows used) | V1e[4][8] | gud[8] (4 used) | G1e[4] | zero[8]
    double *V0d = aux, *Qd = aux + 64, *V1e = aux + 128, *gud = aux + 160, *G1e = aux + 168, *zero = aux + 172;
    // forward-pass staging
    double *zs = aux, *gs = aux + 32;

    if (lane == 0) {
        SM_UNROLL
        for (int s = 0; s < STAGES; ++s) mbar_init(full + s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (lane < 8) zero[lane] = 0.0;
    __syncwarp();

    const int Kn = lti ? 1 : N - 1;
    const double *rec_g = knots + inst * (int64_t)Kn * F;
    const double *tb = term + inst * L::TR;
    double *zb = Z + inst * ((int64_t)N * n + (int64_t)(N - 1) * m);
    double *gb = gains + inst * (int64_t)(N - 1) * GR;
    const int steps = N - 1;

    // ---------------- per-lane constant tables (pointers into stage 0; stage s adds s*F)
    const bool odd = g & 1;
    const int su = (g - 1) >> 1;  // control index of an odd row of tile 1
    // z index of physical position 8 + g (tile 1 row/column of this lane); -1 = unused slot
    const int zc1 = odd ? (su < m ? n + su : -1) : (HAS_X1 && 8 + g / 2 < n ? 8 + g / 2 : -1);
    const double *pf0 = buf + 2 * q + n * g;                         // F[2q..2q+1][x_g]; F[8+q][x_g] at +8-q
    const double *pf1 = buf + 2 * q + n * (zc1 >= 0 ? zc1 : 0);
    const bool has1 = zc1 >= 0;
    // blkdiag(Q, R) entries of this lane's accumulator slots (packed upper storage)
    auto qoff = [](int i, int j) { return L::oQ + (i <= j ? j * (j + 1) / 2 + i : i * (i + 1) / 2 + j); };
    const double *ph00a = buf + qoff(g, 2 * q), *ph00b = buf + qoff(g, 2 * q + 1);
    const double *ph01 = buf + qoff(g, HAS_X1 ? 8 + q : 0);          // column x_{8+q}
    int o11 = L::oQ;
    bool v11 = false;
    if (!odd) {
        if (HAS_X1 && 8 + g / 2 < n) { o11 = qoff(8 + g / 2, 8 + q); v11 = true; }
    } else if (su < m && q < m) {
        o11 = L::oR + (su <= q ? q * (q + 1) / 2 + su : su * (su + 1) / 2 + q);
        v11 = true;
    }
    const double *ph11 = buf + o11;
    const double *pq0 = buf + L::oq + g;
    const double *pq1 = buf + (zc1 >= 0 ? (zc1 < n ? L::oq + zc1 : L::orr + (zc1 - n)) : L::oq);
    // gain store offsets: K0 -> K[q, x_g]; K1 -> K[q, x_{8+g/2}] (g even) or kff[q] (g == 1)
    const int go0 = q < m ? q + m * g : -1;
    const int go1 = q < m ? (odd ? (g == 1 ? m * n + q : -1) : (HAS_X1 && 8 + g / 2 < n ? q + m * (8 + g / 2) : -1)) : -1;
    // control-block staging: every lane reads the whole block and its own two right-hand sides
    const double *rv0 = V0d + 8 * g;
    const double *rv1 = (!odd) ? V1e + 8 * (g >> 1) : ((g == 1 && q < m) ? gud : zero);
    const double *rt10 = g == 1 ? G1e + q : zero;
    // selection fragments of the transposing MMAs (scaled by 1/2 for the symmetrisation)
    const double hsel0 = g == 2 * q ? 0.5 : 0.0, hsel1 = g == 2 * q + 1 ? 0.5 : 0.0;

    // ---------------- terminal cost-to-go  P^ = [Qf qf; qf' 0] in physical positions
    double P[2][2][2];
    SM_UNROLL
    for (int rt = 0; rt < 2; ++rt)
        SM_UNROLL
        for (int ct = 0; ct < 2; ++ct)
            SM_UNROLL
            for (int e = 0; e < 2; ++e) {
                const int pr = 8 * rt + g, pc = 8 * ct + 2 * q + e;
                const int xr = pr < 8 ? pr : (pr == 9 ? -2 : (((pr - 8) & 1) == 0 && 8 + (pr - 8) / 2 < n ? 8 + (pr - 8) / 2 : -1));
                const int xc = pc < 8 ? pc : (pc == 9 ? -2 : (((pc - 8) & 1) == 0 && 8 + (pc - 8) / 2 < n ? 8 + (pc - 8) / 2 : -1));
                double v = 0.0;
                if (xr >= 0 && xc >= 0) v = tb[xr <= xc ? xc * (xc + 1) / 2 + xr : xr * (xr + 1) / 2 + xc];
                else if (xr >= 0 && xc == -2) v = tb[tri(n) + xr];
                else if (xr == -2 && xc >= 0) v = tb[tri(n) + xc];
                P[rt][ct][e] = v;
            }

    auto issue_bwd = [&](int it, int st) {
        const int k = steps - 1 - it;
        mbar_expect_tx(full + st, F * 8);
        bulk_g2s(buf + (size_t)st * F, rec_g + (int64_t)(lti ? 0 : k) * F, F * 8, full + st);
    };
    if (lane == 0) {
        for (int it = 0; it < STAGES - 1 && it < steps; ++it) issue_bwd(it, it);
    }

    int st_all = 0;
    double *gk = gb + (int64_t)(steps - 1) * GR;
    // ---------------- backward pass: k = N-2 .. 0   (src/dynamic_programming.jl:61-64)
    for (int it0 = 0; it0 < steps; it0 += STAGES) {
        const uint32_t par = (it0 / STAGES) & 1;
        SM_UNROLL
        for (int st = 0; st < STAGES; ++st) {
            const int it = it0 + st;
            if (it >= steps) break;
            if (lane == 0 && it + STAGES - 1 < steps) issue_bwd(it + STAGES - 1, (st + STAGES - 1) % STAGES);
            mbar_wait(full + st, par);
            const int so = st * F;  // compile-time after unrolling: loads are [lane pointer + immediate]

            // F fragments: fr[mt][s] = F[kperm(s,q)][z(8mt+g)]  (A fragment of T and B fragment of M)
            double fr[2][3];
            {
                const double2 v = *reinterpret_cast<const double2 *>(pf0 + so);
                fr[0][0] = v.x;
                fr[0][1] = v.y;
                fr[0][2] = KS == 3 ? (pf0 - 2 * q + 8 + q)[so] : 0.0;
                const double2 u = *reinterpret_cast<const double2 *>(pf1 + so);
                const double u2 = KS == 3 ? (pf1 - 2 * q + 8 + q)[so] : 0.0;
                fr[1][0] = has1 ? u.x : 0.0;
                fr[1][1] = has1 ? u.y : 0.0;
                fr[1][2] = has1 ? u2 : 0.0;
            }
            // M accumulators start at blkdiag(Q, R); tile (1,0) is never formed
            double M00[2] = {ph00a[so], ph00b[so]};
            double M01[2] = {HAS_X1 ? ph01[so] : 0.0, 0.0};
            const double h11 = ph11[so];
            double M11[2] = {(!odd && v11) ? h11 : 0.0, (odd && v11) ? h11 : 0.0};
            const double qr0 = pq0[so];
            const double qr1 = has1 ? pq1[so] : 0.0;

            // T = F' P^   (compute_gain! :38,40 — PB and PA at once, plus F'p in position 9)
            double T[2][2][2] = {};
            SM_UNROLL
            for (int s = 0; s < KS; ++s)
                SM_UNROLL
                for (int mt = 0; mt < 2; ++mt)
                    SM_UNROLL
                    for (int nt = 0; nt < 2; ++nt) {
                        const double pb = s == 0 ? P[nt][0][0] : s == 1 ? P[nt][0][1] : P[nt][1][0];
                        mma884(T[mt][nt][0], T[mt][nt][1], fr[mt][s], pb);
                    }
            // M += T F   (E = R + B'PB :39, K = B'PA :41, A'PA :50)
            SM_UNROLL
            for (int s = 0; s < KS; ++s) {
                const double ta0 = s == 0 ? T[0][0][0] : s == 1 ? T[0][0][1] : T[0][1][0];
                const double ta1 = s == 0 ? T[1][0][0] : s == 1 ? T[1][0][1] : T[1][1][0];
                mma884(M00[0], M00[1], ta0, fr[0][s]);
                mma884(M01[0], M01[1], ta0, fr[1][s]);
                mma884(M11[0], M11[1], ta1, fr[1][s]);
            }
            // g^ = [q; r] + F'p : column 9 of T, held by quad lane 0
            const double gh0 = T[0][1][1] + qr0;
            const double gh1 = T[1][1][1] + qr1;

            // ---- stage the control columns
            if (q < m) {
                V0d[8 * g + q] = M01[1];  // Mxu[x_g][u_q]
                if (!odd) V1e[8 * (g >> 1) + q] = M11[1];  // Mxu[x_{8+g/2}][u_q]
                else if (su < m) Qd[8 * su + q] = M11[1];  // Quu[su][q]
            }
            if (q == 0) {
                if (!odd) G1e[g >> 1] = gh1;
                else if (su < m) gud[su] = gh1;
            }
            __syncwarp();
            double a[4][4], v0[4], v1[4];
            SM_UNROLL
            for (int s = 0; s < m; ++s)
                SM_UNROLL
                for (int t = s; t < m; ++t) a[s][t] = Qd[8 * s + t];
            SM_UNROLL
            for (int t = 0; t < m; ++t) {
                v0[t] = rv0[t];
                v1[t] = rv1[t];
            }
            const double t10 = rt10[0];
            double mi[4];
            const int ci = spd_inv_row<m>(a, q, mi);  // chol_solve! :28-31 (E^-1 applied by multiplication)
            if (ci != 0 && st_all == 0) st_all = (steps - it) * 1000 + ci;
            // K[q][pos] = row q of Quu^-1 times [Qux | gu]   (K = E^-1 B'PA :41-43, kff in position 9)
            double K0 = 0.0, K1 = 0.0;
            SM_UNROLL
            for (int t = 0; t < m; ++t) {
                K0 = fma(mi[t], v0[t], K0);
                K1 = fma(mi[t], v1[t], K1);
            }
            if (go0 >= 0) gk[go0] = K0;
            if (go1 >= 0) gk[go1] = K1;
            gk -= GR;

            // ---- P^_ = Mxx^ - [Qxu | gu]' K  (compute_ctg! :50-51 and the affine column in the same MMAs)
            double S00[2] = {M00[0], M00[1]};
            double S01[2] = {M01[0], q == 0 ? gh0 : 0.0};
            double S11[2] = {odd ? t10 : M11[0], (!odd && q == 0) ? gh1 : 0.0};
            const double nV0 = q < m ? -M01[1] : 0.0;
            const double nV1 = q < m ? -rv1[q] : 0.0;  // this lane's own control q
            mma884(S00[0], S00[1], nV0, K0);
            mma884(S01[0], S01[1], nV0, K1);
            mma884(S11[0], S11[1], nV1, K1);
            // Exact symmetrisation.  F'P^F amplifies any antisymmetric rounding residue of P^ by the
            // OPEN-loop dynamics (|A|^2 per knot: 1e-16 -> 5e-8 over 1000 knots of an unstable LTI system),
            // so P^ is kept bitwise symmetric: tile^T = sum_e Sel_e * B(tile, e), Sel_e[r][k] = (r == 2k+e)
            // — a C fragment read as a B fragment is the transpose — 2 DMMAs per tile, all products exact.
            P[0][0][0] = 0.5 * S00[0];
            P[0][0][1] = 0.5 * S00[1];
            mma884(P[0][0][0], P[0][0][1], hsel0, S00[0]);
            mma884(P[0][0][0], P[0][0][1], hsel1, S00[1]);
            P[1][1][0] = 0.5 * S11[0];
            P[1][1][1] = 0.5 * S11[1];
            mma884(P[1][1][0], P[1][1][1], hsel0, S11[0]);
            mma884(P[1][1][0], P[1][1][1], hsel1, S11[1]);
            P[0][1][0] = S01[0];
            P[0][1][1] = S01[1];
            P[1][0][0] = 0.0;
            P[1][0][1] = 0.0;
            mma884(P[1][0][0], P[1][0][1], hsel0 + hsel0, S01[0]);
            mma884(P[1][0][0], P[1][0][1], hsel1 + hsel1, S01[1]);
            __syncwarp();  // every lane is done with this stage and the staging area
        }
    }
    if (info && lane == 0) info[inst] = st_all;
    __syncwarp();
    // ---------------- forward rollout   (src/dynamic_programming.jl:66-70)
    const int AB = n * w;  // doubles of [A B] at the head of a record
    auto issue_fwd = [&](int it) {
        const int st = (steps + it) % STAGES;
        mbar_expect_tx(full + st, AB * 8);
        bulk_g2s(buf + (size_t)st * F, rec_g + (int64_t)(lti ? 0 : it) * F, AB * 8, full + st);
    };
    if (lane == 0) {
        for (int it = 0; it < STAGES - 1 && it < steps; ++it) issue_fwd(it);
    }
    // gains of the next two knots ride in registers (written by this warp; plain loads)
    double ga[2][2];
    SM_UNROLL
    for (int d = 0; d < 2; ++d) {
        const double *gk = gb + (int64_t)d * GR;
        ga[d][0] = (d < steps && lane < GR) ? gk[lane] : 0.0;
        ga[d][1] = (d < steps && lane + 32 < GR) ? gk[lane + 32] : 0.0;
    }
    if (lane < n) zs[lane] = tb[tri(n) + n + lane];
    __syncwarp();
    const int row = lane & 15, half = lane >> 4;
    for (int it = 0; it < steps; ++it) {
        const int git = steps + it;  // position in the stage ring continues from the backward pass
        const int st = git % STAGES;
        double *zc = zs + (it & 1) * 16, *zn = zs + ((it + 1) & 1) * 16;
        if (lane == 0 && it + STAGES - 1 < steps) issue_fwd(it + STAGES - 1);
        // stage this knot's gains, prefetch knot it+2
        gs[lane] = ga[0][0];
        if (lane + 32 < 64) gs[lane + 32] = ga[0][1];
        ga[0][0] = ga[1][0];
        ga[0][1] = ga[1][1];
        {
            const double *gk = gb + (int64_t)(it + 2) * GR;
            ga[1][0] = (it + 2 < steps && lane < GR) ? gk[lane] : 0.0;
            ga[1][1] = (it + 2 < steps && lane + 32 < GR) ? gk[lane + 32] : 0.0;
        }
        __syncwarp();
        double *zk = zb + (int64_t)it * w;
        if (lane < n) __stcs(zk + lane, zc[lane]);
        if (lane < m) {  // u = -K x - kff
            double acc0 = -gs[m * n + lane], acc1 = 0.0;
            SM_UNROLL
            for (int c = 0; c < n; c += 2) {
                acc0 = fma(-gs[lane + m * c], zc[c], acc0);
                acc1 = fma(-gs[lane + m * (c + 1)], zc[c + 1], acc1);
            }
            const double u = acc0 + acc1;
            zc[n + lane] = u;
            __stcs(zk + n + lane, u);
        }
        mbar_wait(full + st, (git / STAGES) & 1);
        __syncwarp();
        const double *rec = buf + (size_t)st * F;
        // x+ = A x + B u : lane (row, half) sums 8 of the 16 columns
        double acc0 = 0.0, acc1 = 0.0;
        if (row < n) {
            SM_UNROLL
            for (int j = 0; j < 8; j += 2) {
                const int c = 8 * half + j;
                if (c < w) acc0 = fma(rec[row + n * c], zc[c], acc0);
                if (c + 1 < w) acc1 = fma(rec[row + n * (c + 1)], zc[c + 1], acc1);
            }
        }
        double xs = acc0 + acc1;
        xs += __shfl_xor_sync(0xffffffffu, xs, 16);
        if (lane < n) zn[lane] = xs;
        __syncwarp();
    }
    if (lane < n) __stcs(zb + (int64_t)steps * w + lane, zs[(steps & 1) * 16 + lane]);
}

}  // namespace rdmma
