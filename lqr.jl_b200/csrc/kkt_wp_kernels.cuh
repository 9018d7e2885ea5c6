// kkt_wp_kernels.cuh — constrained KKT solve for the "quadrotor-sized" class (n = 8 or 12, m <= 4): ONE WARP per
// instance, every n x n block in mma.sync.m8n8k4.f64 accumulator (C-fragment) registers, no matrix ever staged
// in shared memory.
//
// Replaces _solve!(::CholeskySolver) : src/cholesky_solver.jl:166-182 for the stage pattern of the reference's own
// fixtures (test/problems.jl:58-88: initial condition + dynamics + goal, p = [n, 0, ..., 0, n], D2 = [-I 0]; any of the
// three BlockCholesky modes of the cost Hessian — the dense one too: H^-1 is a z-space inverse here):
//   calculate_shur_factors!  src/jacobian_blocks.jl:220-286   S = D H^-1 D', h = D H^-1 g - d
//   cholesky!(chol, shur)    src/cholesky_solve.jl:28-67
//   forward_substitution!    :93-117        backward_substitution! :119-143   (Lambda = -S^-1 h)
//   calculate_primals!       src/cholesky_solver.jl:185-236   res = D'Lambda + g,  dz = -H^-1 res
// Same block-LDL' restatement as kkt_hw_kernels.cuh / kkt_cta_kernels.cuh (explicit SPD inverses so that all n^3
// work is products):  with F = [A B] (or C_N at the last knot), Hi = H_k^-1, T = F Hi,
//   G = T F',   Sigma = Cp + Hi_xx,   Si = Sigma^-1,   Z = T_x Si (the record, = -U'),   v = Si y,
//   Cp <- G - Z T_x' (symmetrised exactly),   dp <- (F hg - d) + T_x v,
// backward  x_{k-1} = v_k + Z_k' x_k,  Lambda = -x,  res_k,  dz_k = -Hi res_k  (Hi comes back from the record: the
// kernel is bound by its serial pivot chains, not by HBM; for the same reason H_{k+1} is inverted in lock step with
// Sigma_k in the forward sweep).
//
// Layout.  A 16 x 16 "physical" index space, tile 0 = x0..x7, tile 1 = [x8 u0 x9 u1 x10 u2 x11 u3] (the map of
// riccati_dmma_kernels.cuh): z-space matrices (H, Hi, F, T) use every slot, x-space matrices (Sigma, Si, Cp, G, Z:
// states or constraint rows) keep the odd slots of tile 1 as identity / zero padding, so a contraction over x is 3
// MMAs per output tile (12 = 3 x 4) and one over z is 4.  A tile lives in C-fragment layout: lane (g = lane >> 2,
// q = lane & 3) holds M[8 rt + g][8 ct + 2 q + e], e = 0, 1.  The identity that makes the chain work without any
// data movement:  C fragments of X as the A operand and C fragments of Y as the B operand of the same step give
// X Y'  (the contraction index of step (ct, e) is column 8 ct + 2 k + e of both) — so with Hi, Si symmetric,
// T = F Hi, G = T F', Z = T Si, Z T' are all "X Y'" products of register-resident operands.  SPD inverses: 2 x 2
// block elimination on the tiles (12 MMAs) around two 8 x 8 Gauss-Jordan inverses done with shuffles; transposes:
// two selection-matrix MMAs per tile.  Lane-level emulator of exactly this arithmetic: tools/emu/kkt_wp_emu.py.
#pragma once
#include "kkt_hw_kernels.cuh"

namespace kwp {
using rdmma::bulk_g2s;
using rdmma::fast_rcp;
using rdmma::mbar_expect_tx;
using rdmma::mbar_init;
using rdmma::mbar_wait;
using rdmma::mma884;

// knot records of the packed data (tile width 1; same row order as every KKT kernel, lqrb200.h):
//   first: H | g | D1 = [A B] | d | C_1 (n x w) | c_1      middle: H | g | D1 | d      last: Q | g | C_N (n x n) | c_N
template <int n, int m, int HESS = LQRB_HESS_BLOCKDIAG>
struct Lay {
    static constexpr int w = n + m;
    // H part: DIAG: w entries | BLOCKDIAG: tri(n) + tri(m) | DENSE: tri(w), upper packed over z = [x; u] (lqrb200.h);
    // the last knot has no controls: n | tri(n) | tri(n)
    static constexpr int HQ = HESS == LQRB_HESS_DIAG ? n : tri(n);
    static constexpr int HR = HESS == LQRB_HESS_DIAG ? m : (HESS == LQRB_HESS_BLOCKDIAG ? tri(m) : tri(w) - tri(n));
    static constexpr int oQ = 0, oR = HQ, og = oR + HR, oD1 = og + w, od = oD1 + n * w, CORE = od + n;
    static constexpr int oC0 = CORE, FIRST = CORE + n * w + n, MID = CORE;
    static constexpr int oCl = HQ + n, LAST = oCl + n * n + n;
    // records may have odd lengths and start on odd doubles: the bulk copies (16-byte pieces) start at the even double
    // before the record and end at the even double after it, see issue() in the kernel
    // ps = stage-constraint rows of every interior knot (C (ps x w) | c (ps) follow d in its record), 0 <= ps <= PSMAX
    static constexpr int PSMAX = 4;
    __host__ __device__ static constexpr int mid(int ps) { return MID + ps * w + ps; }
    __host__ __device__ static constexpr int64_t data_rows(int N, int ps = 0) { return FIRST + (int64_t)(N - 2) * mid(ps) + LAST; }
    __host__ __device__ static constexpr int64_t knot_off(int k, int ps = 0) { return k == 0 ? 0 : FIRST + (int64_t)(k - 1) * mid(ps); }
    __host__ __device__ static constexpr int64_t mult_rows(int N, int ps = 0) { return 2 * n + (int64_t)(N - 1) * n + (int64_t)(N - 2) * ps; }
    __host__ __device__ static constexpr int64_t z_rows(int N) { return (int64_t)N * n + (int64_t)(N - 1) * m; }
    // largest knot record, + 2 doubles: a record that starts on an odd double is copied from the even one before it
    // (rounded up to an even count: every stage of the ring is a 16-byte aligned bulk-copy destination)
    static constexpr int BUF = ((FIRST > MID + PSMAX * (w + 1) ? FIRST : MID + PSMAX * (w + 1)) + 3) & ~1;
};

struct Tile16 {
    double v[2][2][2];  // [row tile][column tile][e]
};

template <int n, int m>
struct Phys {
    static_assert(n == 8 || n == 12, "physical map is written for n = 8, 12");
    static_assert(m >= 1 && m <= 4, "one control per odd slot of tile 1");
    // physical position -> index into z = [x; u]; -1 = unused
    __host__ __device__ static constexpr int zmap(int pos) {
        if (pos < 8) return pos;
        const int j = pos - 8;
        if ((j & 1) == 0) return (8 + j / 2 < n) ? 8 + j / 2 : -1;
        return ((j - 1) / 2 < m) ? n + (j - 1) / 2 : -1;
    }
    __host__ __device__ static constexpr int xmap(int pos) {
        const int z = zmap(pos);
        return (z >= 0 && z < n) ? z : -1;
    }
};

// record of one knot in the scratch array: the real entries of Z in fragment order + v (16 physical slots)
//   [0,32) tile00 e0 | [32,64) tile00 e1 | [64,96) tile01 e0 | [96,112) tile10 e0 (even g) | [112,128) tile10 e1
//   | [128,144) tile11 e0 (even g) | v
// interior knots with ps stage rows add: sd_j (16) | E'_j (16) for j < ps | Bi (16) | c' (4)
// then Hi = H_k^-1 (z space, tiles 00 | 01 | 11 in fragment order, 6 x 32 doubles): the backward sweep reads it back
// instead of inverting H_k a second time (the serial pivot chains, not HBM, bound this kernel);
// interior knots with ps stage rows add: sd_j (16) | E'_j (16) for j < ps | Bi (16) | c' (4)
template <int n>
struct RecW {
    static constexpr int ZR = n > 8 ? 144 : 64, HIO = ZR + 16, REC = HIO + 192;
    __host__ __device__ static constexpr int rec(int ps) { return REC + (ps > 0 ? 32 * ps + 20 : 0); }
};

// X Y' accumulated into out: KS contraction steps (4: z space, 3: x space); UPPER: tile (1,0) is not formed
template <int KS, bool UPPER>
__device__ __forceinline__ void product(Tile16 &out, const Tile16 &X, const Tile16 &Y, double sign) {
    SM_UNROLL
    for (int rt = 0; rt < 2; ++rt)
        SM_UNROLL
        for (int ct = 0; ct < 2; ++ct) {
            if (UPPER && rt == 1 && ct == 0) continue;
            SM_UNROLL
            for (int s = 0; s < KS; ++s) {
                const int kt = s >> 1, e = s & 1;
                mma884(out.v[rt][ct][0], out.v[rt][ct][1], sign * X.v[rt][kt][e], Y.v[ct][kt][e]);
            }
        }
}

// 8 x 8 tiles: d += sign * X Y'
__device__ __forceinline__ void prod8(double (&d)[2], const double (&X)[2], const double (&Y)[2], double sign) {
    mma884(d[0], d[1], sign * X[0], Y[0]);
    mma884(d[0], d[1], sign * X[1], Y[1]);
}

// d += scale * X'  (a C fragment read as a B fragment is the transpose; two selection-matrix MMAs)
__device__ __forceinline__ void transpose8(double (&d)[2], const double (&X)[2], double scale, int g, int q) {
    mma884(d[0], d[1], g == 2 * q ? scale : 0.0, X[0]);
    mma884(d[0], d[1], g == 2 * q + 1 ? scale : 0.0, X[1]);
}

// In-place Gauss-Jordan inverse of an SPD 8 x 8 tile in C-fragment layout (no pivoting; the pivots are the squared
// Cholesky pivots, so the sign test is potrf's).  SKIP_ODD: x-space tile 1 — only its first NEVEN even slots are real,
// the rest is identity padding.  Returns the
// 1-based position of the first non-positive pivot or 0; lo / hi collect the pivots' high words (conditioning
// estimate, integer pipe).
template <bool SKIP_ODD, int NEVEN>
__device__ __forceinline__ int gj8c(double (&a)[2], int g, int q, int &lo, int &hi) {
    int bad = 0;
    SM_UNROLL
    for (int kk = 0; kk < 8; ++kk) {
        if (SKIP_ODD && ((kk & 1) || (kk >> 1) >= NEVEN)) continue;  // identity padding: nothing to eliminate
        const double prow0 = __shfl_sync(0xffffffffu, a[0], 4 * kk + q);
        const double prow1 = __shfl_sync(0xffffffffu, a[1], 4 * kk + q);
        const double src = (kk & 1) ? a[1] : a[0];
        const double pcol = __shfl_sync(0xffffffffu, src, 4 * g + (kk >> 1));
        const double piv = __shfl_sync(0xffffffffu, src, 4 * kk + (kk >> 1));
        if (!(piv > 0.0) && bad == 0) bad = kk + 1;
        lo = min(lo, __double2hiint(piv));
        hi = max(hi, __double2hiint(piv));
        const double p = fast_rcp(piv);
        const double f = pcol * p;
        const bool rowk = g == kk, c0 = 2 * q == kk, c1 = 2 * q + 1 == kk;
        const double u0 = fma(-f, prow0, a[0]), u1 = fma(-f, prow1, a[1]);
        a[0] = rowk ? (c0 ? p : prow0 * p) : (c0 ? -f : u0);
        a[1] = rowk ? (c1 ? p : prow1 * p) : (c1 ? -f : u1);
    }
    return bad;
}

// one pivot step of gj8c (kk is a compile-time constant after unrolling)
__device__ __forceinline__ void gj_step(double (&a)[2], int kk, int g, int q, int &lo, int &hi, int &bad) {
    const double prow0 = __shfl_sync(0xffffffffu, a[0], 4 * kk + q);
    const double prow1 = __shfl_sync(0xffffffffu, a[1], 4 * kk + q);
    const double src = (kk & 1) ? a[1] : a[0];
    const double pcol = __shfl_sync(0xffffffffu, src, 4 * g + (kk >> 1));
    const double piv = __shfl_sync(0xffffffffu, src, 4 * kk + (kk >> 1));
    if (!(piv > 0.0) && bad == 0) bad = kk + 1;
    lo = min(lo, __double2hiint(piv));
    hi = max(hi, __double2hiint(piv));
    const double p = fast_rcp(piv);
    const double f = pcol * p;
    const bool rowk = g == kk, c0 = 2 * q == kk, c1 = 2 * q + 1 == kk;
    const double u0 = fma(-f, prow0, a[0]), u1 = fma(-f, prow1, a[1]);
    a[0] = rowk ? (c0 ? p : prow0 * p) : (c0 ? -f : u0);
    a[1] = rowk ? (c1 ? p : prow1 * p) : (c1 ? -f : u1);
}

// Two independent 8 x 8 inversions pivot by pivot in lock step: the serial chain shuffle -> reciprocal -> FMA of one
// tile fills the latency of the other (the kernel is bound by these chains, not by issue slots).  Tile a is full
// (z space), tile b is an x-space tile 1 with NEVEN real even slots when SKIPB.
template <bool SKIPB, int NEVEN>
__device__ __forceinline__ void gj8c_pair(double (&a)[2], double (&b)[2], int g, int q, int &loa, int &hia, int &bada,
                                          int &lob, int &hib, int &badb) {
    SM_UNROLL
    for (int kk = 0; kk < 8; ++kk) {
        gj_step(a, kk, g, q, loa, hia, bada);
        if (!(SKIPB && ((kk & 1) || (kk >> 1) >= NEVEN))) gj_step(b, kk, g, q, lob, hib, badb);
    }
}

// inv16 of A (z space) and of B (x space) interleaved step by step; returns the bad-pivot positions (1-based) or 0
template <int NX1>
__device__ __forceinline__ void inv16_pair(Tile16 &A, Tile16 &B, int g, int q, int &loa, int &hia, int &bada, int &lob,
                                           int &hib, int &badb) {
    int a0 = 0, b0 = 0, a1 = 0, b1 = 0;
    gj8c_pair<false, 4>(A.v[0][0], B.v[0][0], g, q, loa, hia, a0, lob, hib, b0);
    double Ta[2] = {0.0, 0.0}, Tta[2] = {0.0, 0.0}, Tb[2] = {0.0, 0.0}, Ttb[2] = {0.0, 0.0};
    prod8(Ta, A.v[0][0], A.v[1][0], 1.0);
    prod8(Tb, B.v[0][0], B.v[1][0], 1.0);
    prod8(Tta, A.v[1][0], A.v[0][0], 1.0);
    prod8(Ttb, B.v[1][0], B.v[0][0], 1.0);
    prod8(A.v[1][1], A.v[1][0], Tta, -1.0);
    prod8(B.v[1][1], B.v[1][0], Ttb, -1.0);
    gj8c_pair<true, NX1>(A.v[1][1], B.v[1][1], g, q, loa, hia, a1, lob, hib, b1);
    double Na01[2] = {0.0, 0.0}, Na10[2] = {0.0, 0.0}, Nb01[2] = {0.0, 0.0}, Nb10[2] = {0.0, 0.0};
    prod8(Na01, Ta, A.v[1][1], -1.0);
    prod8(Nb01, Tb, B.v[1][1], -1.0);
    prod8(Na10, A.v[1][1], Ta, -1.0);
    prod8(Nb10, B.v[1][1], Tb, -1.0);
    prod8(A.v[0][0], Na01, Ta, -1.0);
    prod8(B.v[0][0], Nb01, Tb, -1.0);
    A.v[0][1][0] = Na01[0];
    A.v[0][1][1] = Na01[1];
    A.v[1][0][0] = Na10[0];
    A.v[1][0][1] = Na10[1];
    B.v[0][1][0] = Nb01[0];
    B.v[0][1][1] = Nb01[1];
    B.v[1][0][0] = Nb10[0];
    B.v[1][0][1] = Nb10[1];
    bada = a0 != 0 ? a0 : (a1 != 0 ? 8 + a1 : 0);
    badb = b0 != 0 ? b0 : (b1 != 0 ? 8 + b1 : 0);
}

// Inverse of a symmetric positive definite 16 x 16 physical matrix (identity on its pad slots), in place, by 2 x 2
// block elimination on the tiles: 12 MMAs + two 8 x 8 Gauss-Jordan inverses.  Returns the physical position
// (1-based) of the first non-positive pivot or 0.
template <bool XSPACE, int NX1>
__device__ __forceinline__ int inv16(Tile16 &M, int g, int q, int &lo, int &hi) {
    const int bad0 = gj8c<false, 4>(M.v[0][0], g, q, lo, hi);  // I00
    double T1[2] = {0.0, 0.0}, T1t[2] = {0.0, 0.0};
    prod8(T1, M.v[0][0], M.v[1][0], 1.0);   // I00 M01      (M10 = M01')
    prod8(T1t, M.v[1][0], M.v[0][0], 1.0);  // M10 I00 = T1'
    prod8(M.v[1][1], M.v[1][0], T1t, -1.0);  // S = M11 - M10 I00 M01
    const int bad1 = gj8c<XSPACE, NX1>(M.v[1][1], g, q, lo, hi);  // N11 = S^-1
    double N01[2] = {0.0, 0.0}, N10[2] = {0.0, 0.0};
    prod8(N01, T1, M.v[1][1], -1.0);  // -T1 N11
    prod8(N10, M.v[1][1], T1, -1.0);  // -N11 T1'
    prod8(M.v[0][0], N01, T1, -1.0);  // N00 = I00 + T1 N11 T1'
    M.v[0][1][0] = N01[0];
    M.v[0][1][1] = N01[1];
    M.v[1][0][0] = N10[0];
    M.v[1][0][1] = N10[1];
    return bad0 != 0 ? bad0 : (bad1 != 0 ? 8 + bad1 : 0);
}

// out[rt] = sum_c M[8 rt + g][c] x[c]  (x: 16 physical slots in shared memory); every lane of a quad gets the sum
__device__ __forceinline__ void matvec_row(double (&out)[2], const Tile16 &M, const double *x, int q) {
    const double2 x0 = *reinterpret_cast<const double2 *>(x + 2 * q);
    const double2 x1 = *reinterpret_cast<const double2 *>(x + 8 + 2 * q);
    SM_UNROLL
    for (int rt = 0; rt < 2; ++rt) {
        double s = M.v[rt][0][0] * x0.x;
        s = fma(M.v[rt][0][1], x0.y, s);
        s = fma(M.v[rt][1][0], x1.x, s);
        s = fma(M.v[rt][1][1], x1.y, s);
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        out[rt] = s;
    }
}

// the row sums of matvec_row (row 8 rt + g, held by the quad g) -> lane p < 16 gets the value of physical slot p
__device__ __forceinline__ double rows_to_slot(const double (&r)[2], int lane) {
    const double a = __shfl_sync(0xffffffffu, r[0], 4 * (lane & 7));
    const double b = __shfl_sync(0xffffffffu, r[1], 4 * (lane & 7));
    return (lane & 8) ? b : a;
}
// the column sums of matvec_col (column 8 ct + 2 q + e, held by every lane with that q) -> lane p < 16 gets slot p
__device__ __forceinline__ double cols_to_slot(const double (&c)[2][2], int lane) {
    const int p = lane & 15, pq = (p & 7) >> 1;
    const double s00 = __shfl_sync(0xffffffffu, c[0][0], pq), s01 = __shfl_sync(0xffffffffu, c[0][1], pq);
    const double s10 = __shfl_sync(0xffffffffu, c[1][0], pq), s11 = __shfl_sync(0xffffffffu, c[1][1], pq);
    return p < 8 ? ((p & 1) ? s01 : s00) : ((p & 1) ? s11 : s10);
}

// out[ct][e] = sum_r M[r][8 ct + 2 q + e] x[r]  (M' x); every lane gets the sums of its own columns
__device__ __forceinline__ void matvec_col(double (&out)[2][2], const Tile16 &M, const double *x, int g) {
    const double xa = x[g], xb = x[8 + g];
    SM_UNROLL
    for (int ct = 0; ct < 2; ++ct)
        SM_UNROLL
        for (int e = 0; e < 2; ++e) {
            double s = fma(M.v[1][ct][e], xb, M.v[0][ct][e] * xa);
            s += __shfl_xor_sync(0xffffffffu, s, 4);
            s += __shfl_xor_sync(0xffffffffu, s, 8);
            s += __shfl_xor_sync(0xffffffffu, s, 16);
            out[ct][e] = s;
        }
}

// per-warp shared memory in doubles (the launcher sizes the dynamic allocation with it)
template <int n, int m, int HESS>
__host__ __device__ constexpr int warp_smem_doubles() {
    return 2 * Lay<n, m, HESS>::BUF + 496 + 4;
}

template <int n, int m, int HESS, int WARPS, int MINB>
__global__ void __launch_bounds__(WARPS * 32, MINB)
    kkt_wp_kernel(const double *__restrict__ data, double *__restrict__ recs, double *__restrict__ dz,
                  double *__restrict__ mult, double *__restrict__ res, int32_t *__restrict__ info,
                  int32_t *__restrict__ cinfo, int N, int64_t batch, int soc, int ps,
                  const int32_t *__restrict__ pk, const int64_t *__restrict__ koff, const int64_t *__restrict__ moff,
                  int free_final) {
    // ps = stage rows of every interior knot; or, with pk / koff / moff (stage rows per knot, offsets of the knot records
    // and of the multiplier groups [mu_k; lam_k], N + 1 entries each), ps = the largest interior count
    using L = Lay<n, m, HESS>;
    using PH = Phys<n, m>;
    using RW = RecW<n>;
    constexpr int w = L::w;
    constexpr int BUF = L::BUF;
    constexpr int STG = 2;
    // per-warp shared memory (doubles): STG knot buffers | vectors (16 slots each) | stage-constraint work | STG mbarriers
    constexpr int VG = 0, VHG = 16, VY = 32, VV = 48, VX = 64, VXP = 80, VR = 96, VD = 112, NVEC = 128;
    // stage rows j < 4: cz_j (C_j in z slots) | tc_j = Hi C_j' | E_j then E'_j | sd_j | W_j ; B (16) | Bi (16) | ct, c', bc, xi (4 each)
    constexpr int SCZ = NVEC, STC = SCZ + 64, SE = STC + 64, SSD = SE + 64, SW = SSD + 64, SB = SW + 64, SBI = SB + 16,
                  SCT = SBI + 16, SCP = SCT + 4, SBC = SCP + 4, SXI = SBC + 4, NWORK = SXI + 4;
    constexpr int WSM = STG * BUF + NWORK + 2 * STG;
    static_assert(WSM == warp_smem_doubles<n, m, HESS>(), "launcher and kernel disagree on the shared-memory size");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
    const int64_t inst = (int64_t)blockIdx.x * WARPS + warp;
    if (inst >= batch) return;  // whole warp leaves; no CTA-wide barrier is used below
    double *wsm = reinterpret_cast<double *>(smem_raw) + (size_t)warp * WSM;
    double *buf = wsm, *vec = wsm + STG * BUF;
    uint64_t *bars = reinterpret_cast<uint64_t *>(vec + NWORK);
    if (lane == 0) {
        SM_UNROLL
        for (int s = 0; s < STG; ++s) mbar_init(bars + s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();

    const int64_t mrows = moff ? moff[N] : L::mult_rows(N, ps);
    const int64_t doff = inst * (koff ? koff[N] : L::data_rows(N, ps));  // in doubles from `data` (16-byte aligned)
    const int recw = RW::rec(ps);
    double *rb = recs + inst * (int64_t)N * recw;
    double *zb = dz + inst * L::z_rows(N);
    double *mb = mult + inst * mrows;
    double *resb = res ? res + inst * L::z_rows(N) : nullptr;
    const int lstride = n + ps;  // lam_j sits at n + j (n + ps) of the multiplier vector, mu of knot j + 1 right after it

    auto knot_ps = [&](int k) { return (k == 0 || k == N - 1) ? 0 : (pk ? (int)pk[k] : ps); };
    auto knot_off = [&](int k) { return koff ? koff[k] : L::knot_off(k, ps); };
    auto knot_len = [&](int k) { return k == 0 ? L::FIRST : (k == N - 1 ? L::LAST : L::mid(knot_ps(k))); };
    // The whole record of knot k -> buffer st.  Bulk copies move 16-byte pieces: with an odd number of stage rows a
    // record can start on an odd double, so the copy starts at the even double before it (shift 0 or 1) and may
    // carry one double more at the end (the packed array is a whole number of 32-instance tiles: it stays inside).
    auto knot_shift = [&](int k) { return (int)((doff + knot_off(k)) & 1); };
    auto issue = [&](int k, int st) {
        if (lane == 0) {
            const int64_t g0 = doff + knot_off(k);
            const int sh = (int)(g0 & 1);
            const uint32_t bytes = (uint32_t)((knot_len(k) + sh + 1) & ~1) * 8u;
            mbar_expect_tx(bars + st, bytes);
            bulk_g2s(buf + st * BUF, data + (g0 - sh), bytes, bars + st);
        }
    };

    // ---- per-lane physical indices of the 8 tile entries: row position a, column position b
    // z / x indices are recomputed from (g, q) where needed (integer work, off the FP64 pipe)
    auto zrow = [&](int rt) { return rt == 0 ? g : ((g & 1) ? ((g >> 1) < m ? n + (g >> 1) : -1) : (8 + (g >> 1) < n ? 8 + (g >> 1) : -1)); };
    auto zcol = [&](int ct, int e) {
        if (ct == 0) return 2 * q + e;
        return e == 0 ? (8 + q < n ? 8 + q : -1) : (q < m ? n + q : -1);
    };
    auto xrow = [&](int rt) { const int z = zrow(rt); return z < n ? z : -1; };
    auto xcol = [&](int ct, int e) { const int z = zcol(ct, e); return z < n ? z : -1; };
    auto is_diag = [&](int rt, int ct, int e) { return rt == ct && g == 2 * q + e; };

    // H_k (z space) from the knot record; unused slots (and the control slots of the last knot) carry the identity
    auto load_H = [&](Tile16 &H, const double *kp, bool last) {
        const int wk = last ? n : w;
        SM_UNROLL
        for (int rt = 0; rt < 2; ++rt)
            SM_UNROLL
            for (int ct = 0; ct < 2; ++ct)
                SM_UNROLL
                for (int e = 0; e < 2; ++e) {
                    const int za = zrow(rt), zb_ = zcol(ct, e);
                    double v = is_diag(rt, ct, e) ? 1.0 : 0.0;
                    if (!soc && za >= 0 && zb_ >= 0 && za < wk && zb_ < wk) {
                        if (HESS == LQRB_HESS_DENSE)  // whole-matrix mode: cross terms Hux are part of H (src/block_cholesky.jl:55-66)
                            v = kp[sym_idx(za, zb_)];
                        else if (za < n && zb_ < n)
                            v = HESS == LQRB_HESS_DIAG ? (za == zb_ ? kp[L::oQ + za] : 0.0) : kp[L::oQ + sym_idx(za, zb_)];
                        else if (za >= n && zb_ >= n)
                            v = HESS == LQRB_HESS_DIAG ? (za == zb_ ? kp[L::oR + za - n] : 0.0) : kp[L::oR + sym_idx(za - n, zb_ - n)];
                        else
                            v = 0.0;
                    }
                    H.v[rt][ct][e] = v;
                }
    };
    // rows x (constraint rows), columns z: a column-major (n x cols) block at kp + off
    auto load_rows = [&](Tile16 &F, const double *blk, int cols) {
        SM_UNROLL
        for (int rt = 0; rt < 2; ++rt)
            SM_UNROLL
            for (int ct = 0; ct < 2; ++ct)
                SM_UNROLL
                for (int e = 0; e < 2; ++e) {
                    const int r = xrow(rt), z = zcol(ct, e);
                    F.v[rt][ct][e] = (r >= 0 && z >= 0 && z < cols) ? blk[r + n * z] : 0.0;
                }
    };
    // x-space restriction of a z-space symmetric matrix: non-state slots -> identity padding
    auto state_part = [&](const Tile16 &M, int rt, int ct, int e) {
        return (xrow(rt) >= 0 && xcol(ct, e) >= 0) ? M.v[rt][ct][e] : (is_diag(rt, ct, e) ? 1.0 : 0.0);
    };
    auto pad_identity = [&](Tile16 &M) {  // x-space matrix: force the pad slots to the identity
        SM_UNROLL
        for (int rt = 0; rt < 2; ++rt)
            SM_UNROLL
            for (int ct = 0; ct < 2; ++ct)
                SM_UNROLL
                for (int e = 0; e < 2; ++e)
                    if (!(xrow(rt) >= 0 && xcol(ct, e) >= 0)) M.v[rt][ct][e] = is_diag(rt, ct, e) ? 1.0 : 0.0;
    };
    // vectors: lane p < 16 owns physical slot p
    const int zl = lane < 16 ? PH::zmap(lane & 15) : -1;  // z index of this lane's slot
    const int zslot = lane < 8 ? lane : (lane < 16 ? (((lane - 8) & 1) ? ((lane - 9) / 2 < m ? n + (lane - 9) / 2 : -1)
                                                                        : (8 + (lane - 8) / 2 < n ? 8 + (lane - 8) / 2 : -1))
                                                   : -1);
    (void)zl;
    const int xslot = (zslot >= 0 && zslot < n) ? zslot : -1;
    // store the per-row result of matvec_row into a vector (lanes q == 0 own rows 8 rt + g)
    auto put_rows = [&](double *dst, const double (&r)[2]) {
        if (q == 0) {
            dst[g] = r[0];
            dst[8 + g] = r[1];
        }
    };

    issue(0, 0);
    if (N > 1) issue(1, 1);

    int st_all = 0, hcode = 0, lo = 0x7fffffff, hi = 0, spread = 0, hlo = 0x7fffffff, hhi = 0;
    Tile16 Cp;
    SM_UNROLL
    for (int rt = 0; rt < 2; ++rt)
        SM_UNROLL
        for (int ct = 0; ct < 2; ++ct) Cp.v[rt][ct][0] = Cp.v[rt][ct][1] = 0.0;
    if (lane < 16) vec[VD + lane] = 0.0;  // dp
    __syncwarp();
    // H_0^-1; from then on H_{k+1} is inverted in lock step with Sigma_k (they are independent: two serial pivot
    // chains in flight instead of one)
    Tile16 Hnext;
    {
        mbar_wait(bars, 0);
        load_H(Hnext, buf + knot_shift(0), N == 1);
        const int bad = inv16<false, 4>(Hnext, g, q, hlo, hhi);
        if (bad != 0) hcode = 1000 + PH::zmap(bad - 1) + 1;
    }

    // ---------------- forward sweep: k = 0 .. N-1
    for (int k = 0; k < N; ++k) {
        const bool first = k == 0, last = k == N - 1;
        const int st = k & 1;
        mbar_wait(bars + st, (k >> 1) & 1);
        const double *kp = buf + st * BUF + knot_shift(k);
        const int wk = last ? n : w;
        const int psk = knot_ps(k);  // stage rows of this knot (the end knots have their own blocks)
        // g (z slots) -> vec; d (x slots)
        double dv = 0.0;
        if (lane < 16) {
            vec[VG + lane] = (!soc && zslot >= 0 && zslot < wk) ? kp[(last ? L::HQ : L::og) + zslot] : 0.0;
            if (xslot >= 0) dv = last ? kp[L::oCl + n * n + xslot] : kp[L::od + xslot];
        }
        for (int j = 0; j < psk; ++j)  // C_j (row j of the ps x w block, column-major) in z slots
            if (lane < 16) vec[SCZ + 16 * j + lane] = (zslot >= 0 && zslot < w) ? kp[L::CORE + j + psk * zslot] : 0.0;
        Tile16 Hi = Hnext, F;  // H_k^-1 was formed during the previous knot
        load_rows(F, last ? kp + L::oCl : kp + L::oD1, wk);
        {   // Hi -> record (the backward sweep reads it back instead of inverting H_k again)
            double *rh = rb + (int64_t)k * recw + RW::HIO;
            __stcs(rh + lane, Hi.v[0][0][0]);
            __stcs(rh + 32 + lane, Hi.v[0][0][1]);
            __stcs(rh + 64 + lane, Hi.v[0][1][0]);
            __stcs(rh + 96 + lane, Hi.v[0][1][1]);
            __stcs(rh + 128 + lane, Hi.v[1][1][0]);
            __stcs(rh + 160 + lane, Hi.v[1][1][1]);
        }
        __syncwarp();
        double r2[2];
        matvec_row(r2, Hi, vec + VG, q);
        put_rows(vec + VHG, r2);  // hg = Hi g
        for (int j = 0; j < psk; ++j) {  // tc_j = Hi C_j'
            matvec_row(r2, Hi, vec + SCZ + 16 * j, q);
            put_rows(vec + STC + 16 * j, r2);
        }
        Tile16 TF, Gm;
        SM_UNROLL
        for (int rt = 0; rt < 2; ++rt)
            SM_UNROLL
            for (int ct = 0; ct < 2; ++ct) TF.v[rt][ct][0] = TF.v[rt][ct][1] = Gm.v[rt][ct][0] = Gm.v[rt][ct][1] = 0.0;
        product<4, false>(TF, F, Hi, 1.0);  // T = F Hi
        product<4, true>(Gm, TF, F, 1.0);   // G = F Hi F' (upper tiles)
        __syncwarp();                       // hg is published
        matvec_row(r2, F, vec + VHG, q);    // rho = F hg - d
        double rho = 0.0;  // lanes < 16: slot value
        {
            const double rr = rows_to_slot(r2, lane);
            if (lane < 16 && xslot >= 0) rho = rr - dv;
        }
        if (psk > 0) {
            // stage rows as vectors (shur! / copy_shur! for the ps rows, src/jacobian_blocks.jl:231-286):
            //   E_j = F tc_j (x slots),  B = C Hi C',  ct = C hg - c
            for (int j = 0; j < psk; ++j) {
                matvec_row(r2, F, vec + STC + 16 * j, q);
                const double rr = rows_to_slot(r2, lane);
                if (lane < 16) vec[SE + 16 * j + lane] = xslot >= 0 ? rr : 0.0;
            }
            if (lane < psk * psk) {
                const int j = lane / psk, jp = lane % psk;
                double sB = 0.0;
                for (int t = 0; t < 16; ++t) sB = fma(vec[SCZ + 16 * j + t], vec[STC + 16 * jp + t], sB);
                vec[SB + 4 * j + jp] = sB;
            } else if (lane >= 16 && lane < 16 + psk) {
                const int j = lane - 16;
                double sc = -kp[L::CORE + psk * w + j];
                for (int t = 0; t < 16; ++t) sc = fma(vec[SCZ + 16 * j + t], vec[VHG + t], sc);
                vec[SCT + j] = sc;
            }
        }
        Tile16 Sig, T;
        if (first) {
            // first knot, general C_1 (n x w): Sigma = C Hi C', T = -(F Hi C'), y = C hg - c
            Tile16 Cc, TC;
            load_rows(Cc, kp + L::oC0, w);
            SM_UNROLL
            for (int rt = 0; rt < 2; ++rt)
                SM_UNROLL
                for (int ct = 0; ct < 2; ++ct)
                    TC.v[rt][ct][0] = TC.v[rt][ct][1] = Sig.v[rt][ct][0] = Sig.v[rt][ct][1] = T.v[rt][ct][0] = T.v[rt][ct][1] = 0.0;
            product<4, false>(TC, Cc, Hi, 1.0);
            product<4, false>(Sig, TC, Cc, 1.0);
            pad_identity(Sig);
            product<4, false>(T, TF, Cc, -1.0);
            matvec_row(r2, Cc, vec + VHG, q);
            const double rr = rows_to_slot(r2, lane);
            if (lane < 16) vec[VY + lane] = xslot >= 0 ? rr - kp[L::oC0 + n * w + xslot] : 0.0;
        } else {
            SM_UNROLL
            for (int rt = 0; rt < 2; ++rt)
                SM_UNROLL
                for (int ct = 0; ct < 2; ++ct)
                    SM_UNROLL
                    for (int e = 0; e < 2; ++e) Sig.v[rt][ct][e] = Cp.v[rt][ct][e] + state_part(Hi, rt, ct, e);
            T = TF;
            if (lane < 16) vec[VY + lane] = xslot >= 0 ? vec[VD + lane] - vec[VHG + lane] : 0.0;  // y = dp - hg_x
        }
        __syncwarp();  // every read of the knot buffer is done; y is published
        if (k + 2 < N) issue(k + 2, st);
        {
            lo = 0x7fffffff;
            hi = 0;
            int bad = 0, badh = 0;
            if (!last) {
                // H_{k+1} sits in the other buffer (copied two knots ahead); waiting again on a completed phase is free
                mbar_wait(bars + (st ^ 1), ((k + 1) >> 1) & 1);
                load_H(Hnext, buf + (st ^ 1) * BUF + knot_shift(k + 1), k + 1 == N - 1);
                inv16_pair<n - 8>(Hnext, Sig, g, q, hlo, hhi, badh, lo, hi, bad);
            } else {
                bad = inv16<true, n - 8>(Sig, g, q, lo, hi);
            }
            if (bad != 0 && st_all == 0) {
                const int x = PH::xmap(bad - 1);
                st_all = first ? 1000 + 100 + x + 1 : k * 1000 + 200 + x + 1;
            }
            if (badh != 0 && hcode == 0) hcode = (k + 2) * 1000 + PH::zmap(badh - 1) + 1;
            if (lo > 0 && hi >= lo) spread = max(spread, hi - lo);
        }
        Tile16 Zm;
        SM_UNROLL
        for (int rt = 0; rt < 2; ++rt)
            SM_UNROLL
            for (int ct = 0; ct < 2; ++ct) Zm.v[rt][ct][0] = Zm.v[rt][ct][1] = 0.0;
        product<3, false>(Zm, T, Sig, 1.0);  // Z = T_x Si
        matvec_row(r2, Sig, vec + VY, q);    // v = Si y
        {
            const double rr = rows_to_slot(r2, lane);
            if (lane < 16) vec[VV + lane] = xslot >= 0 ? rr : 0.0;
        }
        product<3, true>(Gm, Zm, T, -1.0);  // X = G - Z T_x' (upper tiles)
        // Cp = symmetrised X (an antisymmetric rounding residue is amplified by |A|^2 per knot)
        Cp.v[0][0][0] = 0.5 * Gm.v[0][0][0];
        Cp.v[0][0][1] = 0.5 * Gm.v[0][0][1];
        transpose8(Cp.v[0][0], Gm.v[0][0], 0.5, g, q);
        Cp.v[1][1][0] = 0.5 * Gm.v[1][1][0];
        Cp.v[1][1][1] = 0.5 * Gm.v[1][1][1];
        transpose8(Cp.v[1][1], Gm.v[1][1], 0.5, g, q);
        Cp.v[0][1][0] = Gm.v[0][1][0];
        Cp.v[0][1][1] = Gm.v[0][1][1];
        Cp.v[1][0][0] = Cp.v[1][0][1] = 0.0;
        transpose8(Cp.v[1][0], Gm.v[0][1], 1.0, g, q);
        __syncwarp();  // v is published
        matvec_row(r2, T, vec + VV, q);  // dp' = rho + T_x v   (v is zero on the non-state slots)
        {
            const double rr = rows_to_slot(r2, lane);
            if (lane < 16) vec[VD + lane] = xslot >= 0 ? rho + rr : 0.0;
        }
        if (psk > 0) {
            // eliminate lam_{k-1}:  sd_j = Si D_j (D_j = -(tc_j)_x),  B' = B - D'Si D,  E'_j = E_j + T_x sd_j,
            // c'_j = ct_j - sd_j'y;   eliminate mu_k:  Bi = B'^-1,  Cp -= E'' Bi E',  dp -= E'' Bi c'
            __syncwarp();
            for (int j = 0; j < psk; ++j)
                if (lane < 16) vec[SW + 16 * j + lane] = xslot >= 0 ? -vec[STC + 16 * j + lane] : 0.0;  // D_j (W_j slot as scratch)
            __syncwarp();
            for (int j = 0; j < psk; ++j) {
                matvec_row(r2, Sig, vec + SW + 16 * j, q);
                const double rr = rows_to_slot(r2, lane);
                if (lane < 16) vec[SSD + 16 * j + lane] = xslot >= 0 ? rr : 0.0;
            }
            __syncwarp();
            for (int j = 0; j < psk; ++j) {
                matvec_row(r2, T, vec + SSD + 16 * j, q);
                const double rr = rows_to_slot(r2, lane);
                if (lane < 16) vec[SE + 16 * j + lane] += xslot >= 0 ? rr : 0.0;  // E'_j
            }
            if (lane < psk * psk) {
                const int j = lane / psk, jp = lane % psk;
                double sB = vec[SB + 4 * j + jp];
                for (int t = 0; t < 16; ++t) sB = fma(-vec[SW + 16 * j + t], vec[SSD + 16 * jp + t], sB);
                vec[SB + 4 * j + jp] = sB;  // B'
            } else if (lane >= 16 && lane < 16 + psk) {
                const int j = lane - 16;
                double sc = vec[SCT + j];
                for (int t = 0; t < 16; ++t) sc = fma(-vec[SSD + 16 * j + t], vec[VY + t], sc);
                vec[SCP + j] = sc;  // c'
            }
            __syncwarp();
            if (lane == 0) {  // Bi = B'^-1: Gauss-Jordan on at most 4 x 4, potrf sign test on the pivots
                double bm[4][4];
                for (int a = 0; a < 4; ++a)
                    for (int b = 0; b < 4; ++b) bm[a][b] = (a < psk && b < psk) ? vec[SB + 4 * a + b] : (a == b ? 1.0 : 0.0);
                int badp = 0;
                for (int kk = 0; kk < 4; ++kk) {
                    if (kk >= psk) break;
                    const double piv = bm[kk][kk];
                    if (!(piv > 0.0) && badp == 0) badp = kk + 1;
                    const double pinv = 1.0 / piv;
                    for (int b = 0; b < 4; ++b) bm[kk][b] = b == kk ? pinv : bm[kk][b] * pinv;
                    for (int a = 0; a < 4; ++a) {
                        if (a == kk) continue;
                        const double f = bm[a][kk];
                        for (int b = 0; b < 4; ++b) bm[a][b] = b == kk ? -f * pinv : fma(-f, bm[kk][b], bm[a][b]);
                    }
                }
                for (int a = 0; a < 4; ++a)
                    for (int b = 0; b < 4; ++b) vec[SBI + 4 * a + b] = bm[a][b];
                vec[SXI] = (double)badp;
            }
            __syncwarp();
            {
                const int badp = (int)vec[SXI];
                if (badp != 0 && st_all == 0) st_all = (k + 1) * 1000 + 100 + badp;
            }
            // W_j = sum_j' Bi[j][j'] E'_j' ;  bc = Bi c'
            for (int j = 0; j < psk; ++j)
                if (lane < 16) {
                    double sW = 0.0;
                    for (int jp = 0; jp < psk; ++jp) sW = fma(vec[SBI + 4 * j + jp], vec[SE + 16 * jp + lane], sW);
                    vec[SW + 16 * j + lane] = sW;
                }
            if (lane >= 16 && lane < 16 + psk) {
                const int j = lane - 16;
                double sb = 0.0;
                for (int jp = 0; jp < psk; ++jp) sb = fma(vec[SBI + 4 * j + jp], vec[SCP + jp], sb);
                vec[SBC + j] = sb;
            }
            __syncwarp();
            // Cp -= 1/2 (E'_j W_j' + W_j E'_j')  (products rounded separately: bitwise symmetric);  dp -= sum_j bc_j E'_j
            for (int j = 0; j < psk; ++j) {
                const double *E = vec + SE + 16 * j, *W = vec + SW + 16 * j;
                SM_UNROLL
                for (int rt = 0; rt < 2; ++rt)
                    SM_UNROLL
                    for (int ct = 0; ct < 2; ++ct)
                        SM_UNROLL
                        for (int e = 0; e < 2; ++e) {
                            const int r = 8 * rt + g, c = 8 * ct + 2 * q + e;
                            const double p1 = __dmul_rn(E[r], W[c]), p2 = __dmul_rn(W[r], E[c]);
                            Cp.v[rt][ct][e] = __dadd_rn(Cp.v[rt][ct][e], -0.5 * __dadd_rn(p1, p2));
                        }
                if (lane < 16) vec[VD + lane] -= vec[SBC + j] * E[lane];
            }
            // record: sd_j | E'_j | Bi | c'
            double *rs = rb + (int64_t)k * recw + RW::REC;
            for (int j = 0; j < psk; ++j)
                if (lane < 16) {
                    __stcs(rs + 32 * j + lane, vec[SSD + 16 * j + lane]);
                    __stcs(rs + 32 * j + 16 + lane, vec[SE + 16 * j + lane]);
                }
            if (lane < 16) __stcs(rs + 32 * psk + lane, vec[SBI + lane]);
            if (lane < 4) __stcs(rs + 32 * psk + 16 + lane, vec[SCP + lane]);
        }
        // record: the real entries of Z in fragment order, v
        {
            double *rk = rb + (int64_t)k * recw;
            __stcs(rk + lane, Zm.v[0][0][0]);
            __stcs(rk + 32 + lane, Zm.v[0][0][1]);
            if (n > 8) {
                __stcs(rk + 64 + lane, Zm.v[0][1][0]);
                if (!(g & 1)) {
                    const int hl = (g >> 1) * 4 + q;
                    __stcs(rk + 96 + hl, Zm.v[1][0][0]);
                    __stcs(rk + 112 + hl, Zm.v[1][0][1]);
                    __stcs(rk + 128 + hl, Zm.v[1][1][0]);
                }
            }
            if (lane < 16) __stcs(rk + RW::ZR + lane, vec[VV + lane]);
        }
        __syncwarp();
    }
    // ---------------- last block: mu_N' = Bl'^-1 y_mu   (Cp, dp hold Bl' and y_mu)
    if (free_final) {  // no goal rows (the last knot carried a zero block): mu_N = 0, nothing to invert
        if (lane < 16) {
            vec[VX + lane] = 0.0;
            if (xslot >= 0) __stcs(mb + mrows - n + xslot, 0.0);
        }
    } else {
        pad_identity(Cp);
        lo = 0x7fffffff;
        hi = 0;
        const int bad = inv16<true, n - 8>(Cp, g, q, lo, hi);
        if (bad != 0 && st_all == 0) st_all = N * 1000 + 100 + PH::xmap(bad - 1) + 1;
        if (lo > 0 && hi >= lo) spread = max(spread, hi - lo);
        double r2[2];
        matvec_row(r2, Cp, vec + VD, q);
        const double rr = rows_to_slot(r2, lane);
        if (lane < 16) {
            vec[VX + lane] = xslot >= 0 ? rr : 0.0;
            if (xslot >= 0) __stcs(mb + mrows - n + xslot, -rr);  // mu_N
        }
    }
    if (lane == 0) {
        // the reference factors every H_k before any Schur block: a Hessian failure at any knot takes precedence
        if (info) info[inst] = hcode != 0 ? hcode : st_all;
        cinfo[inst] = spread >> 20;  // log2 of the worst pivot ratio of any Sigma_k
    }
    __syncwarp();

    // ---------------- backward sweep: k = N-1 .. 0     x_{k-1} = v_k + Z_k' x_k,  Lambda = -x
    // the buffer ring continues: knot k uses stage (N-1-k) & 1 with its own phase count
    int uses0 = (N + 1) / 2, uses1 = N / 2;  // completed phases per stage after the forward sweep
    auto issue_b = [&](int it) { issue(N - 1 - it, it & 1); };
    issue_b(0);
    if (N > 1) issue_b(1);
    for (int it = 0; it < N; ++it) {
        const int k = N - 1 - it;
        const bool first = k == 0, last = k == N - 1;
        const int st = it & 1;
        const int wk = last ? n : w;
        // record
        const double *rk = rb + (int64_t)k * recw;
        const int psk = knot_ps(k);
        Tile16 Zm;
        Zm.v[0][0][0] = rk[lane];
        Zm.v[0][0][1] = rk[32 + lane];
        Zm.v[0][1][1] = Zm.v[1][1][1] = 0.0;
        Zm.v[0][1][0] = Zm.v[1][0][0] = Zm.v[1][0][1] = Zm.v[1][1][0] = 0.0;
        if (n > 8) {
            Zm.v[0][1][0] = rk[64 + lane];
            if (!(g & 1)) {
                const int hl = (g >> 1) * 4 + q;
                Zm.v[1][0][0] = rk[96 + hl];
                Zm.v[1][0][1] = rk[112 + hl];
                Zm.v[1][1][0] = rk[128 + hl];
            }
        }
        const double vk = lane < 16 ? rk[RW::ZR + lane] : 0.0;
        double c4[2][2];
        matvec_col(c4, Zm, vec + VX, g);  // Z' x_k : lane (g, q) holds columns 8 ct + 2 q + e
        {
            const double zx = cols_to_slot(c4, lane);
            double xp = xslot >= 0 ? vk + zx : 0.0;  // x_{k-1} (k >= 1) or mu_1'
            if (psk > 0) {
                // xi = Bi (c' - E' x_k)   (mu_k' of the back-substitution);  x_{k-1} -= sum_j xi_j sd_j
                const double *rs = rk + RW::REC;
                if (lane < psk) {
                    double sx = rs[32 * psk + 16 + lane];
                    for (int t = 0; t < 16; ++t) sx = fma(-rs[32 * lane + 16 + t], vec[VX + t], sx);
                    vec[SCP + lane] = sx;
                }
                __syncwarp();
                if (lane < psk) {
                    double sx = 0.0;
                    for (int jp = 0; jp < psk; ++jp) sx = fma(rs[32 * psk + 4 * lane + jp], vec[SCP + jp], sx);
                    vec[SXI + lane] = sx;
                }
                __syncwarp();
                if (lane < 16 && xslot >= 0)
                    for (int j = 0; j < psk; ++j) xp = fma(-vec[SXI + j], rs[32 * j + lane], xp);
            }
            if (lane < 16) vec[VXP + lane] = xp;
        }
        {
            const uint32_t par = (uint32_t)(((st == 0 ? uses0 : uses1) + (it >> 1)) & 1);
            mbar_wait(bars + st, par);
        }
        const double *kp = buf + st * BUF + knot_shift(k);
        if (lane < 16) vec[VG + lane] = (!soc && zslot >= 0 && zslot < wk) ? kp[(last ? L::HQ : L::og) + zslot] : 0.0;
        Tile16 Hi, F;
        {   // H_k^-1 from the record (upper tiles; tile (1,0) is the transpose of tile (0,1))
            const double *rh = rk + RW::HIO;
            Hi.v[0][0][0] = rh[lane];
            Hi.v[0][0][1] = rh[32 + lane];
            Hi.v[0][1][0] = rh[64 + lane];
            Hi.v[0][1][1] = rh[96 + lane];
            Hi.v[1][1][0] = rh[128 + lane];
            Hi.v[1][1][1] = rh[160 + lane];
            Hi.v[1][0][0] = Hi.v[1][0][1] = 0.0;
            transpose8(Hi.v[1][0], Hi.v[0][1], 1.0, g, q);
        }
        load_rows(F, last ? kp + L::oCl : kp + L::oD1, wk);
        __syncwarp();  // x_{k-1}, g are published
        // res_k = g_k + D1' lam_k + D2' lam_{k-1} (+ C_1' mu_1)  with Lambda = -x   (calc_residual! :201-236)
        matvec_col(c4, F, vec + VX, g);
        const double fx = cols_to_slot(c4, lane);
        double cx = 0.0;
        if (first) {
            Tile16 Cc;
            load_rows(Cc, kp + L::oC0, w);
            matvec_col(c4, Cc, vec + VXP, g);
            cx = cols_to_slot(c4, lane);
        }
        double rz = 0.0;
        if (lane < 16 && zslot >= 0 && zslot < wk) {
            rz = vec[VG + lane] - fx;
            if (first) rz -= cx;
            else if (xslot >= 0) rz += vec[VXP + lane];
            for (int j = 0; j < psk; ++j) rz = fma(-vec[SXI + j], kp[L::CORE + j + psk * zslot], rz);  // C' mu_k, mu = -xi
        }
        if (lane < 16) vec[VR + lane] = rz;
        __syncwarp();  // the knot buffer is free, res is published
        if (it + 2 < N) issue_b(it + 2);
        double r2[2];
        matvec_row(r2, Hi, vec + VR, q);  // dz_k = -Hi res_k   (calc_primals! :195-199)
        {
            const double rr = rows_to_slot(r2, lane);
            if (lane < 16 && zslot >= 0 && zslot < wk) {
                __stcs(zb + (int64_t)k * w + zslot, -rr);
                if (resb) __stcs(resb + (int64_t)k * w + zslot, rz);
            }
            // multipliers: [mu_1 (n); lam_1 (n); mu_2 (ps); lam_2; ...; lam_{N-1}; mu_N]; this knot produces lam_{k-1}
            // (k >= 1) or mu_1, and its own stage multipliers mu_k
            const int64_t lo_ = first ? 0 : (moff ? moff[k] - n : (int64_t)n + (int64_t)(k - 1) * lstride);
            if (lane < 16 && xslot >= 0) __stcs(mb + lo_ + xslot, -vec[VXP + lane]);
            if (lane < psk) __stcs(mb + lo_ + n + lane, -vec[SXI + lane]);
        }
        __syncwarp();
        if (lane < 16) vec[VX + lane] = vec[VXP + lane];
        __syncwarp();
    }
}

}  // namespace kwp
