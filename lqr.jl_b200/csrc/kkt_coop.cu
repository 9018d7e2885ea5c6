// kkt_coop.cuh — cooperative (G threads per instance) constrained KKT solve for ANY size / stage
// pattern / explicit D2.  Same two-sweep restructuring of src/cholesky_solver.jl:166-236 as the
// thread-per-instance kernel (see kkt_kernels.cuh), but runtime dimensions, full-storage blocks in a
// per-instance workspace (shared memory when it fits, else an L2-resident global slot), packed
// layout tile width 1.
#include <algorithm>
#include <cstdio>

#include "kkt_coop.cuh"
#include "coop_prims.cuh"
#include "smallmat.cuh"

// ------------------------------------------------------------------ cost Hessian ---------------
// BlockCholesky modes (src/block_cholesky.jl:55-101) on a full-storage w x w workspace matrix.
template <int G>
__device__ __forceinline__ void load_hessian(double *Hf, double *dinv, const double *kp, int n, int mk,
                                             int hess, int soc, int t) {
    const int w = n + mk;
    if (soc) return;
    if (hess == LQRB_HESS_DIAG) {
        for (int i = t; i < w; i += G) dinv[i] = kp[i];
    } else if (hess == LQRB_HESS_BLOCKDIAG) {
        for (int e = t; e < w * w; e += G) {
            const int i = e % w, j = e / w;
            double v = 0.0;
            if (i <= j && j < n) v = kp[tri_idx(i, j)];
            else if (i <= j && i >= n) v = kp[tri(n) + tri_idx(i - n, j - n)];
            Hf[e] = v;
        }
    } else {
        for (int e = t; e < w * w; e += G) {
            const int i = e % w, j = e / w;
            Hf[e] = (i <= j) ? kp[tri_idx(i, j)] : 0.0;
        }
    }
}

template <int G>
__device__ __forceinline__ int factor_hessian(double *Hf, double *dinv, int w, int hess, int soc, int t) {
    if (soc) return 0;
    if (hess == LQRB_HESS_DIAG) {
        for (int i = t; i < w; i += G) dinv[i] = 1.0 / dinv[i];  // stores the inverse (:82-91)
        group_sync<G>();
        return 0;
    }
    return co_chol<G>(Hf, w, w, t);
}

// X (w x nrhs, ld ldx) <- H^-1 X
template <int G>
__device__ __forceinline__ void solve_hessian(const double *Hf, const double *dinv, int w, int hess,
                                              int soc, double *X, int nrhs, int ldx, int t) {
    if (soc || nrhs == 0) return;
    if (hess == LQRB_HESS_DIAG) {
        for (int e = t; e < w * nrhs; e += G) X[(e % w) + (size_t)(e / w) * ldx] *= dinv[e % w];
        group_sync<G>();
        return;
    }
    co_trsm_ut<G>(Hf, w, w, X, nrhs, ldx, t);
    co_trsm_un<G>(Hf, w, w, X, nrhs, ldx, t);
}

struct KktCoopArgs {
    const double *data;
    double *scratch, *dz, *mult, *res;
    int32_t *info;
    const int32_t *p;         // device copy of the stage pattern [N]
    const int64_t *knot_off;  // device: data row offset per knot [N+1]
    const int64_t *rec_off;   // device: record row offset per knot [N+1]
    const int64_t *mult_off;  // device: mult row offset of mu_k per knot [N+1]
    double *gws;              // global workspace (nullptr: shared memory)
    const int32_t *list;      // optional: the instances to process (batch = its length); nullptr = 0..batch-1
    const double *rhs;        // phase 2: per instance [per knot: g (w) | d (p2) | c (ps)], tile width 1
    double *sdump;            // optional: raw Schur blocks S (before cholesky!) in the record layout
    int phase;                // 0 fused, 1 factor only, 2 solve with the kept factor
    int64_t data_stride, mult_stride;  // per-instance strides of data / mult when they are not the shape's own (0: own)
    int n, m, N, hess, d2x, soc;
    int64_t batch;
    int P;  // max p_k
};

template <int G, int THREADS>
__global__ void __launch_bounds__(THREADS) kkt_coop_kernel(KktCoopArgs a) {
    extern __shared__ double smem[];
    constexpr int IPC = THREADS / G;
    const int g = threadIdx.x / G, t = threadIdx.x % G;
    const int n = a.n, m = a.m, N = a.N, P = a.P;
    const size_t wsd = kkt_coop_ws_doubles(n, m, P);
    double *ws = a.gws ? a.gws + ((size_t)blockIdx.x * IPC + g) * wsd : smem + (size_t)g * wsd;
    const int wmax = n + m;
    // carve
    double *Hf = ws, *hg = Hf + wmax * wmax, *dinv = hg + wmax, *z = dinv + wmax, *D1 = z + wmax,
           *D2 = D1 + n * wmax, *Cc = D2 + n * wmax, *WD = Cc + P * wmax, *W2 = WD + wmax * n,
           *WC = W2 + wmax * n, *Ah = WC + wmax * P, *Fh = Ah + n * n, *Cp = Fh + n * n, *Bh = Cp + n * n,
           *Dh = Bh + P * P, *Eh = Dh + n * P, *dp = Eh + n * P, *lamp = dp + n, *lam = lamp + n,
           *lprev = lam + n, *mut = lprev + n, *mu = mut + P, *cvec = mu + P;

    // Groups narrower than a warp synchronise with __syncwarp(): the groups of one warp make the same number of trips,
    // and a group without an instance of its own shadows the last one (same bits written twice).
    constexpr int GPW = G < 32 ? 32 / G : 1;
    for (int64_t base = (int64_t)blockIdx.x * IPC + (g / GPW) * GPW; base < a.batch;
         base += (int64_t)gridDim.x * IPC) {
        const int64_t inst = base + g % GPW < a.batch ? base + g % GPW : a.batch - 1;
        const bool active = true;
        const int64_t ii = a.list ? (int64_t)a.list[inst] : inst;  // optional instance list (re-solve of a subset)
        const int64_t data_rows = a.data_stride ? a.data_stride : a.knot_off[N], rec_rows = a.rec_off[N],
                      mult_rows = a.mult_stride ? a.mult_stride : a.mult_off[N];
        const int64_t NN = (int64_t)N * n + (int64_t)(N - 1) * m;
        const double *db = a.data + ii * data_rows;
        double *sb = a.scratch + inst * rec_rows;  // records by position: a list needs only its own slots
        double *zb = a.dz + ii * NN, *mb = a.mult + ii * mult_rows;
        double *rb = a.res ? a.res + ii * NN : nullptr;
        int st_all = 0, hcode = 0;  // first Schur-block failure, first Hessian failure

        // ======================= forward sweep =======================
        // phase 0: fused solve; 1: factor only (calculate_shur_factors! + cholesky!(U, F), blocks kept in `scratch`);
        // 2: solve with the kept factor and a new right-hand side (a.rhs): only the vector part of
        //    calculate_shur_factors! and forward_substitution! run here, no O(n^3) work.
        const bool fac = a.phase != 2;
        const double *rhsb = a.rhs ? a.rhs + ii * (NN + mult_rows) : nullptr;
        double *sdb = a.sdump ? a.sdump + inst * rec_rows : nullptr;
        for (int k = 0; k < N; ++k) {
            const int mk = k < N - 1 ? m : 0, w = n + mk, p1 = k > 0 ? n : 0, ps = a.p[k],
                      p2 = k < N - 1 ? n : 0;
            const double *kp = db + a.knot_off[k];
            double *rec = sb + a.rec_off[k];
            double *rB = rec, *rD = rB + (int64_t)ps * ps, *rE = rD + (int64_t)p1 * ps, *rF = rE + (int64_t)ps * p2,
                   *rmu = rF + (int64_t)p1 * p2, *rC = rmu + ps, *rl = rC + (int64_t)p1 * p1;
            // raw (unfactored) Schur blocks in the same record layout: B | D | E | F | c | C_{k-1} | d_{k-1}
            double *sd = sdb ? sdb + a.rec_off[k] : nullptr;
            const int hr = hess_rows(n, mk, a.hess);
            const double *D1p = kp + hr + w, *D2p = D1p + p2 * w + p2,
                         *Cp_in = D2p + ((a.d2x && k > 0) ? n * w : 0);
            // right-hand-side rows g | d | c: inside the knot record, or (phase 2) in the separate rhs array
            const double *gp = rhsb ? rhsb + (int64_t)k * (n + m) + a.mult_off[k] : kp + hr;
            const double *dvp = rhsb ? gp + w : D1p + p2 * w;
            const double *cp_in = rhsb ? dvp + p2 : Cp_in + ps * w;
            // ---- load H (full storage), g, D1, D2, C
            load_hessian<G>(Hf, dinv, kp, n, mk, a.hess, a.soc, t);
            for (int e = t; e < w; e += G) hg[e] = a.soc ? 0.0 : gp[e];
            for (int e = t; e < p2 * w; e += G) D1[e] = D1p[e];
            for (int e = t; e < ps * w; e += G) Cc[e] = Cp_in[e];
            if (p1) {
                for (int e = t; e < n * w; e += G) {
                    const int i = e % n, j = e / n;
                    D2[e] = a.d2x ? D2p[e] : (i == j ? -1.0 : 0.0);
                }
            }
            group_sync<G>();
            int st = factor_hessian<G>(Hf, dinv, w, a.hess, a.soc, t);
            if (st && !hcode) hcode = (k + 1) * 1000 + st;
            // ---- W = H^-1 Y' (columns of D2', D1', C') and hg = H^-1 g
            if (fac) {
                for (int e = t; e < w * p1; e += G) W2[e] = D2[(e / w) + (e % w) * n];
                for (int e = t; e < w * p2; e += G) WD[e] = D1[(e / w) + (e % w) * p2];
                for (int e = t; e < w * ps; e += G) WC[e] = Cc[(e / w) + (e % w) * ps];
                group_sync<G>();
            }
            solve_hessian<G>(Hf, dinv, w, a.hess, a.soc, hg, 1, w, t);
            if (fac) {
                solve_hessian<G>(Hf, dinv, w, a.hess, a.soc, W2, p1, w, t);
                solve_hessian<G>(Hf, dinv, w, a.hess, a.soc, WD, p2, w, t);
                solve_hessian<G>(Hf, dinv, w, a.hess, a.soc, WC, ps, w, t);
            }
            // ---- finish block row k-1
            if (p1) {
                if (fac) {
                    co_gemm<G>(0, 0, n, n, w, 1.0, D2, n, W2, w, 1.0, Cp, n, t);  // C_{k-1} += D2 H^-1 D2'
                    for (int e = t; e < n * n; e += G) Ah[e] = Cp[e];
                } else {
                    for (int e = t; e < n * n; e += G) Ah[e] = rC[e];  // the kept factor C^_{k-1}
                }
                co_gemm<G>(0, 0, n, 1, w, 1.0, D2, n, hg, w, 1.0, dp, n, t);  // d_{k-1} += rho1
                for (int e = t; e < n; e += G) lamp[e] = dp[e];
                group_sync<G>();
                if (fac) {
                    if (sd) {
                        // raw S block C_{k-1} = D1 H^-1 D1' (left here by knot k-1) + D2 H^-1 D2', and d_{k-1} likewise
                        double *sC = sd + (int64_t)ps * ps + (int64_t)p1 * ps + (int64_t)ps * p2 + (int64_t)p1 * p2 + ps;
                        co_gemm<G>(0, 0, n, n, w, 1.0, D2, n, W2, w, 1.0, sC, n, t);
                        co_gemm<G>(0, 0, n, 1, w, 1.0, D2, n, hg, w, 1.0, sC + n * n, n, t);
                    }
                    st = co_chol<G>(Ah, n, n, t);
                    if (st && !st_all) st_all = k * 1000 + 200 + st;
                }
                co_trsm_ut<G>(Ah, n, n, lamp, 1, n, t);
                if (active) {
                    if (fac)
                        for (int e = t; e < n * n; e += G) rC[e] = Ah[e];
                    for (int e = t; e < n; e += G) rl[e] = lamp[e];
                }
            }
            if (p1 && p2) {
                if (fac) {
                    co_gemm<G>(0, 0, n, n, w, 1.0, D2, n, WD, w, 0.0, Fh, n, t);  // F = D2 WD
                    if (sd) {
                        double *sF = sd + (int64_t)ps * ps + (int64_t)p1 * ps + (int64_t)ps * p2;
                        for (int e = t; e < n * n; e += G) sF[e] = Fh[e];
                        group_sync<G>();
                    }
                    co_trsm_ut<G>(Ah, n, n, Fh, n, n, t);
                } else {
                    for (int e = t; e < n * n; e += G) Fh[e] = rF[e];
                    group_sync<G>();
                }
            }
            if (ps) {
                if (fac) {
                    co_gemm<G>(0, 0, ps, ps, w, 1.0, Cc, ps, WC, w, 0.0, Bh, ps, t);  // B = C WC
                } else {
                    for (int e = t; e < ps * ps; e += G) Bh[e] = rB[e];
                    for (int e = t; e < p1 * ps; e += G) Dh[e] = rD[e];
                    for (int e = t; e < ps * p2; e += G) Eh[e] = rE[e];
                }
                for (int e = t; e < ps; e += G) cvec[e] = -cp_in[e];
                group_sync<G>();
                co_gemm<G>(0, 0, ps, 1, w, 1.0, Cc, ps, hg, w, 1.0, cvec, ps, t);  // c = rhos - c
                for (int e = t; e < ps; e += G) mut[e] = cvec[e];
                group_sync<G>();
                if (fac) {
                    if (p2) co_gemm<G>(0, 0, ps, p2, w, 1.0, Cc, ps, WD, w, 0.0, Eh, ps, t);  // E = C WD
                    if (p1) co_gemm<G>(0, 0, n, ps, w, 1.0, D2, n, WC, w, 0.0, Dh, n, t);     // D = D2 WC
                    if (sd) {
                        double *s0 = sd;
                        for (int e = t; e < ps * ps; e += G) s0[e] = Bh[e];
                        s0 += (int64_t)ps * ps;
                        for (int e = t; e < p1 * ps; e += G) s0[e] = Dh[e];
                        s0 += (int64_t)p1 * ps;
                        for (int e = t; e < ps * p2; e += G) s0[e] = Eh[e];
                        s0 += (int64_t)ps * p2 + (int64_t)p1 * p2;
                        for (int e = t; e < ps; e += G) s0[e] = cvec[e];
                        group_sync<G>();
                    }
                    if (p1) {
                        co_trsm_ut<G>(Ah, n, n, Dh, ps, n, t);
                        co_gemm<G>(1, 0, ps, ps, n, -1.0, Dh, n, Dh, n, 1.0, Bh, ps, t);
                        if (p2) co_gemm<G>(1, 0, ps, p2, n, -1.0, Dh, n, Fh, n, 1.0, Eh, ps, t);
                    }
                }
                if (p1) co_gemm<G>(1, 0, ps, 1, n, -1.0, Dh, n, lamp, n, 1.0, mut, ps, t);
                if (fac) {
                    st = co_chol<G>(Bh, ps, ps, t);
                    if (st && !st_all) st_all = (k + 1) * 1000 + 100 + st;
                }
                co_trsm_ut<G>(Bh, ps, ps, mut, 1, ps, t);
                if (fac && p2) co_trsm_ut<G>(Bh, ps, ps, Eh, p2, ps, t);
            }
            if (p2) {
                if (fac) co_gemm<G>(0, 0, n, n, w, 1.0, D1, n, WD, w, 0.0, Cp, n, t);  // G22
                for (int e = t; e < n; e += G) dp[e] = -dvp[e];
                group_sync<G>();
                co_gemm<G>(0, 0, n, 1, w, 1.0, D1, n, hg, w, 1.0, dp, n, t);  // rho2 - d
                if (fac && sdb) {
                    // the unfactored parts of C_k and d_k go to knot k+1's slot (the A_{k+1} = C_k aliasing)
                    const int psn = a.p[k + 1], p2n = k + 1 < N - 1 ? n : 0;
                    double *sCn = sdb + a.rec_off[k + 1] + (int64_t)psn * psn + (int64_t)n * psn + (int64_t)psn * p2n +
                                  (int64_t)n * p2n + psn;
                    for (int e = t; e < n * n; e += G) sCn[e] = Cp[e];
                    for (int e = t; e < n; e += G) sCn[n * n + e] = dp[e];
                    group_sync<G>();
                }
                if (p1) {
                    if (fac) co_gemm<G>(1, 0, n, n, n, -1.0, Fh, n, Fh, n, 1.0, Cp, n, t);
                    co_gemm<G>(1, 0, n, 1, n, -1.0, Fh, n, lamp, n, 1.0, dp, n, t);
                }
                if (ps) {
                    if (fac) co_gemm<G>(1, 0, n, n, ps, -1.0, Eh, ps, Eh, ps, 1.0, Cp, n, t);
                    co_gemm<G>(1, 0, n, 1, ps, -1.0, Eh, ps, mut, ps, 1.0, dp, n, t);
                }
            }
            if (active) {
                if (fac) {
                    for (int e = t; e < ps * ps; e += G) rB[e] = Bh[e];
                    for (int e = t; e < p1 * ps; e += G) rD[e] = Dh[e];
                    for (int e = t; e < ps * p2; e += G) rE[e] = Eh[e];
                    for (int e = t; e < p1 * p2; e += G) rF[e] = Fh[e];
                }
                for (int e = t; e < ps; e += G) rmu[e] = mut[e];
            }
            group_sync<G>();
        }
        // the reference factors every H_k before any Schur block: a Hessian failure at any knot takes precedence
        if (active && a.info && t == 0) a.info[ii] = hcode ? hcode : st_all;
        if (a.phase == 1) continue;  // factor only

        // ======================= backward sweep =======================
        for (int k = N - 1; k >= 0; --k) {
            const int mk = k < N - 1 ? m : 0, w = n + mk, p1 = k > 0 ? n : 0, ps = a.p[k],
                      p2 = k < N - 1 ? n : 0;
            const double *kp = db + a.knot_off[k];
            const double *rec = sb + a.rec_off[k];
            const int hr = hess_rows(n, mk, a.hess);
            const double *D1p = kp + hr + w, *D2p = D1p + p2 * w + p2,
                         *Cp_in = D2p + ((a.d2x && k > 0) ? n * w : 0);
            const double *gp = rhsb ? rhsb + (int64_t)k * (n + m) + a.mult_off[k] : kp + hr;
            const double *rB = rec, *rD = rB + (int64_t)ps * ps, *rE = rD + (int64_t)p1 * ps,
                         *rF = rE + (int64_t)ps * p2, *rmu = rF + (int64_t)p1 * p2, *rC = rmu + ps,
                         *rl = rC + (int64_t)p1 * p1;
            // mu' = B^-1 (mu~ - E^ lam')
            for (int e = t; e < ps * ps; e += G) Bh[e] = rB[e];
            for (int i = t; i < ps; i += G) {
                double s = rmu[i];
                for (int l = 0; l < p2; ++l) s = fma(-rE[i + (int64_t)l * ps], lam[l], s);
                mu[i] = s;
            }
            group_sync<G>();
            if (ps) co_trsm_un<G>(Bh, ps, ps, mu, 1, ps, t);
            // lam'_{k-1} = C^-1 (lam~ - D^ mu' - F^ lam')
            if (p1) {
                for (int e = t; e < n * n; e += G) Ah[e] = rC[e];
                for (int i = t; i < n; i += G) {
                    double s = rl[i];
                    for (int l = 0; l < ps; ++l) s = fma(-rD[i + (int64_t)l * n], mu[l], s);
                    for (int l = 0; l < p2; ++l) s = fma(-rF[i + (int64_t)l * n], lam[l], s);
                    lprev[i] = s;
                }
                group_sync<G>();
                co_trsm_un<G>(Ah, n, n, lprev, 1, n, t);
            }
            if (active) {
                double *mm = mb + a.mult_off[k];
                for (int i = t; i < ps; i += G) mm[i] = -mu[i];
                if (p1)
                    for (int i = t; i < n; i += G) mm[i - n] = -lprev[i];
            }
            // res = g - D1'lam' - C'mu' - D2'lprev'
            for (int j = t; j < w; j += G) {
                double s = a.soc ? 0.0 : gp[j];
                for (int i = 0; i < p2; ++i) s = fma(-D1p[i + (int64_t)j * p2], lam[i], s);
                for (int i = 0; i < ps; ++i) s = fma(-Cp_in[i + (int64_t)j * ps], mu[i], s);
                if (p1) {
                    if (a.d2x) {
                        for (int i = 0; i < n; ++i) s = fma(-D2p[i + (int64_t)j * n], lprev[i], s);
                    } else if (j < n) {
                        s += lprev[j];
                    }
                }
                z[j] = s;
                if (active && rb) rb[(int64_t)k * (n + m) + j] = s;
            }
            load_hessian<G>(Hf, dinv, kp, n, mk, a.hess, a.soc, t);
            group_sync<G>();
            factor_hessian<G>(Hf, dinv, w, a.hess, a.soc, t);
            solve_hessian<G>(Hf, dinv, w, a.hess, a.soc, z, 1, w, t);
            if (active)
                for (int j = t; j < w; j += G) zb[(int64_t)k * (n + m) + j] = -z[j];
            for (int i = t; i < p1; i += G) lam[i] = lprev[i];
            group_sync<G>();
        }
    }
}

// device copies of the per-shape offset tables, cached on the handle
using CoopTables = KktTables;

static int32_t get_tables(lqrb_context *h, int n, int m, int N, const int32_t *p, int hess, int d2x,
                          CoopTables *out);
int32_t lqrb_kkt_tables(lqrb_context *h, int n, int m, int N, const int32_t *p, int hess, int d2x, KktTables *out) {
    return get_tables(h, n, m, N, p, hess, d2x, out);
}

static int32_t get_tables(lqrb_context *h, int n, int m, int N, const int32_t *p, int hess, int d2x,
                          CoopTables *out) {
    std::string key = "coop:";
    char buf[64];
    snprintf(buf, sizeof buf, "%d:%d:%d:%d:%d:", n, m, N, hess, d2x);
    key += buf;
    int P = 0;
    for (int k = 0; k < N; ++k) {
        key += std::to_string(p[k]) + ",";
        P = std::max(P, (int)p[k]);
    }
    out->P = P;
    auto it = h->blobs.find(key);
    char *blob = nullptr;
    const size_t off_bytes = (size_t)(N + 1) * sizeof(int64_t);
    const size_t p_bytes = round_up((int64_t)N * sizeof(int32_t), 16);
    if (it != h->blobs.end()) {
        blob = (char *)it->second;
    } else {
        std::vector<char> host(3 * off_bytes + p_bytes);
        int64_t *ko = (int64_t *)host.data(), *ro = ko + (N + 1), *mo = ro + (N + 1);
        int32_t *pp = (int32_t *)(host.data() + 3 * off_bytes);
        int64_t kacc = 0, racc = 0, macc = 0;
        for (int k = 0; k < N; ++k) {
            ko[k] = kacc;
            ro[k] = racc;
            mo[k] = macc;
            pp[k] = p[k];
            kacc = lqrb_kkt_knot_offset(n, m, N, p, hess, d2x, k + 1);
            racc += kkt_coop_rec_knot_rows(k > 0 ? n : 0, p[k], k < N - 1 ? n : 0);
            macc += p[k] + (k < N - 1 ? n : 0);
        }
        ko[N] = kacc;
        ro[N] = racc;
        mo[N] = macc;
        void *d = nullptr;
        LQRB_CUDA(h, cudaMalloc(&d, host.size()));
        LQRB_CUDA(h, cudaMemcpy(d, host.data(), host.size(), cudaMemcpyHostToDevice));
        LQRB_CUDA(h, cudaStreamSynchronize(cudaStreamLegacy));  // pageable source: wait for the staged DMA
        h->blobs[key] = d;
        blob = (char *)d;
    }
    out->knot_off = (const int64_t *)blob;
    out->rec_off = out->knot_off + (N + 1);
    out->mult_off = out->rec_off + (N + 1);
    out->p = (const int32_t *)(blob + 3 * off_bytes);
    return 0;
}

int32_t launch_kkt_coop(lqrb_context *h, int n, int m, int N, const int32_t *p, int hess, int d2x,
                        int flags, int64_t batch, const double *data, double *scratch, double *dz,
                        double *mult, double *res, int32_t *info, Lane lane, const KktCoopExtra *extra) {
    CoopTables tb;
    int32_t rc = get_tables(h, n, m, N, p, hess, d2x, &tb);
    if (rc) return rc;
    KktCoopArgs a;
    a.data = data; a.scratch = scratch; a.dz = dz; a.mult = mult; a.res = res; a.info = info;
    a.p = tb.p; a.knot_off = tb.knot_off; a.rec_off = tb.rec_off; a.mult_off = tb.mult_off;
    a.gws = nullptr;
    a.list = extra ? extra->list : nullptr;
    a.rhs = extra ? extra->rhs : nullptr;
    a.sdump = extra ? extra->sdump : nullptr;
    a.phase = extra ? extra->phase : 0;
    a.data_stride = extra ? extra->data_stride : 0;
    a.mult_stride = extra ? extra->mult_stride : 0;
    a.n = n; a.m = m; a.N = N; a.hess = hess; a.d2x = d2x; a.soc = (flags & LQRB_FLAG_SOC) ? 1 : 0;
    a.batch = batch; a.P = tb.P;
    const size_t wsd = kkt_coop_ws_doubles(n, m, tb.P);
    const size_t smem_cap = 200 * 1024;
    char nm[96];
    if (n + m <= 24) {
        // lanes per instance, measured (N = 101, 8-16 k instances, solves/s at G = 4 / 8 / 16 / 32): (3,2) 1.56e6 / 1.18e6 /
        // 7.6e5 / 4.0e5; (5,2) 5.0e5 / 8.5e5 / 8.3e5 / 5.1e5; (6,3) 3.0e5 / 4.1e5 / 4.7e5 / 2.9e5; (10,3) 1.5e5 / 1.6e5 /
        // 1.75e5 / 1.4e5; (13,4) 5.1e4 / 8.4e4 / 6.2e4 / 7.4e4.  `coop_group` forces one of them.
        int G = n + m <= 5 ? 4 : (n + m <= 7 ? 8 : (n + m <= 13 ? 16 : 32));
        const int64_t force = h->opt("coop_group", 0);
        if (force == 4 || force == 8 || force == 16 || force == 32) G = (int)force;
        constexpr int THREADS = 128;
        const int IPC = THREADS / G;
        size_t smem = wsd * 8 * IPC;
        unsigned grid = (unsigned)std::min<int64_t>((batch + IPC - 1) / IPC, (int64_t)h->sm_count * 64);
        auto kern = G == 4 ? kkt_coop_kernel<4, THREADS>
                           : (G == 8 ? kkt_coop_kernel<8, THREADS> : (G == 16 ? kkt_coop_kernel<16, THREADS> : kkt_coop_kernel<32, THREADS>));
        if (smem > smem_cap) {
            grid = std::min<unsigned>(grid, (unsigned)h->sm_count * 8);  // instances are strided over the grid
            a.gws = (double *)lqrb_scratch(h, SCR_MISC, (size_t)h->sm_count * 8 * IPC * wsd * 8, lane.index);
            if (!a.gws) return 1000 + (int)cudaErrorMemoryAllocation;
            smem = 0;
        } else {
            LQRB_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        }
        kern<<<grid, THREADS, smem, lane.stream>>>(a);
        snprintf(nm, sizeof nm, "kkt_coop<G=%d>(n=%d,m=%d,%s)", G, n, m, a.gws ? "gmem-ws" : "smem-ws");
    } else {
        constexpr int G = 256, THREADS = 256;
        size_t smem = wsd * 8;
        unsigned grid = (unsigned)std::min<int64_t>(batch, (int64_t)h->sm_count * 4);
        auto kern = kkt_coop_kernel<G, THREADS>;
        if (smem > smem_cap) {
            a.gws = (double *)lqrb_scratch(h, SCR_MISC, (size_t)h->sm_count * 4 * wsd * 8, lane.index);
            if (!a.gws) return 1000 + (int)cudaErrorMemoryAllocation;
            smem = 0;
        } else {
            LQRB_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        }
        kern<<<grid, THREADS, smem, lane.stream>>>(a);
        snprintf(nm, sizeof nm, "kkt_coop<G=256>(n=%d,m=%d,%s)", n, m, a.gws ? "gmem-ws" : "smem-ws");
    }
    h->kernel_name = nm;
    LQRB_LAUNCH_CHECK(h, "kkt_coop_kernel");
    return 0;
}
