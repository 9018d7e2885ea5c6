// kkt_kernels.cuh — batched equality-constrained LQR KKT solve, thread-per-instance family.
//
// Replaces _solve!(::CholeskySolver) : src/cholesky_solver.jl:166-182 —
//   calculate_shur_factors!  src/jacobian_blocks.jl:220-229   (shur! :231-242, copy_shur! :249-286)
//   cholesky!(chol, shur)    src/cholesky_solve.jl:28-33,47-67
//   forward_substitution!    src/cholesky_solve.jl:93-117
//   backward_substitution!   src/cholesky_solve.jl:119-143   (negates: Lambda = -S^-1 h)
//   calculate_primals!       src/cholesky_solver.jl:185-236
// and, with SOC, the Ginv=false chain of second_order_correction! (:254-273).
//
// The reference makes five passes over the knots with every block in memory.  Here one thread owns
// one instance and makes TWO sweeps:
//   forward  k = 0..N-1 : load knot k, factor H_k, form its Schur pieces, finish block row k-1 of S
//                         (C_{k-1} += G_k[1,1], the A_k = C_{k-1} aliasing of
//                         src/jacobian_blocks.jl:165-167 becomes a register carry), factor block row
//                         k and forward-substitute; only C^_{k-1} and lam~_{k-1} go to the per-instance
//                         scratch record (tri(n)+n doubles per knot);
//   backward k = N-1..0 : reload knot k and its record, RECOMPUTE the rest of block row k (cheaper
//                         than a round trip through HBM: the kernel is DRAM-bound with the FP64 pipe
//                         under 20 % busy), back-substitute, form the residual and the primal step.
// D2_k = [-I 0] is structural here (test/cartpole.jl:34-42); explicit D2 goes to the cooperative kernel.
#pragma once
#include "smallmat.cuh"

// Knot rows are read either from the packed tile (stride KS = 32 doubles between rows, read-only global
// memory) or from a thread-local array the caller has just filled (KS = 1: the fused SQP kernel linearises
// the knot on the fly instead of streaming it from HBM).
template <int KS>
__device__ __forceinline__ double ldk_keep(const double *p) {
    if constexpr (KS == 32) return ld_keep(p);
    else return *p;
}
template <int KS>
__device__ __forceinline__ double ldk_stream(const double *p) {
    if constexpr (KS == 32) return ld_stream(p);
    else return *p;
}

// ------------------------------------------------------------------ per-knot row layout -------

// rows of one knot in the packed data array (see lqrb200.h): H | g | D1 | d | [D2] | C | c
template <int n, int mk, int ps, int p2, int HESS>
struct KnotRows {
    static constexpr int w = n + mk;
    static constexpr int oH = 0, oG = hess_rows(n, mk, HESS), oD1 = oG + w, od = oD1 + p2 * w,
                         oC = od + p2, oc = oC + ps * w, ROWS = oc + ps;
};

// ------------------------------------------------------------------ cost-Hessian factor -------
// BlockCholesky modes, src/block_cholesky.jl:55-101, factor kept in registers.
template <int n, int mk, int HESS, bool SOC>
struct HFactor {
    static constexpr int w = n + mk;
    static constexpr int NU = SOC ? 1 : (HESS == LQRB_HESS_DIAG ? 1 : hess_rows(n, mk, HESS));
    double u[NU];
    double dinv[w];

    template <int KS = 32>
    __device__ __forceinline__ int load_factor(const double *hp) {
        if constexpr (SOC) {
            return 0;
        } else if constexpr (HESS == LQRB_HESS_DIAG) {  // stores the inverse (:82-91)
            SM_UNROLL
            for (int i = 0; i < w; ++i) dinv[i] = 1.0 / ldk_keep<KS>(hp + i * KS);
            return 0;
        } else if constexpr (HESS == LQRB_HESS_BLOCKDIAG) {  // two potrf (:69-77)
            SM_UNROLL
            for (int e = 0; e < NU; ++e) u[e] = ldk_keep<KS>(hp + e * KS);
            int st = chol_packed<n>(u, dinv);
            if constexpr (mk > 0) {
                const int st2 = chol_packed<mk>(u + tri(n), dinv + n);
                if (st == 0 && st2 != 0) st = n + st2;
            }
            return st;
        } else {  // whole-matrix potrf (:55-66)
            SM_UNROLL
            for (int e = 0; e < NU; ++e) u[e] = ldk_keep<KS>(hp + e * KS);
            return chol_packed<w>(u, dinv);
        }
    }
    // x <- H^-1 x   (ldiv!, :93-96)
    __device__ __forceinline__ void solve(double *x) const {
        if constexpr (SOC) {
        } else if constexpr (HESS == LQRB_HESS_DIAG) {
            SM_UNROLL
            for (int i = 0; i < w; ++i) x[i] *= dinv[i];
        } else if constexpr (HESS == LQRB_HESS_BLOCKDIAG) {
            solve_chol<n>(u, dinv, x);
            if constexpr (mk > 0) solve_chol<mk>(u + tri(n), dinv + n, x + n);
        } else {
            solve_chol<w>(u, dinv, x);
        }
    }
    // Hxx = (H^-1)[0:n,0:n], packed symmetric
    __device__ __forceinline__ void inv_xx(double *Hxx) const {
        if constexpr (SOC) {
            SM_UNROLL
            for (int j = 0; j < n; ++j)
                SM_UNROLL
                for (int i = 0; i <= j; ++i) Hxx[tri_idx(i, j)] = (i == j) ? 1.0 : 0.0;
        } else if constexpr (HESS == LQRB_HESS_DIAG) {
            SM_UNROLL
            for (int j = 0; j < n; ++j)
                SM_UNROLL
                for (int i = 0; i <= j; ++i) Hxx[tri_idx(i, j)] = (i == j) ? dinv[i] : 0.0;
        } else {
            SM_UNROLL
            for (int j = 0; j < n; ++j) {
                double e[w];
                SM_UNROLL
                for (int i = 0; i < w; ++i) e[i] = (i == j) ? 1.0 : 0.0;
                solve(e);
                SM_UNROLL
                for (int i = 0; i <= j; ++i) Hxx[tri_idx(i, j)] = e[i];
            }
        }
    }
};

// state carried from knot k to knot k+1 in the forward sweep
template <int n>
struct FwdCarry {
    double Cp[tri(n)];  // pending C_k = G_k[2,2] - F^'F^ - E^'E^   (+ G_{k+1}[1,1] next)
    double dp[n];       // pending d_k = rho2 - d - F^'lam~ - E^'mu~ (+ rho1_{k+1} next)
};

// Block row k of the factor, everything that depends only on knot k's data and on (A^ = C^_{k-1},
// lam~_{k-1}):   F^ = A^-T F,  D^ = A^-T D,  B^ = chol(B - D^'D^),  E^ = B^-T (E - D^'F^),
//                mu~ = B^-T (c - D^'lam~_{k-1})            (src/cholesky_solve.jl:47-67, :93-117)
// with F = D2*WD = -WD[0:n,:], D = D2*WC = -WC[0:n,:], B = C*WC, E = C*WD  (shur!/copy_shur!,
// src/jacobian_blocks.jl:231-286).  The forward sweep (FWD) also needs G22 = D1*WD and rho2 = D1*hg - d
// to start the next row; the backward sweep calls the same code again instead of reading the row back
// from HBM (the record keeps only C^_{k-1} and lam~_{k-1}).
template <int n, int mk, int p1, int ps, int p2, int HESS, bool SOC, bool FWD>
struct RowFactor {
    static constexpr int w = n + mk;
    double Fh[p1 * p2 + 1];
    double Bh[tri(ps) + 1], Bhinv[ps + 1], Dh[p1 * ps + 1], Eh[ps * p2 + 1], mut[ps + 1];
    double G22[FWD ? tri(p2) + 1 : 1], rho2[FWD ? p2 + 1 : 1];

    template <int KS = 32>
    __device__ __forceinline__ int compute(const double *__restrict__ kp, const HFactor<n, mk, HESS, SOC> &H,
                                           const double *hg, const double *Ah, const double *Ahinv,
                                           const double *lamp) {
        using KR = KnotRows<n, mk, ps, p2, HESS>;
        int info = 0;
        double WD[w * p2 + 1];  // H^-1 D1'   (w x p2, column j = H^-1 * row j of D1)
        if constexpr (p2 > 0) {
            double D1[p2 * w];
            SM_UNROLL
            for (int e = 0; e < p2 * w; ++e) D1[e] = ldk_keep<KS>(kp + (KR::oD1 + e) * KS);
            SM_UNROLL
            for (int j = 0; j < p2; ++j) {
                SM_UNROLL
                for (int i = 0; i < w; ++i) WD[i + j * w] = D1[j + i * p2];
                H.solve(WD + j * w);
            }
            if constexpr (FWD) {
                SM_UNROLL
                for (int j = 0; j < p2; ++j)
                    SM_UNROLL
                    for (int i = 0; i <= j; ++i) {
                        double s = 0.0;
                        SM_UNROLL
                        for (int l = 0; l < w; ++l) s = fma(D1[i + l * p2], WD[l + j * w], s);
                        G22[tri_idx(i, j)] = s;
                    }
                SM_UNROLL
                for (int i = 0; i < p2; ++i) {
                    double s = -ldk_stream<KS>(kp + (KR::od + i) * KS);  // d = r_[3] - d  (copy_shur! :285)
                    SM_UNROLL
                    for (int l = 0; l < w; ++l) s = fma(D1[i + l * p2], hg[l], s);
                    rho2[i] = s;
                }
            }
            if constexpr (p1 > 0) {
                SM_UNROLL
                for (int j = 0; j < p2; ++j) {
                    SM_UNROLL
                    for (int i = 0; i < p1; ++i) Fh[i + j * p1] = -WD[i + j * w];
                    solve_ut<p1>(Ah, Ahinv, Fh + j * p1);  // tri_solve!(U.A, U.F, 'U', 'T')
                }
            }
        }
        if constexpr (ps > 0) {
            double Cc[ps * w], WC[w * ps];
            SM_UNROLL
            for (int e = 0; e < ps * w; ++e) Cc[e] = ldk_keep<KS>(kp + (KR::oC + e) * KS);
            SM_UNROLL
            for (int j = 0; j < ps; ++j) {
                SM_UNROLL
                for (int i = 0; i < w; ++i) WC[i + j * w] = Cc[j + i * ps];
                H.solve(WC + j * w);
            }
            SM_UNROLL
            for (int j = 0; j < ps; ++j)
                SM_UNROLL
                for (int i = 0; i <= j; ++i) {
                    double s = 0.0;
                    SM_UNROLL
                    for (int l = 0; l < w; ++l) s = fma(Cc[i + l * ps], WC[l + j * w], s);
                    Bh[tri_idx(i, j)] = s;  // B = YYt[ips,ips]
                }
            SM_UNROLL
            for (int i = 0; i < ps; ++i) {
                double s = -ldk_stream<KS>(kp + (KR::oc + i) * KS);  // c = r_[2] - c  (:284)
                SM_UNROLL
                for (int l = 0; l < w; ++l) s = fma(Cc[i + l * ps], hg[l], s);
                mut[i] = s;
            }
            if constexpr (p2 > 0) {  // E = C*WD  (ps x p2)
                SM_UNROLL
                for (int j = 0; j < p2; ++j)
                    SM_UNROLL
                    for (int i = 0; i < ps; ++i) {
                        double s = 0.0;
                        SM_UNROLL
                        for (int l = 0; l < w; ++l) s = fma(Cc[i + l * ps], WD[l + j * w], s);
                        Eh[i + j * ps] = s;
                    }
            }
            if constexpr (p1 > 0) {  // D = D2*WC = -WC[0:n,:];  D^ = A^-T D
                SM_UNROLL
                for (int j = 0; j < ps; ++j) {
                    SM_UNROLL
                    for (int i = 0; i < p1; ++i) Dh[i + j * p1] = -WC[i + j * w];
                    solve_ut<p1>(Ah, Ahinv, Dh + j * p1);
                }
                SM_UNROLL
                for (int j = 0; j < ps; ++j)  // B -= D^'D^
                    SM_UNROLL
                    for (int i = 0; i <= j; ++i) {
                        double s = Bh[tri_idx(i, j)];
                        SM_UNROLL
                        for (int l = 0; l < p1; ++l) s = fma(-Dh[l + i * p1], Dh[l + j * p1], s);
                        Bh[tri_idx(i, j)] = s;
                    }
                SM_UNROLL
                for (int i = 0; i < ps; ++i) {  // c - D^'lam~_{k-1}
                    double s = mut[i];
                    SM_UNROLL
                    for (int l = 0; l < p1; ++l) s = fma(-Dh[l + i * p1], lamp[l], s);
                    mut[i] = s;
                }
                if constexpr (p2 > 0) {  // E -= D^'F^
                    SM_UNROLL
                    for (int j = 0; j < p2; ++j)
                        SM_UNROLL
                        for (int i = 0; i < ps; ++i) {
                            double s = Eh[i + j * ps];
                            SM_UNROLL
                            for (int l = 0; l < p1; ++l) s = fma(-Dh[l + i * p1], Fh[l + j * p1], s);
                            Eh[i + j * ps] = s;
                        }
                }
            }
            const int st = chol_packed<ps>(Bh, Bhinv);  // chol!(U.B)
            if (st) info = 100 + st;
            solve_ut<ps>(Bh, Bhinv, mut);               // mu~_k
            if constexpr (p2 > 0) {
                SM_UNROLL
                for (int j = 0; j < p2; ++j) solve_ut<ps>(Bh, Bhinv, Eh + j * ps);  // E^ = B^-T E
            }
        }
        return info;
    }
};

// rows of one knot's record in the scratch array: C^_{k-1} (diag = reciprocals) | lam~_{k-1}
template <int p1>
struct RecRows2 {
    static constexpr int oC = 0, ol = tri(p1), ROWS = ol + p1;
};

// The code a sweep reports, given the one so far and a later knot's: the first failure, except that a Hessian failure
// (stage 0; pivots < 100 at these sizes) takes precedence over a Schur-block one, since the reference factors every H_k
// before any Schur block (src/cholesky_solver.jl:166-182).
__device__ __forceinline__ int kkt_first_failure(int st, int later) {
    const bool hess = st != 0 && st % 1000 < 100, later_hess = later != 0 && later % 1000 < 100;
    return (st == 0 || (later_hess && !hess)) ? later : st;
}

// ------------------------------------------------------------------ forward knot --------------
template <int n, int mk, int p1, int ps, int p2, int HESS, bool SOC, int KS = 32>
__device__ __forceinline__ int kkt_fwd_knot(const double *__restrict__ kp, double *__restrict__ rec,
                                            FwdCarry<n> &cy, int knot) {
    using KR = KnotRows<n, mk, ps, p2, HESS>;
    using RR = RecRows2<p1>;
    constexpr int w = n + mk;
    int info = 0;

    HFactor<n, mk, HESS, SOC> H;
    {
        const int st = H.template load_factor<KS>(kp + KR::oH * KS);
        if (st) info = (knot + 1) * 1000 + st;
    }
    double hg[w];  // H^-1 g  (shur!: r = Y H^-1 g, src/jacobian_blocks.jl:236)
    if constexpr (SOC) {
        SM_UNROLL
        for (int i = 0; i < w; ++i) hg[i] = 0.0;
    } else {
        SM_UNROLL
        for (int i = 0; i < w; ++i) hg[i] = ldk_stream<KS>(kp + (KR::oG + i) * KS);
        H.solve(hg);
    }

    // ---- finish block row k-1: C_{k-1} += G_k[1,1]; d_{k-1} += rho1_k; factor; forward-substitute
    double Ah[tri(p1) + 1], Ahinv[p1 + 1], lamp[p1 + 1];
    if constexpr (p1 > 0) {
        double Hxx[tri(n)];
        H.inv_xx(Hxx);
        SM_UNROLL
        for (int e = 0; e < tri(n); ++e) Ah[e] = cy.Cp[e] + Hxx[e];  // res.A .+= YYt[ip1,ip1]
        SM_UNROLL
        for (int i = 0; i < n; ++i) lamp[i] = cy.dp[i] - hg[i];      // d += next.r_[1], r_[1] = -H^-1g[x]
        const int st = chol_packed<p1>(Ah, Ahinv);                   // chol!(U.C) of row k-1
        if (st && !info) info = knot * 1000 + 200 + st;
        solve_ut<p1>(Ah, Ahinv, lamp);                               // lam~_{k-1}
        SM_UNROLL
        for (int j = 0; j < p1; ++j)
            SM_UNROLL
            for (int i = 0; i <= j; ++i)
                rec[(RR::oC + tri_idx(i, j)) * 32] = (i == j) ? Ahinv[i] : Ah[tri_idx(i, j)];
        SM_UNROLL
        for (int i = 0; i < p1; ++i) rec[(RR::ol + i) * 32] = lamp[i];
    }

    RowFactor<n, mk, p1, ps, p2, HESS, SOC, true> R;
    {
        const int st = R.template compute<KS>(kp, H, hg, Ah, Ahinv, lamp);
        if (st && !info) info = (knot + 1) * 1000 + st;
    }

    // ---- pending C_k, d_k for the next knot to finish
    if constexpr (p2 > 0) {
        SM_UNROLL
        for (int j = 0; j < p2; ++j)
            SM_UNROLL
            for (int i = 0; i <= j; ++i) {
                double s = R.G22[tri_idx(i, j)];
                if constexpr (p1 > 0) {
                    SM_UNROLL
                    for (int l = 0; l < p1; ++l) s = fma(-R.Fh[l + i * p1], R.Fh[l + j * p1], s);
                }
                if constexpr (ps > 0) {
                    SM_UNROLL
                    for (int l = 0; l < ps; ++l) s = fma(-R.Eh[l + i * ps], R.Eh[l + j * ps], s);
                }
                cy.Cp[tri_idx(i, j)] = s;
            }
        SM_UNROLL
        for (int i = 0; i < p2; ++i) {
            double s = R.rho2[i];
            if constexpr (p1 > 0) {
                SM_UNROLL
                for (int l = 0; l < p1; ++l) s = fma(-R.Fh[l + i * p1], lamp[l], s);
            }
            if constexpr (ps > 0) {
                SM_UNROLL
                for (int l = 0; l < ps; ++l) s = fma(-R.Eh[l + i * ps], R.mut[l], s);
            }
            cy.dp[i] = s;
        }
    }
    return info;
}

// ------------------------------------------------------------------ backward knot -------------
// lam holds lam'_k (un-negated back-substitution value) on entry and lam'_{k-1} on exit.
// RS: stride between the record rows (32 = packed tile in global memory, 1 = a thread-local copy)
template <int n, int mk, int p1, int ps, int p2, int HESS, bool SOC, int KS = 32, int RS = 32>
__device__ __forceinline__ void kkt_bwd_knot(const double *__restrict__ kp,
                                             const double *__restrict__ rec, double *lam,
                                             double *__restrict__ dz, double *__restrict__ mult_mu,
                                             double *__restrict__ mult_lprev,
                                             double *__restrict__ res_out, double *dz_reg = nullptr,
                                             double *mult_inf = nullptr) {
    using KR = KnotRows<n, mk, ps, p2, HESS>;
    using RR = RecRows2<p1>;
    constexpr int w = n + mk;

    HFactor<n, mk, HESS, SOC> H;
    H.template load_factor<KS>(kp + KR::oH * KS);
    double g[w], hg[w];
    SM_UNROLL
    for (int i = 0; i < w; ++i) {
        g[i] = SOC ? 0.0 : ldk_stream<KS>(kp + (KR::oG + i) * KS);
        hg[i] = g[i];
    }
    if constexpr (ps > 0) H.solve(hg);  // only mu~ needs H^-1 g here

    // C^_{k-1} and lam~_{k-1} come back from the record; the rest of row k is recomputed
    double Ah[tri(p1) + 1], Ahinv[p1 + 1], lamp[p1 + 1];
    if constexpr (p1 > 0) {
        SM_UNROLL
        for (int j = 0; j < p1; ++j)
            SM_UNROLL
            for (int i = 0; i <= j; ++i) {
                const double v = rec[(RR::oC + tri_idx(i, j)) * RS];
                if (i == j) Ahinv[i] = v;
                Ah[tri_idx(i, j)] = v;
            }
        SM_UNROLL
        for (int i = 0; i < p1; ++i) lamp[i] = rec[(RR::ol + i) * RS];
    }
    RowFactor<n, mk, p1, ps, p2, HESS, SOC, false> R;
    R.template compute<KS>(kp, H, hg, Ah, Ahinv, lamp);

    // mu'_k = B^-1 (mu~ - E^ lam'_k)      (backward_substitution! :130-134)
    double mu[ps + 1];
    if constexpr (ps > 0) {
        SM_UNROLL
        for (int i = 0; i < ps; ++i) {
            double s = R.mut[i];
            if constexpr (p2 > 0) {
                SM_UNROLL
                for (int l = 0; l < p2; ++l) s = fma(-R.Eh[i + l * ps], lam[l], s);
            }
            mu[i] = s;
        }
        solve_un<ps>(R.Bh, R.Bhinv, mu);
    }
    // lam'_{k-1} = C^_{k-1}^-1 (lam~_{k-1} - D^ mu'_k - F^ lam'_k)   (:127-129)
    double lprev[p1 + 1];
    if constexpr (p1 > 0) {
        SM_UNROLL
        for (int i = 0; i < p1; ++i) {
            double s = lamp[i];
            if constexpr (ps > 0) {
                SM_UNROLL
                for (int l = 0; l < ps; ++l) s = fma(-R.Dh[i + l * p1], mu[l], s);
            }
            if constexpr (p2 > 0) {
                SM_UNROLL
                for (int l = 0; l < p2; ++l) s = fma(-R.Fh[i + l * p1], lam[l], s);
            }
            lprev[i] = s;
        }
        solve_un<p1>(Ah, Ahinv, lprev);
    }
    // multipliers (negated, :140-141): mu_k and lam_{k-1}
    SM_UNROLL
    for (int i = 0; i < ps; ++i) __stcs(mult_mu + i * 32, -mu[i]);
    SM_UNROLL
    for (int i = 0; i < p1; ++i) __stcs(mult_lprev + i * 32, -lprev[i]);
    if (mult_inf) {  // running ||Lambda||_inf for the caller's merit penalty
        SM_UNROLL
        for (int i = 0; i < ps; ++i) *mult_inf = fmax(*mult_inf, fabs(mu[i]));
        SM_UNROLL
        for (int i = 0; i < p1; ++i) *mult_inf = fmax(*mult_inf, fabs(lprev[i]));
    }

    // res_k = D1'lam_k + C'mu_k + D2'lam_{k-1} + g_k  (calc_residual! :201-236), with the final
    // (negated) multipliers; D2 = [-I 0].
    double z[w];
    SM_UNROLL
    for (int j = 0; j < w; ++j) {
        double s = g[j];
        if constexpr (p2 > 0) {
            SM_UNROLL
            for (int i = 0; i < p2; ++i) s = fma(-ldk_keep<KS>(kp + (KR::oD1 + i + j * p2) * KS), lam[i], s);
        }
        if constexpr (ps > 0) {
            SM_UNROLL
            for (int i = 0; i < ps; ++i) s = fma(-ldk_keep<KS>(kp + (KR::oC + i + j * ps) * KS), mu[i], s);
        }
        if constexpr (p1 > 0) {
            if (j < n) s += lprev[j];  // D2' lam_{k-1} = -(-lam'_{k-1})
        }
        z[j] = s;
    }
    if (res_out) {
        SM_UNROLL
        for (int j = 0; j < w; ++j) __stcs(res_out + j * 32, z[j]);
    }
    // dz_k = -H_k^-1 res_k   (calc_primals! :195-199)
    H.solve(z);
    SM_UNROLL
    for (int j = 0; j < w; ++j) __stcs(dz + j * 32, -z[j]);
    if (dz_reg) {
        SM_UNROLL
        for (int j = 0; j < w; ++j) dz_reg[j] = -z[j];
    }
    if constexpr (p1 > 0) {
        SM_UNROLL
        for (int i = 0; i < p1; ++i) lam[i] = lprev[i];
    }
}

// ------------------------------------------------------------------ kernel --------------------
// stage-constraint pattern: p[0] = P1, p[1..N-2] = PM, p[N-1] = PN.
template <int n, int m, int P1, int PM, int PN, int HESS>
struct KktLayout {
    using KF = KnotRows<n, m, P1, n, HESS>;
    using KM = KnotRows<n, m, PM, n, HESS>;
    using KL = KnotRows<n, 0, PN, 0, HESS>;
    using RF = RecRows2<0>;
    using RM = RecRows2<n>;
    using RL = RecRows2<n>;
    __host__ __device__ static constexpr int64_t data_rows(int N) {
        return KF::ROWS + (int64_t)(N - 2) * KM::ROWS + KL::ROWS;
    }
    __host__ __device__ static constexpr int64_t rec_rows(int N) {
        return RF::ROWS + (int64_t)(N - 2) * RM::ROWS + RL::ROWS;
    }
    __host__ __device__ static constexpr int64_t mult_rows(int N) {
        return P1 + PN + (int64_t)(N - 2) * PM + (int64_t)(N - 1) * n;
    }
    __host__ __device__ static constexpr int64_t z_rows(int N) { return (int64_t)N * n + (int64_t)(N - 1) * m; }
};

// Launch bound: for w = n+m <= 5 ask for 8 CTAs of 64 threads per SM (<= 128 registers, 16 warps/SM):
// measured on B200 (262,144 Dubins instances) 6.42 -> 6.20 ms, cartpole 1.29 -> 1.05 ms; the kernel is
// DRAM-bound, so residency beats the few spilled bytes.  Larger sizes keep all 255 registers.
template <int n, int m, int P1, int PM, int PN, int HESS, bool SOC, int THREADS>
__global__ void __launch_bounds__(THREADS, (n + m <= 5) ? 8 : 1)
    kkt_tpi_kernel(const double *__restrict__ data, double *__restrict__ scratch,
                   double *__restrict__ dz, double *__restrict__ mult, double *__restrict__ res,
                   int32_t *__restrict__ info, int N, int64_t batch) {
    using L = KktLayout<n, m, P1, PM, PN, HESS>;
    const int64_t inst = (int64_t)blockIdx.x * THREADS + threadIdx.x;
    if (inst >= batch) return;
    const int64_t tile = inst >> 5;
    const int lane = (int)(inst & 31);
    const double *db = data + tile * L::data_rows(N) * 32 + lane;
    double *sb = scratch + tile * L::rec_rows(N) * 32 + lane;
    double *zb = dz + tile * L::z_rows(N) * 32 + lane;
    double *mb = mult + tile * L::mult_rows(N) * 32 + lane;
    double *rb = res ? res + tile * L::z_rows(N) * 32 + lane : nullptr;

    // ---------------- forward sweep
    FwdCarry<n> cy;
    int st = kkt_fwd_knot<n, m, 0, P1, n, HESS, SOC>(db, sb, cy, 0);
    for (int k = 1; k < N - 1; ++k) {
        const int s2 = kkt_fwd_knot<n, m, n, PM, n, HESS, SOC>(
            db + ((int64_t)L::KF::ROWS + (int64_t)(k - 1) * L::KM::ROWS) * 32,
            sb + ((int64_t)L::RF::ROWS + (int64_t)(k - 1) * L::RM::ROWS) * 32, cy, k);
        st = kkt_first_failure(st, s2);
    }
    const int64_t dlast = (int64_t)L::KF::ROWS + (int64_t)(N - 2) * L::KM::ROWS;
    const int64_t rlast = (int64_t)L::RF::ROWS + (int64_t)(N - 2) * L::RM::ROWS;
    {
        const int s2 = kkt_fwd_knot<n, 0, n, PN, 0, HESS, SOC>(db + dlast * 32, sb + rlast * 32, cy, N - 1);
        st = kkt_first_failure(st, s2);
    }
    if (info) info[inst] = st;

    // ---------------- backward sweep
    double lam[n];
    // mult rows: [mu_0 (P1); lam_0 (n); mu_1 (PM); lam_1; ...; mu_{N-1} (PN)]
    const int64_t mlast = (int64_t)P1 + n + (int64_t)(N - 2) * (PM + n);
    const int64_t zlast = (int64_t)(N - 1) * (n + m);
    kkt_bwd_knot<n, 0, n, PN, 0, HESS, SOC>(db + dlast * 32, sb + rlast * 32, lam, zb + zlast * 32,
                                            mb + mlast * 32, mb + (mlast - n) * 32,
                                            rb ? rb + zlast * 32 : nullptr);
    for (int k = N - 2; k >= 1; --k) {
        const int64_t mo = (int64_t)P1 + n + (int64_t)(k - 1) * (PM + n);
        const int64_t zo = (int64_t)k * (n + m);
        kkt_bwd_knot<n, m, n, PM, n, HESS, SOC>(
            db + ((int64_t)L::KF::ROWS + (int64_t)(k - 1) * L::KM::ROWS) * 32,
            sb + ((int64_t)L::RF::ROWS + (int64_t)(k - 1) * L::RM::ROWS) * 32, lam, zb + zo * 32,
            mb + mo * 32, mb + (mo - n) * 32, rb ? rb + zo * 32 : nullptr);
    }
    kkt_bwd_knot<n, m, 0, P1, n, HESS, SOC>(db, sb, lam, zb, mb, mb, rb);
}
