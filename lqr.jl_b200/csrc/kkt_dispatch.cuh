// kkt_dispatch.cuh — what the translation units of the constrained-KKT path share: the shape descriptor, the size
// lists of the tuned kernel families and the family launchers (kkt_tpi.cu, kkt_hw.cu, kkt_wp.cu, kkt_cta.cu — one
// translation unit per family so that they compile in parallel); dispatch and the C ABI are in kkt.cu.
#pragma once
#include <algorithm>
#include <cstdio>
#include <string>
#include <vector>

#include "kkt_coop.cuh"

// default of the `kkt_cond_bits` option: instances whose worst Schur-block pivot ratio reaches 2^bits are solved again
// by the Cholesky-based kernel (see kkt_resolve_ill_conditioned).  Calibrated with tools/stress_scales.py
// (profiles/r2_conditioning_calibration.txt): the error of the explicit-inverse kernels is about 2^bits times that of
// the reference's U'U order; every grid case where they miss 1e-10 while the reference order meets it has bits >= 7,
// the BASELINE configs at their own scaling have bits 2-3.
#define LQRB_KKT_COND_BITS 6

// ------------------------------------------------------------------ size classes --------------
// thread-per-instance instantiations: (n, m, P1, PM, PN) with p = [P1, PM, ..., PM, PN].
//   cartpole (test/problems.jl:58-88): 4,1 init+goal          dubins: 3,2 init+goal (+1 mid row)
//   DoubleIntegrator(3) (test/problems.jl:14-56): 6,3 init, 1 mid row, goal;  D=2: 4,2
#define KKT_TPI_SIZES_A(X) \
    X(4, 1, 4, 0, 4) X(3, 2, 3, 0, 3) X(3, 2, 3, 1, 3) X(2, 1, 2, 0, 2) X(4, 2, 4, 1, 4) X(6, 3, 6, 1, 6)
// the other small shapes (n <= 6, m <= 3), init + goal rows and 0 or 1 stage row per interior knot
#define KKT_TPI_SIZES_B(X)                                                                                          \
    X(4, 2, 4, 0, 4) X(6, 3, 6, 0, 6) X(2, 2, 2, 0, 2) X(2, 2, 2, 1, 2) X(3, 1, 3, 0, 3) X(3, 3, 3, 0, 3) X(3, 3, 3, 1, 3) \
    X(5, 1, 5, 0, 5) X(6, 1, 6, 0, 6)
#define KKT_TPI_SIZES_C(X) \
    X(5, 2, 5, 0, 5) X(5, 2, 5, 1, 5) X(6, 2, 6, 0, 6) X(6, 2, 6, 1, 6) X(4, 3, 4, 0, 4) X(4, 3, 4, 1, 4) X(5, 3, 5, 0, 5) X(5, 3, 5, 1, 5)
// the same shapes without goal rows (p_N = 0: free final state, the MPC form)
#define KKT_TPI_SIZES_D(X)                                                                                          \
    X(4, 1, 4, 0, 0) X(3, 2, 3, 0, 0) X(3, 2, 3, 1, 0) X(2, 1, 2, 0, 0) X(4, 2, 4, 0, 0) X(4, 2, 4, 1, 0) X(6, 3, 6, 0, 0) \
    X(6, 3, 6, 1, 0) X(2, 2, 2, 0, 0) X(2, 2, 2, 1, 0) X(3, 1, 3, 0, 0) X(3, 3, 3, 0, 0) X(3, 3, 3, 1, 0)
#define KKT_TPI_SIZES_E(X)                                                                                          \
    X(5, 1, 5, 0, 0) X(6, 1, 6, 0, 0) X(5, 2, 5, 0, 0) X(5, 2, 5, 1, 0) X(6, 2, 6, 0, 0) X(6, 2, 6, 1, 0) X(4, 3, 4, 0, 0) \
    X(4, 3, 4, 1, 0) X(5, 3, 5, 0, 0) X(5, 3, 5, 1, 0)
#define KKT_TPI_SIZES(X) KKT_TPI_SIZES_A(X) KKT_TPI_SIZES_B(X) KKT_TPI_SIZES_C(X) KKT_TPI_SIZES_D(X) KKT_TPI_SIZES_E(X)

struct KktShape {
    int n, m, N, hess, d2x;
    const int32_t *p;
    bool uniform;  // p = [P1, PM.., PN]
    int P1, PM, PN;
    int PMAX;  // largest interior count
    // set on the padded shape of a problem WITHOUT goal rows (p_N = 0): its last knot carries a zero goal block
    // (PN = n), the tuned kernel leaves mu_N = 0 instead of inverting the (zero) last Schur block
    bool free_final = false;
};

inline KktShape make_shape(int n, int m, int N, const int32_t *p, int hess, int d2x) {
    KktShape s{n, m, N, hess, d2x, p, true, p[0], N > 2 ? p[1] : 0, p[N - 1], 0};
    for (int k = 1; k < N - 1; ++k) {
        if (p[k] != s.PM) s.uniform = false;
        s.PMAX = std::max(s.PMAX, (int)p[k]);
    }
    return s;
}

// half-warp-per-instance instantiations: p = [n, 0, ..., 0, n], block-diagonal Hessian, structural D2
#define KKT_HW_SIZES(X) X(12, 4) X(8, 4)

// warp-per-instance FP64 tensor-core instantiations (kkt_wp_kernels.cuh; same stage pattern)
#define KKT_WP_SIZES(X) X(12, 4) X(8, 4) X(12, 3) X(8, 3) X(12, 2) X(8, 2) X(12, 1) X(8, 1)

// CTA-per-instance FP64 tensor-core instantiations (same stage pattern)
#define KKT_CTA_SIZES(X) X(64, 16) X(48, 16) X(32, 16) X(32, 8) X(24, 16) X(24, 8) X(16, 16) X(16, 8)

struct KktSizes {
    int64_t NN, P, data_rows, rec_rows;
    int64_t sC, sc, sD2;
};

inline KktSizes kkt_sizes(const KktShape &s) {
    KktSizes z{};
    z.NN = lqrb_num_vars(s.n, s.m, s.N);
    z.P = lqrb_num_cons(s.n, s.N, s.p);
    z.data_rows = lqrb_kkt_data_rows(s.n, s.m, s.N, s.p, s.hess, s.d2x);
    for (int k = 0; k < s.N; ++k) {
        const int w = s.n + (k < s.N - 1 ? s.m : 0);
        z.sC += (int64_t)s.p[k] * w;
        z.sc += s.p[k];
        if (k > 0) z.sD2 += (int64_t)s.n * w;
    }
    z.rec_rows = kkt_coop_rec_rows(s.n, s.m, s.N, s.p);  // an upper bound that also fits the TPI records
    return z;
}


// Family launchers.  kkt_launch_tpi runs a whole batch.  The tuned families (kkt_*_chunk) launch one chunk of `cb`
// instances (every pointer at the chunk's first instance, scratch reused by every chunk), name the kernel in
// h->kernel_name and return in *cinfo the chunk's conditioning estimates (device memory inside scratch); the chunk loop
// and the re-solve of ill-conditioned instances are in kkt.cu.  LQRB_NO_KERNEL if no instantiation matches.
// *_scratch_per_instance: doubles of scratch one instance needs (0: not in the size list).
#define LQRB_NO_KERNEL (-12345)
int32_t kkt_launch_tpi(lqrb_context *h, const KktShape &s, int64_t batch, int flags, const double *data, double *scratch,
                       double *dz, double *mult, double *res, int32_t *info, cudaStream_t st);
int32_t kkt_hw_chunk(lqrb_context *h, const KktShape &s, int64_t cb, int soc, const double *data, double *scratch,
                     double *dz, double *mult, double *res, int32_t *info, int32_t **cinfo, cudaStream_t st);
int32_t kkt_wp_chunk(lqrb_context *h, const KktShape &s, int64_t cb, int soc, const double *data, double *scratch,
                     double *dz, double *mult, double *res, int32_t *info, int32_t **cinfo, cudaStream_t st);
int32_t kkt_cta_chunk(lqrb_context *h, const KktShape &s, int64_t cb, int soc, const double *data, double *scratch,
                      double *dz, double *mult, double *res, int32_t *info, int32_t **cinfo, cudaStream_t st);
size_t kkt_hw_scratch_per_instance(const KktShape &s);
size_t kkt_wp_scratch_per_instance(const KktShape &s);
size_t kkt_cta_scratch_per_instance(const KktShape &s);
