// kkt_coop.cuh — declarations of the cooperative KKT path (kernel in kkt_coop.cu).
#pragma once
#include "common.cuh"

// rows of one knot's factor record (full-storage blocks): B^ | D^ | E^ | F^ | mu~ | C^_{k-1} | lam~_{k-1}
__host__ __device__ inline int64_t kkt_coop_rec_knot_rows(int p1, int ps, int p2) {
    return (int64_t)ps * ps + (int64_t)p1 * ps + (int64_t)ps * p2 + (int64_t)p1 * p2 + ps + (int64_t)p1 * p1 + p1;
}

static inline int64_t kkt_coop_rec_rows(int n, int m, int N, const int32_t *p) {
    int64_t r = 0;
    for (int k = 0; k < N; ++k) r += kkt_coop_rec_knot_rows(k > 0 ? n : 0, p[k], k < N - 1 ? n : 0);
    return r;
}

__host__ __device__ inline size_t kkt_coop_ws_doubles(int n, int m, int P) {
    const size_t w = n + m;
    return w * w + 3 * w + 2 * n * w + P * w + 2 * w * n + w * P + 3 * (size_t)n * n + (size_t)P * P +
           2 * (size_t)n * P + 4 * n + 3 * P + 16;
}

// phase 0: fused solve (default); 1: factor only — calculate_shur_factors! (src/jacobian_blocks.jl:220-229) +
// cholesky!(U, F) (src/cholesky_solve.jl:28-33), the block rows of U stay in `scratch`; 2: forward / backward
// substitution + calculate_primals! with the kept U and the right-hand-side rows `rhs` ([per knot: g | d | c] per
// instance).  `sdump` (phases 0, 1): the unfactored Schur blocks S and h in the record layout (copy_shur_factors!).
struct KktCoopExtra {
    int phase = 0;
    const double *rhs = nullptr;
    double *sdump = nullptr;
    const int32_t *list = nullptr;  // device list of instance indices to process (batch = its length)
    // per-instance strides (doubles) of `data` and `mult` when the arrays belong to a larger layout than this shape's
    // (the re-solve of a free-final-state problem that a tuned kernel ran with a zero goal block); 0: the shape's own
    int64_t data_stride = 0, mult_stride = 0;
};

int32_t launch_kkt_coop(lqrb_context *h, int n, int m, int N, const int32_t *p, int hess, int d2x,
                        int flags, int64_t batch, const double *data, double *scratch, double *dz,
                        double *mult, double *res, int32_t *info, Lane lane,
                        const KktCoopExtra *extra = nullptr);

// device copies of the per-shape tables (cached on the handle): p[N], and N + 1 prefix offsets of the knot records in the
// packed data (T = 1 layout), of the factor records and of the multiplier groups [mu_k; lam_k]
struct KktTables {
    const int32_t *p;
    const int64_t *knot_off, *rec_off, *mult_off;
    int P;  // max p[k]
};
int32_t lqrb_kkt_tables(lqrb_context *h, int n, int m, int N, const int32_t *p, int hess, int d2x, KktTables *out);
