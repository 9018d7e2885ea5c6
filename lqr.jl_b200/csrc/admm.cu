// admm.cu — host side of the box-constrained LTI MPC solve by ADMM on the cached Riccati factor (DESIGN §4.12).  The
// cache itself (lqrb_admm_cache_f64) is built in dare.cu, next to the DARE launch it runs.
#include <cmath>
#include <cstdio>

#include "admm_kernels.cuh"

namespace {
constexpr size_t ADMM_SMEM_MAX = 227 * 1024;

template <int G>
int32_t admm_launch(lqrb_context *h, size_t per, int64_t batch, cudaStream_t s, const double *cache, const double *x0,
                    const double *xref, const double *uref, const double *umin, const double *umax, const double *xmin,
                    const double *xmax, double *state, int warm, double *Z, int32_t *iters, double *res,
                    int32_t *info, int n, int m, int N, const lqrb_admm_options_t &o) {
    // one warp per block: as many instances as fit in 227 KB, at most 32 / G
    const int ipb = (int)std::min<size_t>(32 / G, ADMM_SMEM_MAX / per);
    const size_t smem = per * ipb;
    LQRB_CUDA(h, cudaFuncSetAttribute(admm_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    admm_kernel<G><<<(unsigned)((batch + ipb - 1) / ipb), ipb * G, smem, s>>>(
        cache, x0, xref, uref, umin, umax, xmin, xmax, state, warm, Z, iters, res, info, n, m, N, o.max_iter,
        o.eps_pri, o.eps_dual, batch, ipb);
    char nm[64];
    snprintf(nm, sizeof nm, "admm<G=%d>(n=%d)", G, n);
    h->kernel_name = nm;
    LQRB_LAUNCH_CHECK(h, "admm kernel");
    return 0;
}
}  // namespace

extern "C" int32_t lqrb_admm_solve_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, int64_t batch, int32_t flags,
                                       const lqrb_admm_options_t *opts, const double *cache, const double *x0,
                                       const double *xref, const double *uref, const double *umin,
                                       const double *umax, const double *xmin, const double *xmax, double *state,
                                       double *Z, int32_t *iters, double *res, int32_t *info) {
    if (!h) return -1;
    if (n < 1 || n > 32) return lqrb_fail(h, -2, "n out of range [1,32]");
    if (m < 1 || m > n) return lqrb_fail(h, -3, "m out of range [1,n]");
    if (N < 2) return lqrb_fail(h, -4, "N must be >= 2");
    const size_t per = admm_smem_doubles(n, m, N) * sizeof(double);
    if (per > ADMM_SMEM_MAX) return lqrb_fail(h, -4, "N too long: one instance's working set exceeds 227 KB");
    if (batch < 0) return lqrb_fail(h, -5, "batch must be >= 0");
    if (flags & ~LQRB_FLAG_WARM_START) return lqrb_fail(h, -6, "flags other than LQRB_FLAG_WARM_START");
    if ((flags & LQRB_FLAG_WARM_START) && !state) return lqrb_fail(h, -6, "LQRB_FLAG_WARM_START without a state");
    if (!opts || opts->max_iter < 1 || !(opts->eps_pri >= 0.0) || !(opts->eps_dual >= 0.0))
        return lqrb_fail(h, -7, "opts NULL, max_iter < 1, or eps_pri / eps_dual negative or NaN");
    if (!cache) return lqrb_fail(h, -8, "cache is NULL");
    if (!x0) return lqrb_fail(h, -9, "x0 is NULL");
    if (!Z) return lqrb_fail(h, -17, "Z is NULL");
    if (batch == 0) return 0;
    LQRB_CUDA(h, cudaSetDevice(h->device));
    const int warm = (flags & LQRB_FLAG_WARM_START) ? 1 : 0;
    const lqrb_admm_options_t o = *opts;
    const int64_t Kn = N - 1, sx = 8ll * n, su = 8ll * m;
    const int64_t sstate = 16 * Kn * (n + m), sZ = 8 * ((int64_t)N * n + Kn * m);
    return lqrb_for_chunks(
        h, batch, 0,
        {{cache, admm_cache_doubles(n, m) * 8}, {x0, sx}, {xref, sx * N}, {uref, su * Kn}, {umin, su * Kn},
         {umax, su * Kn}, {xmin, sx * Kn}, {xmax, sx * Kn}, {warm ? state : nullptr, sstate}},
        {{state, sstate}, {Z, sZ}, {iters, 4}, {res, 16}, {info, 4}},
        [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
            const double *const *a = (const double *const *)in;
            double *st = (double *)out[0], *z = (double *)out[1], *r = (double *)out[3];
            int32_t *it = (int32_t *)out[2], *inf = (int32_t *)out[4];
            switch (admm_group(n)) {
                case 4:
                    return admm_launch<4>(h, per, cb, lane.stream, a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], st,
                                          warm, z, it, r, inf, n, m, N, o);
                case 8:
                    return admm_launch<8>(h, per, cb, lane.stream, a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], st,
                                          warm, z, it, r, inf, n, m, N, o);
                case 16:
                    return admm_launch<16>(h, per, cb, lane.stream, a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], st,
                                           warm, z, it, r, inf, n, m, N, o);
                default:
                    return admm_launch<32>(h, per, cb, lane.stream, a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], st,
                                           warm, z, it, r, inf, n, m, N, o);
            }
        });
}
