// dare.cu — host side of the batched discrete algebraic Riccati equation and its gradient (DESIGN §4.11), and of the
// ADMM cache built on it (DESIGN §4.12).
#include <cmath>
#include <cstdio>

#include "admm_kernels.cuh"

namespace {
// Launch shape of both kernels, as launch_coop (riccati.cu): a warp per instance, four instances per 128-thread
// block, up to n = 24 (four slices then take at most 111 KB); a CTA of 256 threads per instance above that.  At
// n = 64 one forward slice is 6 n^2 doubles = 192 KB, one gradient slice at (64, 16) 212 KB, both under 227 KB.
constexpr int DARE_WARP_MAX_N = 24;

// every kernel argument after the launch shape is forwarded as given
template <typename... Params, typename... Args>
int32_t dare_launch(lqrb_context *h, const char *what, void (*warp_kern)(Params...), void (*cta_kern)(Params...),
                    size_t per, int n, int64_t batch, cudaStream_t s, Args... args) {
    const bool warp = n <= DARE_WARP_MAX_N;
    auto kern = warp ? warp_kern : cta_kern;
    const size_t smem = warp ? per * 4 : per;
    if (smem > 227 * 1024) return lqrb_fail(h, -2, "n, m too large for the shared-memory DARE kernels");
    LQRB_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned grid = (unsigned)(warp ? (batch + 3) / 4 : batch);
    kern<<<grid, warp ? 128 : 256, smem, s>>>(args...);
    char nm[64];
    snprintf(nm, sizeof nm, "%s<G=%d>(n=%d)", what, warp ? 32 : 256, n);
    h->kernel_name = nm;
    LQRB_LAUNCH_CHECK(h, "dare kernel");
    return 0;
}

int32_t check_dare_dims(lqrb_context *h, int n, int m, int64_t batch) {
    if (!h) return -1;
    if (n < 1 || n > 64) return lqrb_fail(h, -2, "n out of range [1,64]");
    if (m < 1 || m > n) return lqrb_fail(h, -3, "m out of range [1,n]");
    if (batch < 0) return lqrb_fail(h, -4, "batch must be >= 0");
    return 0;
}
}  // namespace

extern "C" int32_t lqrb_dare_f64(lqrb_handle_t h, int32_t n, int32_t m, int64_t batch, const double *A,
                                 const double *B, const double *Q, const double *R, double *P, double *K,
                                 int32_t *iters, int32_t *info) {
    int32_t rc = check_dare_dims(h, n, m, batch);
    if (rc) return rc;
    if (!A) return lqrb_fail(h, -5, "A is NULL");
    if (!B) return lqrb_fail(h, -6, "B is NULL");
    if (!Q) return lqrb_fail(h, -7, "Q is NULL");
    if (!R) return lqrb_fail(h, -8, "R is NULL");
    if (!P && !K) return lqrb_fail(h, -9, "P and K are both NULL");
    if (batch == 0) return 0;
    LQRB_CUDA(h, cudaSetDevice(h->device));
    const int64_t sA = (int64_t)n * n * 8, sB = (int64_t)n * m * 8, sR = (int64_t)m * m * 8;
    const size_t per = dare_smem_doubles(n) * sizeof(double);
    return lqrb_for_chunks(
        h, batch, 0, {{A, sA}, {B, sB}, {Q, sA}, {R, sR}}, {{P, sA}, {K, sB}, {iters, 4}, {info, 4}},
        [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
            const double *const *a = (const double *const *)in;
            return dare_launch(h, "dare", dare_kernel<32, 128>, dare_kernel<256, 256>, per, n, cb, lane.stream, a[0],
                               a[1], a[2], a[3], (double *)out[0], (double *)out[1], (int32_t *)out[2],
                               (int32_t *)out[3], n, m, cb);
        });
}

extern "C" int32_t lqrb_dare_grad_f64(lqrb_handle_t h, int32_t n, int32_t m, int64_t batch, const double *A,
                                      const double *B, const double *R, const double *P, const double *dP,
                                      const double *dK, double *gA, double *gB, double *gQ, double *gR,
                                      int32_t *info) {
    int32_t rc = check_dare_dims(h, n, m, batch);
    if (rc) return rc;
    if (!A) return lqrb_fail(h, -5, "A is NULL");
    if (!B) return lqrb_fail(h, -6, "B is NULL");
    if (!R) return lqrb_fail(h, -7, "R is NULL");
    if (!P) return lqrb_fail(h, -8, "P is NULL");
    if (!dP && !dK) return lqrb_fail(h, -9, "dP and dK are both NULL");
    if (!gA && !gB && !gQ && !gR) return lqrb_fail(h, -11, "every gradient output is NULL");
    if (batch == 0) return 0;
    LQRB_CUDA(h, cudaSetDevice(h->device));
    const int64_t sA = (int64_t)n * n * 8, sB = (int64_t)n * m * 8, sR = (int64_t)m * m * 8;
    const size_t per = dare_grad_smem_doubles(n, m) * sizeof(double);
    return lqrb_for_chunks(
        h, batch, 0, {{A, sA}, {B, sB}, {R, sR}, {P, sA}, {dP, sA}, {dK, sB}},
        {{gA, sA}, {gB, sB}, {gQ, sA}, {gR, sR}, {info, 4}},
        [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
            const double *const *a = (const double *const *)in;
            double *const *g = (double *const *)out;
            return dare_launch(h, "dare_grad", dare_grad_kernel<32, 128>, dare_grad_kernel<256, 256>, per, n, cb,
                               lane.stream, a[0], a[1], a[2], a[3], a[4], a[5], g[0], g[1], g[2], g[3],
                               (int32_t *)out[4], n, m, cb);
        });
}

extern "C" int32_t lqrb_admm_cache_f64(lqrb_handle_t h, int32_t n, int32_t m, int64_t batch, double rho,
                                       const double *A, const double *B, const double *Q, const double *R,
                                       double *cache, int32_t *info) {
    if (!h) return -1;
    if (n < 1 || n > 32) return lqrb_fail(h, -2, "n out of range [1,32]");
    if (m < 1 || m > n) return lqrb_fail(h, -3, "m out of range [1,n]");
    if (batch < 0) return lqrb_fail(h, -4, "batch must be >= 0");
    if (!(rho > 0.0) || !std::isfinite(rho)) return lqrb_fail(h, -5, "rho must be finite and > 0");
    if (!A) return lqrb_fail(h, -6, "A is NULL");
    if (!B) return lqrb_fail(h, -7, "B is NULL");
    if (!Q) return lqrb_fail(h, -8, "Q is NULL");
    if (!R) return lqrb_fail(h, -9, "R is NULL");
    if (!cache) return lqrb_fail(h, -10, "cache is NULL");
    if (batch == 0) return 0;
    LQRB_CUDA(h, cudaSetDevice(h->device));
    const int64_t sA = (int64_t)n * n * 8, sB = (int64_t)n * m * 8, sR = (int64_t)m * m * 8;
    const size_t per = dare_smem_doubles(n) * sizeof(double);
    const size_t cache_smem = 4 * ((size_t)n * n + 2 * n * m + 2 * m * m) * sizeof(double);
    return lqrb_for_chunks(
        h, batch, 0, {{A, sA}, {B, sB}, {Q, sA}, {R, sR}}, {{cache, admm_cache_doubles(n, m) * 8}, {info, 4}},
        [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
            const double *const *a = (const double *const *)in;
            // scratch: Q + rho I | R + rho I | P | K | DARE info
            const size_t nd = (size_t)cb * (2 * n * n + m * m + n * m);
            double *Qt = (double *)lqrb_scratch(h, SCR_ADMM_CACHE, nd * 8 + (size_t)cb * 4, lane.index);
            if (!Qt) return 1000 + (int)cudaErrorMemoryAllocation;
            double *Rt = Qt + cb * n * n, *P = Rt + cb * m * m, *K = P + cb * n * n;
            int32_t *dinfo = (int32_t *)(K + cb * n * m);
            const int64_t total = cb * (n * n + m * m);
            admm_shift_kernel<<<(unsigned)std::min<int64_t>((total + 255) / 256, 4096), 256, 0, lane.stream>>>(
                a[2], a[3], rho, Qt, Rt, n, m, cb);
            LQRB_LAUNCH_CHECK(h, "admm_shift_kernel");
            int32_t rc = dare_launch(h, "dare", dare_kernel<32, 128>, dare_kernel<256, 256>, per, n, cb, lane.stream,
                                     a[0], a[1], (const double *)Qt, (const double *)Rt, P, K, (int32_t *)nullptr,
                                     dinfo, n, m, cb);
            if (rc) return rc;
            LQRB_CUDA(h, cudaFuncSetAttribute(admm_cache_kernel<32, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                              (int)cache_smem));
            admm_cache_kernel<32, 128><<<(unsigned)((cb + 3) / 4), 128, cache_smem, lane.stream>>>(
                a[0], a[1], a[2], a[3], Rt, P, K, dinfo, rho, (double *)out[0], (int32_t *)out[1], n, m, cb);
            h->kernel_name = "admm_cache";
            LQRB_LAUNCH_CHECK(h, "admm_cache_kernel");
            return 0;
        });
}
