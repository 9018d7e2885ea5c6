// riccati.cu — host side of the batched Riccati entry points (dispatch, packing, host-buffer path).
#include <algorithm>
#include <cstdio>

#include "riccati_kernels.cuh"
#include "riccati_dmma_kernels.cuh"
#include "riccati_cta_kernels.cuh"
#include "riccati_grad_kernels.cuh"
#include "riccati_gain_grad_kernels.cuh"

// ------------------------------------------------------------------ routing -------------------
// The sizes with a kernel of their own, by family: Tpi thread per instance (registers only), Dmma warp per instance on
// the FP64 tensor cores (n in {8,12}, m <= 4, even record length), Cta CTA per instance on the tensor cores (large
// state).  The Dmma and Cta entries, in this order, are also the padding targets.
#define RICCATI_SIZES(X)                                                                                              \
    X(Tpi, 2, 1) X(Tpi, 3, 2) X(Tpi, 4, 1) X(Tpi, 4, 2) X(Tpi, 6, 3) X(Tpi, 2, 2) X(Tpi, 3, 1) X(Tpi, 3, 3)           \
    X(Tpi, 4, 3) X(Tpi, 5, 1) X(Tpi, 5, 2) X(Tpi, 5, 3) X(Tpi, 6, 1) X(Tpi, 6, 2)                                     \
    X(Dmma, 8, 1) X(Dmma, 8, 2) X(Dmma, 8, 3) X(Dmma, 8, 4) X(Dmma, 12, 1) X(Dmma, 12, 2) X(Dmma, 12, 3)              \
    X(Dmma, 12, 4)                                                                                                    \
    X(Cta, 16, 8) X(Cta, 16, 16) X(Cta, 24, 8) X(Cta, 24, 16) X(Cta, 32, 8) X(Cta, 32, 16) X(Cta, 48, 16) X(Cta, 64, 16)

namespace {
enum class RiccatiFamily { Tpi, Dmma, Cta, Pad, Coop };
struct RiccatiRoute {
    RiccatiFamily family;
    int n2 = 0, m2 = 0;  // Pad: the tuned size class
};
}  // namespace

// Which kernel family solves (n, m): the only reader of the options that steer the choice.
//   riccati_variant = 2: the cooperative kernel for every shape (the tests' reference); any other value: the default.
//   riccati_pad = 0: a size without a kernel of its own goes to the cooperative kernel instead of being padded.
// The tensor-core kernels and the padded path read the packed records with 16-byte loads: misaligned data goes to
// riccati_tpi or riccati_coop.
static RiccatiRoute riccati_route(const lqrb_context *h, int n, int m, bool data_aligned) {
    if (h->opt("riccati_variant", 0) == 2) return {RiccatiFamily::Coop};
    RiccatiFamily own = RiccatiFamily::Coop;
#define X(F_, N_, M_) \
    if (n == N_ && m == M_) own = RiccatiFamily::F_;
    RICCATI_SIZES(X)
#undef X
    if (own == RiccatiFamily::Tpi || (data_aligned && own != RiccatiFamily::Coop)) return {own};
    if (data_aligned && h->opt("riccati_pad", 1) != 0) {
#define X(F_, N_, M_) \
    if (RiccatiFamily::F_ != RiccatiFamily::Tpi && n <= N_ && m <= M_) return {RiccatiFamily::Pad, N_, M_};
        RICCATI_SIZES(X)
#undef X
    }
    return {RiccatiFamily::Coop};
}

int lqrb_riccati_tile(const lqrb_context *h, int n, int m) {
    return riccati_route(h, n, m, true).family == RiccatiFamily::Tpi ? LQRB_TILE : 1;
}

// ------------------------------------------------------------------ row maps ------------------
// source array ids: 0 A, 1 B, 2 Q, 3 R, 4 q, 5 r, 6 Qf, 7 qf, 8 x0
static std::vector<RowMap> riccati_knot_map(int n, int m, int N, int flags) {
    const int Kn = (flags & LQRB_FLAG_LTI) ? 1 : N - 1;
    std::vector<RowMap> map;
    map.reserve((size_t)Kn * (n * n + n * m + tri(n) + tri(m) + n + m));
    for (int k = 0; k < Kn; ++k) {
        for (int e = 0; e < n * n; ++e) map.push_back({0, k * n * n + e, 0.0});
        for (int e = 0; e < n * m; ++e) map.push_back({1, k * n * m + e, 0.0});
        for (int j = 0; j < n; ++j)
            for (int i = 0; i <= j; ++i) map.push_back({2, k * n * n + i + j * n, 0.0});
        for (int j = 0; j < m; ++j)
            for (int i = 0; i <= j; ++i) map.push_back({3, k * m * m + i + j * m, 0.0});
        for (int e = 0; e < n; ++e) map.push_back({4, k * n + e, 0.0});
        for (int e = 0; e < m; ++e) map.push_back({5, k * m + e, 0.0});
        if (lqrb_riccati_knot_rows(n, m) > n * n + n * m + tri(n) + tri(m) + n + m) map.push_back({-1, 0, 0.0});  // padding
    }
    return map;
}

static std::vector<RowMap> riccati_term_map(int n) {
    std::vector<RowMap> map;
    for (int j = 0; j < n; ++j)
        for (int i = 0; i <= j; ++i) map.push_back({6, i + j * n, 0.0});
    for (int e = 0; e < n; ++e) map.push_back({7, e, 0.0});
    for (int e = 0; e < n; ++e) map.push_back({8, e, 0.0});
    return map;
}

// The adjoint problem of lqrb_riccati_grad_f64: the forward A, B, Q, R with q̂_k, r̂_k taken from dZ, always packed as
// LTV (q̂ varies per knot; under LTI every knot points at record 0 of A, B, Q, R).
// source array ids: 0 A, 1 B, 2 Q, 3 R, 4 dZ, 6 Qf
static std::vector<RowMap> riccati_adjoint_knot_map(int n, int m, int N, int flags) {
    const bool lti = (flags & LQRB_FLAG_LTI) != 0;
    std::vector<RowMap> map;
    map.reserve((size_t)(N - 1) * lqrb_riccati_knot_rows(n, m));
    for (int k = 0; k < N - 1; ++k) {
        const int kk = lti ? 0 : k, z = k * (n + m);
        for (int e = 0; e < n * n; ++e) map.push_back({0, kk * n * n + e, 0.0});
        for (int e = 0; e < n * m; ++e) map.push_back({1, kk * n * m + e, 0.0});
        for (int j = 0; j < n; ++j)
            for (int i = 0; i <= j; ++i) map.push_back({2, kk * n * n + i + j * n, 0.0});
        for (int j = 0; j < m; ++j)
            for (int i = 0; i <= j; ++i) map.push_back({3, kk * m * m + i + j * m, 0.0});
        for (int e = 0; e < n; ++e) map.push_back({4, z + e, 0.0});
        for (int e = 0; e < m; ++e) map.push_back({4, z + n + e, 0.0});
        if (lqrb_riccati_knot_rows(n, m) > n * n + n * m + tri(n) + tri(m) + n + m) map.push_back({-1, 0, 0.0});  // padding
    }
    return map;
}

// Qf | q̂f = dZ[x_{N-1}] | x̂0 = 0
static std::vector<RowMap> riccati_adjoint_term_map(int n, int m, int N) {
    std::vector<RowMap> map;
    for (int j = 0; j < n; ++j)
        for (int i = 0; i <= j; ++i) map.push_back({6, i + j * n, 0.0});
    for (int e = 0; e < n; ++e) map.push_back({4, (N - 1) * (n + m) + e, 0.0});
    for (int e = 0; e < n; ++e) map.push_back({-1, 0, 0.0});
    return map;
}

// gains packed rows -> K (array 0), kff (array 1)
static std::vector<RowMap> riccati_gain_map(int n, int m, int N) {
    std::vector<RowMap> map;
    for (int k = 0; k < N - 1; ++k) {
        for (int e = 0; e < m * n; ++e) map.push_back({0, k * m * n + e, 0.0});
        for (int e = 0; e < m; ++e) map.push_back({1, k * m + e, 0.0});
    }
    return map;
}

static std::string key(const char *tag, int a, int b, int c, int d) {
    char buf[96];
    snprintf(buf, sizeof buf, "%s:%d:%d:%d:%d", tag, a, b, c, d);
    return buf;
}

static int32_t check_dims(lqrb_context *h, int n, int m, int N, int64_t batch) {
    if (!h) return -1;
    if (n < 1 || n > 128) return lqrb_fail(h, -2, "n out of range [1,128]");
    if (m < 1 || m > n) return lqrb_fail(h, -3, "m out of range [1,n]");
    if (N < 2) return lqrb_fail(h, -4, "N must be >= 2");
    if (batch < 0) return lqrb_fail(h, -5, "batch must be >= 0");
    return 0;
}

// ------------------------------------------------------------------ solve (packed, device) ----
// Launch shapes.  The headline batch (65,536 = 2,048 warps) must fit in ONE wave: 148 SMs x 16 warps
// = 2,368 resident warps needs <= 128 registers per thread (ncu, round 1: at 154 registers only 12
// warps/SM fit -> 1.15 waves and a tail that ran at 1/7 occupancy).  Small sizes take the tight
// bound (64 threads x 8 CTAs); the register-heavy sizes keep the loose one (128 x 1).
template <int n, int m>
static int32_t launch_tpi(lqrb_context *h, int N, int64_t batch, int lti, const double *knots,
                          const double *term, double *Z, double *gains, int32_t *info,
                          cudaStream_t s) {
    constexpr bool SMALL = (n * n + n * m) <= 20;
    constexpr int THREADS = SMALL ? 64 : 128, MINB = SMALL ? 8 : 1;
    const unsigned grid = (unsigned)((batch + THREADS - 1) / THREADS);
    if (lti) riccati_tpi_kernel<n, m, true, THREADS, MINB><<<grid, THREADS, 0, s>>>(knots, term, Z, gains, info, N, batch);
    else riccati_tpi_kernel<n, m, false, THREADS, MINB><<<grid, THREADS, 0, s>>>(knots, term, Z, gains, info, N, batch);
    char nm[64];
    snprintf(nm, sizeof nm, "riccati_tpi<%d,%d>%s%s", n, m, lti ? "[lti]" : "", SMALL ? "[64x8]" : "[128x1]");
    h->kernel_name = nm;
    LQRB_LAUNCH_CHECK(h, "riccati_tpi_kernel");
    return 0;
}

static int32_t launch_coop(lqrb_context *h, int n, int m, int N, int64_t batch, int lti,
                           const double *knots, const double *term, double *Z, double *gains,
                           int32_t *info, cudaStream_t s) {
    const size_t per = riccati_coop_smem_doubles(n, m) * sizeof(double);
    char nm[64];
    if (n + m <= 24) {
        constexpr int G = 32, THREADS = 128;
        const size_t smem = per * (THREADS / G);
        auto kern = riccati_coop_kernel<G, THREADS>;
        LQRB_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const unsigned grid = (unsigned)((batch + THREADS / G - 1) / (THREADS / G));
        kern<<<grid, THREADS, smem, s>>>(knots, term, Z, gains, info, n, m, N, lti, batch);
        snprintf(nm, sizeof nm, "riccati_coop<G=32>(n=%d,m=%d)", n, m);
    } else {
        constexpr int G = 256, THREADS = 256;
        if (per > 227 * 1024) return lqrb_fail(h, -2, "n,m too large for the shared-memory Riccati kernel");
        auto kern = riccati_coop_kernel<G, THREADS>;
        LQRB_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)per));
        kern<<<(unsigned)batch, THREADS, per, s>>>(knots, term, Z, gains, info, n, m, N, lti, batch);
        snprintf(nm, sizeof nm, "riccati_coop<G=256>(n=%d,m=%d)", n, m);
    }
    h->kernel_name = nm;
    LQRB_LAUNCH_CHECK(h, "riccati_coop_kernel");
    return 0;
}

template <int n, int m>
static int32_t launch_dmma(lqrb_context *h, int N, int64_t batch, int lti, const double *knots,
                           const double *term, double *Z, double *gains, int32_t *info,
                           cudaStream_t s) {
    // 3 stages x 4 warps: 34 KB per CTA -> 6 CTAs = 24 warps per SM (<= 85 registers per thread).  m >= 2 takes 5
    // CTAs = 20 warps (<= 102 registers): the LDL' of the control block needs more live values, and at 85 registers
    // it spilled in the knot loop (5a-R +6 %); with 5 CTAs nothing spills and 5a-R is as fast as before.
    constexpr int STAGES = 3, WARPS = 4, MINB = m == 1 ? 6 : 5;
    const size_t smem = rdmma::riccati_dmma_warp_smem(rdmma::Map<n, m>::F, STAGES) * WARPS;
    auto kern = rdmma::riccati_dmma_kernel<n, m, STAGES, WARPS, MINB>;
    LQRB_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned grid = (unsigned)((batch + WARPS - 1) / WARPS);
    kern<<<grid, WARPS * 32, smem, s>>>(knots, term, Z, gains, info, N, lti, batch);
    char nm[64];
    snprintf(nm, sizeof nm, "riccati_dmma<%d,%d>%s", n, m, lti ? "[lti]" : "");
    h->kernel_name = nm;
    LQRB_LAUNCH_CHECK(h, "riccati_dmma_kernel");
    return 0;
}

template <int n, int m>
static int32_t launch_cta(lqrb_context *h, int N, int64_t batch, int lti, const double *knots,
                          const double *term, double *Z, double *gains, int32_t *info, cudaStream_t s) {
    using C = rcta::Cfg<n, m>;
    auto kern = rcta::riccati_cta_kernel<n, m>;
    LQRB_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
    kern<<<(unsigned)batch, C::THREADS, C::SMEM, s>>>(knots, term, Z, gains, info, N, lti, batch);
    char nm[64];
    snprintf(nm, sizeof nm, "riccati_cta_dmma<%d,%d>%s", n, m, lti ? "[lti]" : "");
    h->kernel_name = nm;
    LQRB_LAUNCH_CHECK(h, "riccati_cta_kernel");
    return 0;
}

template <RiccatiFamily F, int n, int m>
static int32_t launch_sized(lqrb_context *h, int N, int64_t batch, int lti, const double *knots, const double *term,
                            double *Z, double *gains, int32_t *info, cudaStream_t s) {
    if constexpr (F == RiccatiFamily::Tpi) return launch_tpi<n, m>(h, N, batch, lti, knots, term, Z, gains, info, s);
    else if constexpr (F == RiccatiFamily::Dmma) return launch_dmma<n, m>(h, N, batch, lti, knots, term, Z, gains, info, s);
    else return launch_cta<n, m>(h, N, batch, lti, knots, term, Z, gains, info, s);
}

// the kernel of a (family, n, m) entry of RICCATI_SIZES
static int32_t launch_tuned(lqrb_context *h, RiccatiFamily family, int n, int m, int N, int64_t batch, int lti,
                            const double *knots, const double *term, double *Z, double *gains, int32_t *info,
                            cudaStream_t s) {
#define X(F_, N_, M_)                                                     \
    if (family == RiccatiFamily::F_ && n == N_ && m == M_)                \
        return launch_sized<RiccatiFamily::F_, N_, M_>(h, N, batch, lti, knots, term, Z, gains, info, s);
    RICCATI_SIZES(X)
#undef X
    return lqrb_fail(h, 1, "no tuned Riccati kernel for this size");
}

// ------------------------------------------------------------------ padding into a tuned size class ----
// A size without a tensor-core kernel of its own (n = 7, 9..11, 13.., or m > 4 at n <= 12, ...) is embedded in the next
// tuned size class (n2, m2): pad states with A = 0, B = 0, Q = Qf = I, x0 = 0 and pad controls with R = I stay exactly
// zero and leave the original recursion untouched.  The packed arrays are expanded on the device, the tuned kernel runs,
// Z and the gains are compacted back.

namespace {
struct RiccatiPadMaps {
    std::vector<RowMap> knots, term, z, gains;
};
}

static RiccatiPadMaps riccati_pad_maps(int n, int m, int N, int Kn, int n2, int m2) {
    RiccatiPadMaps M;
    const int F = lqrb_riccati_knot_rows(n, m), F2 = lqrb_riccati_knot_rows(n2, m2);
    const int nn = n * n, nm = n * m, tn = tri(n), tm = tri(m);
    for (int k = 0; k < Kn; ++k) {
        const int32_t b = k * F;
        const size_t start = M.knots.size();
        for (int j = 0; j < n2; ++j)  // A' = blkdiag(A, 0)
            for (int i = 0; i < n2; ++i) M.knots.push_back((i < n && j < n) ? RowMap{0, b + i + j * n, 0.0} : RowMap{-1, 0, 0.0});
        for (int j = 0; j < m2; ++j)  // B' = [B 0; 0 0]
            for (int i = 0; i < n2; ++i)
                M.knots.push_back((i < n && j < m) ? RowMap{0, b + nn + i + j * n, 0.0} : RowMap{-1, 0, 0.0});
        for (int j = 0; j < n2; ++j)  // Q' = blkdiag(Q, I), upper packed
            for (int i = 0; i <= j; ++i)
                M.knots.push_back(j < n ? RowMap{0, b + nn + nm + j * (j + 1) / 2 + i, 0.0} : RowMap{-1, 0, i == j ? 1.0 : 0.0});
        for (int j = 0; j < m2; ++j)  // R' = blkdiag(R, I)
            for (int i = 0; i <= j; ++i)
                M.knots.push_back(j < m ? RowMap{0, b + nn + nm + tn + j * (j + 1) / 2 + i, 0.0} : RowMap{-1, 0, i == j ? 1.0 : 0.0});
        for (int i = 0; i < n2; ++i) M.knots.push_back(i < n ? RowMap{0, b + nn + nm + tn + tm + i, 0.0} : RowMap{-1, 0, 0.0});
        for (int i = 0; i < m2; ++i) M.knots.push_back(i < m ? RowMap{0, b + nn + nm + tn + tm + n + i, 0.0} : RowMap{-1, 0, 0.0});
        while (M.knots.size() - start < (size_t)F2) M.knots.push_back(RowMap{-1, 0, 0.0});  // record padding
    }
    for (int j = 0; j < n2; ++j)  // Qf' = blkdiag(Qf, I)
        for (int i = 0; i <= j; ++i) M.term.push_back(j < n ? RowMap{0, j * (j + 1) / 2 + i, 0.0} : RowMap{-1, 0, i == j ? 1.0 : 0.0});
    for (int i = 0; i < n2; ++i) M.term.push_back(i < n ? RowMap{0, tn + i, 0.0} : RowMap{-1, 0, 0.0});
    for (int i = 0; i < n2; ++i) M.term.push_back(i < n ? RowMap{0, tn + n + i, 0.0} : RowMap{-1, 0, 0.0});
    // outputs: rows of the padded arrays -> offsets in the original ones (skipped when pad)
    for (int k = 0; k < N; ++k) {
        for (int i = 0; i < n2; ++i) M.z.push_back(i < n ? RowMap{0, k * (n + m) + i, 0.0} : RowMap{-1, 0, 0.0});
        if (k < N - 1)
            for (int i = 0; i < m2; ++i) M.z.push_back(i < m ? RowMap{0, k * (n + m) + n + i, 0.0} : RowMap{-1, 0, 0.0});
    }
    const int GR = m * n + m;
    for (int k = 0; k < N - 1; ++k) {
        for (int j = 0; j < n2; ++j)
            for (int c = 0; c < m2; ++c) M.gains.push_back((c < m && j < n) ? RowMap{0, k * GR + c + m * j, 0.0} : RowMap{-1, 0, 0.0});
        for (int c = 0; c < m2; ++c) M.gains.push_back(c < m ? RowMap{0, k * GR + m * n + c, 0.0} : RowMap{-1, 0, 0.0});
    }
    return M;
}

static int32_t riccati_solve_padded(lqrb_context *h, int n, int m, int N, int n2, int m2, int64_t batch, int flags,
                                    const double *knots, const double *term, double *Z, double *gains, int32_t *info,
                                    Lane lane) {
    const RiccatiFamily family = riccati_route(h, n2, m2, true).family;
    if (family != RiccatiFamily::Dmma && family != RiccatiFamily::Cta)
        return lqrb_fail(h, 1, "padded Riccati size has no tensor-core kernel");
    const int lti = (flags & LQRB_FLAG_LTI) ? 1 : 0;
    const int Kn = lti ? 1 : N - 1;
    const int64_t F = lqrb_riccati_knot_rows(n, m), F2 = lqrb_riccati_knot_rows(n2, m2);
    const int64_t TR = tri(n) + 2 * n, TR2 = tri(n2) + 2 * n2;
    const int64_t ZR = (int64_t)N * n + (int64_t)(N - 1) * m, ZR2 = (int64_t)N * n2 + (int64_t)(N - 1) * m2;
    const int64_t GR = (int64_t)(N - 1) * (m * n + m), GR2 = (int64_t)(N - 1) * (m2 * n2 + m2);
    const std::string k0 = key("rpad", n, m, N, Kn) + key("->", n2, m2, 0, 0);
    DevMap mk, mt, mz, mg;
    if (h->maps.find(k0 + ":g") == h->maps.end()) {
        const RiccatiPadMaps M = riccati_pad_maps(n, m, N, Kn, n2, m2);
        mk = lqrb_get_map(h, k0 + ":k", M.knots);
        mt = lqrb_get_map(h, k0 + ":t", M.term);
        mz = lqrb_get_map(h, k0 + ":z", M.z);
        mg = lqrb_get_map(h, k0 + ":g", M.gains);
    } else {
        mk = h->maps[k0 + ":k"];
        mt = h->maps[k0 + ":t"];
        mz = h->maps[k0 + ":z"];
        mg = h->maps[k0 + ":g"];
    }
    if (mk.rows != Kn * F2 || mt.rows != TR2 || mz.rows != ZR2 || mg.rows != GR2) return lqrb_fail(h, 1, "pad map size mismatch");
    // chunks of at most ~2 GB of padded arrays
    const int64_t per = Kn * F2 + TR2 + ZR2 + GR2;
    int64_t chunk = std::max<int64_t>(LQRB_TILE, ((int64_t)2 << 30) / (per * 8) / LQRB_TILE * LQRB_TILE);
    chunk = std::min(chunk, lqrb_padded_batch(batch));
    const size_t slice = ((size_t)chunk * per * 8 + 255) / 256 * 256;
    char *base = (char *)lqrb_scratch(h, SCR_RICCATI_PAD, slice, lane.index);
    if (!base) return 1000 + (int)cudaErrorMemoryAllocation;
    double *knots2 = (double *)base, *term2 = knots2 + chunk * Kn * F2, *Z2 = term2 + chunk * TR2, *gains2 = Z2 + chunk * ZR2;
    std::string name;
    for (int64_t first = 0; first < batch; first += chunk) {
        const int64_t cb = std::min(chunk, batch - first);
        ArrayTable src = {};
        src.ptr[0] = knots + first * Kn * F;
        src.stride[0] = Kn * F;
        int32_t rc = lqrb_gather_pack(h, mk, src, cb, 1, knots2, lane.stream);
        if (rc) return rc;
        src.ptr[0] = term + first * TR;
        src.stride[0] = TR;
        rc = lqrb_gather_pack(h, mt, src, cb, 1, term2, lane.stream);
        if (rc) return rc;
        rc = launch_tuned(h, family, n2, m2, N, cb, lti, knots2, term2, Z2, gains2, info ? info + first : nullptr,
                          lane.stream);
        if (rc) return rc;
        name = h->kernel_name;
        ArrayTableOut o = {};
        o.ptr[0] = Z + first * ZR;
        o.stride[0] = ZR;
        rc = lqrb_scatter_unpack(h, mz, o, cb, 1, Z2, lane.stream);
        if (rc) return rc;
        o.ptr[0] = gains + first * GR;
        o.stride[0] = GR;
        rc = lqrb_scatter_unpack(h, mg, o, cb, 1, gains2, lane.stream);
        if (rc) return rc;
    }
    char nm[64];
    snprintf(nm, sizeof nm, " <- (%d,%d) padded", n, m);
    h->kernel_name = name + nm;
    return 0;
}

static int32_t riccati_solve_on(lqrb_context *h, int n, int m, int N, int64_t batch, int flags,
                                const double *knots, const double *term, double *Z, double *gains,
                                int32_t *info, Lane lane) {
    if (batch == 0) return 0;
    const RiccatiRoute r = riccati_route(h, n, m, ((uintptr_t)knots & 15) == 0);
    const int lti = (flags & LQRB_FLAG_LTI) ? 1 : 0;
    switch (r.family) {
    case RiccatiFamily::Pad:
        return riccati_solve_padded(h, n, m, N, r.n2, r.m2, batch, flags, knots, term, Z, gains, info, lane);
    case RiccatiFamily::Tpi:
    case RiccatiFamily::Dmma:
    case RiccatiFamily::Cta:
        return launch_tuned(h, r.family, n, m, N, batch, lti, knots, term, Z, gains, info, lane.stream);
    case RiccatiFamily::Coop:
        break;
    }
    return launch_coop(h, n, m, N, batch, lti, knots, term, Z, gains, info, lane.stream);
}

extern "C" int32_t lqrb_riccati_solve_packed_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N,
                                                 int64_t batch, int32_t flags, const double *knots,
                                                 const double *term, double *Z, double *gains,
                                                 int32_t *info) {
    int32_t rc = check_dims(h, n, m, N, batch);
    if (rc) return rc;
    if (!knots) return lqrb_fail(h, -7, "knots is NULL");
    if (!term) return lqrb_fail(h, -8, "term is NULL");
    if (!Z) return lqrb_fail(h, -9, "Z is NULL");
    LQRB_CUDA(h, cudaSetDevice(h->device));
    if (!gains) {
        const size_t bytes = (size_t)lqrb_padded_batch(batch) * (N - 1) * (m * n + m) * sizeof(double);
        gains = (double *)lqrb_scratch(h, SCR_GAINS, bytes);
        if (!gains) return 1000 + (int)cudaErrorMemoryAllocation;
    }
    return riccati_solve_on(h, n, m, N, batch, flags, knots, term, Z, gains, info, Lane{h->stream, 0});
}

// ------------------------------------------------------------------ pack (device) -------------
static int32_t riccati_pack_on(lqrb_context *h, int n, int m, int N, int64_t batch, int flags,
                               const double *A, const double *B, const double *Q, const double *R,
                               const double *q, const double *r, const double *Qf, const double *qf,
                               const double *x0, double *knots, double *term, cudaStream_t s) {
    const int Kn = (flags & LQRB_FLAG_LTI) ? 1 : N - 1;
    const int tile = lqrb_riccati_tile(h, n, m);
    ArrayTable t = {};
    const double *ptrs[9] = {A, B, Q, R, q, r, Qf, qf, x0};
    const int64_t strides[9] = {(int64_t)Kn * n * n, (int64_t)Kn * n * m, (int64_t)Kn * n * n,
                                (int64_t)Kn * m * m, (int64_t)Kn * n,     (int64_t)Kn * m,
                                (int64_t)n * n,      n,                   n};
    for (int i = 0; i < 9; ++i) {
        t.ptr[i] = ptrs[i];
        t.stride[i] = strides[i];
    }
    DevMap km = lqrb_get_map(h, key("rk", n, m, N, flags & LQRB_FLAG_LTI), riccati_knot_map(n, m, N, flags));
    DevMap tm = lqrb_get_map(h, key("rt", n, 0, 0, 0), riccati_term_map(n));
    int32_t rc = lqrb_gather_pack(h, km, t, batch, tile, knots, s);
    if (rc) return rc;
    return lqrb_gather_pack(h, tm, t, batch, tile, term, s);
}

extern "C" int32_t lqrb_riccati_pack_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N,
                                         int64_t batch, int32_t flags, const double *A,
                                         const double *B, const double *Q, const double *R,
                                         const double *q, const double *r, const double *Qf,
                                         const double *qf, const double *x0, double *knots,
                                         double *term) {
    int32_t rc = check_dims(h, n, m, N, batch);
    if (rc) return rc;
    if (!A) return lqrb_fail(h, -7, "A is NULL");
    if (!B) return lqrb_fail(h, -8, "B is NULL");
    if (!Q) return lqrb_fail(h, -9, "Q is NULL");
    if (!R) return lqrb_fail(h, -10, "R is NULL");
    if (!Qf) return lqrb_fail(h, -13, "Qf is NULL");
    if (!x0) return lqrb_fail(h, -15, "x0 is NULL");
    if (!knots) return lqrb_fail(h, -16, "knots is NULL");
    if (!term) return lqrb_fail(h, -17, "term is NULL");
    LQRB_CUDA(h, cudaSetDevice(h->device));
    return riccati_pack_on(h, n, m, N, batch, flags, A, B, Q, R, q, r, Qf, qf, x0, knots, term, h->stream);
}

// ------------------------------------------------------------------ unpack helpers ------------
static int32_t riccati_unpack_on(lqrb_context *h, int n, int m, int N, int64_t batch,
                                 const double *Zp, const double *gains, double *Z, double *K,
                                 double *kff, cudaStream_t s) {
    const int tile = lqrb_riccati_tile(h, n, m);
    const int64_t NN = lqrb_num_vars(n, m, N);
    ArrayTableOut t = {};
    t.ptr[0] = Z;
    t.stride[0] = NN;
    int32_t rc = lqrb_scatter_unpack(h, lqrb_identity_map(h, NN), t, batch, tile, Zp, s);
    if (rc) return rc;
    if (K || kff) {
        ArrayTableOut g = {};
        g.ptr[0] = K;
        g.stride[0] = (int64_t)(N - 1) * m * n;
        g.ptr[1] = kff;
        g.stride[1] = (int64_t)(N - 1) * m;
        rc = lqrb_scatter_unpack(h, lqrb_get_map(h, key("rg", n, m, N, 0), riccati_gain_map(n, m, N)), g,
                                 batch, tile, gains, s);
    }
    return rc;
}

extern "C" int32_t lqrb_riccati_tile_width(lqrb_handle_t h, int32_t n, int32_t m) {
    if (!h) return -1;
    if (n < 1) return -2;
    if (m < 1) return -3;
    return lqrb_riccati_tile(h, n, m);
}

extern "C" int32_t lqrb_riccati_unpack_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, int64_t batch,
                                           const double *Zp, const double *gains, double *Z, double *K,
                                           double *kff) {
    int32_t rc = check_dims(h, n, m, N, batch);
    if (rc) return rc;
    if (!Zp) return lqrb_fail(h, -6, "packed Z is NULL");
    if ((K || kff) && !gains) return lqrb_fail(h, -7, "K / kff requested but the packed gains are NULL");
    if (!Z) return lqrb_fail(h, -8, "Z is NULL");
    LQRB_CUDA(h, cudaSetDevice(h->device));
    return riccati_unpack_on(h, n, m, N, batch, Zp, gains, Z, K, kff, h->stream);
}

// ------------------------------------------------------------------ full call -----------------
extern "C" int32_t lqrb_riccati_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, int64_t batch,
                                    int32_t flags, const double *A, const double *B, const double *Q,
                                    const double *R, const double *q, const double *r,
                                    const double *Qf, const double *qf, const double *x0, double *Z,
                                    double *K, double *kff, int32_t *info) {
    int32_t rc = check_dims(h, n, m, N, batch);
    if (rc) return rc;
    if (!A) return lqrb_fail(h, -7, "A is NULL");
    if (!B) return lqrb_fail(h, -8, "B is NULL");
    if (!Q) return lqrb_fail(h, -9, "Q is NULL");
    if (!R) return lqrb_fail(h, -10, "R is NULL");
    if (!Qf) return lqrb_fail(h, -13, "Qf is NULL");
    if (!x0) return lqrb_fail(h, -15, "x0 is NULL");
    if (!Z) return lqrb_fail(h, -16, "Z is NULL");
    if (batch == 0) return 0;
    LQRB_CUDA(h, cudaSetDevice(h->device));

    lqrb_riccati_layout_t L;
    lqrb_riccati_layout(n, m, N, flags, &L);
    const int64_t Kn = L.knot_count, NN = L.z_rows, GRN = L.gain_rows;
    // bytes per instance of the instance-major arrays (q, r and qf count when absent too: they fix the chunk size)
    const int64_t sA = Kn * n * n * 8, sB = Kn * n * m * 8, sR = Kn * m * m * 8, sq = Kn * n * 8, sr = Kn * m * 8,
                  sQf = (int64_t)n * n * 8, sx = (int64_t)n * 8;
    return lqrb_for_chunks(
        h, batch, 0, {{A, sA}, {B, sB}, {Q, sA}, {R, sR}, {q, sq}, {r, sr}, {Qf, sQf}, {qf, sx}, {x0, sx}},
        {{Z, NN * 8}, {K, (int64_t)(N - 1) * m * n * 8}, {kff, (int64_t)(N - 1) * m * 8}, {info, 4}},
        [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
            const int64_t ldb = lqrb_padded_batch(cb);
            double *knots = (double *)lqrb_scratch(h, SCR_PACK_IN, (size_t)ldb * Kn * L.rows_per_knot * 8, lane.index);
            double *term = (double *)lqrb_scratch(h, SCR_PACK_IN2, (size_t)ldb * L.term_rows * 8, lane.index);
            double *Zp = (double *)lqrb_scratch(h, SCR_PACK_OUT, (size_t)ldb * NN * 8, lane.index);
            double *gains = (double *)lqrb_scratch(h, SCR_GAINS, (size_t)ldb * GRN * 8, lane.index);
            if (!knots || !term || !Zp || !gains) return 1000 + (int)cudaErrorMemoryAllocation;
            const double *const *a = (const double *const *)in;
            int32_t rc = riccati_pack_on(h, n, m, N, cb, flags, a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], a[8],
                                         knots, term, lane.stream);
            if (rc) return rc;
            rc = riccati_solve_on(h, n, m, N, cb, flags, knots, term, Zp, gains, (int32_t *)out[3], lane);
            if (rc) return rc;
            return riccati_unpack_on(h, n, m, N, cb, Zp, gains, (double *)out[0], (double *)out[1], (double *)out[2],
                                     lane.stream);
        });
}

// ------------------------------------------------------------------ gradient ------------------
template <int G, int R>
static int32_t launch_grad(lqrb_context *h, int n, int m, int N, int64_t batch, bool lti, const RiccatiGradArgs &a,
                           cudaStream_t s) {
    constexpr int THREADS = 128;
    int threads = THREADS;
    size_t smem = 0;
    if (lti) {
        // one accumulator slice per group, fewer groups per block when the slices are large
        const size_t per = (size_t)(2 * n * n + n * m + m * m) * sizeof(double), cap = 227 * 1024;
        if (per > cap) return lqrb_fail(h, -2, "n, m too large for the LTI gradient accumulators");
        const int groups = (int)std::min<size_t>(THREADS / G, cap / per);
        threads = groups * G;
        smem = per * groups;
    }
    const int per_block = threads / G;
    const unsigned grid = (unsigned)((batch + per_block - 1) / per_block);
    if (lti) {
        auto kern = riccati_grad_kernel<G, R, true>;
        LQRB_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, threads, smem, s>>>(a, n, m, N, batch);
    } else {
        riccati_grad_kernel<G, R, false><<<grid, threads, 0, s>>>(a, n, m, N, batch);
    }
    char nm[64];
    snprintf(nm, sizeof nm, "riccati_grad<G=%d,R=%d>%s", G, R, lti ? "[lti]" : "");
    h->kernel_name += std::string(" + ") + nm;
    LQRB_LAUNCH_CHECK(h, "riccati_grad_kernel");
    return 0;
}

// The solve accepts n <= 84 (riccati_coop_kernel's shared memory bounds the sizes without a tuned kernel), so three
// rows per lane cover every size that reaches the sweep.
static int32_t launch_grad_sized(lqrb_context *h, int n, int m, int N, int64_t batch, bool lti,
                                 const RiccatiGradArgs &a, cudaStream_t s) {
    if (n <= 4) return launch_grad<4, 1>(h, n, m, N, batch, lti, a, s);
    if (n <= 8) return launch_grad<8, 1>(h, n, m, N, batch, lti, a, s);
    if (n <= 16) return launch_grad<16, 1>(h, n, m, N, batch, lti, a, s);
    if (n <= 32) return launch_grad<32, 1>(h, n, m, N, batch, lti, a, s);
    if (n <= 64) return launch_grad<32, 2>(h, n, m, N, batch, lti, a, s);
    if (n <= 96) return launch_grad<32, 3>(h, n, m, N, batch, lti, a, s);
    return lqrb_fail(h, -2, "n too large for the Riccati gradient sweep");
}

// Gradient of ℓ(Z) through lqrb_riccati_f64 for one chunk (DESIGN §4.8): the adjoint LQR (same A, B, Q, R, Qf; linear
// terms dZ; x̂0 = 0) is packed and solved by the forward dispatch, its solution unpacked to Ẑ, and one backward sweep
// forms the costates of both problems and every gradient.  `in` holds A, B, Q, R, q, r, Qf, qf, Z, dZ and `out` gA, gB,
// gQ, gR, gq, gr, gQf, gqf, gx0, info, as chunk pointers of lqrb_for_chunks.
static int32_t riccati_grad_chunk(lqrb_context *h, int n, int m, int N, int flags, Lane lane, int64_t cb,
                                  const void *const *in, void *const *out) {
    const bool lti = (flags & LQRB_FLAG_LTI) != 0;
    lqrb_riccati_layout_t L;
    lqrb_riccati_layout(n, m, N, 0, &L);  // the adjoint problem is always packed as LTV
    const int64_t Kn = lti ? 1 : N - 1, NN = L.z_rows;
    const int64_t sA = Kn * n * n, sB = Kn * n * m, sR = Kn * m * m, sQf = (int64_t)n * n;
    const int64_t ldb = lqrb_padded_batch(cb);
    double *knots = (double *)lqrb_scratch(h, SCR_PACK_IN, (size_t)ldb * L.knot_count * L.rows_per_knot * 8, lane.index);
    double *term = (double *)lqrb_scratch(h, SCR_PACK_IN2, (size_t)ldb * L.term_rows * 8, lane.index);
    double *Zp = (double *)lqrb_scratch(h, SCR_PACK_OUT, (size_t)ldb * NN * 8, lane.index);
    double *gains = (double *)lqrb_scratch(h, SCR_GAINS, (size_t)ldb * L.gain_rows * 8, lane.index);
    double *Zh = (double *)lqrb_scratch(h, SCR_ADJOINT_Z, (size_t)cb * NN * 8, lane.index);
    if (!knots || !term || !Zp || !gains || !Zh) return 1000 + (int)cudaErrorMemoryAllocation;
    const double *const *a = (const double *const *)in;
    const int tile = lqrb_riccati_tile(h, n, m);
    ArrayTable t = {};
    const double *ptrs[7] = {a[0], a[1], a[2], a[3], a[9], nullptr, a[6]};
    const int64_t strides[7] = {sA, sB, sA, sR, NN, 0, sQf};
    for (int i = 0; i < 7; ++i) {
        t.ptr[i] = ptrs[i];
        t.stride[i] = strides[i];
    }
    DevMap km = lqrb_get_map(h, key("rak", n, m, N, lti ? 1 : 0), riccati_adjoint_knot_map(n, m, N, flags));
    DevMap tm = lqrb_get_map(h, key("rat", n, m, N, 0), riccati_adjoint_term_map(n, m, N));
    int32_t rc = lqrb_gather_pack(h, km, t, cb, tile, knots, lane.stream);
    if (rc) return rc;
    rc = lqrb_gather_pack(h, tm, t, cb, tile, term, lane.stream);
    if (rc) return rc;
    rc = riccati_solve_on(h, n, m, N, cb, 0, knots, term, Zp, gains, (int32_t *)out[9], lane);
    if (rc) return rc;
    ArrayTableOut o = {};
    o.ptr[0] = Zh;
    o.stride[0] = NN;
    rc = lqrb_scatter_unpack(h, lqrb_identity_map(h, NN), o, cb, tile, Zp, lane.stream);
    if (rc) return rc;
    double *const *g = (double *const *)out;
    // the sweep reads K_k from the adjoint solve's gains (the adjoint problem has the forward A, B, Q, R, Qf, so the
    // same K_k), in the solve's packed layout: tiled for the thread-per-instance family, instance-major otherwise
    const RiccatiGradArgs ga = {a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], a[8], Zh, a[9], gains, tile,
                                g[0], g[1], g[2], g[3], g[4], g[5], g[6], g[7], g[8]};
    return launch_grad_sized(h, n, m, N, cb, lti, ga, lane.stream);
}

extern "C" int32_t lqrb_riccati_grad_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, int64_t batch,
                                         int32_t flags, const double *A, const double *B, const double *Q,
                                         const double *R, const double *q, const double *r, const double *Qf,
                                         const double *qf, const double *Z, const double *dZ, double *gA, double *gB,
                                         double *gQ, double *gR, double *gq, double *gr, double *gQf, double *gqf,
                                         double *gx0, int32_t *info) {
    int32_t rc = check_dims(h, n, m, N, batch);
    if (rc) return rc;
    if (flags & ~(LQRB_FLAG_LTI | LQRB_FLAG_NO_AFFINE)) return lqrb_fail(h, -6, "flags: only LTI and NO_AFFINE apply");
    if (!A) return lqrb_fail(h, -7, "A is NULL");
    if (!B) return lqrb_fail(h, -8, "B is NULL");
    if (!Q) return lqrb_fail(h, -9, "Q is NULL");
    if (!R) return lqrb_fail(h, -10, "R is NULL");
    if (!Qf) return lqrb_fail(h, -13, "Qf is NULL");
    if (!Z) return lqrb_fail(h, -15, "Z is NULL");
    if (!dZ) return lqrb_fail(h, -16, "dZ is NULL");
    if (!gA && !gB && !gQ && !gR && !gq && !gr && !gQf && !gqf && !gx0)
        return lqrb_fail(h, -17, "every gradient output is NULL");
    if (batch == 0) return 0;
    LQRB_CUDA(h, cudaSetDevice(h->device));
    if (flags & LQRB_FLAG_NO_AFFINE) q = r = qf = nullptr;

    const int64_t Kn = (flags & LQRB_FLAG_LTI) ? 1 : N - 1, NN = lqrb_num_vars(n, m, N);
    const int64_t sA = Kn * n * n * 8, sB = Kn * n * m * 8, sR = Kn * m * m * 8, sq = Kn * n * 8, sr = Kn * m * 8,
                  sQf = (int64_t)n * n * 8, sx = (int64_t)n * 8;
    return lqrb_for_chunks(
        h, batch, 0,
        {{A, sA}, {B, sB}, {Q, sA}, {R, sR}, {q, sq}, {r, sr}, {Qf, sQf}, {qf, sx}, {Z, NN * 8}, {dZ, NN * 8}},
        {{gA, sA}, {gB, sB}, {gQ, sA}, {gR, sR}, {gq, sq}, {gr, sr}, {gQf, sQf}, {gqf, sx}, {gx0, sx}, {info, 4}},
        [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
            return riccati_grad_chunk(h, n, m, N, flags, lane, cb, in, out);
        });
}

// ------------------------------------------------------------------ gradient through the gains -----
// Instances per block of riccati_gain_grad_kernel<G>: up to 128 threads, as many groups as their shared-memory slices
// allow, in whole warps; 0 when one warp's groups do not fit.
static int gain_grad_groups(int G, int n, int m) {
    const size_t per = (size_t)gain_grad_smem_doubles(n, m) * sizeof(double), cap = 227 * 1024;
    const int whole = 32 / G;  // groups per warp
    const int groups = (int)std::min<size_t>(128 / G, cap / per) / whole * whole;
    return groups;
}

template <int G, int R>
static int32_t launch_gain_grad(lqrb_context *h, int n, int m, int N, int64_t batch, bool lti,
                                const RiccatiGainGradArgs &a, cudaStream_t s) {
    const int groups = gain_grad_groups(G, n, m);
    if (groups == 0) return lqrb_fail(h, -2, "n, m too large for the gain gradient sweep");
    const size_t smem = (size_t)gain_grad_smem_doubles(n, m) * sizeof(double) * groups;
    const unsigned grid = (unsigned)((batch + groups - 1) / groups);
    auto kern = lti ? riccati_gain_grad_kernel<G, R, true> : riccati_gain_grad_kernel<G, R, false>;
    LQRB_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, groups * G, smem, s>>>(a, n, m, N, batch);
    char nm[64];
    snprintf(nm, sizeof nm, "riccati_gain_grad<G=%d,R=%d>%s", G, R, lti ? "[lti]" : "");
    h->kernel_name = h->kernel_name.empty() ? std::string(nm) : h->kernel_name + " + " + nm;
    LQRB_LAUNCH_CHECK(h, "riccati_gain_grad_kernel");
    return 0;
}

// the lane configuration of riccati_grad_kernel (launch_grad_sized): lanes per instance and rows per lane
static void gain_grad_lanes(int n, int *G, int *R) {
    *G = n <= 4 ? 4 : n <= 8 ? 8 : n <= 16 ? 16 : 32;
    *R = n <= 32 ? 1 : n <= 64 ? 2 : 3;
}

static int32_t launch_gain_grad_sized(lqrb_context *h, int n, int m, int N, int64_t batch, bool lti,
                                      const RiccatiGainGradArgs &a, cudaStream_t s) {
    if (n <= 4) return launch_gain_grad<4, 1>(h, n, m, N, batch, lti, a, s);
    if (n <= 8) return launch_gain_grad<8, 1>(h, n, m, N, batch, lti, a, s);
    if (n <= 16) return launch_gain_grad<16, 1>(h, n, m, N, batch, lti, a, s);
    if (n <= 32) return launch_gain_grad<32, 1>(h, n, m, N, batch, lti, a, s);
    if (n <= 64) return launch_gain_grad<32, 2>(h, n, m, N, batch, lti, a, s);
    if (n <= 96) return launch_gain_grad<32, 3>(h, n, m, N, batch, lti, a, s);
    return lqrb_fail(h, -2, "n too large for the gain gradient sweep");
}

// The code lqrb_riccati_f64 returns for a shape it cannot solve (0 when it can): only the cooperative kernel at
// n + m > 24 has a size limit, its shared memory (launch_coop).
static int32_t riccati_size_code(lqrb_context *h, int n, int m) {
    if (riccati_route(h, n, m, true).family == RiccatiFamily::Coop && n + m > 24 &&
        riccati_coop_smem_doubles(n, m) * sizeof(double) > 227 * 1024)
        return lqrb_fail(h, -2, "n,m too large for the shared-memory Riccati kernel");
    return 0;
}

// Gradient of ℓ(Z, K, kff) through lqrb_riccati_f64 (DESIGN §4.10): the Z part is lqrb_riccati_grad_f64's chunk body
// (or zeroed outputs without dZ), then riccati_gain_grad_kernel recomputes the recursion into a per-knot tape and
// adds the adjoint of the recursion driven by dK, dkff.
extern "C" int32_t lqrb_riccati_grad_gains_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, int64_t batch,
                                               int32_t flags, const double *A, const double *B, const double *Q,
                                               const double *R, const double *q, const double *r, const double *Qf,
                                               const double *qf, const double *Z, const double *dZ, const double *dK,
                                               const double *dkff, double *gA, double *gB, double *gQ, double *gR,
                                               double *gq, double *gr, double *gQf, double *gqf, double *gx0,
                                               int32_t *info) {
    int32_t rc = check_dims(h, n, m, N, batch);
    if (rc) return rc;
    if (flags & ~(LQRB_FLAG_LTI | LQRB_FLAG_NO_AFFINE)) return lqrb_fail(h, -6, "flags: only LTI and NO_AFFINE apply");
    if (!A) return lqrb_fail(h, -7, "A is NULL");
    if (!B) return lqrb_fail(h, -8, "B is NULL");
    if (!Q) return lqrb_fail(h, -9, "Q is NULL");
    if (!R) return lqrb_fail(h, -10, "R is NULL");
    if (!Qf) return lqrb_fail(h, -13, "Qf is NULL");
    if (dZ && !Z) return lqrb_fail(h, -15, "Z is NULL while dZ is given");
    if (!dZ && !dK && !dkff) return lqrb_fail(h, -16, "every cotangent (dZ, dK, dkff) is NULL");
    if (!gA && !gB && !gQ && !gR && !gq && !gr && !gQf && !gqf && !gx0)
        return lqrb_fail(h, -19, "every gradient output is NULL");
    if (batch == 0) return 0;
    LQRB_CUDA(h, cudaSetDevice(h->device));
    if (flags & LQRB_FLAG_NO_AFFINE) q = r = qf = nullptr;
    if (!dZ) Z = nullptr;
    if (!dZ && (rc = riccati_size_code(h, n, m))) return rc;

    const bool lti = (flags & LQRB_FLAG_LTI) != 0;
    const int64_t Kn = lti ? 1 : N - 1, NN = lqrb_num_vars(n, m, N);
    const int64_t sA = Kn * n * n * 8, sB = Kn * n * m * 8, sR = Kn * m * m * 8, sq = Kn * n * 8, sr = Kn * m * 8,
                  sQf = (int64_t)n * n * 8, sx = (int64_t)n * 8;
    const int64_t sK = (int64_t)(N - 1) * m * n * 8, skff = (int64_t)(N - 1) * m * 8;
    int G, Rr;
    gain_grad_lanes(n, &G, &Rr);
    const int groups = std::max(1, gain_grad_groups(G, n, m));
    return lqrb_for_chunks(
        h, batch, 0,
        {{A, sA}, {B, sB}, {Q, sA}, {R, sR}, {q, sq}, {r, sr}, {Qf, sQf}, {qf, sx}, {Z, NN * 8}, {dZ, NN * 8},
         {dK, sK}, {dkff, skff}},
        {{gA, sA}, {gB, sB}, {gQ, sA}, {gR, sR}, {gq, sq}, {gr, sr}, {gQf, sQf}, {gqf, sx}, {gx0, sx}, {info, 4}},
        [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
            int32_t rc = 0;
            h->kernel_name.clear();
            if (dZ) {
                rc = riccati_grad_chunk(h, n, m, N, flags, lane, cb, in, out);
                if (rc) return rc;
            } else {
                const int64_t bytes[10] = {sA, sB, sA, sR, sq, sr, sQf, sx, sx, 4};
                for (int i = 0; i < 10; ++i)
                    if (out[i]) LQRB_CUDA(h, cudaMemsetAsync(out[i], 0, (size_t)(cb * bytes[i]), lane.stream));
            }
            if (!dK && !dkff) return 0;
            const int64_t slots = round_up(cb, groups);  // groups past the batch write a slot of their own
            double *tape = (double *)lqrb_scratch(h, SCR_GAIN_TAPE,
                                                  (size_t)slots * (N - 1) * gain_grad_tape_doubles(n, m) * 8,
                                                  lane.index);
            if (!tape) return 1000 + (int)cudaErrorMemoryAllocation;
            const double *const *a = (const double *const *)in;
            double *const *g = (double *const *)out;
            const RiccatiGainGradArgs ga = {a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], a[10], a[11], tape,
                                            g[0], g[1], g[2], g[3], g[4], g[5], g[6], g[7], (int32_t *)out[9]};
            return launch_gain_grad_sized(h, n, m, N, cb, lti, ga, lane.stream);
        });
}

// ------------------------------------------------------------------ rollout -------------------
// rollout!(X, U) : src/least_squares.jl:195-202, one WARP per instance (n <= 32): lane i owns row i of A_k, B_k, so
// every load of a column of [A B] is one contiguous piece (the instance-major arrays are column-major), x_k and u_k
// travel by shuffle, and X is written as contiguous n-double pieces.  The thread-per-instance kernel below read A
// with a stride of Kn n^2 doubles between lanes (every lane its own 32-byte sector).
__global__ void __launch_bounds__(128)
    rollout_warp_kernel(const double *__restrict__ A, const double *__restrict__ B, const double *__restrict__ x0,
                        const double *__restrict__ U, double *__restrict__ X, int n, int m, int N, int lti,
                        int64_t batch) {
    const int64_t inst = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (inst >= batch) return;
    const int Kn = lti ? 1 : N - 1;
    const double *Ai = A + inst * (int64_t)Kn * n * n, *Bi = B + inst * (int64_t)Kn * n * m;
    const double *Ui = U + inst * (int64_t)(N - 1) * m;
    double *Xi = X + inst * (int64_t)N * n;
    double x = lane < n ? x0[inst * n + lane] : 0.0;
    if (lane < n) Xi[lane] = x;
    double un = lane < m ? Ui[lane] : 0.0;  // u_0, one knot ahead of its use
    for (int k = 0; k < N - 1; ++k) {
        const double *Ak = Ai + (int64_t)(lti ? 0 : k) * n * n, *Bk = Bi + (int64_t)(lti ? 0 : k) * n * m;
        const double u = un;
        if (k + 1 < N - 1) un = lane < m ? Ui[(int64_t)(k + 1) * m + lane] : 0.0;
        double s0 = 0.0, s1 = 0.0;
        for (int l = 0; l + 1 < n; l += 2) {
            const double a0 = lane < n ? Ak[lane + l * n] : 0.0, a1 = lane < n ? Ak[lane + (l + 1) * n] : 0.0;
            s0 = fma(a0, __shfl_sync(0xffffffffu, x, l), s0);
            s1 = fma(a1, __shfl_sync(0xffffffffu, x, l + 1), s1);
        }
        if (n & 1) s0 = fma(lane < n ? Ak[lane + (n - 1) * n] : 0.0, __shfl_sync(0xffffffffu, x, n - 1), s0);
        for (int l = 0; l < m; ++l) s1 = fma(lane < n ? Bk[lane + l * n] : 0.0, __shfl_sync(0xffffffffu, u, l), s1);
        x = s0 + s1;
        if (lane < n) Xi[(int64_t)(k + 1) * n + lane] = x;
    }
}

// the same for n > 32: one thread per instance, the state lives in the output array
__global__ void rollout_kernel(const double *__restrict__ A, const double *__restrict__ B,
                               const double *__restrict__ x0, const double *__restrict__ U,
                               double *__restrict__ X, int n, int m, int N, int lti, int64_t batch) {
    const int64_t inst = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= batch) return;
    const int Kn = lti ? 1 : N - 1;
    const double *Ai = A + inst * (int64_t)Kn * n * n, *Bi = B + inst * (int64_t)Kn * n * m;
    const double *Ui = U + inst * (int64_t)(N - 1) * m;
    double *Xi = X + inst * (int64_t)N * n;
    for (int i = 0; i < n; ++i) Xi[i] = x0[inst * n + i];
    for (int k = 0; k < N - 1; ++k) {
        const double *Ak = Ai + (int64_t)(lti ? 0 : k) * n * n, *Bk = Bi + (int64_t)(lti ? 0 : k) * n * m;
        const double *xk = Xi + (int64_t)k * n, *uk = Ui + (int64_t)k * m;
        double *xn = Xi + (int64_t)(k + 1) * n;
        for (int i = 0; i < n; ++i) {
            double s = 0.0;
            for (int l = 0; l < n; ++l) s = fma(Ak[i + l * n], xk[l], s);
            for (int l = 0; l < m; ++l) s = fma(Bk[i + l * n], uk[l], s);
            xn[i] = s;
        }
    }
}

extern "C" int32_t lqrb_rollout_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, int64_t batch,
                                    int32_t flags, const double *A, const double *B, const double *x0,
                                    const double *U, double *X) {
    int32_t rc = check_dims(h, n, m, N, batch);
    if (rc) return rc;
    if (!A) return lqrb_fail(h, -7, "A is NULL");
    if (!B) return lqrb_fail(h, -8, "B is NULL");
    if (!x0) return lqrb_fail(h, -9, "x0 is NULL");
    if (!U) return lqrb_fail(h, -10, "U is NULL");
    if (!X) return lqrb_fail(h, -11, "X is NULL");
    if (batch == 0) return 0;
    LQRB_CUDA(h, cudaSetDevice(h->device));
    const int lti = (flags & LQRB_FLAG_LTI) ? 1 : 0;
    const int64_t Kn = lti ? 1 : N - 1;
    return lqrb_for_chunks(
        h, batch, batch, {{A, Kn * n * n * 8}, {B, Kn * n * m * 8}, {x0, (int64_t)n * 8}, {U, (int64_t)(N - 1) * m * 8}},
        {{X, (int64_t)N * n * 8}},
        [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
            const double *const *a = (const double *const *)in;
            double *dX = (double *)out[0];
            if (n <= 32) {
                rollout_warp_kernel<<<(unsigned)((cb + 3) / 4), 128, 0, lane.stream>>>(a[0], a[1], a[2], a[3], dX, n, m,
                                                                                       N, lti, cb);
                h->kernel_name = "rollout_warp";
            } else {
                rollout_kernel<<<(unsigned)((cb + 127) / 128), 128, 0, lane.stream>>>(a[0], a[1], a[2], a[3], dX, n, m,
                                                                                      N, lti, cb);
                h->kernel_name = "rollout_tpi";
            }
            LQRB_LAUNCH_CHECK(h, "rollout_kernel");
            return 0;
        });
}
