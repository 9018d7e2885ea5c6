// kkt_wp.cu — launcher of the warp-per-instance tensor-core KKT kernel (kkt_wp_kernels.cuh); size list in kkt_dispatch.cuh.
#include "kkt_dispatch.cuh"
#include "kkt_wp_kernels.cuh"

// warp-per-instance FP64 tensor-core kernel (kkt_wp_kernels.cuh): H^-1 is formed in the kernel, so there is no
// pre-pass and no Hi array (scratch: the records and the conditioning estimates)
template <int n, int m, int HESS>
static int32_t launch_kkt_wp(lqrb_context *h, const KktShape &s, int64_t cb, int soc, const double *data,
                             double *scratch, double *dz, double *mult, double *res, int32_t *info, int32_t **cinfo_out,
                             cudaStream_t st) {
    using RW = kwp::RecW<n>;
    const int N = s.N;
    constexpr int WARPS = 4, MINB = 3;  // 168 registers: 12 warps per SM
    constexpr size_t smem = (size_t)WARPS * kwp::warp_smem_doubles<n, m, HESS>() * sizeof(double);
    const int ps = s.PMAX;
    // uniform interior pattern: offsets are closed forms; else the per-knot tables of the general path
    KktTables tb{};
    if (!s.uniform) {
        int32_t trc = lqrb_kkt_tables(h, n, m, N, s.p, HESS, 0, &tb);
        if (trc) return trc;
    }
    auto kern = kwp::kkt_wp_kernel<n, m, HESS, WARPS, MINB>;
    LQRB_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // scratch: [records: cb x N x REC] [cinfo: cb]
    double *recs = scratch;
    int32_t *cinfo = reinterpret_cast<int32_t *>(recs + (size_t)cb * N * RW::rec(ps));
    kern<<<(unsigned)((cb + WARPS - 1) / WARPS), WARPS * 32, smem, st>>>(
        data, recs, dz, mult, res, info, cinfo, N, cb, soc, ps, s.uniform ? nullptr : tb.p,
        s.uniform ? nullptr : tb.knot_off, s.uniform ? nullptr : tb.mult_off, s.free_final ? 1 : 0);
    LQRB_LAUNCH_CHECK(h, "kkt_wp_kernel");
    *cinfo_out = cinfo;
    char nm[128];
    if (s.uniform)
        snprintf(nm, sizeof nm, "kkt_wp_dmma<%d,%d,p=%d/%d/%d,hess=%d%s>", n, m, n, ps, n, HESS, soc ? ",soc" : "");
    else
        snprintf(nm, sizeof nm, "kkt_wp_dmma<%d,%d,p=%d/per-knot<=%d/%d,hess=%d%s>", n, m, n, ps, n, HESS, soc ? ",soc" : "");
    h->kernel_name = nm;
    return 0;
}

int32_t kkt_wp_chunk(lqrb_context *h, const KktShape &s, int64_t cb, int soc, const double *data, double *scratch,
                     double *dz, double *mult, double *res, int32_t *info, int32_t **cinfo, cudaStream_t st) {
#define X(N_, M_)                                                                                                          \
    if (s.n == N_ && s.m == M_) {                                                                                          \
        if (s.hess == LQRB_HESS_DIAG)                                                                                      \
            return launch_kkt_wp<N_, M_, LQRB_HESS_DIAG>(h, s, cb, soc, data, scratch, dz, mult, res, info, cinfo, st);      \
        if (s.hess == LQRB_HESS_BLOCKDIAG)                                                                                 \
            return launch_kkt_wp<N_, M_, LQRB_HESS_BLOCKDIAG>(h, s, cb, soc, data, scratch, dz, mult, res, info, cinfo, st); \
        return launch_kkt_wp<N_, M_, LQRB_HESS_DENSE>(h, s, cb, soc, data, scratch, dz, mult, res, info, cinfo, st);         \
    }
    KKT_WP_SIZES(X)
#undef X
    return LQRB_NO_KERNEL;
}

size_t kkt_wp_scratch_per_instance(const KktShape &s) {
#define X(N_, M_) \
    if (s.n == N_ && s.m == M_) return (size_t)s.N * kwp::RecW<N_>::rec(s.PMAX) + 1;
    KKT_WP_SIZES(X)
#undef X
    return 0;
}
