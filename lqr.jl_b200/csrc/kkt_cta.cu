// kkt_cta.cu — launcher of the CTA-per-instance tensor-core KKT kernels (kkt_cta_kernels.cuh); size list in kkt_dispatch.cuh.
#include "kkt_dispatch.cuh"
#include "kkt_cta_kernels.cuh"

template <int n, int m, int HESS>
static int32_t launch_kkt_cta(lqrb_context *h, const KktShape &s, int64_t cb, int soc, const double *data,
                              double *scratch, double *dz, double *mult, double *res, int32_t *info, int32_t **cinfo_out,
                              cudaStream_t st) {
    using L = kcta::Lay<n, m, HESS>;
    const int N = s.N, ps = s.PM;
    // the stage-row work areas are allocated only when there are stage rows (config 5b-K keeps its footprint)
    const size_t psm = (size_t)(ps ? L::PREP_TOTAL_ST : L::PREP_TOTAL) * sizeof(double),
                 msm = (size_t)(ps ? L::MAIN_TOTAL_ST : L::MAIN_TOTAL) * sizeof(double);
    auto pk = ps ? kcta::kkt_cta_prep_kernel<n, m, HESS, true> : kcta::kkt_cta_prep_kernel<n, m, HESS, false>;
    auto mk = ps ? kcta::kkt_cta_kernel<n, m, HESS, true> : kcta::kkt_cta_kernel<n, m, HESS, false>;
    LQRB_CUDA(h, cudaFuncSetAttribute(pk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psm));
    LQRB_CUDA(h, cudaFuncSetAttribute(mk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msm));
    // scratch: [records: cb x N x REC] [pre-pass slots: cb x prep_rows] [hinfo: cb] [cinfo: cb]
    double *recs = scratch;
    double *prep = recs + (size_t)cb * N * L::rec(ps);
    int32_t *hinfo = reinterpret_cast<int32_t *>(prep + (size_t)cb * L::prep_rows(N, ps));
    int32_t *cinfo = hinfo + cb;  // conditioning estimates (the "+ 1" double per instance holds both)
    LQRB_CUDA(h, cudaMemsetAsync(hinfo, 0x7f, (size_t)cb * sizeof(int32_t), st));
    LQRB_CUDA(h, cudaMemsetAsync(cinfo, 0, (size_t)cb * sizeof(int32_t), st));
    kcta::kkt_cta_ri_kernel<n, m, HESS><<<(unsigned)((cb * (N - 1) + 7) / 8), 128, 0, st>>>(data, prep, hinfo, N, cb, soc, ps);
    LQRB_LAUNCH_CHECK(h, "kkt_cta_ri_kernel");
    pk<<<(unsigned)(cb * N), L::THREADS, psm, st>>>(data, prep, hinfo, cinfo, N, cb, soc, ps);
    LQRB_LAUNCH_CHECK(h, "kkt_cta_prep_kernel");
    mk<<<(unsigned)cb, L::THREADS, msm, st>>>(data, prep, hinfo, recs, dz, mult, res, info, cinfo, N, cb, soc, ps,
                                              s.free_final ? 1 : 0);
    LQRB_LAUNCH_CHECK(h, "kkt_cta_kernel");
    *cinfo_out = cinfo;
    char nm[128];
    snprintf(nm, sizeof nm, "kkt_cta_dmma<%d,%d,p=%d/%d/%d,hess=%d%s>", n, m, n, ps, n, HESS, soc ? ",soc" : "");
    h->kernel_name = nm;
    return 0;
}

int32_t kkt_cta_chunk(lqrb_context *h, const KktShape &s, int64_t cb, int soc, const double *data, double *scratch,
                      double *dz, double *mult, double *res, int32_t *info, int32_t **cinfo, cudaStream_t st) {
#define X(N_, M_)                                                                                                    \
    if (s.n == N_ && s.m == M_)                                                                                      \
        return s.hess == LQRB_HESS_DIAG                                                                              \
                   ? launch_kkt_cta<N_, M_, LQRB_HESS_DIAG>(h, s, cb, soc, data, scratch, dz, mult, res, info, cinfo, st) \
                   : launch_kkt_cta<N_, M_, LQRB_HESS_BLOCKDIAG>(h, s, cb, soc, data, scratch, dz, mult, res, info, cinfo, st);
    KKT_CTA_SIZES(X)
#undef X
    return LQRB_NO_KERNEL;
}

size_t kkt_cta_scratch_per_instance(const KktShape &s) {
#define X(N_, M_)               \
    if (s.n == N_ && s.m == M_) \
        return (size_t)s.N * kcta::Lay<N_, M_>::rec(s.PMAX) + kcta::Lay<N_, M_>::prep_rows(s.N, s.PMAX) + 1;
    KKT_CTA_SIZES(X)
#undef X
    return 0;
}
