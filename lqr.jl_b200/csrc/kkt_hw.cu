// kkt_hw.cu — launcher of the half-warp-per-instance KKT kernel (kkt_hw_kernels.cuh); size list in kkt_dispatch.cuh.
#include "kkt_dispatch.cuh"
#include "kkt_hw_kernels.cuh"

template <int n, int m, int HESS>
static int32_t launch_kkt_hw(lqrb_context *h, const KktShape &s, int64_t cb, int soc, const double *data,
                             double *scratch, double *dz, double *mult, double *res, int32_t *info, int32_t **cinfo_out,
                             cudaStream_t st) {
    using L = khw::Lay<n, m, HESS>;
    const int N = s.N;
    // Three 4-warp CTAs per SM at 168 registers: eight 2-warp CTAs at 128 registers (16 warps, a few spills) were
    // 3.5 % slower in an A/B on one box (48.95 vs 47.2 ms) — the kernel is not latency-bound.
    constexpr int WARPS = 4, MINB = 3;
    const size_t smem = (size_t)WARPS * (2 * L::INST2 + 4) * sizeof(double);
    auto kern = khw::kkt_hw2_kernel<n, m, HESS, WARPS, MINB>;
    LQRB_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // scratch: [records: cb x N x REC] [Hi: cb x N x HI] [hinfo: cb] [cinfo: cb]
    double *recs = scratch;
    double *hinv = recs + (size_t)cb * N * L::REC;
    int32_t *hinfo = reinterpret_cast<int32_t *>(hinv + (size_t)cb * N * L::HI);
    int32_t *cinfo = hinfo + cb;  // conditioning estimates (the "+ 1" double per instance holds both)
    LQRB_CUDA(h, cudaMemsetAsync(hinfo, 0x7f, (size_t)cb * sizeof(int32_t), st));
    const int64_t total = cb * N;
    khw::kkt_hinv_kernel<n, m, HESS><<<(unsigned)((total + 127) / 128), 128, 0, st>>>(data, hinv, hinfo, N, cb, soc);
    LQRB_LAUNCH_CHECK(h, "kkt_hinv_kernel");
    const int64_t pairs = (cb + 1) / 2;
    kern<<<(unsigned)((pairs + WARPS - 1) / WARPS), WARPS * 32, smem, st>>>(data, hinv, hinfo, recs, dz, mult, res, info,
                                                                            cinfo, N, cb, soc);
    LQRB_LAUNCH_CHECK(h, "kkt_hw_kernel");
    *cinfo_out = cinfo;
    char nm[128];
    snprintf(nm, sizeof nm, "kkt_hw<%d,%d,p=%d/0/%d,hess=%d%s>", n, m, n, n, HESS, soc ? ",soc" : "");
    h->kernel_name = nm;
    return 0;
}

int32_t kkt_hw_chunk(lqrb_context *h, const KktShape &s, int64_t cb, int soc, const double *data, double *scratch,
                     double *dz, double *mult, double *res, int32_t *info, int32_t **cinfo, cudaStream_t st) {
#define X(N_, M_)                                                                                                   \
    if (s.n == N_ && s.m == M_)                                                                                     \
        return s.hess == LQRB_HESS_DIAG                                                                             \
                   ? launch_kkt_hw<N_, M_, LQRB_HESS_DIAG>(h, s, cb, soc, data, scratch, dz, mult, res, info, cinfo, st) \
                   : launch_kkt_hw<N_, M_, LQRB_HESS_BLOCKDIAG>(h, s, cb, soc, data, scratch, dz, mult, res, info, cinfo, st);
    KKT_HW_SIZES(X)
#undef X
    return LQRB_NO_KERNEL;
}

size_t kkt_hw_scratch_per_instance(const KktShape &s) {
#define X(N_, M_) \
    if (s.n == N_ && s.m == M_) return (size_t)s.N * (khw::Lay<N_, M_>::REC + khw::Lay<N_, M_>::HI) + 1;
    KKT_HW_SIZES(X)
#undef X
    return 0;
}
