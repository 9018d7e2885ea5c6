// residual.cu — stationarity residual of the KKT system for GIVEN multipliers.
//
// Replaces residual(solver; recalculate) : src/cholesky_solver.jl:238-252, i.e. calc_residual! (:201-236) on
// the kept multipliers of the last solve and freshly evaluated Jacobians / gradients:
//     res_k = D1_k' lam_k + C_k' mu_k + D2_k' lam_{k-1} + g_k          (g skipped when Ginv = false, :229-231)
//     residual = || ( ||res_k|| )_k ||  =  || res ||_2                 (:246-251)
// This is the feas_d of step! (:126-134).  Fully parallel over (instance, entry of Z): one CTA per instance,
// threads stride over the NN entries, instance-major inputs read in place (no packing — every input is read
// exactly once, column j of a Jacobian block is contiguous).
#include "common.cuh"

#include <vector>

namespace {

struct ResArgs {
    const double *q, *r, *A, *B, *D2, *C, *mult;
    double *res, *norms;
    const int64_t *mo, *co;  // per knot: start of mu_k inside mult, start of C_k inside C
    const int32_t *p;
    int n, m, N, grad;
    int64_t NN, P, sC, sD2, batch;
};

template <int THREADS>
__global__ void __launch_bounds__(THREADS) kkt_residual_kernel(ResArgs a) {
    const int64_t b = blockIdx.x;
    const int n = a.n, m = a.m, N = a.N, w = n + m;
    const double *q = a.q ? a.q + b * (int64_t)n * N : nullptr;
    const double *r = a.r ? a.r + b * (int64_t)m * (N - 1) : nullptr;
    const double *A = a.A + b * (int64_t)n * n * (N - 1);
    const double *B = a.B + b * (int64_t)n * m * (N - 1);
    const double *D2 = a.D2 ? a.D2 + b * a.sD2 : nullptr;
    const double *C = a.C ? a.C + b * a.sC : nullptr;
    const double *mult = a.mult + b * a.P;
    double acc = 0.0;
    for (int64_t e = threadIdx.x; e < a.NN; e += THREADS) {
        const int k = (int)min((int64_t)(N - 1), e / w);
        const int j = (int)(e - (int64_t)k * w);
        const int pk = a.p[k];
        const double *mu = mult + a.mo[k];
        const double *lam = mu + pk;
        double s = 0.0;
        if (a.grad) s = j < n ? q[(int64_t)k * n + j] : r[(int64_t)k * m + (j - n)];
        if (k < N - 1) {  // D1_k = [A_k B_k]
            const double *col = j < n ? A + (int64_t)k * n * n + (int64_t)n * j : B + (int64_t)k * n * m + (int64_t)n * (j - n);
            for (int i = 0; i < n; ++i) s = fma(col[i], lam[i], s);
        }
        if (pk > 0) {
            const int wk = k < N - 1 ? w : n;
            (void)wk;
            const double *col = C + a.co[k] + (int64_t)pk * j;
            for (int i = 0; i < pk; ++i) s = fma(col[i], mu[i], s);
        }
        if (k > 0) {
            const double *lp = mult + a.mo[k - 1] + a.p[k - 1];  // lam_{k-1}
            if (D2) {
                const double *col = D2 + (int64_t)(k - 1) * n * w + (int64_t)n * j;
                for (int i = 0; i < n; ++i) s = fma(col[i], lp[i], s);
            } else if (j < n) {
                s -= lp[j];  // D2 = [-I 0]
            }
        }
        if (a.res) a.res[b * a.NN + e] = s;
        acc = fma(s, s, acc);
    }
    if (a.norms) {
        __shared__ double red[THREADS / 32];
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int i = 0; i < THREADS / 32; ++i) t += red[i];
            a.norms[b] = sqrt(t);
        }
    }
}

}  // namespace

extern "C" int32_t lqrb_kkt_residual_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, int64_t batch,
                                         const int32_t *p, int32_t flags, const double *q, const double *r,
                                         const double *A, const double *B, const double *D2, const double *C,
                                         const double *mult, double *res, double *norms) {
    if (!h) return -1;
    if (n < 1 || n > 128) return lqrb_fail(h, -2, "n out of range [1,128]");
    if (m < 1 || m > n) return lqrb_fail(h, -3, "m out of range [1,n]");
    if (N < 2) return lqrb_fail(h, -4, "N must be >= 2");
    if (batch < 0) return lqrb_fail(h, -5, "batch must be >= 0");
    if (!p) return lqrb_fail(h, -6, "p is NULL");
    for (int k = 0; k < N; ++k)
        if (p[k] < 0 || p[k] > n + m) return lqrb_fail(h, -6, "p[k] out of range [0, n+m]");
    const bool grad = (flags & LQRB_FLAG_SOC) == 0;
    if (grad && (!q || !r)) return lqrb_fail(h, -8, "q/r is NULL (only allowed with LQRB_FLAG_SOC)");
    if (!A || !B) return lqrb_fail(h, -10, "A/B is NULL");
    if (!mult) return lqrb_fail(h, -14, "mult is NULL");
    if (!res && !norms) return lqrb_fail(h, -15, "res and norms are both NULL");
    if (batch == 0) return 0;
    LQRB_CUDA(h, cudaSetDevice(h->device));

    const int w = n + m;
    const int64_t K1 = N - 1, NN = lqrb_num_vars(n, m, N), P = lqrb_num_cons(n, N, p);
    int64_t sC = 0;
    for (int k = 0; k < N; ++k) sC += (int64_t)p[k] * (k < N - 1 ? w : n);
    const int64_t sD2 = K1 > 0 ? (K1 - 1) * (int64_t)n * w + (int64_t)n * n : 0;
    if (sC > 0 && !C) return lqrb_fail(h, -13, "C is NULL but p has non-zero entries");

    // offset tables, cached per shape
    std::string key = "res:" + std::to_string(n) + ":" + std::to_string(m) + ":" + std::to_string(N) + ":";
    for (int k = 0; k < N; ++k) key += std::to_string(p[k]) + ",";
    const size_t off_bytes = (size_t)N * sizeof(int64_t);
    char *blob = nullptr;
    auto it = h->blobs.find(key);
    if (it != h->blobs.end()) {
        blob = (char *)it->second;
    } else {
        std::vector<char> host(2 * off_bytes + (size_t)N * sizeof(int32_t));
        int64_t *mo = (int64_t *)host.data(), *co = mo + N;
        int32_t *pp = (int32_t *)(host.data() + 2 * off_bytes);
        int64_t macc = 0, cacc = 0;
        for (int k = 0; k < N; ++k) {
            mo[k] = macc;
            co[k] = cacc;
            pp[k] = p[k];
            macc += p[k] + (k < N - 1 ? n : 0);
            cacc += (int64_t)p[k] * (k < N - 1 ? w : n);
        }
        void *d = nullptr;
        LQRB_CUDA(h, cudaMalloc(&d, host.size()));
        LQRB_CUDA(h, cudaMemcpy(d, host.data(), host.size(), cudaMemcpyHostToDevice));
        LQRB_CUDA(h, cudaStreamSynchronize(cudaStreamLegacy));  // pageable source: wait for the staged DMA
        h->blobs[key] = d;
        blob = (char *)d;
    }

    ResArgs a{};
    a.mo = (const int64_t *)blob;
    a.co = a.mo + N;
    a.p = (const int32_t *)(blob + 2 * off_bytes);
    a.n = n; a.m = m; a.N = N; a.grad = grad ? 1 : 0;
    a.NN = NN; a.P = P; a.sC = sC; a.sD2 = sD2;
    // bytes per instance; the staged chunks hold about 256 MB of input plus output (or `host_chunk` instances)
    const int64_t per[7] = {grad ? (int64_t)n * N * 8 : 0, grad ? (int64_t)m * K1 * 8 : 0, (int64_t)n * n * K1 * 8,
                            (int64_t)n * m * K1 * 8,       D2 ? sD2 * 8 : 0,               sC * 8, P * 8};
    const double *src[7] = {q, r, A, B, D2, C, mult};
    std::vector<HostArray> inputs(7);
    int64_t io_bytes = (NN + 1) * 8;
    for (int i = 0; i < 7; ++i) {
        inputs[i] = {src[i], per[i]};
        io_bytes += per[i];
    }
    int64_t chunk = h->opt("host_chunk", 0);
    if (chunk <= 0) chunk = std::max<int64_t>(1, (256ll << 20) / io_bytes);
    return lqrb_for_chunks(h, batch, chunk, inputs, {{res, NN * 8}, {norms, 8}},
                           [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
                               constexpr int THREADS = 128;
                               const double *const *d = (const double *const *)in;
                               a.q = d[0]; a.r = d[1]; a.A = d[2]; a.B = d[3]; a.D2 = d[4]; a.C = d[5]; a.mult = d[6];
                               a.res = (double *)out[0];
                               a.norms = (double *)out[1];
                               a.batch = cb;
                               kkt_residual_kernel<THREADS><<<(unsigned)cb, THREADS, 0, lane.stream>>>(a);
                               LQRB_LAUNCH_CHECK(h, "kkt_residual_kernel");
                               h->kernel_name = "kkt_residual";
                               return 0;
                           });
}
