// block_cholesky.cu — batched BlockCholesky entry points.
//
// Replaces cholesky!(chol, A, B[, C]) (src/block_cholesky.jl:55-91) and ldiv!(chol, b) / chol \ b
// (:93-101) for a batch of independent M = [A C'; C B] blocks in the reference's own instance-major,
// column-major storage.  Inside the KKT kernels the same three modes run in registers
// (HFactor in kkt_kernels.cuh); these standalone entry points exist so a caller holding
// BlockCholesky / InvertedQuadratic objects (update_cholesky!, :155-159) can swap them in.
// One thread per instance; the matrix is factored in place in global memory (L1-resident, w <= 128).
#include "common.cuh"

__device__ static int potrf_u_inplace(double *a, int k, int lda) {
    for (int j = 0; j < k; ++j) {
        double s = a[j + j * lda];
        for (int l = 0; l < j; ++l) s = fma(-a[l + j * lda], a[l + j * lda], s);
        if (!(s > 0.0)) return j + 1;
        s = sqrt(s);
        a[j + j * lda] = s;
        for (int i = j + 1; i < k; ++i) {
            double t = a[j + i * lda];
            for (int l = 0; l < j; ++l) t = fma(-a[l + j * lda], a[l + i * lda], t);
            a[j + i * lda] = t / s;
        }
    }
    return 0;
}

__global__ void block_cholesky_kernel(const double *__restrict__ A, const double *__restrict__ B,
                                      const double *__restrict__ C, double *__restrict__ M,
                                      int32_t *__restrict__ info, int n, int m, int mode, int64_t batch) {
    const int64_t inst = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= batch) return;
    const int w = n + m;
    const double *Ai = A + inst * (int64_t)n * n, *Bi = B ? B + inst * (int64_t)m * m : nullptr;
    const double *Ci = C ? C + inst * (int64_t)m * n : nullptr;
    double *Mi = M + inst * (int64_t)w * w;
    for (int e = 0; e < w * w; ++e) Mi[e] = 0.0;
    int st = 0;
    if (mode == LQRB_HESS_DIAG) {  // stores the inverse (:82-91)
        for (int i = 0; i < n; ++i) Mi[i + i * w] = 1.0 / Ai[i + i * n];
        for (int i = 0; i < m; ++i) Mi[(n + i) + (n + i) * w] = 1.0 / Bi[i + i * m];
    } else {
        for (int j = 0; j < n; ++j)
            for (int i = 0; i < n; ++i) Mi[i + j * w] = Ai[i + j * n];
        for (int j = 0; j < m; ++j)
            for (int i = 0; i < m; ++i) Mi[(n + i) + (n + j) * w] = Bi[i + j * m];
        if (mode == LQRB_HESS_BLOCKDIAG) {  // two potrf (:69-77)
            st = potrf_u_inplace(Mi, n, w);
            if (!st) {
                st = potrf_u_inplace(Mi + n + n * w, m, w);
                if (st) st += n;
            }
        } else {  // whole-matrix potrf (:55-66)
            if (Ci)
                for (int j = 0; j < n; ++j)
                    for (int i = 0; i < m; ++i) {
                        Mi[(n + i) + j * w] = Ci[i + j * m];
                        Mi[j + (n + i) * w] = Ci[i + j * m];
                    }
            st = potrf_u_inplace(Mi, w, w);
        }
        // like the reference's chol.F.U view, only the upper triangle is meaningful: clear the rest
        for (int j = 0; j < w; ++j)
            for (int i = j + 1; i < w; ++i) Mi[i + j * w] = 0.0;
    }
    if (info) info[inst] = st;
}

__global__ void block_ldiv_kernel(const double *__restrict__ M, double *__restrict__ b, int n, int m,
                                  int mode, int nrhs, int64_t batch) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= batch * nrhs) return;
    const int64_t inst = idx / nrhs;
    const int w = n + m;
    const double *U = M + inst * (int64_t)w * w;
    double *x = b + idx * (int64_t)w;
    if (mode == LQRB_HESS_DIAG) {  // b .*= chol.M.diag (:95-96)
        for (int i = 0; i < w; ++i) x[i] *= U[i + i * w];
        return;
    }
    for (int i = 0; i < w; ++i) {  // U' y = b
        double s = x[i];
        for (int l = 0; l < i; ++l) s = fma(-U[l + i * w], x[l], s);
        x[i] = s / U[i + i * w];
    }
    for (int i = w - 1; i >= 0; --i) {  // U x = y
        double s = x[i];
        for (int l = i + 1; l < w; ++l) s = fma(-U[i + l * w], x[l], s);
        x[i] = s / U[i + i * w];
    }
}

extern "C" int32_t lqrb_block_cholesky_f64(lqrb_handle_t h, int32_t n, int32_t m, int64_t batch,
                                           int32_t mode, const double *A, const double *B,
                                           const double *C, double *M, int32_t *info) {
    if (!h) return -1;
    if (n < 1 || n > 128) return lqrb_fail(h, -2, "n out of range");
    if (m < 0 || n + m > 192) return lqrb_fail(h, -3, "m out of range");
    if (batch < 0) return lqrb_fail(h, -4, "batch < 0");
    if (mode < 0 || mode > 2) return lqrb_fail(h, -5, "bad mode");
    if (!A) return lqrb_fail(h, -6, "A is NULL");
    if (m > 0 && !B) return lqrb_fail(h, -7, "B is NULL");
    if (!M) return lqrb_fail(h, -9, "M is NULL");
    if (batch == 0) return 0;
    LQRB_CUDA(h, cudaSetDevice(h->device));
    const int w = n + m;
    return lqrb_for_chunks(
        h, batch, batch, {{A, (int64_t)n * n * 8}, {B, (int64_t)m * m * 8}, {C, (int64_t)m * n * 8}},
        {{M, (int64_t)w * w * 8}, {info, 4}},
        [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
            block_cholesky_kernel<<<(unsigned)((cb + 63) / 64), 64, 0, lane.stream>>>(
                (const double *)in[0], (const double *)in[1], (const double *)in[2], (double *)out[0], (int32_t *)out[1],
                n, m, mode, cb);
            h->kernel_name = "block_cholesky";
            LQRB_LAUNCH_CHECK(h, "block_cholesky_kernel");
            return 0;
        });
}

extern "C" int32_t lqrb_block_ldiv_f64(lqrb_handle_t h, int32_t n, int32_t m, int64_t batch,
                                       int32_t mode, const double *M, int32_t nrhs, double *b) {
    if (!h) return -1;
    if (n < 1 || n > 128) return lqrb_fail(h, -2, "n out of range");
    if (m < 0 || n + m > 192) return lqrb_fail(h, -3, "m out of range");
    if (batch < 0) return lqrb_fail(h, -4, "batch < 0");
    if (mode < 0 || mode > 2) return lqrb_fail(h, -5, "bad mode");
    if (!M) return lqrb_fail(h, -6, "M is NULL");
    if (nrhs < 0) return lqrb_fail(h, -7, "nrhs < 0");
    if (!b) return lqrb_fail(h, -8, "b is NULL");
    if (batch == 0 || nrhs == 0) return 0;
    LQRB_CUDA(h, cudaSetDevice(h->device));
    const int w = n + m;
    const int64_t bb = (int64_t)w * nrhs * 8;
    // b is updated in place
    return lqrb_for_chunks(h, batch, batch, {{M, (int64_t)w * w * 8}, {b, bb}}, {{b, bb}},
                           [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
                               const int64_t tot = cb * nrhs;
                               block_ldiv_kernel<<<(unsigned)((tot + 63) / 64), 64, 0, lane.stream>>>(
                                   (const double *)in[0], (double *)out[0], n, m, mode, nrhs, cb);
                               h->kernel_name = "block_ldiv";
                               LQRB_LAUNCH_CHECK(h, "block_ldiv_kernel");
                               return 0;
                           });
}
