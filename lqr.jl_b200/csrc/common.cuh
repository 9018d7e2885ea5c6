// common.cuh — shared host/device helpers of liblqrb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <functional>
#include <map>
#include <string>
#include <vector>

#include "../../include/lqrb200.h"

// ------------------------------------------------------------------ packed layout -------------
// Every device-resident array is "tiled batch-minor": [tile][row][T] doubles, where a tile holds T
// consecutive instances.  T = 32 for the thread-per-instance kernels (a warp reads one row of its
// tile as one 256-byte line, and a whole knot of a tile is ONE contiguous chunk that a single
// cp.async.bulk moves), T = 1 (plain instance-major records) for the cooperative kernels, where a
// group of threads owns an instance and reads its rows contiguously.
#define LQRB_TILE 32

__host__ __device__ __forceinline__ int64_t packed_index(int64_t rows, int tile_w, int64_t row,
                                                         int64_t inst) {
    return ((inst / tile_w) * rows + row) * tile_w + (inst % tile_w);
}

__host__ __device__ constexpr int tri(int k) { return k * (k + 1) / 2; }
// upper-packed column-major index of (i,j), i <= j
__host__ __device__ constexpr int tri_idx(int i, int j) { return j * (j + 1) / 2 + i; }
__host__ __device__ constexpr int sym_idx(int i, int j) { return i <= j ? tri_idx(i, j) : tri_idx(j, i); }

// rows the cost Hessian of one knot takes in the packed KKT data (see lqrb200.h)
__host__ __device__ constexpr int hess_rows(int n, int mk, int hess) {
    return hess == LQRB_HESS_DIAG ? n + mk : hess == LQRB_HESS_BLOCKDIAG ? tri(n) + tri(mk) : tri(n + mk);
}

// ------------------------------------------------------------------ context -------------------
// Device scratch: one grow-only allocation per (slot, lane); see `Lane`.
enum ScratchSlot {
    SCR_GAINS = 0,
    SCR_FACT,
    SCR_STAGE_A,  // lqrb_for_chunks: staged inputs of a chunk
    SCR_STAGE_B,  //                  staged outputs of a chunk
    SCR_PACK_IN,
    SCR_PACK_IN2,
    SCR_PACK_OUT,
    SCR_PACK_OUT2,
    SCR_PACK_OUT3,
    SCR_MISC,
    SCR_SQP0,
    SCR_SQP1,
    SCR_SQP2,
    SCR_SQP3,
    SCR_KEEP_DATA,    // lqrb_kkt_factor_f64: packed matrices of the kept factorisation
    SCR_KEEP_REC,     //                      block rows of U (BlockUpperTriangular3 records)
    SCR_REFINE,       // records of the instances re-solved by the Cholesky-based kernel (ill-conditioned blocks)
    SCR_REFINE_LIST,  // their indices
    SCR_RICCATI_PAD,  // Riccati problems embedded in a tuned size class: padded knots, term, Z, gains
    SCR_ADJOINT_Z,    // lqrb_riccati_grad_f64 / lqrb_kkt_grad_f64: the adjoint solution, instance-major (read by the
                      // gradient kernels)
    SCR_ADJOINT_MULT, // lqrb_kkt_grad_f64: the adjoint multipliers, instance-major
    SCR_GAIN_TAPE,    // lqrb_riccati_grad_gains_f64: P_{k+1}, p_{k+1}, K_k, kff_k and the factor of G_k per knot
    SCR_ADMM_CACHE,   // lqrb_admm_cache_f64: Q + rho I, R + rho I, and the DARE's P, K, info of a chunk
    SCR_COUNT
};

// Where a piece of work runs: its stream and which per-lane scratch it owns.  A staged call (lqrb_for_chunks) runs its
// chunks alternately on lanes {copy_stream[0], 0} and {copy_stream[1], 1}; a device-resident call runs on
// {h->stream, 0}.  Sharing lane 0 between h->stream and copy stream 0 is safe: a staged call waits for h->stream before
// its first chunk and synchronises both copy streams before it returns, so work of two calls never overlaps on it.
struct Lane {
    cudaStream_t stream;
    int index;  // 0 or 1
};

struct RowMap;
struct DevMap {
    const RowMap *dev = nullptr;
    int64_t rows = 0;
};

struct lqrb_context {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;      // stream all work is ordered on
    cudaStream_t own_stream = nullptr;  // created by the handle
    cudaStream_t copy_stream[2] = {nullptr, nullptr};
    cudaEvent_t ev[8] = {};
    std::string err;
    std::string kernel_name;
    int64_t launches = 0;
    void *scratch[SCR_COUNT][2] = {};
    size_t scratch_bytes[SCR_COUNT][2] = {};
    void *pinned[2] = {};
    size_t pinned_bytes[2] = {};
    std::map<std::string, int64_t> options;
    std::map<std::string, struct DevMap> maps;  // cached device copies of row maps
    std::map<std::string, void *> blobs;        // cached device tables (cooperative KKT offsets)
    std::vector<int32_t> last_cond;             // conditioning estimates (log2 pivot ratio) per instance of the last
                                                // KKT solve call that ran a tuned kernel
    int64_t last_refined = 0;                   // instances of that call re-solved by the Cholesky-based kernel
    std::string kept_key;                       // shape + flags of the factorisation kept by lqrb_kkt_factor_f64
    int64_t kept_batch = 0;

    int64_t opt(const char *name, int64_t dflt) const {
        auto it = options.find(name);
        return it == options.end() ? dflt : it->second;
    }
};

int32_t lqrb_fail(lqrb_context *h, int32_t code, const std::string &msg);
int32_t lqrb_cuda_fail(lqrb_context *h, cudaError_t e, const char *what);
// grow-only scratch of one lane; returns nullptr and records the error on failure
void *lqrb_scratch(lqrb_context *h, int slot, size_t bytes, int lane = 0);
void *lqrb_pinned(lqrb_context *h, int lane, size_t bytes);

// ------------------------------------------------------------------ host / device staging (host_io.cu) ----
// One instance-major caller array: its pointer (NULL: absent) and its bytes per instance (0: absent).
struct HostArray {
    const void *ptr;
    int64_t bytes;
};
// Runs one chunk of `cb` instances (chunks run in instance order).  `in` / `out` hold device pointers to the chunk's
// part of every listed array, in list order; absent arrays are NULL.
using ChunkBody = std::function<int32_t(Lane lane, int64_t cb, const void *const *in, void *const *out)>;
// Runs `body` over the batch.  A call is device-resident when every present array, inputs and outputs alike, is device
// or managed memory: then `body` runs once on {h->stream, 0} with the caller's own pointers, without synchronising.
// Otherwise the call is staged: chunks of `chunk` instances alternate over the two copy streams; each copies its part
// of every present input into the lane's staging scratch, runs `body`, and copies every present output back; the call
// returns when both streams are done.  An output with the same pointer as an input is updated in place (in/out arrays).
// chunk = 0 picks the size: the `host_chunk` option if set, otherwise about 64 MB of input (counting every listed
// input, present or not), rounded up to LQRB_TILE.
int32_t lqrb_for_chunks(lqrb_context *h, int64_t batch, int64_t chunk, const std::vector<HostArray> &inputs,
                        const std::vector<HostArray> &outputs, const ChunkBody &body);

#define LQRB_CUDA(h, call)                                              \
    do {                                                                \
        cudaError_t e__ = (call);                                       \
        if (e__ != cudaSuccess) return lqrb_cuda_fail((h), e__, #call); \
    } while (0)

#define LQRB_LAUNCH_CHECK(h, name)                                                    \
    do {                                                                              \
        (h)->launches++;                                                              \
        cudaError_t e__ = cudaGetLastError();                                         \
        if (e__ != cudaSuccess) return lqrb_cuda_fail((h), e__, "launch of " name);   \
    } while (0)

static inline int64_t round_up(int64_t a, int64_t b) { return (a + b - 1) / b * b; }

// ------------------------------------------------------------------ gather/scatter maps -------
// One packed row = one element of one instance-major source array.
// Doubles per knot record of the packed Riccati layout: A | B | Q (upper packed) | R (upper packed) | q | r, plus one
// padding double for the warp-per-instance tensor-core size class (n = 8, 12, m <= 4) when that count is odd — its
// records travel by 16-byte bulk copies and are read with 16-byte shared loads (m = 2, 3 at both n).
__host__ __device__ constexpr int lqrb_riccati_knot_rows(int n, int m) {
    const int f = n * n + n * m + n * (n + 1) / 2 + m * (m + 1) / 2 + n + m;
    return ((n == 8 || n == 12) && m <= 4) ? ((f + 1) & ~1) : f;
}

struct RowMap {
    int32_t array;   // index into the source pointer table (-1: constant fill)
    int32_t offset;  // element offset inside that array's per-instance record
    double fill;     // value when array < 0
};
#define LQRB_MAX_ARRAYS 16
struct ArrayTable {
    const double *ptr[LQRB_MAX_ARRAYS];
    int64_t stride[LQRB_MAX_ARRAYS];  // per-instance record length (doubles)
};
struct ArrayTableOut {
    double *ptr[LQRB_MAX_ARRAYS];
    int64_t stride[LQRB_MAX_ARRAYS];
};

// cached upload of a row map; `build` is called only on a cache miss
DevMap lqrb_get_map(lqrb_context *h, const std::string &key, std::vector<RowMap> (*build)(const int *),
                    const int *args);
DevMap lqrb_get_map(lqrb_context *h, const std::string &key, const std::vector<RowMap> &map);
// identity row map: packed [rows] <-> instance-major [rows, batch]
DevMap lqrb_identity_map(lqrb_context *h, int64_t rows);
// instance-major sources -> packed [tile][rows][tile_w]
int32_t lqrb_gather_pack(lqrb_context *h, const DevMap &map, const ArrayTable &src, int64_t batch,
                         int tile_w, double *packed, cudaStream_t s);
// packed -> instance-major destinations (rows with array < 0 are skipped)
int32_t lqrb_scatter_unpack(lqrb_context *h, const DevMap &map, const ArrayTableOut &dst,
                            int64_t batch, int tile_w, const double *packed, cudaStream_t s);

// which tile width the library uses for a size class (32: thread-per-instance, 1: cooperative)
int lqrb_riccati_tile(const lqrb_context *h, int n, int m);
int lqrb_kkt_tile(const lqrb_context *h, int n, int m, int N, const int32_t *p, int hess_mode,
                  int explicit_d2);
// lqrb_kkt_solve_packed_f64 on a given lane (the SQP driver calls it from inside its own staged call)
int32_t lqrb_kkt_solve_packed_on(lqrb_context *h, int n, int m, int N, int64_t batch, const int32_t *p, int hess_mode,
                                 int explicit_d2, int flags, const double *data, double *dz, double *mult, double *res,
                                 int32_t *info, Lane lane);

