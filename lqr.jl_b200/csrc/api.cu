// api.cu — handle management, error reporting, scratch, and the pack / unpack (layout) kernels.
#include <cstdio>
#include <cstring>

#include "common.cuh"

// ------------------------------------------------------------------ errors / scratch ----------
int32_t lqrb_fail(lqrb_context *h, int32_t code, const std::string &msg) {
    if (h) h->err = msg;
    return code;
}

int32_t lqrb_cuda_fail(lqrb_context *h, cudaError_t e, const char *what) {
    if (h) h->err = std::string(what) + ": " + cudaGetErrorString(e);
    return 1000 + (int32_t)e;
}

void *lqrb_scratch(lqrb_context *h, int slot, size_t bytes, int lane) {
    if (bytes == 0) bytes = 16;
    void *&cur = h->scratch[slot][lane];
    size_t &have = h->scratch_bytes[slot][lane];
    if (have >= bytes) return cur;
    if (cur) {
        cudaDeviceSynchronize();  // the slot may still be in use on the handle's streams
        cudaFree(cur);
        cur = nullptr;
        have = 0;
    }
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
        lqrb_cuda_fail(h, e, "cudaMalloc(scratch)");
        return nullptr;
    }
    cur = p;
    have = bytes;
    return p;
}

void *lqrb_pinned(lqrb_context *h, int lane, size_t bytes) {
    if (bytes == 0) bytes = 16;
    if (h->pinned_bytes[lane] >= bytes) return h->pinned[lane];
    if (h->pinned[lane]) {
        cudaStreamSynchronize(h->stream);
        cudaFreeHost(h->pinned[lane]);
        h->pinned[lane] = nullptr;
        h->pinned_bytes[lane] = 0;
    }
    void *p = nullptr;
    cudaError_t e = cudaMallocHost(&p, bytes);
    if (e != cudaSuccess) {
        lqrb_cuda_fail(h, e, "cudaMallocHost");
        return nullptr;
    }
    h->pinned[lane] = p;
    h->pinned_bytes[lane] = bytes;
    return p;
}

// ------------------------------------------------------------------ library / handle ----------
extern "C" int32_t lqrb_version(void) { return LQRB_VERSION; }

extern "C" int32_t lqrb_device_count(int32_t *count) {
    if (!count) return -1;
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *count = 0;
        return 1000 + (int32_t)e;
    }
    *count = c;
    return 0;
}

extern "C" int32_t lqrb_create(lqrb_handle_t *handle, int32_t device) {
    if (!handle) return -1;
    *handle = nullptr;
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return 1000 + (int32_t)e;
    }
    if (device < 0 || device >= c) return -2;
    lqrb_context *h = new lqrb_context();
    h->device = device;
    if ((e = cudaSetDevice(device)) != cudaSuccess) {
        delete h;
        return 1000 + (int32_t)e;
    }
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
        delete h;
        return 1000 + (int32_t)e;
    }
    if (prop.major != 10) {
        // sm_100a cubins only: fail loudly instead of falling back to anything else
        delete h;
        return -2;
    }
    h->sm_count = prop.multiProcessorCount;
    cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&h->copy_stream[0], cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&h->copy_stream[1], cudaStreamNonBlocking);
    for (auto &ev : h->ev) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    h->stream = h->own_stream;
    *handle = h;
    return 0;
}

extern "C" int32_t lqrb_destroy(lqrb_handle_t h) {
    if (!h) return -1;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (auto &slot : h->scratch)
        for (void *p : slot)
            if (p) cudaFree(p);
    for (void *p : h->pinned)
        if (p) cudaFreeHost(p);
    for (auto &kv : h->maps)
        if (kv.second.dev) cudaFree((void *)kv.second.dev);
    for (auto &kv : h->blobs)
        if (kv.second) cudaFree(kv.second);
    for (auto &ev : h->ev)
        if (ev) cudaEventDestroy(ev);
    cudaStreamDestroy(h->own_stream);
    cudaStreamDestroy(h->copy_stream[0]);
    cudaStreamDestroy(h->copy_stream[1]);
    delete h;
    return 0;
}

extern "C" const char *lqrb_last_error_string(lqrb_handle_t h) {
    return h ? h->err.c_str() : "null handle";
}

extern "C" int32_t lqrb_set_stream(lqrb_handle_t h, void *s) {
    if (!h) return -1;
    h->stream = s ? (cudaStream_t)s : h->own_stream;
    return 0;
}

extern "C" int32_t lqrb_synchronize(lqrb_handle_t h) {
    if (!h) return -1;
    LQRB_CUDA(h, cudaSetDevice(h->device));
    LQRB_CUDA(h, cudaStreamSynchronize(h->stream));
    return 0;
}

extern "C" int64_t lqrb_launch_count(lqrb_handle_t h) { return h ? h->launches : -1; }

extern "C" const char *lqrb_last_kernel_name(lqrb_handle_t h) {
    return h ? h->kernel_name.c_str() : "";
}

extern "C" int32_t lqrb_set_option(lqrb_handle_t h, const char *name, int64_t value) {
    if (!h) return -1;
    if (!name) return -2;
    h->options[name] = value;
    return 0;
}

// ------------------------------------------------------------------ layout queries ------------
extern "C" int64_t lqrb_padded_batch(int64_t batch) { return round_up(batch, LQRB_TILE); }

extern "C" int64_t lqrb_num_vars(int32_t n, int32_t m, int32_t N) {
    return (int64_t)N * n + (int64_t)(N - 1) * m;
}

extern "C" int64_t lqrb_num_cons(int32_t n, int32_t N, const int32_t *p) {
    int64_t P = (int64_t)(N - 1) * n;
    if (p)
        for (int k = 0; k < N; ++k) P += p[k];
    return P;
}

extern "C" int32_t lqrb_riccati_layout(int32_t n, int32_t m, int32_t N, int32_t flags,
                                       lqrb_riccati_layout_t *out) {
    if (n < 1) return -1;
    if (m < 1) return -2;
    if (N < 2) return -3;
    if (!out) return -5;
    out->rows_per_knot = lqrb_riccati_knot_rows(n, m);  // one padding double for (8 | 12, 2 | 3)
    out->knot_count = (flags & LQRB_FLAG_LTI) ? 1 : N - 1;
    out->term_rows = tri(n) + 2 * n;
    out->z_rows = lqrb_num_vars(n, m, N);
    out->gain_rows = (int64_t)(N - 1) * (m * n + m);
    return 0;
}

// ------------------------------------------------------------------ pack / unpack kernels -----
// gather: instance-major -> packed.  grid (instance tiles of 32, row chunks of 32), block (32, 8).
template <int TILE_W>
__global__ void __launch_bounds__(256) gather_pack_kernel(const RowMap *__restrict__ map, ArrayTable src,
                                                          int64_t rows, int64_t batch,
                                                          double *__restrict__ packed) {
    __shared__ double sm[32][33];
    const int64_t row0 = (int64_t)blockIdx.y * 32, inst0 = (int64_t)blockIdx.x * 32;
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int64_t row = row0 + tx;
    RowMap rm;
    rm.array = -1;
    rm.offset = 0;
    rm.fill = 0.0;
    if (row < rows) rm = map[row];
    const double *base = rm.array >= 0 ? src.ptr[rm.array] : nullptr;
    const int64_t stride = rm.array >= 0 ? src.stride[rm.array] : 0;
#pragma unroll
    for (int j = ty; j < 32; j += 8) {
        const int64_t inst = inst0 + j;
        double v = rm.fill;
        if (base != nullptr && inst < batch) v = base[inst * stride + rm.offset];
        sm[j][tx] = v;
    }
    __syncthreads();
    if (TILE_W == 32) {
        // thread (tx = instance lane, ty = row)
#pragma unroll
        for (int j = ty; j < 32; j += 8) {
            const int64_t r = row0 + j;
            if (r < rows) packed[((int64_t)blockIdx.x * rows + r) * 32 + tx] = sm[tx][j];
        }
    } else {
        // T = 1: packed[inst*rows + row]; thread (tx = row, ty = instance)
#pragma unroll
        for (int j = ty; j < 32; j += 8) {
            const int64_t inst = inst0 + j;
            if (row < rows && inst < batch) packed[inst * rows + row] = sm[j][tx];
        }
    }
}

template <int TILE_W>
__global__ void __launch_bounds__(256) scatter_unpack_kernel(const RowMap *__restrict__ map, ArrayTableOut dst,
                                                             int64_t rows, int64_t batch,
                                                             const double *__restrict__ packed) {
    __shared__ double sm[32][33];
    const int64_t row0 = (int64_t)blockIdx.y * 32, inst0 = (int64_t)blockIdx.x * 32;
    const int tx = threadIdx.x, ty = threadIdx.y;
    if (TILE_W == 32) {
#pragma unroll
        for (int j = ty; j < 32; j += 8) {
            const int64_t r = row0 + j;
            sm[tx][j] = (r < rows) ? packed[((int64_t)blockIdx.x * rows + r) * 32 + tx] : 0.0;
        }
    } else {
        const int64_t row = row0 + tx;
#pragma unroll
        for (int j = ty; j < 32; j += 8) {
            const int64_t inst = inst0 + j;
            sm[j][tx] = (row < rows && inst < batch) ? packed[inst * rows + row] : 0.0;
        }
    }
    __syncthreads();
    const int64_t row = row0 + tx;
    if (row >= rows) return;
    const RowMap rm = map[row];
    if (rm.array < 0) return;
    double *base = dst.ptr[rm.array];
    if (base == nullptr) return;
    const int64_t stride = dst.stride[rm.array];
#pragma unroll
    for (int j = ty; j < 32; j += 8) {
        const int64_t inst = inst0 + j;
        if (inst < batch) base[inst * stride + rm.offset] = sm[j][tx];
    }
}

DevMap lqrb_get_map(lqrb_context *h, const std::string &key, const std::vector<RowMap> &map) {
    auto it = h->maps.find(key);
    if (it != h->maps.end()) return it->second;
    DevMap d;
    d.rows = (int64_t)map.size();
    void *p = nullptr;
    const size_t bytes = map.size() * sizeof(RowMap) + 16;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) {
        e = cudaMemcpy(p, map.data(), map.size() * sizeof(RowMap), cudaMemcpyHostToDevice);
        // a pageable-source cudaMemcpy may return while the DMA from its staging buffer is still in flight on
        // the legacy stream; the kernels that read the map run on non-blocking streams, so wait for it here
        // (once per map shape)
        if (e == cudaSuccess) e = cudaStreamSynchronize(cudaStreamLegacy);
        if (e != cudaSuccess) cudaFree(p);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        lqrb_cuda_fail(h, e, "row map upload");
        d.dev = nullptr;  // rows stays > 0: the pack / unpack launchers report the failure instead of skipping
        return d;
    }
    d.dev = (const RowMap *)p;
    h->maps[key] = d;
    return d;
}

DevMap lqrb_get_map(lqrb_context *h, const std::string &key, std::vector<RowMap> (*build)(const int *),
                    const int *args) {
    auto it = h->maps.find(key);
    if (it != h->maps.end()) return it->second;
    return lqrb_get_map(h, key, build(args));
}

int32_t lqrb_gather_pack(lqrb_context *h, const DevMap &map, const ArrayTable &src, int64_t batch,
                         int tile_w, double *packed, cudaStream_t s) {
    const int64_t rows = map.rows;
    if (rows > 0 && !map.dev) return 1000 + (int)cudaErrorMemoryAllocation;  // failed row-map upload (lqrb_get_map)
    if (rows == 0 || batch == 0) return 0;
    dim3 grid((unsigned)((batch + 31) / 32), (unsigned)((rows + 31) / 32)), block(32, 8);
    if (tile_w == 32)
        gather_pack_kernel<32><<<grid, block, 0, s>>>(map.dev, src, rows, batch, packed);
    else
        gather_pack_kernel<1><<<grid, block, 0, s>>>(map.dev, src, rows, batch, packed);
    LQRB_LAUNCH_CHECK(h, "gather_pack_kernel");
    return 0;
}

int32_t lqrb_scatter_unpack(lqrb_context *h, const DevMap &map, const ArrayTableOut &dst,
                            int64_t batch, int tile_w, const double *packed, cudaStream_t s) {
    const int64_t rows = map.rows;
    if (rows > 0 && !map.dev) return 1000 + (int)cudaErrorMemoryAllocation;  // failed row-map upload (lqrb_get_map)
    if (rows == 0 || batch == 0) return 0;
    dim3 grid((unsigned)((batch + 31) / 32), (unsigned)((rows + 31) / 32)), block(32, 8);
    if (tile_w == 32)
        scatter_unpack_kernel<32><<<grid, block, 0, s>>>(map.dev, dst, rows, batch, packed);
    else
        scatter_unpack_kernel<1><<<grid, block, 0, s>>>(map.dev, dst, rows, batch, packed);
    LQRB_LAUNCH_CHECK(h, "scatter_unpack_kernel");
    return 0;
}

DevMap lqrb_identity_map(lqrb_context *h, int64_t rows) {
    std::vector<RowMap> m((size_t)rows);
    for (int64_t r = 0; r < rows; ++r) m[(size_t)r] = RowMap{0, (int32_t)r, 0.0};
    return lqrb_get_map(h, "id" + std::to_string(rows), m);
}

extern "C" int32_t lqrb_unpack_rows_f64(lqrb_handle_t h, int64_t rows, int64_t batch, int32_t tile,
                                        const double *packed, double *instance_major) {
    if (!h) return -1;
    if (rows < 0) return -2;
    if (batch < 0) return -3;
    if (tile != 1 && tile != LQRB_TILE) return lqrb_fail(h, -4, "tile must be 1 or 32 (lqrb_*_tile_width)");
    if (!packed) return -5;
    if (!instance_major) return -6;
    LQRB_CUDA(h, cudaSetDevice(h->device));
    ArrayTableOut t = {};
    t.ptr[0] = instance_major;
    t.stride[0] = rows;
    return lqrb_scatter_unpack(h, lqrb_identity_map(h, rows), t, batch, tile, packed, h->stream);
}

extern "C" int32_t lqrb_pack_rows_f64(lqrb_handle_t h, int64_t rows, int64_t batch, int32_t tile,
                                      const double *instance_major, double *packed) {
    if (!h) return -1;
    if (rows < 0) return -2;
    if (batch < 0) return -3;
    if (tile != 1 && tile != LQRB_TILE) return lqrb_fail(h, -4, "tile must be 1 or 32 (lqrb_*_tile_width)");
    if (!instance_major) return -5;
    if (!packed) return -6;
    LQRB_CUDA(h, cudaSetDevice(h->device));
    ArrayTable t = {};
    t.ptr[0] = instance_major;
    t.stride[0] = rows;
    return lqrb_gather_pack(h, lqrb_identity_map(h, rows), t, batch, tile, packed, h->stream);
}
