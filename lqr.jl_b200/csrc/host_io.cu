// host_io.cu — moving the caller's instance-major arrays between host and device: the one rule that tells a
// device-resident call from a staged one, and the chunk driver every entry point runs its work through.
#include "common.cuh"

static bool lqrb_is_device_ptr(const void *p) {
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

static bool present(const HostArray &a) { return a.ptr && a.bytes > 0; }

int32_t lqrb_for_chunks(lqrb_context *h, int64_t batch, int64_t chunk, const std::vector<HostArray> &inputs,
                        const std::vector<HostArray> &outputs, const ChunkBody &body) {
    if (batch <= 0) return 0;
    const size_t ni = inputs.size(), no = outputs.size();
    std::vector<const void *> din(ni, nullptr);
    std::vector<void *> dout(no, nullptr);

    bool resident = true;
    for (const HostArray &a : inputs) resident = resident && (!present(a) || lqrb_is_device_ptr(a.ptr));
    for (const HostArray &a : outputs) resident = resident && (!present(a) || lqrb_is_device_ptr(a.ptr));
    if (resident) {
        for (size_t i = 0; i < ni; ++i) din[i] = present(inputs[i]) ? inputs[i].ptr : nullptr;
        for (size_t j = 0; j < no; ++j) dout[j] = present(outputs[j]) ? const_cast<void *>(outputs[j].ptr) : nullptr;
        return body(Lane{h->stream, 0}, batch, din.data(), dout.data());
    }

    if (chunk <= 0) {
        int64_t in_bytes = 0;
        for (const HostArray &a : inputs) in_bytes += a.bytes;
        chunk = h->opt("host_chunk", 0);
        // ~64 MB of input per chunk keeps both copy engines and the SMs busy
        if (chunk <= 0) chunk = (64ll << 20) / std::max<int64_t>(in_bytes, 1) / LQRB_TILE * LQRB_TILE;
        chunk = std::max<int64_t>(LQRB_TILE, round_up(chunk, LQRB_TILE));
    }
    chunk = std::min(chunk, batch);

    // staging of one lane: a 256-byte aligned slice of `chunk` instances per present array; an output that is also an
    // input uses the input's slice
    std::vector<size_t> in_off(ni), out_off(no);
    std::vector<int> alias(no, -1);
    size_t in_total = 0, out_total = 0;
    for (size_t i = 0; i < ni; ++i) {
        if (!present(inputs[i])) continue;
        in_off[i] = in_total;
        in_total += (size_t)round_up(chunk * inputs[i].bytes, 256);
    }
    for (size_t j = 0; j < no; ++j) {
        if (!present(outputs[j])) continue;
        for (size_t i = 0; i < ni; ++i)
            if (present(inputs[i]) && inputs[i].ptr == outputs[j].ptr) alias[j] = (int)i;
        if (alias[j] >= 0) continue;
        out_off[j] = out_total;
        out_total += (size_t)round_up(chunk * outputs[j].bytes, 256);
    }

    LQRB_CUDA(h, cudaEventRecord(h->ev[0], h->stream));
    for (int i = 0; i < 2; ++i) LQRB_CUDA(h, cudaStreamWaitEvent(h->copy_stream[i], h->ev[0], 0));
    int index = 0;
    for (int64_t first = 0; first < batch; first += chunk, index ^= 1) {
        const int64_t cb = std::min(chunk, batch - first);
        const Lane lane{h->copy_stream[index], index};
        char *si = (char *)lqrb_scratch(h, SCR_STAGE_A, in_total, index);
        char *so = (char *)lqrb_scratch(h, SCR_STAGE_B, out_total, index);
        if (!si || !so) return 1000 + (int)cudaErrorMemoryAllocation;
        for (size_t i = 0; i < ni; ++i) {
            const HostArray &a = inputs[i];
            if (!present(a)) continue;
            din[i] = si + in_off[i];
            LQRB_CUDA(h, cudaMemcpyAsync(si + in_off[i], (const char *)a.ptr + first * a.bytes, (size_t)(cb * a.bytes),
                                         cudaMemcpyDefault, lane.stream));
        }
        for (size_t j = 0; j < no; ++j)
            if (present(outputs[j])) dout[j] = alias[j] >= 0 ? const_cast<void *>(din[alias[j]]) : so + out_off[j];
        int32_t rc = body(lane, cb, din.data(), dout.data());
        if (rc) return rc;
        for (size_t j = 0; j < no; ++j) {
            const HostArray &a = outputs[j];
            if (!present(a)) continue;
            LQRB_CUDA(h, cudaMemcpyAsync((char *)const_cast<void *>(a.ptr) + first * a.bytes, dout[j],
                                         (size_t)(cb * a.bytes), cudaMemcpyDefault, lane.stream));
        }
    }
    for (int i = 0; i < 2; ++i) LQRB_CUDA(h, cudaStreamSynchronize(h->copy_stream[i]));
    return 0;
}
