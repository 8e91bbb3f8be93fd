// dab_api.cu — handle lifecycle, uploads, error reporting for libdiskann_b200.so.
#include "dab_common.cuh"

#include <algorithm>

#include <cstdlib>

#include <vector>

namespace dab {

std::atomic<uint64_t> g_launches{0};

char* error_buffer() {
    static thread_local char buf[512] = {0};
    return buf;
}

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(error_buffer(), 512, fmt, ap);
    va_end(ap);
    return code;
}

int Scratch::reserve(size_t n) {
    if (n <= bytes) return DAB_OK;
    release();
    size_t want = n + n / 4;
    cudaError_t e = pinned_host ? cudaMallocHost(&p, want) : cudaMalloc(&p, want);
    if (e != cudaSuccess) {
        p = nullptr;
        bytes = 0;
        return fail(DAB_ERR_OUT_OF_MEMORY, "scratch allocation of %zu bytes failed: %s", want,
                    cudaGetErrorString(e));
    }
    bytes = want;
    return DAB_OK;
}

void Scratch::release() {
    if (p) {
        if (pinned_host)
            cudaFreeHost(p);
        else
            cudaFree(p);
    }
    p = nullptr;
    bytes = 0;
}

// repack [count][src_stride] -> [count][dst_stride], zero padded
__global__ void repack_rows_kernel(const uint8_t* __restrict__ src, size_t src_stride,
                                   uint8_t* __restrict__ dst, size_t dst_stride, size_t row_bytes,
                                   uint64_t count) {
    const uint64_t total = count * dst_stride;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total;
         i += (uint64_t)gridDim.x * blockDim.x) {
        uint64_t r = i / dst_stride;
        size_t c = i % dst_stride;
        dst[i] = c < row_bytes ? src[r * src_stride + c] : 0;
    }
}

void TestHooks::load() {
    const char* t = getenv("DAB_TEST_VISITED_LOG2");
    const long v = t ? atol(t) : 0;
    test_visited_log2 = v >= 8 && v <= 30 ? (int)v : 0;
    pq_global_lut = getenv("DAB_TEST_PQ_GLOBAL_LUT") != nullptr;
}

}  // namespace dab

using namespace dab;

extern "C" {

const char* dab_last_error(void) { return error_buffer(); }
uint64_t dab_launch_count(void) { return g_launches.load(); }

int dab_create(dab_index** out, int dtype, int metric, uint32_t dim, uint64_t n_points,
               uint32_t n_start, uint32_t max_degree, int device) {
    if (!out) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_create: out is NULL");
    *out = nullptr;
    if (dtype < DAB_F32 || dtype > DAB_U8) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_create: unknown dtype %d", dtype);
    if (metric < DAB_COSINE || metric > DAB_COSINE_NORMALIZED)
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_create: unknown metric %d", metric);
    if (dim == 0) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_create: dim must be > 0");
    if (n_points + n_start == 0 || n_points + n_start >= 0x7FFFFFFFull)
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_create: n_points + n_start must be in [1, 2^31-1)");
    if (max_degree == 0 || max_degree > 1024)
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_create: max_degree must be in [1, 1024]");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(DAB_ERR_NO_DEVICE, "dab_create: no CUDA device visible (the product path has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_create: device %d out of range", device);
    DAB_CUDA(cudaSetDevice(device));
    dab_index* idx = new dab_index();
    idx->dtype = dtype;
    idx->metric = metric;
    idx->dim = dim;
    idx->n_points = n_points;
    idx->n_start = n_start;
    idx->max_degree = max_degree;
    idx->device = device;
    cudaDeviceGetAttribute(&idx->sm_count, cudaDevAttrMultiProcessorCount, device);
    idx->row_stride = round_up((size_t)dim * elem_size(dtype), 32);
    idx->adj_stride = (uint32_t)round_up((size_t)max_degree + 1, 8);
    idx->h_stage.pinned_host = true;
    idx->h_counters.pinned_host = true;
    idx->hooks.load();
    cudaError_t e = cudaStreamCreateWithFlags(&idx->own_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete idx;
        return fail(DAB_ERR_CUDA, "cudaStreamCreate failed: %s", cudaGetErrorString(e));
    }
    idx->stream = idx->own_stream;
    const uint64_t total = idx->n_total();
    e = cudaMalloc(&idx->d_vectors, total * idx->row_stride);
    if (e == cudaSuccess) e = cudaMalloc(&idx->d_adj, total * (size_t)idx->adj_stride * 4 + 512);  // +slack: kernels read whole 128 B lines of the last row
    if (e != cudaSuccess) {
        dab_destroy(idx);
        return fail(DAB_ERR_OUT_OF_MEMORY, "dab_create: device allocation failed: %s", cudaGetErrorString(e));
    }
    cudaMemsetAsync(idx->d_vectors, 0, total * idx->row_stride, idx->stream);
    cudaMemsetAsync(idx->d_adj, 0, total * (size_t)idx->adj_stride * 4, idx->stream);
    cudaStreamSynchronize(idx->stream);
    *out = idx;
    return DAB_OK;
}

void dab_destroy(dab_index* idx) {
    if (!idx) return;
    cudaSetDevice(idx->device);
    if (idx->own_stream) cudaStreamSynchronize(idx->own_stream);
    search_slots_release(idx);
    comm_release(idx);
    tc_release(idx);
    cudaFree(idx->d_vectors);
    cudaFree(idx->d_adj);
    cudaFree(idx->d_pivots);
    cudaFree(idx->d_offsets);
    cudaFree(idx->d_codes);
    cudaFree(idx->d_sq_shift);
    cudaFree(idx->d_sq_codes);
    cudaFree(idx->d_sq_comp);
    idx->s_queries.release();
    idx->s_ids.release();
    idx->s_out.release();
    idx->s_out2.release();
    idx->s_tables.release();
    idx->s_counters.release();
    idx->s_stats.release();
    idx->h_stage.release();
    idx->h_counters.release();
    if (idx->own_stream) cudaStreamDestroy(idx->own_stream);
    delete idx;
}

int dab_set_stream(dab_index* idx, void* cuda_stream) {
    if (!idx) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_set_stream: idx is NULL");
    idx->stream = cuda_stream ? (cudaStream_t)cuda_stream : idx->own_stream;
    return DAB_OK;
}

static int upload_rows(dab_index* idx, const void* rows, uint64_t first, uint64_t count, bool on_device) {
    if (!idx || (!rows && count)) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_upload_vectors: NULL argument");
    if (first + count > idx->n_total())
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_upload_vectors: rows [%llu, %llu) out of range (%llu rows)",
                    (unsigned long long)first, (unsigned long long)(first + count), (unsigned long long)idx->n_total());
    if (count == 0) return DAB_OK;
    DAB_CUDA(cudaSetDevice(idx->device));
    const size_t row_bytes = (size_t)idx->dim * elem_size(idx->dtype);
    uint8_t* dst = idx->d_vectors + first * idx->row_stride;
    if (!on_device) {
        DAB_CUDA(cudaMemcpy2DAsync(dst, idx->row_stride, rows, row_bytes, row_bytes, count, cudaMemcpyHostToDevice,
                                   idx->stream));
    } else {
        DAB_CUDA(cudaMemcpy2DAsync(dst, idx->row_stride, rows, row_bytes, row_bytes, count, cudaMemcpyDeviceToDevice,
                                   idx->stream));
    }
    DAB_CUDA(cudaStreamSynchronize(idx->stream));
    idx->vectors_ready = true;
    ++idx->vectors_version;
    return DAB_OK;
}

int dab_upload_vectors(dab_index* idx, const void* rows, uint64_t first, uint64_t count) {
    return upload_rows(idx, rows, first, count, false);
}
int dab_upload_vectors_device(dab_index* idx, const void* d_rows, uint64_t first, uint64_t count) {
    return upload_rows(idx, d_rows, first, count, true);
}

// degree check of rows that are already on the device (the host path checks before copying): first offending row, or ~0
__global__ void __launch_bounds__(256) graph_degree_check_kernel(const uint32_t* __restrict__ adj, uint32_t src_stride, uint64_t count,
                                                                  uint32_t max_degree, unsigned long long* __restrict__ first_bad) {
    for (uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; r < count; r += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t len = adj[r * (size_t)src_stride];
        if (len > max_degree || len + 1 > src_stride) atomicMin(first_bad, (unsigned long long)r);
    }
}

static int upload_graph(dab_index* idx, const uint32_t* adj, uint32_t src_stride, uint64_t first, uint64_t count,
                        bool on_device) {
    if (!idx || (!adj && count)) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_upload_graph: NULL argument");
    if (first + count > idx->n_total()) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_upload_graph: rows out of range");
    if (src_stride == 0) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_upload_graph: src_stride is 0");
    if (count == 0) return DAB_OK;
    DAB_CUDA(cudaSetDevice(idx->device));
    const size_t copy_words = src_stride < idx->adj_stride ? src_stride : idx->adj_stride;
    if (!on_device) {
        // validate degrees on the host: a row's length must fit the device row
        for (uint64_t r = 0; r < count; ++r) {
            uint32_t len = adj[r * (size_t)src_stride];
            if (len > idx->max_degree || len + 1 > src_stride)
                return fail(DAB_ERR_INVALID_ARGUMENT, "dab_upload_graph: row %llu has degree %u > max_degree %u",
                            (unsigned long long)(first + r), len, idx->max_degree);
        }
    } else {
        int rc;
        if ((rc = idx->s_counters.reserve(16))) return rc;
        unsigned long long* d_bad = (unsigned long long*)idx->s_counters.p;
        DAB_CUDA(cudaMemsetAsync(d_bad, 0xFF, 8, idx->stream));
        const int grid = (int)std::min<uint64_t>((count + 255) / 256, (uint64_t)idx->sm_count * 8);
        graph_degree_check_kernel<<<grid, 256, 0, idx->stream>>>(adj, src_stride, count, idx->max_degree, d_bad);
        DAB_LAUNCHED();
        DAB_CUDA(cudaGetLastError());
        unsigned long long bad = 0;
        DAB_CUDA(cudaMemcpyAsync(&bad, d_bad, 8, cudaMemcpyDeviceToHost, idx->stream));
        DAB_CUDA(cudaStreamSynchronize(idx->stream));
        if (bad != ~0ull)
            return fail(DAB_ERR_INVALID_ARGUMENT, "dab_upload_graph_device: row %llu has a degree > max_degree %u (or beyond src_stride %u)",
                        (unsigned long long)(first + bad), idx->max_degree, src_stride);
    }
    DAB_CUDA(cudaMemcpy2DAsync(idx->d_adj + first * idx->adj_stride, (size_t)idx->adj_stride * 4, adj,
                               (size_t)src_stride * 4, copy_words * 4, count,
                               on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, idx->stream));
    DAB_CUDA(cudaStreamSynchronize(idx->stream));
    idx->graph_ready = true;
    return DAB_OK;
}

int dab_upload_graph(dab_index* idx, const uint32_t* adj, uint32_t src_stride, uint64_t first, uint64_t count) {
    return upload_graph(idx, adj, src_stride, first, count, false);
}
int dab_upload_graph_device(dab_index* idx, const uint32_t* d_adj, uint32_t src_stride, uint64_t first,
                            uint64_t count) {
    return upload_graph(idx, d_adj, src_stride, first, count, true);
}

int dab_download_graph(dab_index* idx, uint32_t* adj, uint32_t dst_stride, uint64_t first, uint64_t count) {
    if (!idx || (!adj && count)) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_download_graph: NULL argument");
    if (first + count > idx->n_total()) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_download_graph: rows out of range");
    if (dst_stride < idx->max_degree + 1)
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_download_graph: dst_stride %u < max_degree + 1", dst_stride);
    if (count == 0) return DAB_OK;
    DAB_CUDA(cudaSetDevice(idx->device));
    DAB_CUDA(cudaMemcpy2DAsync(adj, (size_t)dst_stride * 4, idx->d_adj + first * idx->adj_stride,
                               (size_t)idx->adj_stride * 4, ((size_t)idx->max_degree + 1) * 4, count,
                               cudaMemcpyDeviceToHost, idx->stream));
    DAB_CUDA(cudaStreamSynchronize(idx->stream));
    return DAB_OK;
}

int dab_upload_pq(dab_index* idx, const float* pivots, uint32_t n_centers, const uint64_t* offsets,
                  uint32_t n_chunks, const uint8_t* codes) {
    if (!idx || !pivots || !offsets) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_upload_pq: NULL argument");
    if (n_centers == 0 || n_centers > 256)
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_upload_pq: n_centers must be in [1, 256] (got %u)", n_centers);
    if (n_chunks == 0 || n_chunks > idx->dim)
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_upload_pq: n_chunks must be in [1, dim]");
    // ChunkOffsets invariants (fixed_chunk_pq_table.rs:112-124)
    if (offsets[0] != 0 || offsets[n_chunks] != idx->dim)
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_upload_pq: offsets must start at 0 and end at dim");
    std::vector<uint32_t> off32(n_chunks + 1);
    for (uint32_t c = 0; c <= n_chunks; ++c) {
        if (c && offsets[c] <= offsets[c - 1])
            return fail(DAB_ERR_INVALID_ARGUMENT, "dab_upload_pq: offsets must be strictly increasing");
        off32[c] = (uint32_t)offsets[c];
    }
    DAB_CUDA(cudaSetDevice(idx->device));
    cudaFree(idx->d_pivots);
    cudaFree(idx->d_offsets);
    cudaFree(idx->d_codes);
    idx->d_pivots = nullptr;
    idx->d_offsets = nullptr;
    idx->d_codes = nullptr;
    DAB_CUDA(cudaMalloc(&idx->d_pivots, (size_t)n_centers * idx->dim * 4));
    DAB_CUDA(cudaMalloc(&idx->d_offsets, (size_t)(n_chunks + 1) * 4));
    DAB_CUDA(cudaMalloc(&idx->d_codes, idx->n_total() * (size_t)n_chunks));
    DAB_CUDA(cudaMemcpy(idx->d_pivots, pivots, (size_t)n_centers * idx->dim * 4, cudaMemcpyHostToDevice));
    DAB_CUDA(cudaMemcpy(idx->d_offsets, off32.data(), (size_t)(n_chunks + 1) * 4, cudaMemcpyHostToDevice));
    if (codes)
        DAB_CUDA(cudaMemcpy(idx->d_codes, codes, idx->n_total() * (size_t)n_chunks, cudaMemcpyHostToDevice));
    else
        DAB_CUDA(cudaMemset(idx->d_codes, 0, idx->n_total() * (size_t)n_chunks));
    idx->pq_chunks = n_chunks;
    idx->pq_centers = n_centers;
    idx->pq_uniform_len = off32[1] - off32[0];
    for (uint32_t c = 1; c < n_chunks; ++c)
        if (off32[c + 1] - off32[c] != idx->pq_uniform_len) idx->pq_uniform_len = 0;
    idx->pq_codes_ready = codes != nullptr;
    return DAB_OK;
}

}  // extern "C"
