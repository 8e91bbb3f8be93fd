// dab_common.cuh — shared host-side plumbing for libdiskann_b200.so (index handle, error
// reporting, launch accounting).  Compiled for sm_100a only.
#pragma once

#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>

#include "../../include/diskann_b200.h"

struct dab_index;

namespace dab {

constexpr uint32_t kNoId = 0xFFFFFFFFu;

// thread-local error message (dab_last_error)
char* error_buffer();
int fail(int code, const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;
void comm_release(struct ::dab_index* idx);  // replicate.cu
void tc_release(struct ::dab_index* idx);    // flat_tc.cu
void search_slots_release(struct ::dab_index* idx);  // search_kernel.cu

#define DAB_CUDA(expr)                                                                        \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess)                                                                \
            return ::dab::fail(_e == cudaErrorMemoryAllocation ? DAB_ERR_OUT_OF_MEMORY         \
                                                               : DAB_ERR_CUDA,               \
                               "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),        \
                               __FILE__, __LINE__);                                           \
    } while (0)

#define DAB_LAUNCHED() (::dab::g_launches.fetch_add(1, std::memory_order_relaxed))

inline size_t elem_size(int dtype) {
    switch (dtype) {
        case DAB_F32: return 4;
        case DAB_F16: return 2;
        default: return 1;
    }
}
inline size_t round_up(size_t x, size_t m) { return (x + m - 1) / m * m; }

// A grow-only device (or pinned host) scratch buffer.
struct Scratch {
    void* p = nullptr;
    size_t bytes = 0;
    bool pinned_host = false;
    int reserve(size_t n);
    void release();
};

// Test hooks, read from the environment once at dab_create.  They let tests reach paths that small
// inputs never select; none changes a result.
struct TestHooks {
    int test_visited_log2 = 0;  // DAB_TEST_VISITED_LOG2: visited tables small enough to take the overflow / re-run paths
    bool pq_global_lut = false;  // DAB_TEST_PQ_GLOBAL_LUT: per-query PQ tables in global memory (search_kernel_pq MODE 0,
                                 // pq_lut_kernel + pq_adc_kernel) even where they fit shared memory
    void load();
};

}  // namespace dab

struct dab_index {
    int dtype = 0, metric = 0;
    uint32_t dim = 0;
    uint64_t n_points = 0;
    uint32_t n_start = 0;
    uint32_t max_degree = 0;
    int device = 0;
    int sm_count = 148;

    cudaStream_t stream = nullptr;      // stream in use
    cudaStream_t own_stream = nullptr;  // library-created

    // HBM-resident snapshot
    uint8_t* d_vectors = nullptr;  // (n_points + n_start) rows, row_stride bytes apart
    size_t row_stride = 0;         // round_up(dim * sizeof(T), 32): rows start on sector bounds
    uint32_t* d_adj = nullptr;     // (n_points + n_start) rows of adj_stride words: [len, ids...]
    uint32_t adj_stride = 0;       // round_up(max_degree + 1, 8) words (32 B multiple)
    bool vectors_ready = false, graph_ready = false;

    // product quantization
    float* d_pivots = nullptr;     // [n_centers][dim]
    uint32_t* d_offsets = nullptr; // [n_chunks + 1]
    uint8_t* d_codes = nullptr;    // [n_total][n_chunks]
    uint32_t pq_chunks = 0, pq_centers = 0;
    uint32_t pq_uniform_len = 0;   // every chunk has this many dimensions (0: lengths differ)
    bool pq_codes_ready = false;   // codes uploaded (dab_upload_pq) or produced (dab_pq_encode_all)
    // scalar-quantized store (providers inmem/scalar.rs SQStore<NBITS>): dense N-bit codes, one 16 B-aligned
    // row per point, compensations apart (only the inner-product epilogue reads them)
    int sq_nbits = 0;
    float sq_scale = 0.0f, sq_shift_square_norm = 0.0f, sq_mean_norm = 0.0f;
    float* d_sq_shift = nullptr;   // [dim]
    uint8_t* d_sq_codes = nullptr; // [n_total][sq_stride]
    float* d_sq_comp = nullptr;    // [n_total]
    uint32_t sq_row_bytes = 0, sq_stride = 0;
    bool sq_codes_ready = false;

    // scratch (grow-only)
    dab::Scratch s_queries, s_ids, s_out, s_out2, s_tables, s_counters, s_stats;
    dab::Scratch h_stage;  // pinned host staging
    dab::Scratch h_counters;  // pinned: the four counters a search pass reports
    void* slots[DAB_MAX_SLOTS] = {};  // batches in flight (dab_search_batch_async), search_kernel.cu

    // search-side state learned across calls
    uint32_t hint_l = 0, hint_beam = 0, hint_visited = 0;  // largest visited set seen at (L, beam)
    uint32_t pq_hint_l = 0, pq_hint_beam = 0, pq_hint_visited = 0; int pq_hint_mode = 0;  // the same for the PQ traversal kernel
    uint32_t v3_overflow_l = 0, v3_overflow_beam = 0;      // share of queries that outgrew the shared-memory
    float v3_overflow_frac = 0.0f;                         // tables at (L, beam): search_kernel_v3 is skipped when large
    void* l2_window_ptr = nullptr;       // current persisting-L2 window (visited tables)
    size_t l2_window_bytes = 0;
    cudaStream_t l2_window_stream = nullptr;

    uint64_t rec_truncated = 0;  // build: searches whose expanded-node record was cut at its capacity
    dab::TestHooks hooks;

    // tensor-core exhaustive scan (flat_tc.cu): bf16 operand copy of the rows + score coefficients
    void* d_tc_base = nullptr;
    void* d_tc_coef = nullptr;
    uint64_t tc_version = 0, vectors_version = 1;  // the copy is rebuilt when rows were uploaded since

    // replication (replicate.cu): NCCL communicator of a one-process-per-GPU host
    void* nccl_comm = nullptr;
    int nccl_rank = 0, nccl_ranks = 0;

    uint64_t n_total() const { return n_points + n_start; }
};
