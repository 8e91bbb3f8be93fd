// search_v3.cuh — launch parameters of search_kernel_v3 (visited set in shared memory), shared by
// the kernel (search_kernel_v3.cu) and the host dispatcher (run_search, search_kernel.cu).
#pragma once

#include "dab_common.cuh"

namespace dab {

constexpr int kV3Warps = 4;  // warps per CTA; every warp owns one query at a time

struct SearchParamsV3 {
    const uint8_t* vectors;
    size_t row_stride;
    const uint32_t* adj;
    uint32_t adj_stride;
    uint64_t n_points;
    uint32_t n_start;
    uint32_t dim;
    uint32_t max_degree;
    const void* queries;
    const uint32_t* query_rows;
    const uint32_t* query_list;
    uint32_t n_work;
    uint32_t k, cap, beam;
    uint32_t* out_ids;
    float* out_dists;
    uint32_t* out_counts;
    uint32_t* out_cmps;
    uint32_t* out_hops;
    uint32_t* counters;       // [0] work counter, [1] overflow count, [2] max visited
    uint32_t* overflow_list;  // queries whose visited set outgrew the shared-memory table
    uint32_t* rec_ids;
    float* rec_dists;
    uint32_t* rec_counts;
    uint32_t rec_cap;
    // visited set: 16-bit entries per warp in shared memory (search_smem.cuh): n_buckets buckets of 16 tags
    uint32_t n_buckets, tag_kmask, tag_magic, tag_shift, visited_limit;
    uint32_t fast_nm;  // f32 rows of 32 * fast_nm <= 128 elements: register-resident query, 8 rows per step (0: generic path)
    // per-warp shared memory layout (bytes)
    uint32_t warp_smem, off_q, off_qd, off_qi, off_cid, off_cd, off_beam, off_adj, off_table;
    uint32_t adj_words;  // words of an adjacency row prefetched into shared memory (0: off)
};

struct V3Launch {
    void (*kern)(const SearchParamsV3);
    size_t smem_block;
    int grid;         // resident CTAs on the device
    uint32_t capacity;  // ids a table holds before the query is handed to the global-table kernel
};

// Returns 1 when this configuration is not covered by v3 (caller uses v2 / the generic kernel),
// 0 on success with `out` filled.  `visited_need` = ids the table should hold (0: unknown).
int v3_prepare(const dab_index* idx, uint32_t l_search, uint32_t beam, uint32_t visited_need, SearchParamsV3& p, V3Launch& out);

}  // namespace dab
