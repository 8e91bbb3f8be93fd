// search_v2.cuh — launch parameters of search_kernel_v2, shared by the kernel
// (search_kernel_v2.cu) and the host dispatcher (run_search, search_kernel.cu).
#pragma once

#include "dab_common.cuh"

namespace dab {

constexpr int kV2Warps = 1;  // warps per CTA (each warp owns a query)

struct SearchParamsV2 {
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
    uint32_t* tables;
    uint32_t n_buckets;   // visited table: buckets of 8 ids (32 B) per warp, any count >= 16
    // level 1 of the visited set: per-warp table of 16-bit quotient tags in shared memory (search_common.cuh)
    uint32_t t1_buckets;  // buckets of 16 tags (0: off — ids too wide for 14-bit tags, or disabled)
    uint32_t t1_limit;    // ids after which level 1 takes no more (87.5 % of its slots)
    uint32_t tag_kmask, tag_magic, tag_shift, off_t1;
    uint32_t* counters;
    uint32_t* overflow_list;
    uint32_t* rec_ids;
    float* rec_dists;
    uint32_t* rec_counts;
    uint32_t rec_cap;
    // per-warp shared memory layout (bytes)
    uint32_t warp_smem, off_q, off_qd, off_qi, off_cid, off_cd, off_beam, off_rows, off_adj;
    uint32_t adj_words;   // words of an adjacency row prefetched into shared memory (0: L2 prefetch only)
    uint32_t row_bytes;   // bytes copied per row (multiple of 16)
    uint32_t row_slot;    // bytes between staged rows
    uint32_t stage_rows;  // rows staged per round (multiple of kGroup)
};

struct V2Launch {
    void (*kern)(const SearchParamsV2);
    size_t smem_block;
    int grid;
};

// Returns 1 when this configuration is not covered by v2 (caller falls back to the generic
// kernel), 0 on success with `out` filled, or a negative DAB error code.
// `level1`: give the visited set its shared-memory level (see search_kernel_v2.cu) when the configuration allows it.
int v2_prepare(const dab_index* idx, uint32_t l_search, uint32_t beam, bool level1, SearchParamsV2& p, V2Launch& out);

}  // namespace dab
