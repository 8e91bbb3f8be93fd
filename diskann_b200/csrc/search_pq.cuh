// search_pq.cuh — parameter block shared by the quantized-traversal kernels (search_kernel_pq.cu: per-warp table in
// global memory, SQ, DirectCosine; search_kernel_pqs.cu: pivots resident in shared memory).
#pragma once

#include "dab_common.cuh"

namespace dab {

constexpr int kPqWarps = 4;

struct SearchParamsPq {
    const uint8_t* vectors;  // only for the f32 view of the query rows in build-free search: unused
    const uint32_t* adj;
    uint32_t adj_stride;
    uint64_t n_points;
    uint32_t n_start;
    uint32_t dim;
    uint32_t max_degree;
    int dtype;
    const void* queries;
    const uint32_t* query_list;
    uint32_t n_work;
    uint32_t k, cap, beam;
    const float* pivots;
    const uint32_t* offsets;
    const uint8_t* codes;
    uint32_t n_chunks, n_centers;
    int ip_table;  // 1: TableIP (entries -dot), 0: TableL2
    int direct_cosine;  // 1: Metric::Cosine -> QueryComputer::DirectCosine (no table): resumable cosine over the gathered pivot chunks
    float* luts;   // [warps][n_chunks * n_centers]
    uint32_t* out_ids;
    float* out_dists;
    uint32_t* out_counts;
    uint32_t* out_cmps;
    uint32_t* out_hops;
    uint32_t* tables;
    uint32_t n_buckets;
    uint32_t* counters;
    uint32_t* overflow_list;
    // optional: the whole candidate list (best.iter()) for the rerank stage
    uint32_t* list_ids;     // [nq][list_cap]
    uint32_t* list_counts;  // [nq]
    uint32_t list_cap;
    // MODE 1: scalar-quantized store
    const uint8_t* sq_codes;  // [n_total][sq_stride], dense N-bit codes, zero padded to 16 B
    const float* sq_comp;     // [n_total]
    const float* sq_shift;    // [dim]
    uint32_t sq_stride;
    int sq_nbits, sq_metric;
    float sq_scale, sq_scale_squared, sq_shift_square_norm, sq_mean_norm;
    uint32_t warp_smem, off_q, off_qd, off_qi, off_cid, off_cd, off_beam, off_qc, off_nrow;
    // search_kernel_pqs: the pivot table of the CTA in shared memory
    uint32_t piv_stride;  // floats between pivot rows (odd multiple of 4: rows of different centres start in different 16-byte bank groups)
    uint32_t piv_bytes;   // n_centers * piv_stride * 4, the per-warp slices follow
};

// search_kernel_pqs.cu — the shape of one launch of the shared-memory-pivot kernel
struct PqsPlan {
    int warps;         // warps (= queries in flight) per CTA, one CTA per SM
    int grid;
    size_t smem;       // dynamic shared memory per CTA
    uint32_t piv_stride, piv_bytes;
    int chunk_len;     // 4 / 8: every chunk has this length (float4 loads, folded arithmetic); 0: generic
};
// false: this index / call does not fit the kernel (pivot table too large for shared memory, > 32 chunks, ...)
bool pqs_plan(const dab_index* idx, uint32_t warp_smem, uint32_t nq, PqsPlan* out);
int pqs_launch(dab_index* idx, const SearchParamsPq& p, const PqsPlan& plan, uint32_t cap);



}  // namespace dab
