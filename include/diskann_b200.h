/*
 * diskann_b200.h — C ABI of the B200-native distance hot path for microsoft/DiskANN (DiskANN3).
 *
 * This is the drop-in boundary (SURVEY.md §8b): a plain-C shared library
 * (libdiskann_b200.so, sm_100a CUDA inside) whose entry points are what a Rust `-sys` crate
 * for this path binds.  Conventions mirror the reference's only FFI precedent,
 * diskann-garnet/src/lib.rs:262-630: opaque handle, (pointer, length) pairs, integer status,
 * no unwinding across the boundary, caller owns every host buffer, the library owns device
 * memory.  INTEGRATION.md shows the reference-side binding.
 *
 * Each entry point cites the reference interface it replaces (paths relative to the
 * reference checkout).
 *
 * Value conventions are the reference's (diskann-vector/src/distance/distance_provider.rs:
 * 30-43, implementations.rs:217-404): L2 -> sum (x-y)^2 (no sqrt); InnerProduct -> -sum xy;
 * Cosine -> 1 - cos (clamped); CosineNormalized -> 1 - sum xy (== Cosine for i8/u8).
 * Float results are bit-identical to the reference's x86-64-v3 SIMD order; integer and PQ
 * results are exact.
 */
#ifndef DISKANN_B200_H
#define DISKANN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* element types: diskann/src/utils/vector_repr.rs:117-190 (f32, f16, i8, u8) */
enum { DAB_F32 = 0, DAB_F16 = 1, DAB_I8 = 2, DAB_U8 = 3 };

/* diskann-vector/src/distance/metric.rs:8-20, #[repr(C)] values */
enum { DAB_COSINE = 0, DAB_INNER_PRODUCT = 1, DAB_L2 = 2, DAB_COSINE_NORMALIZED = 3 };

/* status codes (0 == ok); dab_last_error() has the message (maps to ANNError::message) */
enum {
    DAB_OK = 0,
    DAB_ERR_INVALID_ARGUMENT = 1, /* bad dtype/metric/length: layers/full.rs:203-213, 306-314 */
    DAB_ERR_CUDA = 2,
    DAB_ERR_OUT_OF_MEMORY = 3,
    DAB_ERR_VISITED_OVERFLOW = 4, /* per-query visited set exceeded its capacity (retried internally) */
    DAB_ERR_NOT_READY = 5,        /* e.g. search before vectors/graph were uploaded */
    DAB_ERR_NO_DEVICE = 6
};

typedef struct dab_index dab_index; /* opaque */

/* ------------------------------------------------------------------ lifecycle */

/* Replaces diskann_inmem::Provider::new(layer, config, start_points)
 * (diskann-inmem/src/provider.rs:71-131) + layers::Full::<T>::new(dim, metric)
 * (diskann-inmem/src/layers/full.rs:368-504) for the device-resident snapshot:
 * n_points data rows (ids [0, n_points)) + n_start frozen start rows
 * (ids [n_points, n_points + n_start)), adjacency rows of max_degree + 1 words. */
int dab_create(dab_index** out, int dtype, int metric, uint32_t dim, uint64_t n_points,
               uint32_t n_start, uint32_t max_degree, int device);
void dab_destroy(dab_index* idx);

/* thread-local message of the last failing call on this thread */
const char* dab_last_error(void);

/* Launch on the caller's CUDA stream (cudaStream_t passed as void*); NULL restores the
 * library's own stream. */
int dab_set_stream(dab_index* idx, void* cuda_stream);

/* number of kernels this library has launched in this process (bench.py "gpu_launches") */
uint64_t dab_launch_count(void);

/* ------------------------------------------------------------------ data upload */

/* layers::Set<T>::set(element, bytes) (diskann-inmem/src/layers/mod.rs:79-96) /
 * Provider::set_element (provider.rs:341-372): dense row-major rows of dim elements, no
 * tags.  `first` may address start rows (first >= n_points).  Host or device source. */
int dab_upload_vectors(dab_index* idx, const void* rows, uint64_t first, uint64_t count);
int dab_upload_vectors_device(dab_index* idx, const void* d_rows, uint64_t first, uint64_t count);

/* Neighbors buffer (diskann-inmem/src/neighbors.rs:69-163): row = [len, id_0 .. id_{len-1}],
 * src_stride words between source rows (>= max_degree + 1). */
int dab_upload_graph(dab_index* idx, const uint32_t* adj, uint32_t src_stride, uint64_t first,
                     uint64_t count);
int dab_upload_graph_device(dab_index* idx, const uint32_t* d_adj, uint32_t src_stride,
                            uint64_t first, uint64_t count);
int dab_download_graph(dab_index* idx, uint32_t* adj, uint32_t dst_stride, uint64_t first,
                       uint64_t count);

/* FixedChunkPQTable::new(dim, pq_table, chunk_offsets)
 * (diskann-providers/src/model/pq/fixed_chunk_pq_table.rs:104-135) + the compressed
 * vectors of the quant store: pivots [n_centers][dim] f32, offsets [n_chunks + 1],
 * codes [(n_points + n_start)][n_chunks] (may be NULL, then call dab_pq_encode_all; a PQ
 * traversal before that returns DAB_ERR_NOT_READY). */
int dab_upload_pq(dab_index* idx, const float* pivots, uint32_t n_centers,
                  const uint64_t* offsets, uint32_t n_chunks, const uint8_t* codes);

/* train_pq (diskann-providers/src/index/diskann_async.rs:61-89 -> model/pq/pq_construction.rs:163-243
 * -> diskann-quantization/src/product/train.rs): per chunk k-means++ seeding
 * (algorithms/kmeans/plusplus.rs:381-498) and `lloyds_reps` Lloyd iterations (lloyds.rs:372-426; the
 * benchmark uses 5) over n host training rows [n][dim] f32, entirely on the device, arithmetic in the
 * reference's order.  Chunk offsets are ChunkOffsets::partition (quantization/src/views.rs:226-243).
 * The random draws come from SplitMix64(seed + chunk) (the reference's StdRng is not reproduced).
 * Replaces the resident table; codes are cleared until dab_pq_encode_all. */
int dab_pq_train(dab_index* idx, const float* train, uint64_t n, uint32_t n_chunks, uint32_t n_centers,
                 uint32_t lloyds_reps, uint64_t seed);
/* BasicTable::compress_into (product/tables/basic.rs:161-194) for every uploaded row (converted to
 * f32, T: Into<f32>) into the resident codes — the quant store of a quantized build. */
int dab_pq_encode_all(dab_index* idx);
/* copies the resident table back: pivots [n_centers][dim], offsets [n_chunks + 1], codes
 * [(n_points + n_start)][n_chunks]; any pointer may be NULL. */
int dab_pq_download(dab_index* idx, float* pivots, uint64_t* offsets, uint8_t* codes);

/* ------------------------------------------------------------------ replication across GPUs */

/* The index is replicated, the query batch is sharded, the search path has no collective
 * (benchmark-core/src/search/api.rs:410-419 partitions queries over tasks the same way; SURVEY.md §8e).
 * One NCCL broadcast per resident buffer (vectors, adjacency, PQ table and codes) at load.  NCCL is
 * resolved with dlopen("libnccl.so.2") at first use; DAB_ERR_NOT_READY if it cannot be loaded.
 * One process per GPU: rank 0 calls dab_comm_unique_id and ships the 128 bytes to the other ranks,
 * every rank calls dab_comm_init on its own handle (created with the same shape), then
 * dab_broadcast_index(idx, root).  dab_destroy releases the communicator. */
int dab_comm_unique_id(char* out_id128);
int dab_comm_init(dab_index* idx, const char* id128, int n_ranks, int rank);
int dab_broadcast_index(dab_index* idx, int root);
int dab_comm_destroy(dab_index* idx);
/* One process driving several GPUs: per_gpu[0] is the root, per_gpu[i] lives on its own device. */
int dab_broadcast(dab_index* const* per_gpu, int n_gpus);

/* ------------------------------------------------------------------ (1) per-pair / per-query distances */

/* DistanceProvider::distance_comparer(metric, dim) -> Distance<T,U>::call
 * (diskann-vector/src/distance/distance_provider.rs:44-46, 86) and
 * layers::Distance::evaluate(x, y) (diskann-inmem/src/layers/mod.rs:68-77): n independent
 * pairs x[i] . y[i], host buffers, dense rows.  Supported (dtype_x, dtype_y): (f32,f32)
 * (f16,f16) (f32,f16) (i8,i8) (u8,u8).  Stateless: no index needed. */
int dab_pair_distances(int dtype_x, int dtype_y, int metric, uint32_t dim, const void* x,
                       const void* y, uint64_t n, float* out, int device);

/* SearchAccessor::expand_beam's distance stage batched over queries
 * (diskann-inmem/src/provider.rs:436-479, 620-690; glue.rs:210-219):
 * out[q][j] = QueryDistance(query q).evaluate(row ids[q][j]); ids == UINT32_MAX are skipped
 * (out = NaN).  Queries have the index dtype (f16 queries are widened once,
 * layers/full.rs:421-423). */
int dab_distances(dab_index* idx, const void* queries, uint32_t nq, const uint32_t* ids,
                  uint32_t c, float* out);
int dab_distances_device(dab_index* idx, const void* d_queries, uint32_t nq,
                         const uint32_t* d_ids, uint32_t c, float* d_out);

/* PruneAccessor::fill + Distance: DistanceFunction<ElementRef, ElementRef>
 * (diskann/src/graph/glue.rs:855-906; index.rs:2623-2625): data x data distances.
 * out[i] = Distance<T,T>(row a[i], row b[i]). */
int dab_row_pair_distances(dab_index* idx, const uint32_t* a, const uint32_t* b, uint64_t n,
                           float* out);
/* candidate x candidate block for robust_prune: out[i][j] = Distance<T,T>(ids[i], ids[j]) */
int dab_pairwise(dab_index* idx, const uint32_t* ids, uint32_t n, float* out);

/* ------------------------------------------------------------------ (3') batched greedy search */

/* DiskANNIndex::search_internal + Knn::search + post-process for a whole query batch
 * (diskann/src/graph/index.rs:1933-2000; graph/search/knn_search.rs:170-190;
 * diskann-inmem/src/provider.rs:907-950), i.e. benchmark_core::search::graph::KNN::search
 * (diskann-benchmark-core/src/search/graph/knn.rs:208-238) for every query at once.
 * Results exclude start points; rows are padded with id UINT32_MAX / distance +inf;
 * out_counts/out_cmps/out_hops may be NULL.  cmps/hops follow SearchStats
 * (index.rs:1990-1991). */
int dab_search_batch(dab_index* idx, const void* queries, uint32_t nq, uint32_t k, uint32_t l_search,
                     uint32_t beam_width, uint32_t* out_ids, float* out_dists,
                     uint32_t* out_counts, uint32_t* out_cmps, uint32_t* out_hops);
int dab_search_batch_device(dab_index* idx, const void* d_queries, uint32_t nq, uint32_t k,
                            uint32_t l_search, uint32_t beam_width, uint32_t* d_out_ids,
                            float* d_out_dists, uint32_t* d_out_counts, uint32_t* d_out_cmps,
                            uint32_t* d_out_hops);

/* Batches in flight.  The reference keeps every core busy by handing each query to a task of a
 * thread pool (diskann-benchmark-core/src/search/api.rs:410-419: `search_all` spawns one task per
 * query partition and joins them); the device equivalent is to keep more than one BATCH in flight:
 * `dab_search_batch_async` queues the copy of the queries, the search and the copy of the results
 * on a stream owned by `slot` (0 <= slot < DAB_MAX_SLOTS) and returns without waiting, `dab_wait`
 * joins the slot.  Batches on different slots overlap: the host<->device copies of one run under
 * the kernel of another, and the CTAs of the next batch fill the SMs that the draining tail of the
 * previous one leaves idle.  Results, statistics and error behaviour are those of dab_search_batch;
 * the host buffers (pinned memory makes the copies asynchronous) and the device buffers of the
 * `_device_` flavour must stay valid and untouched until `dab_wait(slot)` returns.  A slot holds
 * one batch at a time (DAB_ERR_INVALID_ARGUMENT otherwise); waiting on an idle slot is a no-op. */
#define DAB_MAX_SLOTS 4
int dab_search_batch_async(dab_index* idx, uint32_t slot, const void* queries, uint32_t nq, uint32_t k,
                           uint32_t l_search, uint32_t beam_width, uint32_t* out_ids, float* out_dists,
                           uint32_t* out_counts, uint32_t* out_cmps, uint32_t* out_hops);
int dab_search_batch_device_async(dab_index* idx, uint32_t slot, const void* d_queries, uint32_t nq, uint32_t k,
                                  uint32_t l_search, uint32_t beam_width, uint32_t* d_out_ids,
                                  float* d_out_dists, uint32_t* d_out_counts, uint32_t* d_out_cmps,
                                  uint32_t* d_out_hops);
int dab_wait(dab_index* idx, uint32_t slot);

/* ------------------------------------------------------------------ product quantization */

/* FixedChunkPQTable::populate_chunk_distances / populate_chunk_inner_products
 * (fixed_chunk_pq_table.rs:152-218): lut[q][chunk][center]; metric L2 or InnerProduct. */
int dab_pq_populate_lut(dab_index* idx, const float* queries, uint32_t nq, int metric, float* out_lut);

/* QueryComputer::evaluate_similarity over gathered codes
 * (pq/distance/dynamic.rs:63-103; pq_dist_lookup_single, fixed_chunk_pq_table.rs:82-98;
 * compute_pq_distance :617-670): out[q][j] for ids[q][j].  Queries are f32. */
int dab_pq_distances(dab_index* idx, const float* queries, uint32_t nq, const uint32_t* ids,
                     uint32_t c, float* out);

/* DistanceComputer::evaluate_similarity(code, code) (pq/distance/dynamic.rs:101-140; the PQ prune path):
 * FixedChunkPQTable::{qq_l2_distance, qq_inner_product, qq_cosine_distance}
 * (fixed_chunk_pq_table.rs:285-361) between the stored codes of rows a[i] and b[i] under the index
 * metric (CosineNormalized -> cosine, VTable dynamic.rs:126-131).  Resumable accumulation across chunks. */
int dab_pq_self_distances(dab_index* idx, const uint32_t* ids_a, const uint32_t* ids_b, uint64_t n, float* out);

/* The providers' PQ traversal: QuantAccessor::expand_beam with
 * `computer.evaluate_similarity(aux_vectors[i])`
 * (diskann-providers/src/model/graph/provider/async_/inmem/product.rs:311-340) inside
 * search_internal — dab_search_batch with every traversal distance an ADC lookup over the
 * uploaded codes (start points included).  Queries have the index dtype and are converted to
 * f32 (T: Into<f32>); L2 / CosineNormalized use TableL2, InnerProduct TableIP; Metric::Cosine
 * runs QueryComputer::DirectCosine (pq/distance/cosine.rs:16-70: no table, the resumable cosine
 * over the pivot chunks a code selects).  No rerank: distances returned are the traversal values. */
int dab_search_batch_pq(dab_index* idx, const void* queries, uint32_t nq, uint32_t k, uint32_t l_search,
                        uint32_t beam_width, uint32_t* out_ids, float* out_dists,
                        uint32_t* out_counts, uint32_t* out_cmps, uint32_t* out_hops);

/* The same followed by the quantized providers' default post-processing
 * Pipeline<FilterStartPoints, Rerank> (inmem/product.rs:391-400; full_precision.rs:356-399): every
 * entry of the candidate list that is not a start point is re-scored with the full-precision
 * Distance<T, T> over the uploaded rows, the list is ordered by that distance (ties keep their
 * traversal order; the reference leaves them unspecified) and the first k are returned — what
 * `use_fp_for_search: false` runs in diskann-benchmark (src/index/inmem/product.rs:233-239).
 * Every row type and metric of the index: f32 / f16 / i8 / u8 (f16 x f16 and Metric::Cosine over float rows use the
 * schemas with two accumulators, simd.rs:424-483). */
int dab_search_batch_pq_rerank(dab_index* idx, const void* queries, uint32_t nq, uint32_t k, uint32_t l_search,
                               uint32_t beam_width, uint32_t* out_ids, float* out_dists,
                               uint32_t* out_counts, uint32_t* out_cmps, uint32_t* out_hops);
/* device-pointer variant of both (rerank = 0 / 1); results stay in HBM */
int dab_search_batch_pq_device(dab_index* idx, const void* d_queries, uint32_t nq, uint32_t k, uint32_t l_search,
                               uint32_t beam_width, int rerank, uint32_t* d_out_ids, float* d_out_dists,
                               uint32_t* d_out_counts, uint32_t* d_out_cmps, uint32_t* d_out_hops);

/* BasicTable::compress_into (diskann-quantization/src/product/tables/basic.rs:161-194) for n
 * host vectors (f32): codes [n][n_chunks].  Returns DAB_ERR_INVALID_ARGUMENT if a chunk's
 * minimum distance is infinite/NaN (first offending row/chunk in the message). */
int dab_pq_encode(dab_index* idx, const float* vectors, uint64_t n, uint8_t* out_codes);

/* ------------------------------------------------------------------ scalar quantization */

/* ScalarQuantizer::compress_into (diskann-quantization/src/scalar/quantizer.rs:190-239,
 * 407-430): codes one per byte in [0, 2^nbits), compensation per vector. */
int dab_sq_compress(int device, const float* shift, float scale, uint32_t dim, int nbits,
                    const float* vectors, uint64_t n, uint8_t* out_codes, float* out_comp);

/* CompensatedSquaredL2 / CompensatedIP / CompensatedCosineNormalized
 * (scalar/vectors.rs:206-237, 310-376, 380-460) for n code pairs. */
int dab_sq_distances(int device, int metric, int nbits, float scale_squared, float shift_square_norm,
                     uint32_t dim, const uint8_t* x, const float* comp_x, const uint8_t* y,
                     const float* comp_y, uint64_t n, float* out);

/* The scalar-quantized store of an index (diskann-providers/src/model/graph/provider/async_/inmem/
 * scalar.rs:60-258, SQStore<NBITS>): the quantizer (ScalarQuantizer: shift[dim], scale, and the two
 * derived fields quantizer.shift_square_norm() and quantizer.mean_norm(), 0 when None) and one row
 * per point (data + start points) in the reference's canonical-front layout (diskann-quantization/
 * src/meta/vector.rs:478-507): 4 bytes f32 compensation, then ceil(dim * nbits / 8) bytes of
 * Dense-packed codes (bits/slice.rs:261-323) — what set_quant_vector (:193-212) stores.  rows may
 * be NULL when dab_sq_encode_all follows.  nbits in {1, 2, 4, 8}. */
int dab_upload_sq(dab_index* idx, int nbits, const float* shift, float scale, float shift_square_norm,
                  float mean_norm, const uint8_t* rows);
/* SQStore::set_vector (scalar.rs:150-175) for every resident row (any dtype, as_f32 first). */
int dab_sq_encode_all(dab_index* idx);
/* rows back in the canonical-front layout: (n_points + n_start) x (4 + ceil(dim * nbits / 8)) */
int dab_sq_download(dab_index* idx, uint8_t* rows);

/* KNN::search through the scalar-quantized accessor (scalar.rs:449-570): the query is compressed
 * with the store's quantizer (query_computer, :227-253; rescaled to mean_norm for InnerProduct) and
 * every traversal distance is Compensated{SquaredL2, IP, CosineNormalized} over the packed codes
 * (scalar/vectors.rs:206-460; integer cores bits/distances.rs:397, 979).  rerank = 0: the
 * quant-only strategy (RemoveDeletedIdsAndCopy: first k of the candidate list with their quantized
 * distances, scalar.rs:640-670); rerank = 1: Pipeline<FilterStartPoints, Rerank> with the
 * full-precision rows (:596-610).  Metric::Cosine is rejected like SQStore::distance_computer
 * (:214-226).  Outputs as dab_search_batch. */
int dab_search_batch_sq(dab_index* idx, const void* queries, uint32_t nq, uint32_t k, uint32_t l_search,
                        uint32_t beam_width, int rerank, uint32_t* out_ids, float* out_dists,
                        uint32_t* out_counts, uint32_t* out_cmps, uint32_t* out_hops);
int dab_search_batch_sq_device(dab_index* idx, const void* d_queries, uint32_t nq, uint32_t k, uint32_t l_search,
                               uint32_t beam_width, int rerank, uint32_t* d_out_ids, float* d_out_dists,
                               uint32_t* d_out_counts, uint32_t* d_out_cmps, uint32_t* d_out_hops);

/* ------------------------------------------------------------------ MinMax quantization */

/* The per-vector N-bit quantizer of diskann-quantization/src/minmax (NBITS = 1, 2, 4, 8; Transform::Null).  Rows use the
 * reference's canonical-front layout of minmax::Data<NBITS> (meta/vector.rs:377-392): MinMaxCompensation
 * {dim: u32, b, n, a, norm_squared} (vectors.rs:43-52, 20 bytes) followed by ceil(dim * NBITS / 8) bytes of dense codes,
 * value i at bit i * NBITS — so rows written here can be handed to DataRef::from_canonical_front and back. */
uint32_t dab_minmax_row_bytes(uint32_t dim, int nbits);  /* Data::<NBITS>::canonical_bytes(dim); 0 for an unsupported width */

/* MinMaxQuantizer::new(Transform::Null(dim), grid_scale) + CompressInto<&[f32], DataMutRef<NBITS>> for n vectors
 * (quantizer.rs:153-228, get_range :117-151): out_rows [n][dab_minmax_row_bytes], out_loss [n] (L2Loss, may be NULL).
 * An input vector containing NaN makes the call fail (InputContainsNaN, naming the first such vector) after every row
 * has been written, the way the reference sets the meta before returning the error. */
int dab_minmax_compress(int device, float grid_scale, uint32_t dim, int nbits, const float* vectors, uint64_t n,
                        uint8_t* out_rows, float* out_loss);

/* PureDistanceFunction<DataRef<NBITS>, DataRef<MBITS>, distances::Result<f32>> for MinMaxL2Squared / MinMaxIP (negated) /
 * MinMaxCosine / MinMaxCosineNormalized (vectors.rs:206-455), selected by `metric` (Metric repr): out[i] = d(x_rows[i],
 * y_rows[i]).  Widths: N x N, and 8 x N (the pairings the reference instantiates).  Rows whose stored dimension differs
 * from `dim` give NaN (UnequalLengths). */
int dab_minmax_distances(int device, int metric, int nbits_x, int nbits_y, uint32_t dim, const uint8_t* x_rows,
                         const uint8_t* y_rows, uint64_t n, float* out);

/* The query side of the minmax-exhaustive-search benchmark (diskann-benchmark/src/exhaustive/minmax.rs): queries stay
 * full precision — CompressInto<&[f32], FullQueryMut> (quantizer.rs:369-417: FullQueryMeta {sum, norm_squared}) — and
 * PureDistanceFunction<FullQueryRef, DataRef<NBITS>, distances::Result<f32>> for the four MinMax distances
 * (vectors.rs:272-305, 347-392, 417-476) is evaluated for every (query, row) pair: out [nq][n].  The f32 x N-bit inner
 * product follows the reference's x86-64-v3 kernels lane for lane (bits/distances.rs:2295-2725).  A query containing NaN
 * fails the call (InputContainsNaN). */
int dab_minmax_query_distances(int device, int metric, int nbits, uint32_t dim, const float* queries, uint32_t nq,
                               const uint8_t* rows, uint64_t n, float* out);

/* ------------------------------------------------------------------ build-side reuse */

/* PruneAccessor::fill + robust_prune (diskann/src/graph/index.rs:2349-2380, 2565-2650;
 * graph/internal/prune.rs:106-259; PruneKind graph/config/mod.rs:80-103) for n_pools
 * independent candidate pools: pool p has pool_lens[p] (id, source distance) entries in
 * pool_ids/pool_dists[p * pool_cap ...] (any order; sorted by distance then arrival order and
 * truncated to max_occlusion_size = 750 like SortedNeighbors::new), locations[p] is the node
 * being pruned (excluded from its own pool).  Candidate x candidate distances are
 * Distance<T,T> over the uploaded rows.  out_ids [n_pools][degree] (padded UINT32_MAX). */
int dab_robust_prune(dab_index* idx, const uint32_t* pool_ids, const float* pool_dists,
                     const uint32_t* pool_lens, const uint32_t* locations, uint32_t n_pools,
                     uint32_t pool_cap, uint32_t degree, float alpha, uint32_t* out_ids,
                     uint32_t* out_counts);

/* Batched Vamana construction on the device (the rows SURVEY.md §8f.2 marks "next"):
 * DiskANNIndex::multi_insert semantics (diskann/src/graph/index.rs:815) — batches of inserts
 * searched with the same search kernel, pruned with robust_prune
 * (graph/internal/prune.rs:106-259) and back-edges merged per destination (aggregate_backedges :123, one
 * add_edge_and_prune per target: extend with every source, prune once).  intra_batch_candidates = None; the
 * bootstrap routine (index.rs:589-747, run by the reference while a batch's back-edges reach <= 8 x batch distinct
 * targets) is NOT run: batch_size = 1 is DiskANNIndex::insert point by point, larger batches grow as inserted / 8 up
 * to batch_size (0: a default from the index size) so that no point is inserted blind.  Uses the uploaded vectors
 * (including start rows) and overwrites the adjacency. */
int dab_build(dab_index* idx, uint32_t pruned_degree, uint32_t l_build, float alpha,
              uint32_t batch_size);

/* exact k-NN by exhaustive scan (diskann/src/flat; ground truth for recall):
 * out_ids [nq][k] ascending distance, ties by lower id. */
int dab_flat_knn(dab_index* idx, const void* queries, uint32_t nq, uint32_t k, uint32_t* out_ids,
                 float* out_dists);

/* The same scan on the tensor cores (BASELINE.json north_star: "the query x neighbour distance batch is a
 * tcgen05 tensor-core GEMM ... with TMA-staged vector tiles and fused ||x||^2 + ||y||^2 expansion"):
 * bf16 operands (f32 / f16 rows as a 3-product hi/lo split, i8 / u8 exact), fp32 accumulation in TMEM,
 * fused score expansion and per-row candidate selection in the epilogue; the candidates are then
 * re-scored with the exact reference-order kernel, so out_dists are bit-identical to dab_flat_knn and
 * out_ids equal it unless approximate scores (~1e-5 relative) displace a true neighbour by more than
 * the selection slack.  k <= 24. */
int dab_flat_knn_tc(dab_index* idx, const void* queries, uint32_t nq, uint32_t k, uint32_t* out_ids,
                    float* out_dists);

#ifdef __cplusplus
}
#endif
#endif
