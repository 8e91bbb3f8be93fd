// search_kernel.cu — batched greedy (beam) search kept entirely on the device.
//
// Restates DiskANNIndex::search_internal (diskann/src/graph/index.rs:1933-2000) with the
// reference's NeighborPriorityQueue semantics (diskann/src/neighbor/queue.rs:130-318) and the
// inmem expand_beam (diskann-inmem/src/provider.rs:436-479, 620-690), one warp per query:
//
//   * persistent warps pull queries from an atomic work counter (grid = SMs x resident CTAs);
//   * the sorted candidate list (capacity L + #start, scratch.rs:195-208) lives in shared
//     memory, inserted warp-cooperatively at the lower bound (new item before equal
//     distances; a full queue rejects only `last < new`; NaN ignored);
//   * the visited set (a HashSet in the reference) is an exact open-addressed table per warp
//     in global memory — sized from the reference's own estimate
//     (graph/search/scratch.rs:186-192), overflow is detected and the query is re-run with a
//     larger table, so membership semantics stay exact;
//   * adjacency rows ([len, ids...], diskann-inmem/src/neighbors.rs:69-163) are fetched with
//     coalesced 128 B loads, filtered against the visited set in adjacency order, and the
//     surviving rows are gathered straight from HBM into the bit-exact distance chains of
//     distance_device.cuh (U rows in flight per team);
//   * cmps / hops follow SearchStats (index.rs:1990-1991).
//
// HBM-gather bound by design: per (query, candidate) the kernel must move dim*sizeof(T) row
// bytes for ~2-3 flop/element — no tensor cores.
#include "dab_common.cuh"
#include "distance_device.cuh"
#include "search_v2.cuh"
#include "search_v3.cuh"

#include <algorithm>
#include <cstdlib>

namespace dab {

constexpr int kSearchWarps = 4;          // warps per CTA (independent queries)
constexpr uint32_t kEmpty = 0xFFFFFFFFu; // empty slot of the visited table
constexpr uint32_t kVisitedFlag = 0x80000000u;
constexpr int kRowsInFlight = 4;         // U: rows per team per pass

struct SearchParams {
    const uint8_t* vectors;
    size_t row_stride;
    const uint32_t* adj;
    uint32_t adj_stride;
    uint64_t n_points;
    uint32_t n_start;
    uint32_t dim;
    uint32_t max_degree;
    const void* queries;          // [nq][dim] of the index dtype, or NULL when query_rows is set
    const uint32_t* query_rows;   // build mode: the query is row query_rows[q] of the index
    const uint32_t* query_list;   // optional indirection (retry pass): work item -> query index
    uint32_t n_work;
    uint32_t k, cap, beam;
    uint32_t* out_ids;
    float* out_dists;
    uint32_t* out_counts;
    uint32_t* out_cmps;
    uint32_t* out_hops;
    uint32_t* tables;
    uint32_t hcap_log2;
    uint32_t* counters;           // [0] work counter, [1] overflow count, [2] max visited
    uint32_t* overflow_list;      // query indices whose visited table overflowed
    // optional record of expanded nodes (VisitedSearchRecord, used by the device build)
    uint32_t* rec_ids;
    float* rec_dists;
    uint32_t* rec_counts;
    uint32_t rec_cap;
    // shared-memory layout (bytes, per warp)
    uint32_t warp_smem, off_qd, off_qi, off_cid, off_cd, off_beam;
};

__device__ __forceinline__ uint32_t hash_id(uint32_t id, uint32_t log2cap) {
    return (id * 0x9E3779B1u) >> (32u - log2cap);
}

// returns true when `id` was not yet in the set (HashSet::insert)
__device__ __forceinline__ bool visited_insert(uint32_t* table, uint32_t log2cap, uint32_t id) {
    const uint32_t mask = (1u << log2cap) - 1u;
    uint32_t h = hash_id(id, log2cap);
    for (uint32_t probes = 0; probes <= mask; ++probes) {  // bounded: a full table can never hang the device
        // plain L2 read first (L1 bypassed: the table is updated by L2 atomics): most probes hit
        // an id that is already present and must not dirty the sector
        uint32_t old = __ldcg(table + h);
        if (old == kEmpty) old = atomicCAS(table + h, kEmpty, id);
        if (old == kEmpty) return true;
        if (old == id) return false;
        h = (h + 1) & mask;
    }
    return false;
}

// NeighborPriorityQueue::insert, queue.rs:130-171 (warp-uniform arguments)
__device__ __forceinline__ void queue_insert(float* qd, uint32_t* qi, uint32_t cap, uint32_t& size,
                                             uint32_t& cursor, uint32_t id, float d, int lane) {
    if (d != d) return;
    if (size == cap && qd[size - 1] < d) return;
    uint32_t pos = 0;
    for (uint32_t b = 0; b < size; b += 32) {
        const uint32_t i = b + lane;
        const bool lt = i < size && qd[i] < d;
        const unsigned m = __ballot_sync(kFull, lt);
        pos += __popc(m);
        if (m != kFull) break;
    }
    if (size == cap) --size;
    if (pos < size) {
        for (int b = (int)((size - 1) & ~31u); b >= (int)(pos & ~31u); b -= 32) {
            const uint32_t i = (uint32_t)b + lane;
            const bool mv = i >= pos && i < size;
            float v = 0.0f;
            uint32_t w = 0;
            if (mv) {
                v = qd[i];
                w = qi[i];
            }
            __syncwarp();
            if (mv) {
                qd[i + 1] = v;
                qi[i + 1] = w;
            }
            __syncwarp();
        }
    }
    __syncwarp();  // orders the reads above against the write below when nothing was moved (racecheck)
    if (lane == 0) {
        qd[pos] = d;
        qi[pos] = id;
    }
    __syncwarp();
    ++size;
    if (pos < cursor) cursor = pos;
}

template <typename TD, int NA, int KIND, int POST, bool IS_INT, bool SIGNED>
__global__ void __launch_bounds__(kSearchWarps * 32) search_kernel(const SearchParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    uint8_t* base = smem + (size_t)wib * p.warp_smem;
    float* qf = reinterpret_cast<float*>(base);
    uint8_t* qb = base;
    float* qd = reinterpret_cast<float*>(base + p.off_qd);
    uint32_t* qi = reinterpret_cast<uint32_t*>(base + p.off_qi);
    uint32_t* cid = reinterpret_cast<uint32_t*>(base + p.off_cid);
    float* cd = reinterpret_cast<float*>(base + p.off_cd);
    uint32_t* beam_ids = reinterpret_cast<uint32_t*>(base + p.off_beam);

    const uint32_t warp_slot = blockIdx.x * kSearchWarps + wib;
    uint32_t* table = p.tables + ((size_t)warp_slot << p.hcap_log2);
    const uint32_t hcap = 1u << p.hcap_log2;
    const uint32_t hlimit = hcap - (hcap >> 2);  // 75 % load
    const uint64_t n_total = p.n_points + p.n_start;
    const int dim = (int)p.dim;
    constexpr int S = 8 * NA, TEAMS = IS_INT ? 1 : 32 / S;
    constexpr int U = kRowsInFlight;
    const int team = IS_INT ? 0 : lane / S, slot = IS_INT ? lane : lane % S;

    for (;;) {
        uint32_t w = 0;
        if (lane == 0) w = atomicAdd(p.counters, 1u);
        w = __shfl_sync(kFull, w, 0);
        if (w >= p.n_work) break;
        const uint32_t qidx = p.query_list ? p.query_list[w] : w;

        // ---- stage the query (f16 widened to f32 once: layers/full.rs:421-423)
        __syncwarp();
        {
            const uint8_t* src = p.query_rows
                                     ? p.vectors + (size_t)p.query_rows[qidx] * p.row_stride
                                     : reinterpret_cast<const uint8_t*>(p.queries) + (size_t)qidx * dim * sizeof(TD);
            if constexpr (IS_INT) {
                const int qbytes = (dim + 3) & ~3;
                for (int e = lane; e < qbytes; e += 32) qb[e] = e < dim ? src[e] : 0;
            } else {
                const TD* s = reinterpret_cast<const TD*>(src);
                for (int e = lane; e < dim; e += 32) qf[e] = to_f32(s[e]);
            }
        }
        // ---- clear the visited table
        {
            uint4 e4 = make_uint4(kEmpty, kEmpty, kEmpty, kEmpty);
            uint4* t4 = reinterpret_cast<uint4*>(table);
            for (uint32_t i = lane; i < (hcap >> 2); i += 32) t4[i] = e4;
        }
        __syncwarp();
        int qq = 0;
        if constexpr (IS_INT && KIND != KIND_IP) qq = warp_int_self<SIGNED>(qb, dim, lane);

        uint32_t size = 0, cursor = 0, cmps = 0, hops = 0, nvisited = 0, nrec = 0;
        bool overflow = false;

        // ---- start points: SearchAccessor::start_point_distances (provider.rs:406-433)
        for (uint32_t s = 0; s < p.n_start; ++s) {
            const uint32_t id = (uint32_t)p.n_points + s;
            if (lane == 0) visited_insert(table, p.hcap_log2, id);
            ++nvisited;
            float r[1];
            if constexpr (IS_INT) {
                const uint8_t* rows[1] = {p.vectors + (size_t)id * p.row_stride};
                warp_int_multi<SIGNED, KIND, 1>(qb, rows, dim, lane, qq, r);
            } else {
                const TD* rows[1] = {reinterpret_cast<const TD*>(p.vectors + (size_t)id * p.row_stride)};
                team_float_multi<NA, KIND, 1>(qf, rows, dim, slot, r);
                r[0] = __shfl_sync(kFull, r[0], 0);
            }
            __syncwarp();
            queue_insert(qd, qi, p.cap, size, cursor, id, post_op<POST>(r[0]), lane);
            ++cmps;
        }

        // ---- greedy loop
        while (cursor < min(p.cap, size)) {
            // closest_notvisited x beam_width (queue.rs:297-313)
            uint32_t nb = 0;
            while (nb < p.beam && cursor < min(p.cap, size)) {
                const uint32_t cur = cursor;
                const uint32_t id = qi[cur];
                __syncwarp();
                if (lane == 0) {
                    qi[cur] = id | kVisitedFlag;
                    beam_ids[nb] = id;
                    if (p.rec_ids && nrec < p.rec_cap) {
                        p.rec_ids[(size_t)qidx * p.rec_cap + nrec] = id;
                        p.rec_dists[(size_t)qidx * p.rec_cap + nrec] = qd[cur];
                    }
                }
                ++nrec;
                ++nb;
                __syncwarp();
                ++cursor;
                while (cursor < size && (qi[cursor] & kVisitedFlag)) ++cursor;
            }

            // expand_beam: adjacency fetch + visited filter, adjacency order preserved
            uint32_t ncand = 0;
            for (uint32_t b = 0; b < nb; ++b) {
                const uint32_t node = beam_ids[b];
                const uint32_t* row = p.adj + (size_t)node * p.adj_stride;
                // words [0..31], [32..63], [64..95] issued together; word 0 is the degree
                uint32_t w0 = __ldg(row + lane);
                uint32_t w1 = 32 + lane < p.adj_stride ? __ldg(row + 32 + lane) : kEmpty;
                uint32_t w2 = 64 + lane < p.adj_stride ? __ldg(row + 64 + lane) : kEmpty;
                uint32_t deg = __shfl_sync(kFull, w0, 0);
                deg = min(deg, p.max_degree);
                for (uint32_t c0 = 0; c0 < deg + 1; c0 += 32) {
                    uint32_t word;
                    if (c0 == 0) word = w0;
                    else if (c0 == 32) word = w1;
                    else if (c0 == 64) word = w2;
                    else word = c0 + lane < p.adj_stride ? __ldg(row + c0 + lane) : kEmpty;
                    const uint32_t j = c0 + lane;  // word index; neighbour index j - 1
                    const bool valid = j >= 1 && j <= deg;
                    bool inserted = false;
                    if (valid) inserted = visited_insert(table, p.hcap_log2, word);
                    const bool isnew = inserted && word < n_total;  // is_in_bounds
                    const unsigned mi = __ballot_sync(kFull, inserted);
                    const unsigned mn = __ballot_sync(kFull, isnew);
                    if (isnew) cid[ncand + __popc(mn & ((1u << lane) - 1u))] = word;
                    ncand += __popc(mn);
                    nvisited += __popc(mi);
                }
                if (nvisited + p.max_degree + 32 > hlimit) {  // the next node could pass the load limit: stop expanding now
                    overflow = true;
                    break;
                }
            }
            if (overflow) break;
            __syncwarp();

            // gather + distance for the surviving candidates
            for (uint32_t c0 = 0; c0 < ncand; c0 += TEAMS * U) {
                float r[U];
                uint32_t cc[U];
                if constexpr (IS_INT) {
                    const uint8_t* rows[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        cc[u] = c0 + u;
                        const uint32_t id = cid[min(cc[u], ncand - 1)];
                        rows[u] = p.vectors + (size_t)id * p.row_stride;
                    }
                    warp_int_multi<SIGNED, KIND, U>(qb, rows, dim, lane, qq, r);
                } else {
                    const TD* rows[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        cc[u] = c0 + u * TEAMS + team;
                        const uint32_t id = cid[min(cc[u], ncand - 1)];
                        rows[u] = reinterpret_cast<const TD*>(p.vectors + (size_t)id * p.row_stride);
                    }
                    team_float_multi<NA, KIND, U>(qf, rows, dim, slot, r);
                }
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (slot == 0 && cc[u] < ncand) cd[cc[u]] = post_op<POST>(r[u]);
            }
            __syncwarp();

            // best.insert for every neighbour in order (index.rs:1986-1988)
            for (uint32_t c = 0; c < ncand; ++c) queue_insert(qd, qi, p.cap, size, cursor, cid[c], cd[c], lane);
            cmps += ncand;
            hops += nb;
        }

        if (overflow) {
            if (lane == 0) {
                uint32_t o = atomicAdd(p.counters + 1, 1u);
                p.overflow_list[o] = qidx;
            }
            continue;
        }

        // ---- post-process: drop start points, first k (provider.rs:907-950)
        {
            const uint32_t n = min(p.cap, size);
            uint32_t count = 0;
            for (uint32_t b = 0; b < n && count < p.k; b += 32) {
                const uint32_t i = b + lane;
                uint32_t id = i < n ? (qi[i] & ~kVisitedFlag) : kEmpty;
                const bool keep = i < n && id < p.n_points;
                const unsigned m = __ballot_sync(kFull, keep);
                const uint32_t pos = count + __popc(m & ((1u << lane) - 1u));
                if (keep && pos < p.k) {
                    p.out_ids[(size_t)qidx * p.k + pos] = id;
                    p.out_dists[(size_t)qidx * p.k + pos] = qd[i];
                }
                count += __popc(m);
            }
            count = min(count, p.k);
            for (uint32_t i = count + lane; i < p.k; i += 32) {
                p.out_ids[(size_t)qidx * p.k + i] = kEmpty;
                p.out_dists[(size_t)qidx * p.k + i] = __int_as_float(0x7F800000);
            }
            if (lane == 0) {
                atomicMax(p.counters + 2, nvisited);
                if (p.out_counts) p.out_counts[qidx] = count;
                if (p.out_cmps) p.out_cmps[qidx] = cmps;
                if (p.out_hops) p.out_hops[qidx] = hops;
                if (p.rec_counts) {
                    p.rec_counts[qidx] = min(nrec, p.rec_cap);
                    if (nrec > p.rec_cap) atomicAdd(p.counters + 3, 1u);  // expanded nodes beyond the record: reported by dab_build
                }
            }
        }
    }
}

// ------------------------------------------------------------------ host side

static uint32_t next_pow2_log2(uint64_t v) {
    uint32_t l = 0;
    while ((1ull << l) < v) ++l;
    return l;
}

// Keep the visited tables L2-resident: they are hit ~max_degree times per hop with random
// 4-byte probes, while vector rows stream through.  cudaAccessPolicyWindow on the stream.
// The generic kernel keeps its tables L2-resident with a persisting access-policy window on the
// stream; search_kernel_v2 marks its table accesses evict_last / row copies evict_first per
// instruction instead (search_common.cuh) and runs measurably slower with the window on top, so
// the window is dropped (`bytes == 0`) whenever v2 is dispatched.
static void pin_tables_in_l2(dab_index* idx, size_t bytes) {
    void* want = bytes ? idx->s_tables.p : nullptr;
    if (idx->l2_window_ptr == want && idx->l2_window_bytes == bytes && (bytes == 0 || idx->l2_window_stream == idx->stream)) return;
    cudaStreamAttrValue attr;
    memset(&attr, 0, sizeof(attr));
    if (bytes == 0) {
        attr.accessPolicyWindow.num_bytes = 0;
        attr.accessPolicyWindow.hitProp = cudaAccessPropertyNormal;
        attr.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
        if (cudaStreamSetAttribute(idx->l2_window_stream, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess) cudaGetLastError();
        idx->l2_window_ptr = nullptr;
        idx->l2_window_bytes = 0;
        return;
    }
    int max_persist = 0, max_window = 0;
    cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, idx->device);
    cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, idx->device);
    if (max_persist <= 0 || max_window <= 0) return;
    cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)max_persist);
    attr.accessPolicyWindow.base_ptr = idx->s_tables.p;
    attr.accessPolicyWindow.num_bytes = std::min<size_t>(bytes, (size_t)max_window);
    attr.accessPolicyWindow.hitRatio = bytes <= (size_t)max_persist ? 1.0f : (float)((double)max_persist / (double)bytes);
    attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    if (cudaStreamSetAttribute(idx->stream, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess) {
        cudaGetLastError();
        return;
    }
    idx->l2_window_ptr = idx->s_tables.p;
    idx->l2_window_bytes = bytes;
    idx->l2_window_stream = idx->stream;
}

template <typename K>
static int launch_one(K kern, const dab_index* idx, SearchParams& p, size_t smem_block, int& grid_out) {
    DAB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_block));
    int per_sm = 0;
    DAB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kSearchWarps * 32, smem_block));
    if (per_sm < 1) return fail(DAB_ERR_INVALID_ARGUMENT, "search kernel does not fit: %zu B shared memory per CTA", smem_block);
    grid_out = per_sm * idx->sm_count;
    return DAB_OK;
}

// ---- one batch of searches as a resumable job ------------------------------------------------
// A batch is launched (`launch`: kernel + read-back of the four counters into pinned memory, nothing
// waits) and later completed (`finish`: waits, learns the visited-set size, re-runs the few queries
// whose visited set outgrew its table).  The synchronous entry points run launch + finish on the
// handle's stream; dab_search_batch_async / dab_wait keep several batches in flight on slot-owned
// streams so the tail of one batch (workers running out of queries) is filled by the next batch's
// CTAs and the host<->device copies of neighbouring batches overlap the kernel.
struct SearchJob {
    dab_index* idx = nullptr;
    cudaStream_t stream = nullptr;
    Scratch* tables = nullptr;
    Scratch* counters = nullptr;
    uint32_t* h_counters = nullptr;  // pinned, 4 words
    bool use_window = false;         // persisting-L2 window for the generic kernel's tables (default stream only)
    bool full_grid = false;          // batches in flight: launch every resident worker (the next batch fills what this one leaves)

    uint32_t nq = 0, l_search = 0, beam = 0;
    bool recording = false;
    SearchParams p;
    SearchParamsV2 p2;
    SearchParamsV3 p3;
    void (*kern)(const SearchParams) = nullptr;
    size_t smem_block = 0;
    int grid = 0;
    bool use_v2 = false;
    V2Launch v2;
    V3Launch v3;
    uint64_t slots = 0;
    int stage = 1;  // 0: search_kernel_v3 pass in flight, 1: global-table pass in flight
    int pass = 0;
    Scratch retry_list;
    uint32_t *d_counters = nullptr, *d_overflow = nullptr;

    int prepare(const void* d_queries, const uint32_t* d_query_rows, uint32_t nq_, uint32_t k, uint32_t l_search_, uint32_t beam_,
                uint32_t* d_ids, float* d_dists, uint32_t* d_counts, uint32_t* d_cmps, uint32_t* d_hops, uint32_t* rec_ids,
                float* rec_dists, uint32_t* rec_counts, uint32_t rec_cap);
    int launch();
    int finish();
    ~SearchJob() { retry_list.release(); }
};

int SearchJob::prepare(const void* d_queries, const uint32_t* d_query_rows, uint32_t nq_, uint32_t k, uint32_t l_search_,
                       uint32_t beam_, uint32_t* d_ids, float* d_dists, uint32_t* d_counts, uint32_t* d_cmps, uint32_t* d_hops,
                       uint32_t* rec_ids, float* rec_dists, uint32_t* rec_counts, uint32_t rec_cap) {
    nq = nq_, l_search = l_search_, beam = beam_;
    recording = rec_ids != nullptr;
    const bool is_int = idx->dtype == DAB_I8 || idx->dtype == DAB_U8;
    const MetricPlan plan = plan_for(idx->metric, is_int);

    memset(&p, 0, sizeof(p));
    p.vectors = idx->d_vectors;
    p.row_stride = idx->row_stride;
    p.adj = idx->d_adj;
    p.adj_stride = idx->adj_stride;
    p.n_points = idx->n_points;
    p.n_start = idx->n_start;
    p.dim = idx->dim;
    p.max_degree = idx->max_degree;
    p.queries = d_queries;
    p.query_rows = d_query_rows;
    p.k = k;
    p.cap = l_search + idx->n_start;  // scratch.rs:195-208
    p.beam = beam;
    p.out_ids = d_ids;
    p.out_dists = d_dists;
    p.out_counts = d_counts;
    p.out_cmps = d_cmps;
    p.out_hops = d_hops;
    p.rec_ids = rec_ids;
    p.rec_dists = rec_dists;
    p.rec_counts = rec_counts;
    p.rec_cap = rec_cap;

    // shared memory layout per warp
    size_t off = 0;
    const size_t qbytes = is_int ? round_up(idx->dim, 4) : (size_t)idx->dim * 4;
    off = round_up(qbytes, 16);
    p.off_qd = (uint32_t)off;
    off += round_up((size_t)p.cap * 4, 16);
    p.off_qi = (uint32_t)off;
    off += round_up((size_t)p.cap * 4, 16);
    const size_t ncand_max = (size_t)beam * idx->max_degree;
    p.off_cid = (uint32_t)off;
    off += round_up(ncand_max * 4, 16);
    p.off_cd = (uint32_t)off;
    off += round_up(ncand_max * 4, 16);
    p.off_beam = (uint32_t)off;
    off += round_up((size_t)beam * 4, 16);
    p.warp_smem = (uint32_t)off;
    smem_block = off * kSearchWarps;
    if (smem_block > 220 * 1024)
        return fail(DAB_ERR_INVALID_ARGUMENT, "search: L=%u, beam=%u, dim=%u need %zu B shared memory per CTA (> 220 KiB)",
                    l_search, beam, idx->dim, smem_block);

    // the generic kernel (every dtype / metric / L; also the target of overflow re-runs)
    int rc = DAB_OK;
#define PICK(TD, NA, K, P, II, SG)                               \
    do {                                                         \
        kern = search_kernel<TD, NA, K, P, II, SG>;              \
        rc = launch_one(kern, idx, p, smem_block, grid);         \
    } while (0)
#define PICK_FLOAT(TD)                                                                   \
    do {                                                                                 \
        if (plan.kind == KIND_L2) PICK(TD, 4, KIND_L2, POST_ID, false, false);            \
        else if (plan.kind == KIND_IP && plan.post == POST_NEG) PICK(TD, 4, KIND_IP, POST_NEG, false, false); \
        else if (plan.kind == KIND_IP) PICK(TD, 4, KIND_IP, POST_ONE_MINUS, false, false); \
        else PICK(TD, 2, KIND_COS, POST_ONE_MINUS, false, false);                         \
    } while (0)
#define PICK_INT(SG)                                                                     \
    do {                                                                                 \
        if (plan.kind == KIND_L2) PICK(uint8_t, 4, KIND_L2, POST_ID, true, SG);           \
        else if (plan.kind == KIND_IP) PICK(uint8_t, 4, KIND_IP, POST_NEG, true, SG);     \
        else PICK(uint8_t, 4, KIND_COS, POST_ONE_MINUS, true, SG);                        \
    } while (0)
    switch (idx->dtype) {
        case DAB_F32: PICK_FLOAT(float); break;
        case DAB_F16: PICK_FLOAT(__half); break;  // f32 query x f16 rows (Strategy4x2 / 2x4)
        case DAB_I8: PICK_INT(true); break;
        default: PICK_INT(false); break;
    }
#undef PICK
#undef PICK_FLOAT
#undef PICK_INT
    if (rc) return rc;

    // the latency-restructured kernel covers the NA = 4 schemas up to L + S = 256
    memset(&p2, 0, sizeof(p2));
    use_v2 = v2_prepare(idx, l_search, beam, full_grid, p2, v2) == 0;
    if (use_v2) {
        p2.vectors = p.vectors;
        p2.row_stride = p.row_stride;
        p2.adj = p.adj;
        p2.adj_stride = p.adj_stride;
        p2.n_points = p.n_points;
        p2.n_start = p.n_start;
        p2.dim = p.dim;
        p2.max_degree = p.max_degree;
        p2.queries = p.queries;
        p2.query_rows = p.query_rows;
        p2.k = p.k;
        p2.cap = p.cap;
        p2.beam = p.beam;
        p2.out_ids = p.out_ids;
        p2.out_dists = p.out_dists;
        p2.out_counts = p.out_counts;
        p2.out_cmps = p.out_cmps;
        p2.out_hops = p.out_hops;
        p2.rec_ids = p.rec_ids;
        p2.rec_dists = p.rec_dists;
        p2.rec_counts = p.rec_counts;
        p2.rec_cap = p.rec_cap;
        grid = v2.grid;
    }

    // visited-table capacity: the reference's estimate (scratch.rs:186-192:
    // 1.1 * max_degree * 1.3 * L), never more than the index, at least 256 slots
    double est = 1.1 * idx->max_degree * 1.3 * (double)l_search;
    const bool hinted = idx->hint_visited > 0 && l_search <= idx->hint_l && beam <= idx->hint_beam;
    if (hinted) {
        // later batches: 1.15x the largest visited set seen at this (or a larger) L (visited sets
        // grow monotonically with L); queries that still overflow are re-run with a larger table
        const double seen = ((double)idx->hint_visited * 1.15 + idx->max_degree) / (use_v2 ? 0.875 : 0.75) + 8.0;
        if (seen < est) est = seen;
    }
    if (est > (double)idx->n_total() * 1.34) est = (double)idx->n_total() * 1.34;
    slots = std::max<uint64_t>(256, (uint64_t)est + 1);
    if (idx->hooks.test_visited_log2) slots = 1ull << idx->hooks.test_visited_log2;  // tests force the overflow/retry path

    if ((rc = counters->reserve(16 + (size_t)nq * 4))) return rc;
    d_counters = (uint32_t*)counters->p;
    d_overflow = d_counters + 4;
    p.counters = d_counters;
    p.overflow_list = d_overflow;
    p.n_work = nq;
    p.query_list = nullptr;
    p2.counters = d_counters;
    p2.overflow_list = d_overflow;

    // first pass with the visited sets in shared memory (search_kernel_v3) where it is the faster
    // kernel; queries that outgrow their table are re-run on global tables
    stage = 1;
    pass = 0;
    uint32_t need = 0;
    if (hinted) need = (uint32_t)std::min<double>((double)idx->hint_visited * 1.15, 4.0e9);
    if (idx->hooks.test_visited_log2) need = (1u << idx->hooks.test_visited_log2) / 2;
    const bool skip = idx->v3_overflow_l == l_search && idx->v3_overflow_beam == beam && idx->v3_overflow_frac > 0.25f;
    memset(&p3, 0, sizeof(p3));
    if (!skip && v3_prepare(idx, l_search, beam, need, p3, v3) == 0) {
        stage = 0;
        p3.vectors = p.vectors, p3.row_stride = p.row_stride, p3.adj = p.adj, p3.adj_stride = p.adj_stride;
        p3.n_points = p.n_points, p3.n_start = p.n_start, p3.dim = p.dim, p3.max_degree = p.max_degree;
        p3.queries = p.queries, p3.query_rows = p.query_rows, p3.query_list = nullptr, p3.n_work = nq;
        p3.k = p.k, p3.cap = p.cap, p3.beam = p.beam;
        p3.out_ids = p.out_ids, p3.out_dists = p.out_dists, p3.out_counts = p.out_counts;
        p3.out_cmps = p.out_cmps, p3.out_hops = p.out_hops;
        p3.rec_ids = p.rec_ids, p3.rec_dists = p.rec_dists, p3.rec_counts = p.rec_counts, p3.rec_cap = p.rec_cap;
        p3.counters = d_counters, p3.overflow_list = d_overflow;
    }
    return DAB_OK;
}

// launch the pass of the current stage and queue the read-back of its counters
int SearchJob::launch() {
    DAB_CUDA(cudaMemsetAsync(d_counters, 0, 16, stream));
    if (stage == 0) {
        // persistent workers: size the grid so every resident worker runs the same number of queries
        const uint64_t max_workers = (uint64_t)v3.grid * kV3Warps;
        const uint64_t rounds = (nq + max_workers - 1) / max_workers;
        const uint64_t need_warps = (nq + rounds - 1) / rounds;
        const int launch_grid = (int)((need_warps + kV3Warps - 1) / kV3Warps);
        v3.kern<<<launch_grid, kV3Warps * 32, v3.smem_block, stream>>>(p3);
    } else {
        // slots per warp: a power of two for the generic kernel, any multiple of 8 (32-byte buckets) for v2
        const uint32_t warps = (uint32_t)grid * (use_v2 ? kV2Warps : kSearchWarps);
        const uint32_t hlog = std::max<uint32_t>(use_v2 ? 8 : 10, next_pow2_log2(slots));
        const uint32_t n_buckets = (uint32_t)((slots + 7) / 8);
        const size_t words_per_warp = use_v2 ? (size_t)n_buckets * 8 : ((size_t)1 << hlog);
        int rc;
        if ((rc = tables->reserve((size_t)warps * words_per_warp * 4))) return rc;
        p.tables = (uint32_t*)tables->p;
        p.hcap_log2 = hlog;
        if (use_window) pin_tables_in_l2(idx, use_v2 ? 0 : (size_t)warps * words_per_warp * 4);
        if (use_v2) {
            // one warp per query, persistent: size the grid so every resident warp runs the same
            // number of queries (10K queries on 3108 slots would otherwise pay for 4 full rounds
            // with the last one 22 % full)
            const uint64_t max_warps = (uint64_t)grid * kV2Warps;
            const uint64_t rounds = (p.n_work + max_warps - 1) / max_warps;
            const uint64_t need = (p.n_work + rounds - 1) / rounds;
            int launch_grid = (int)((need + kV2Warps - 1) / kV2Warps);
            if (full_grid) launch_grid = (int)std::min<uint64_t>((uint64_t)grid, ((uint64_t)p.n_work + kV2Warps - 1) / kV2Warps);
            p2.tables = p.tables;
            p2.n_buckets = n_buckets;
            p2.query_list = p.query_list;
            p2.n_work = p.n_work;
            v2.kern<<<launch_grid, kV2Warps * 32, v2.smem_block, stream>>>(p2);
        } else {
            const int launch_grid = (int)std::min<uint64_t>((uint64_t)grid, ((uint64_t)p.n_work + kSearchWarps - 1) / kSearchWarps);
            kern<<<launch_grid, kSearchWarps * 32, smem_block, stream>>>(p);
        }
    }
    DAB_LAUNCHED();
    DAB_CUDA(cudaGetLastError());
    DAB_CUDA(cudaMemcpyAsync(h_counters, d_counters, 16, cudaMemcpyDeviceToHost, stream));
    return DAB_OK;
}

int SearchJob::finish() {
    for (;;) {
        DAB_CUDA(cudaStreamSynchronize(stream));
        idx->rec_truncated += h_counters[3];
        const uint32_t n_over = h_counters[1];
        if (!recording) {  // build-time searches run on a growing graph: do not learn from them
            if (l_search != idx->hint_l || beam != idx->hint_beam) {
                idx->hint_l = l_search;
                idx->hint_beam = beam;
                idx->hint_visited = 0;
            }
            idx->hint_visited = std::max(idx->hint_visited, h_counters[2]);
            if (stage == 0) {
                idx->v3_overflow_l = l_search;
                idx->v3_overflow_beam = beam;
                idx->v3_overflow_frac = (float)n_over / (float)nq;
            }
        }
        if (n_over == 0) {
            retry_list.release();
            return DAB_OK;
        }
        // re-run the overflowed queries on (larger) global tables
        Scratch next;
        int rc;
        if ((rc = next.reserve((size_t)n_over * 4))) return rc;
        DAB_CUDA(cudaMemcpyAsync(next.p, d_overflow, (size_t)n_over * 4, cudaMemcpyDeviceToDevice, stream));
        DAB_CUDA(cudaStreamSynchronize(stream));
        retry_list.release();
        retry_list = next;
        p.query_list = (const uint32_t*)retry_list.p;
        p.n_work = n_over;
        if (stage == 0) {
            // the overflowed queries are the largest: size the global tables from the estimate again
            stage = 1;
            pass = 0;
            if (!idx->hooks.test_visited_log2)
                slots = std::max<uint64_t>(slots, std::min<uint64_t>((uint64_t)(1.1 * idx->max_degree * 1.3 * (double)l_search) + 1,
                                                                        (uint64_t)((double)idx->n_total() * 1.34) + 1));
        } else {
            if (++pass >= 6) {
                retry_list.release();
                return fail(DAB_ERR_VISITED_OVERFLOW, "search: visited set still overflowing after 6 passes");
            }
            slots *= 4;
            if (slots > 4 * idx->n_total() + 4096) slots = 2 * idx->n_total() + 2048;
        }
        if ((rc = launch())) return rc;
    }
}

static int check_search_args(const dab_index* idx, uint32_t k, uint32_t l_search, uint32_t beam) {
    if (!idx->vectors_ready || !idx->graph_ready) return fail(DAB_ERR_NOT_READY, "search: vectors and graph must be uploaded first");
    if (k == 0 || l_search == 0 || beam == 0) return fail(DAB_ERR_INVALID_ARGUMENT, "search: k, l_search and beam_width must be > 0");
    if (beam > 64) return fail(DAB_ERR_INVALID_ARGUMENT, "search: beam_width %u > 64", beam);
    return DAB_OK;
}

// Runs the search over work items on the handle's stream and waits; device pointers only.  `rec_*` optional.
int run_search(dab_index* idx, const void* d_queries, const uint32_t* d_query_rows, uint32_t nq, uint32_t k,
               uint32_t l_search, uint32_t beam, uint32_t* d_ids, float* d_dists, uint32_t* d_counts, uint32_t* d_cmps,
               uint32_t* d_hops, uint32_t* rec_ids, float* rec_dists, uint32_t* rec_counts, uint32_t rec_cap) {
    int rc;
    if ((rc = check_search_args(idx, k, l_search, beam))) return rc;
    if (nq == 0) return DAB_OK;
    if ((rc = idx->h_counters.reserve(16))) return rc;
    SearchJob job;
    job.idx = idx;
    job.stream = idx->stream;
    job.tables = &idx->s_tables;
    job.counters = &idx->s_counters;
    job.h_counters = (uint32_t*)idx->h_counters.p;
    job.use_window = true;
    if ((rc = job.prepare(d_queries, d_query_rows, nq, k, l_search, beam, d_ids, d_dists, d_counts, d_cmps, d_hops, rec_ids,
                          rec_dists, rec_counts, rec_cap)))
        return rc;
    if ((rc = job.launch())) return rc;
    return job.finish();
}

// ---- batches in flight (dab_search_batch_async / dab_search_batch_device_async / dab_wait) ----
struct AsyncHostOut {  // host destinations of a pending host-buffer call
    uint32_t* ids;
    float* dists;
    uint32_t *counts, *cmps, *hops;
    uint32_t nq, k;
};

struct SearchSlot {
    cudaStream_t stream = nullptr;
    Scratch tables, counters, queries, out, stats, h_counters;
    SearchJob* job = nullptr;
    AsyncHostOut host_out{};
    bool has_host_out = false;
};

void search_slots_release(dab_index* idx) {
    for (int i = 0; i < DAB_MAX_SLOTS; ++i) {
        SearchSlot* s = (SearchSlot*)idx->slots[i];
        if (!s) continue;
        if (s->stream) cudaStreamSynchronize(s->stream);
        delete s->job;
        s->tables.release(), s->counters.release(), s->queries.release(), s->out.release(), s->stats.release(), s->h_counters.release();
        if (s->stream) cudaStreamDestroy(s->stream);
        delete s;
        idx->slots[i] = nullptr;
    }
}

static int slot_of(dab_index* idx, uint32_t slot, SearchSlot** out) {
    if (slot >= DAB_MAX_SLOTS) return fail(DAB_ERR_INVALID_ARGUMENT, "search: slot %u out of range (DAB_MAX_SLOTS = %d)", slot, DAB_MAX_SLOTS);
    SearchSlot* s = (SearchSlot*)idx->slots[slot];
    if (!s) {
        s = new SearchSlot();
        s->h_counters.pinned_host = true;
        if (cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete s;
            return fail(DAB_ERR_CUDA, "search: cannot create the stream of slot %u", slot);
        }
        idx->slots[slot] = s;
    }
    *out = s;
    return DAB_OK;
}

static int slot_launch(dab_index* idx, SearchSlot* s, const void* d_queries, uint32_t nq, uint32_t k, uint32_t l_search, uint32_t beam,
                       uint32_t* d_ids, float* d_dists, uint32_t* d_counts, uint32_t* d_cmps, uint32_t* d_hops) {
    int rc;
    if ((rc = s->h_counters.reserve(16))) return rc;
    SearchJob* job = new SearchJob();
    job->idx = idx;
    job->stream = s->stream;
    job->tables = &s->tables;
    job->counters = &s->counters;
    job->h_counters = (uint32_t*)s->h_counters.p;
    job->full_grid = true;
    if ((rc = job->prepare(d_queries, nullptr, nq, k, l_search, beam, d_ids, d_dists, d_counts, d_cmps, d_hops, nullptr, nullptr,
                           nullptr, 0)) ||
        (rc = job->launch())) {
        delete job;
        return rc;
    }
    s->job = job;
    return DAB_OK;
}

}  // namespace dab

using namespace dab;

extern "C" {

int dab_search_batch_device(dab_index* idx, const void* d_queries, uint32_t nq, uint32_t k, uint32_t l_search,
                            uint32_t beam_width, uint32_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts,
                            uint32_t* d_out_cmps, uint32_t* d_out_hops) {
    if (!idx) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch: idx is NULL");
    if (nq && (!d_queries || !d_out_ids || !d_out_dists)) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch: NULL argument");
    DAB_CUDA(cudaSetDevice(idx->device));
    return run_search(idx, d_queries, nullptr, nq, k, l_search, beam_width, d_out_ids, d_out_dists, d_out_counts,
                      d_out_cmps, d_out_hops, nullptr, nullptr, nullptr, 0);
}

int dab_search_batch(dab_index* idx, const void* queries, uint32_t nq, uint32_t k, uint32_t l_search,
                     uint32_t beam_width, uint32_t* out_ids, float* out_dists, uint32_t* out_counts,
                     uint32_t* out_cmps, uint32_t* out_hops) {
    if (!idx) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch: idx is NULL");
    if (nq == 0) return DAB_OK;
    if (!queries || !out_ids || !out_dists) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch: NULL argument");
    if (k == 0) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch: k must be > 0");
    DAB_CUDA(cudaSetDevice(idx->device));
    const size_t qbytes = (size_t)nq * idx->dim * elem_size(idx->dtype);
    const size_t rbytes = (size_t)nq * k * 4;
    int rc;
    if ((rc = idx->s_queries.reserve(qbytes))) return rc;
    if ((rc = idx->s_out.reserve(2 * rbytes))) return rc;
    if ((rc = idx->s_stats.reserve((size_t)nq * 12))) return rc;
    uint32_t* d_ids = (uint32_t*)idx->s_out.p;
    float* d_dists = (float*)((uint8_t*)idx->s_out.p + rbytes);
    uint32_t* d_counts = (uint32_t*)idx->s_stats.p;
    uint32_t* d_cmps = d_counts + nq;
    uint32_t* d_hops = d_cmps + nq;
    DAB_CUDA(cudaMemcpyAsync(idx->s_queries.p, queries, qbytes, cudaMemcpyHostToDevice, idx->stream));
    if ((rc = run_search(idx, idx->s_queries.p, nullptr, nq, k, l_search, beam_width, d_ids, d_dists, d_counts, d_cmps,
                         d_hops, nullptr, nullptr, nullptr, 0)))
        return rc;
    DAB_CUDA(cudaMemcpyAsync(out_ids, d_ids, rbytes, cudaMemcpyDeviceToHost, idx->stream));
    DAB_CUDA(cudaMemcpyAsync(out_dists, d_dists, rbytes, cudaMemcpyDeviceToHost, idx->stream));
    if (out_counts) DAB_CUDA(cudaMemcpyAsync(out_counts, d_counts, (size_t)nq * 4, cudaMemcpyDeviceToHost, idx->stream));
    if (out_cmps) DAB_CUDA(cudaMemcpyAsync(out_cmps, d_cmps, (size_t)nq * 4, cudaMemcpyDeviceToHost, idx->stream));
    if (out_hops) DAB_CUDA(cudaMemcpyAsync(out_hops, d_hops, (size_t)nq * 4, cudaMemcpyDeviceToHost, idx->stream));
    DAB_CUDA(cudaStreamSynchronize(idx->stream));
    return DAB_OK;
}

// ---- asynchronous batches: launch on a slot, collect with dab_wait ---------------------------
// Host-buffer flavour: the queries are copied from `queries` on the slot's stream (pinned memory makes
// the copy asynchronous), the kernel follows, and the results are copied into the host outputs; all of
// it is queued by this call when no query can overflow its visited table on the way, i.e. nothing waits.
// dab_wait(slot) blocks until the slot's batch is complete (and, in the rare overflow case, re-runs the
// affected queries and repeats the result copies).  The buffers must stay valid until dab_wait returns.
static int queue_result_copies(SearchSlot* s, const AsyncHostOut& o) {
    const size_t rbytes = (size_t)o.nq * o.k * 4;
    uint32_t* d_ids = (uint32_t*)s->out.p;
    float* d_dists = (float*)((uint8_t*)s->out.p + rbytes);
    uint32_t* d_counts = (uint32_t*)s->stats.p;
    DAB_CUDA(cudaMemcpyAsync(o.ids, d_ids, rbytes, cudaMemcpyDeviceToHost, s->stream));
    DAB_CUDA(cudaMemcpyAsync(o.dists, d_dists, rbytes, cudaMemcpyDeviceToHost, s->stream));
    if (o.counts) DAB_CUDA(cudaMemcpyAsync(o.counts, d_counts, (size_t)o.nq * 4, cudaMemcpyDeviceToHost, s->stream));
    if (o.cmps) DAB_CUDA(cudaMemcpyAsync(o.cmps, d_counts + o.nq, (size_t)o.nq * 4, cudaMemcpyDeviceToHost, s->stream));
    if (o.hops) DAB_CUDA(cudaMemcpyAsync(o.hops, d_counts + 2 * (size_t)o.nq, (size_t)o.nq * 4, cudaMemcpyDeviceToHost, s->stream));
    return DAB_OK;
}

int dab_search_batch_async(dab_index* idx, uint32_t slot, const void* queries, uint32_t nq, uint32_t k, uint32_t l_search,
                           uint32_t beam_width, uint32_t* out_ids, float* out_dists, uint32_t* out_counts, uint32_t* out_cmps,
                           uint32_t* out_hops) {
    if (!idx) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_async: idx is NULL");
    if (nq && (!queries || !out_ids || !out_dists)) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_async: NULL argument");
    int rc;
    if ((rc = check_search_args(idx, k, l_search, beam_width))) return rc;
    DAB_CUDA(cudaSetDevice(idx->device));
    SearchSlot* s = nullptr;
    if ((rc = slot_of(idx, slot, &s))) return rc;
    if (s->job) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_async: slot %u still has a batch in flight (call dab_wait)", slot);
    if (nq == 0) return DAB_OK;
    const size_t qbytes = (size_t)nq * idx->dim * elem_size(idx->dtype);
    const size_t rbytes = (size_t)nq * k * 4;
    if ((rc = s->queries.reserve(qbytes))) return rc;
    if ((rc = s->out.reserve(2 * rbytes))) return rc;
    if ((rc = s->stats.reserve((size_t)nq * 12))) return rc;
    uint32_t* d_ids = (uint32_t*)s->out.p;
    float* d_dists = (float*)((uint8_t*)s->out.p + rbytes);
    uint32_t* d_counts = (uint32_t*)s->stats.p;
    DAB_CUDA(cudaMemcpyAsync(s->queries.p, queries, qbytes, cudaMemcpyHostToDevice, s->stream));
    if ((rc = slot_launch(idx, s, s->queries.p, nq, k, l_search, beam_width, d_ids, d_dists, d_counts, d_counts + nq, d_counts + 2 * (size_t)nq)))
        return rc;
    s->host_out = AsyncHostOut{out_ids, out_dists, out_counts, out_cmps, out_hops, nq, k};
    s->has_host_out = true;
    // optimistic copies: valid as they are unless a query overflowed (then dab_wait repeats them)
    return queue_result_copies(s, s->host_out);
}

int dab_search_batch_device_async(dab_index* idx, uint32_t slot, const void* d_queries, uint32_t nq, uint32_t k, uint32_t l_search,
                                  uint32_t beam_width, uint32_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts,
                                  uint32_t* d_out_cmps, uint32_t* d_out_hops) {
    if (!idx) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_device_async: idx is NULL");
    if (nq && (!d_queries || !d_out_ids || !d_out_dists)) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_device_async: NULL argument");
    int rc;
    if ((rc = check_search_args(idx, k, l_search, beam_width))) return rc;
    DAB_CUDA(cudaSetDevice(idx->device));
    SearchSlot* s = nullptr;
    if ((rc = slot_of(idx, slot, &s))) return rc;
    if (s->job) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_device_async: slot %u still has a batch in flight (call dab_wait)", slot);
    if (nq == 0) return DAB_OK;
    s->has_host_out = false;
    return slot_launch(idx, s, d_queries, nq, k, l_search, beam_width, d_out_ids, d_out_dists, d_out_counts, d_out_cmps, d_out_hops);
}

int dab_wait(dab_index* idx, uint32_t slot) {
    if (!idx) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_wait: idx is NULL");
    if (slot >= DAB_MAX_SLOTS) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_wait: slot %u out of range (DAB_MAX_SLOTS = %d)", slot, DAB_MAX_SLOTS);
    SearchSlot* s = (SearchSlot*)idx->slots[slot];
    if (!s || !s->job) return DAB_OK;
    DAB_CUDA(cudaSetDevice(idx->device));
    SearchJob* job = s->job;
    s->job = nullptr;
    DAB_CUDA(cudaStreamSynchronize(s->stream));
    const bool overflowed = job->h_counters[1] != 0;
    int rc = job->finish();
    delete job;
    if (rc) return rc;
    if (overflowed && s->has_host_out) {
        if ((rc = queue_result_copies(s, s->host_out))) return rc;
        DAB_CUDA(cudaStreamSynchronize(s->stream));
    }
    return DAB_OK;
}

}  // extern "C"
