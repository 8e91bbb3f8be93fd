// search_kernel_v3.cu — batched greedy search with the visited set in SHARED memory.
//
// Same semantics and bit-identical results as search_kernel.cu / search_kernel_v2.cu
// (DiskANNIndex::search_internal, index.rs:1933-2000; NeighborPriorityQueue, queue.rs:130-318;
// expand_beam, provider.rs:436-479, 620-690).  What changes against v2 is the number of
// dependent GLOBAL-memory round trips a hop costs — v2 has three (bucket probe, CAS, row
// copy), and its per-warp tables (62 MB for 3334 resident warps) do not stay in L2, so ≈3 GB of
// the 8.8 GB a launch moves is random 32-byte table sectors (profiles/r01_table_footprint.md):
//
//   * the visited set of a query is an exact open-addressed table of 16-bit quotient tags in
//     the warp's own shared memory (id -> (bucket, tag) is a bijection for ids < 2^K, so only
//     the tag is stored: 16 entries per 32-byte bucket, displacement <= 2 buckets recorded in
//     the tag's top two bits).  A probe is two LDS.128, an insert one 32-bit shared-memory CAS;
//     a query that outgrows its table is handed to the global-table kernel (exactness is kept,
//     only speed is lost);
//   * the only HBM round trip left on a hop's critical path is the row gather itself: rows are
//     read straight into registers with 16-byte loads, 8 (f32) / 4 (f16) lanes per row and up
//     to 16 rows in flight per warp, each lane running the FMA chains of the SIMD slots it
//     loaded (the lane mapping of frontier_wide_kernel, which reaches 0.84-0.96 of the measured
//     HBM peak) — no staging buffer, which is what makes room for the table;
//   * i8 / u8 rows use the same structure with exact i32 dot products (dp4a);
//   * the adjacency row of the predicted next node is copied into shared memory while the
//     current hop runs (as in v2), so a hop normally starts without a global round trip.
#include "dab_common.cuh"
#include "distance_device.cuh"
#include "search_common.cuh"
#include "search_smem.cuh"
#include "search_v3.cuh"

#include <algorithm>
#include <cstdlib>
#include <type_traits>

namespace dab {

namespace {

// ---- f32 rows of 32 * nm <= 128 elements (the headline shapes: 128-d, 96-d) ------------------
// Same lane mapping and association as wide_distances, with the per-hop overheads removed: the
// 16 query elements a lane ever multiplies live in registers (packed pairs), and a step covers 4
// rows (one pass, 8 lanes per row) whose nm 16-byte loads per lane are issued back to back.  The
// reduction is xor 2 and xor 4 for (s0+s1)+(s2+s3), xor 1 for x_i + x_{i+4}, then (t0+t2)+(t1+t3).
template <int KIND, int POST>
__device__ __forceinline__ void wide_distances_f32_fast(const uint64_t (&q2)[8], int nm, const uint8_t* __restrict__ vectors,
                                                        size_t row_stride, const uint32_t* __restrict__ cid, uint32_t n,
                                                        float* __restrict__ cd, int lane) {
    const int team = lane >> 3, tl = lane & 7;
    // one pass per step measured faster than two passes reduced by a butterfly (2.71 vs 2.90 ms on C2)
    if (n > 4) prefetch_rows(vectors, row_stride, cid, n, (uint32_t)nm * 128u, lane);
    for (uint32_t j0 = 0; j0 < n; j0 += 4) {
        const uint8_t* row0 = vectors + (size_t)cid[min(j0 + team, n - 1)] * row_stride + 16 * tl;
        uint4 v0[4];
#pragma unroll
        for (int m = 0; m < 4; ++m)
            if (m < nm) v0[m] = ldg16(row0 + m * 128);
        uint64_t a0[2] = {0ull, 0ull};
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            if (m < nm) {
                a0[0] = step2<KIND>(a0[0], q2[2 * m], pack2(__uint_as_float(v0[m].x), __uint_as_float(v0[m].y)));
                a0[1] = step2<KIND>(a0[1], q2[2 * m + 1], pack2(__uint_as_float(v0[m].z), __uint_as_float(v0[m].w)));
            }
        }
        float acc[4];
        unpack2(a0[0], acc[0], acc[1]);
        unpack2(a0[1], acc[2], acc[3]);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            acc[i] = __fadd_rn(acc[i], __shfl_xor_sync(kFull, acc[i], 2));
            acc[i] = __fadd_rn(acc[i], __shfl_xor_sync(kFull, acc[i], 4));
        }
        float ts[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) ts[i] = __fadd_rn(acc[i], __shfl_xor_sync(kFull, acc[i], 1));
        const float r = __fadd_rn(__fadd_rn(ts[0], ts[2]), __fadd_rn(ts[1], ts[3]));
        if (tl == 0 && j0 + team < n) cd[j0 + team] = post_op<POST>(r);
    }
}

template <typename T>
struct IsInt {
    static constexpr bool value = std::is_same<T, int8_t>::value || std::is_same<T, uint8_t>::value;
};

constexpr int kV3MinCtas = 4;  // resident CTAs per SM the register budget is sized for
constexpr int kV3PassesF32 = 2;  // f32 rows: passes (of 4 rows, 4 x 16-byte loads per lane each) in flight
constexpr int kV3PassesF16 = 2;  // f16 rows: passes (of 8 rows) in flight
constexpr int kV3LoadsF16 = 4;   // f16 rows: 16-byte loads per lane per pass in flight
constexpr int kV3PassesInt = 4;  // i8 / u8 rows: passes (of 4 rows, one 16-byte load per lane each) in flight

}  // namespace

template <typename TD, int KIND, int POST, int QT, bool FAST>
__global__ void __launch_bounds__(kV3Warps * 32, kV3MinCtas) search_kernel_v3(const SearchParamsV3 p) {
    extern __shared__ __align__(128) uint8_t smem[];
    constexpr bool kInt = IsInt<TD>::value;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    uint8_t* base = smem + (size_t)wib * p.warp_smem;
    float* qf = reinterpret_cast<float*>(base + p.off_q);
    float* qd = reinterpret_cast<float*>(base + p.off_qd);
    uint32_t* qi = reinterpret_cast<uint32_t*>(base + p.off_qi);
    uint32_t* cid = reinterpret_cast<uint32_t*>(base + p.off_cid);
    float* cd = reinterpret_cast<float*>(base + p.off_cd);
    uint32_t* beam_ids = reinterpret_cast<uint32_t*>(base + p.off_beam);
    uint32_t* adjbuf = reinterpret_cast<uint32_t*>(base + p.off_adj);
    const uint32_t adjbuf_a = smem_addr(adjbuf);
    uint32_t* table = reinterpret_cast<uint32_t*>(base + p.off_table);
    const uint32_t nbk = p.n_buckets;
    const Tag16Map tmap{p.tag_kmask, nbk, p.tag_magic, p.tag_shift};
    auto visit = [&](uint32_t id, bool& ovf) -> bool {
        uint32_t bk, tg;
        tag16_of(id, tmap, bk, tg);
        return smem16_insert(table, nbk, bk, tg, ovf);
    };
    const uint64_t n_total = p.n_points + p.n_start;
    const int dim = (int)p.dim;

    for (;;) {
        uint32_t w = 0;
        if (lane == 0) w = atomicAdd(p.counters, 1u);
        w = __shfl_sync(kFull, w, 0);
        if (w >= p.n_work) break;
        const uint32_t qidx = p.query_list ? p.query_list[w] : w;

        __syncwarp();
        {
            const TD* s = p.query_rows ? reinterpret_cast<const TD*>(p.vectors + (size_t)p.query_rows[qidx] * p.row_stride)
                                       : reinterpret_cast<const TD*>(p.queries) + (size_t)qidx * dim;
            if constexpr (kInt) {
                uint8_t* qb = reinterpret_cast<uint8_t*>(qf);
                const int qbytes = (dim + 15) & ~15;
                for (int e = lane; e < qbytes; e += 32) qb[e] = e < dim ? reinterpret_cast<const uint8_t*>(s)[e] : 0;
            } else {
                for (int e = lane; e < dim; e += 32) qf[e] = to_f32(s[e]);
            }
            const uint4 e4 = make_uint4(kEmptyV2, kEmptyV2, kEmptyV2, kEmptyV2);
            for (uint32_t i = lane; i < nbk * 2; i += 32) reinterpret_cast<uint4*>(table)[i] = e4;
        }
        __syncwarp();
        int qq = 0;  // sum x^2 of an integer query (unused by inner product)
        if constexpr (kInt) {
            if (KIND != KIND_IP) qq = warp_int_self<std::is_same<TD, int8_t>::value>(reinterpret_cast<const uint8_t*>(qf), dim, lane);
        }
        (void)qq;
        // fast f32 path: the 16 query elements this lane multiplies, as packed pairs
        uint64_t q2[8] = {0ull, 0ull, 0ull, 0ull, 0ull, 0ull, 0ull, 0ull};
        if constexpr (FAST) {
            {
#pragma unroll
                for (int m = 0; m < 4; ++m) {
                    if (m < (int)p.fast_nm) {
                        const float4 x = *reinterpret_cast<const float4*>(qf + 32 * m + 4 * (lane & 7));
                        q2[2 * m] = pack2(x.x, x.y);
                        q2[2 * m + 1] = pack2(x.z, x.w);
                    }
                }
            }
        }

        uint32_t size = 0, cursor_lo = 0, cmps = 0, hops = 0, nvisited = 0, nrec = 0;
        uint32_t pred = kEmptyV2;  // node whose adjacency row sits in adjbuf
        bool overflow = false;

        auto distances = [&](uint32_t c0, uint32_t n) {
            if constexpr (kInt) {
                wide_distances_int<std::is_same<TD, int8_t>::value, KIND, POST, kV3PassesInt>(reinterpret_cast<const uint8_t*>(qf), qq, p.vectors,
                                                                                 p.row_stride, cid + c0, n, cd + c0, dim, lane);
            } else if constexpr (sizeof(TD) == 2) {
                wide_distances<TD, KIND, POST, kV3PassesF16, kV3LoadsF16>(qf, p.vectors, p.row_stride, cid + c0, n, cd + c0, dim, lane);
            } else if constexpr (FAST) {
                wide_distances_f32_fast<KIND, POST>(q2, (int)p.fast_nm, p.vectors, p.row_stride, cid + c0, n, cd + c0, lane);
            } else {
                wide_distances<TD, KIND, POST, kV3PassesF32, 4>(qf, p.vectors, p.row_stride, cid + c0, n, cd + c0, dim, lane);
            }
            __syncwarp();
        };

        // ---- start points (SearchAccessor::start_point_distances, provider.rs:406-433)
        for (uint32_t s0 = 0; s0 < p.n_start; s0 += 32) {
            const uint32_t n = min(32u, p.n_start - s0);
            bool ovf = false;
            if ((uint32_t)lane < n) {
                const uint32_t id = (uint32_t)p.n_points + s0 + lane;
                cid[lane] = id;
                visit(id, ovf);
            }
            if (__any_sync(kFull, ovf)) overflow = true;
            __syncwarp();
            distances(0, n);
            merge_round<QT>(qd, qi, p.cap, size, cursor_lo, cid, cd, 0, n, lane);
            nvisited += n;
            cmps += n;
        }
        if (nvisited > p.visited_limit) overflow = true;

        // ---- greedy loop (index.rs:1961-1992)
        while (!overflow) {
            const uint32_t lim = min(p.cap, size);
            uint32_t nb = 0;
            while (nb < p.beam) {  // closest_notvisited x beam_width (queue.rs:297-313)
                const uint32_t idx = first_unvisited(qi, cursor_lo, lim, lane);
                if (idx >= lim) break;
                const uint32_t id = qi[idx];
                __syncwarp();
                if (lane == 0) {
                    qi[idx] = id | kFlagV2;
                    beam_ids[nb] = id;
                    if (p.rec_ids && nrec < p.rec_cap) {
                        p.rec_ids[(size_t)qidx * p.rec_cap + nrec] = id;
                        p.rec_dists[(size_t)qidx * p.rec_cap + nrec] = qd[idx];
                    }
                }
                cursor_lo = idx + 1;
                ++nrec;
                ++nb;
                __syncwarp();
            }
            if (nb == 0) break;

            uint32_t ncand = 0;
            for (uint32_t b = 0; b < nb; ++b) {
                const uint32_t node = beam_ids[b];
                const uint32_t* row = p.adj + (size_t)node * p.adj_stride;
                uint32_t wd[3];
                if (b == 0 && p.adj_words) {
                    // the speculative copy of the previous hop must be drained before the buffer
                    // is read or re-targeted
                    asm volatile("cp.async.wait_group 0;" ::: "memory");
                    __syncwarp();
                }
                if (b == 0 && node == pred) {
                    wd[0] = adjbuf[lane];
                    wd[1] = 32 + lane < p.adj_words ? adjbuf[32 + lane] : kEmptyV2;
                    wd[2] = 64 + lane < p.adj_words ? adjbuf[64 + lane] : kEmptyV2;
                    __syncwarp();
                } else {
                    wd[0] = __ldg(row + lane);
                    wd[1] = 32 + lane < p.adj_stride ? __ldg(row + 32 + lane) : kEmptyV2;
                    wd[2] = 64 + lane < p.adj_stride ? __ldg(row + 64 + lane) : kEmptyV2;
                }
                if (b == 0) {
                    // speculative: the next hop most likely expands the now-first unvisited entry
                    const uint32_t nxt = first_unvisited(qi, cursor_lo, lim, lane);
                    pred = kEmptyV2;
                    if (nxt < lim && p.adj_words) {
                        const uint32_t nid = qi[nxt] & ~kFlagV2;
                        const uint32_t* nrow = p.adj + (size_t)nid * p.adj_stride;
                        pred = nid;
                        if ((uint32_t)lane * 4 < p.adj_words)
                            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(adjbuf_a + lane * 16), "l"(nrow + lane * 4) : "memory");
                        asm volatile("cp.async.commit_group;" ::: "memory");
                    }
                }
                const uint32_t deg = min(__shfl_sync(kFull, wd[0], 0), p.max_degree);
                if (nvisited + deg > p.visited_limit) {  // the table could pass its load limit: global-table kernel
                    overflow = true;
                    break;
                }
                bool ovf = false;
                auto filter = [&](uint32_t word, uint32_t j) {
                    bool inserted = false;
                    // ids beyond 2^K cannot be in bounds and never reach the outputs: not tracked
                    if (j >= 1 && j <= deg && word <= tmap.kmask) inserted = visit(word, ovf);
                    const bool isnew = inserted && word < n_total;  // is_in_bounds
                    const unsigned mi = __ballot_sync(kFull, inserted);
                    const unsigned mn = __ballot_sync(kFull, isnew);
                    if (isnew) cid[ncand + __popc(mn & ((1u << lane) - 1u))] = word;
                    ncand += __popc(mn);
                    nvisited += __popc(mi);
                };
#pragma unroll
                for (int c = 0; c < 3; ++c)
                    if ((uint32_t)c * 32 <= deg) filter(wd[c], c * 32 + lane);
                // adjacency rows longer than 95 neighbours: remaining chunks
                for (uint32_t c0 = 96; c0 < deg + 1; c0 += 32) {
                    const uint32_t j = c0 + lane;
                    filter(j < p.adj_stride ? __ldg(row + j) : kEmptyV2, j);
                }
                if (__any_sync(kFull, ovf)) {
                    overflow = true;
                    break;
                }
            }
            if (overflow) break;
            __syncwarp();

            distances(0, ncand);

            // best.insert for every neighbour in adjacency order (index.rs:1986-1988)
            for (uint32_t c0 = 0; c0 < ncand; c0 += 32)
                merge_round<QT>(qd, qi, p.cap, size, cursor_lo, cid, cd, c0, min(32u, ncand - c0), lane);
            cmps += ncand;
            hops += nb;
        }

        if (overflow) {
            if (p.adj_words) asm volatile("cp.async.wait_group 0;" ::: "memory");
            if (lane == 0) {
                const uint32_t o = atomicAdd(p.counters + 1, 1u);
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
                const uint32_t id = i < n ? (qi[i] & ~kFlagV2) : kEmptyV2;
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
                p.out_ids[(size_t)qidx * p.k + i] = kEmptyV2;
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
int v3_prepare(const dab_index* idx, uint32_t l_search, uint32_t beam, uint32_t visited_need, SearchParamsV3& p, V3Launch& out) {
    // v3 wins for short candidate lists (C2: 1.11 vs 1.67 ms at L = 15) and loses at the headline L = 100
    // (2.94 vs 2.68 ms); the measured crossover is L ~ 25 on both the 128-d f32 and the 768-d f16 shape
    // (profiles/r02_sweep_l.txt): longer lists go to the global-table kernel
    if (l_search + idx->n_start > 24) return 1;
    const bool is_int = idx->dtype == DAB_I8 || idx->dtype == DAB_U8;
    const MetricPlan plan = plan_for(idx->metric, is_int);
    if (plan.kind == KIND_COS && !is_int) return 1;  // float cosine: NA = 2 schema, generic kernel
    const uint32_t cap = l_search + idx->n_start;
    if (cap > 256 || idx->max_degree > 1000) return 1;
    if ((idx->row_stride & 15) != 0) return 1;
    // quotient tags: ids < 2^K, tag = h / n_buckets must fit 14 bits
    uint32_t K = 8;
    while (((uint64_t)1 << K) < idx->n_total()) ++K;
    if (K > 30) return 1;
    const uint64_t min_buckets = std::max<uint64_t>(16, (((uint64_t)1 << K) + 16383) >> 14);

    size_t off = 0;
    p.off_q = (uint32_t)off;
    off += is_int ? round_up((size_t)idx->dim, 16) : round_up((size_t)idx->dim * 4, 16);
    const size_t ncand_max = std::max<size_t>((size_t)beam * idx->max_degree, std::min<uint32_t>(32, idx->n_start));
    p.off_cid = (uint32_t)off;
    off += round_up(ncand_max * 4, 16);
    p.off_cd = (uint32_t)off;
    off += round_up(ncand_max * 4, 16);
    p.off_beam = (uint32_t)off;
    off += round_up((size_t)beam * 4, 16);
    p.adj_words = idx->adj_stride % 4 == 0 ? (uint32_t)std::min<size_t>(idx->adj_stride, 96) : 0;
    p.off_adj = (uint32_t)off;
    off += (size_t)p.adj_words * 4;
    const size_t cap_pad = round_up(cap, 4);
    p.off_qd = (uint32_t)off;
    off += cap_pad * 4;
    p.off_qi = (uint32_t)off;
    off += cap_pad * 4;
    off = round_up(off, 32);
    p.off_table = (uint32_t)off;
    const size_t fixed = off;

    const size_t smem_sm = 227 * 1024;  // per SM, 1 KB per CTA is reserved by the system
    auto table_bytes_at = [&](int ctas) -> long long {
        const long long per_cta = (long long)(smem_sm / ctas) - 1024;
        return (per_cta / kV3Warps - (long long)fixed) / 32 * 32;
    };
    // registers bound the residency (kV3MinCtas CTAs per SM), so the table takes all the shared
    // memory that residency leaves: a smaller table would only overflow more often
    long long tbytes = table_bytes_at(kV3MinCtas);
    if (idx->hooks.test_visited_log2 && visited_need)  // tests: a table small enough to overflow
        tbytes = (long long)round_up((size_t)((visited_need + idx->max_degree) / 0.875) * 2 + 32, 32);
    if (tbytes < (long long)min_buckets * 32) tbytes = (long long)min_buckets * 32;
    if (tbytes > table_bytes_at(1)) return 1;
    uint64_t nbk = (uint64_t)tbytes / 32;
    uint32_t sbits = 0;
    while (((uint64_t)1 << sbits) < nbk) ++sbits;
    if (K + sbits > 32) return 1;
    p.n_buckets = (uint32_t)nbk;
    p.tag_kmask = (uint32_t)(((uint64_t)1 << K) - 1);
    p.tag_shift = K + sbits;
    p.tag_magic = (uint32_t)((((uint64_t)1 << (K + sbits)) + nbk - 1) / nbk);
    p.visited_limit = (uint32_t)(nbk * 14);  // 87.5 % of 16 tags per bucket
    p.fast_nm = (idx->dtype == DAB_F32 && idx->dim % 32 == 0 && idx->dim <= 128) ? idx->dim / 32 : 0;
    out.capacity = p.visited_limit > idx->max_degree ? p.visited_limit - idx->max_degree : 0;
    if (out.capacity < 4 * idx->max_degree) return 1;
    p.warp_smem = (uint32_t)round_up(fixed + (size_t)tbytes, 128);
    out.smem_block = (size_t)p.warp_smem * kV3Warps;

#define PICK2(TD, K_, P_, Q_)                                                              \
    do {                                                                                   \
        if (std::is_same<TD, float>::value && p.fast_nm) out.kern = search_kernel_v3<float, K_, P_, Q_, true>; \
        else out.kern = search_kernel_v3<TD, K_, P_, Q_, false>;                            \
    } while (0)
#define PICK_Q(TD, K_, P_)                 \
    do {                                   \
        if (cap <= 128) PICK2(TD, K_, P_, 4); \
        else PICK2(TD, K_, P_, 8);         \
    } while (0)
#define PICK_T(TD)                                                       \
    do {                                                                 \
        if (plan.kind == KIND_L2) PICK_Q(TD, KIND_L2, POST_ID);           \
        else if (plan.post == POST_NEG) PICK_Q(TD, KIND_IP, POST_NEG);    \
        else PICK_Q(TD, KIND_IP, POST_ONE_MINUS);                         \
    } while (0)
#define PICK_I(TD)                                                       \
    do {                                                                 \
        if (plan.kind == KIND_L2) PICK_Q(TD, KIND_L2, POST_ID);           \
        else if (plan.kind == KIND_IP) PICK_Q(TD, KIND_IP, POST_NEG);     \
        else PICK_Q(TD, KIND_COS, POST_ONE_MINUS);                        \
    } while (0)
    if (idx->dtype == DAB_F32) PICK_T(float);
    else if (idx->dtype == DAB_F16) PICK_T(__half);
    else if (idx->dtype == DAB_I8) PICK_I(int8_t);
    else PICK_I(uint8_t);
#undef PICK_I
#undef PICK_T
#undef PICK_Q
#undef PICK2
    if (cudaFuncSetAttribute(out.kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)out.smem_block) != cudaSuccess) {
        cudaGetLastError();
        return 1;
    }
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, out.kern, kV3Warps * 32, out.smem_block) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        return 1;
    }
    out.grid = per_sm * idx->sm_count;
    return 0;
}

}  // namespace dab
