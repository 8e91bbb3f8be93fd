// search_kernel_v2.cu — latency-restructured batched greedy search for float rows
// (f32 x f32 and f32-widened x f16; L2 / InnerProduct / CosineNormalized schemas, NA = 4).
//
// Same semantics as search_kernel.cu (DiskANNIndex::search_internal, index.rs:1933-2000;
// NeighborPriorityQueue, queue.rs:130-318; expand_beam, provider.rs:436-479) and bit-identical
// results; what changes is how many dependent memory round trips a hop costs:
//
//   * rows of the surviving candidates of a hop are staged in shared memory with cp.async
//     (16 B per lane, eight lanes per row: one warp instruction moves 128 B of four rows and no
//     lane needs another lane's address; no registers tied up), a stage of
//     rows in flight at once (a TMA bulk-copy variant was measured slower: UBLKCP takes
//     warp-uniform operands, so per-row copies serialise);
//   * distances are computed from shared memory (lane s <-> SIMD slot s, conflict-free) for 8
//     rows per pass and reduced with a transpose-butterfly in the reference's association
//     (xor 8, 16, [remainder], 4, 2, 1) — 9 shuffles per 8 rows;
//   * the sorted candidate list lives in shared memory and a whole round of candidates is merged
//     at once by rank (search_common.cuh), equivalent to the reference's sequential inserts;
//   * all visited-set probes of an adjacency row are issued together (one 256-bit evict_last
//     load per 8-id bucket); the adjacency row of the next-best unvisited candidate is copied
//     into shared memory while the current hop runs, so the next hop usually starts without a
//     global round trip;
//   * the distance arithmetic advances two rows per instruction (packed f32x2 FADD2 / FFMA2).
#include "dab_common.cuh"
#include "distance_device.cuh"
#include "search_common.cuh"
#include "search_v2.cuh"

#include <algorithm>
#include <cstdlib>
#include <type_traits>

namespace dab {

constexpr int kGroup = 8;  // rows reduced together
// resident CTAs (one warp each) per SM the register budget is sized for
constexpr int kV2MinCtas = 21;
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// transpose-butterfly stage over M live values (see flat_kernels.cu)
template <int M>
__device__ __forceinline__ void bfly8(float (&v)[kGroup], int lane, int bit) {
    const bool up = (lane & bit) != 0;
#pragma unroll
    for (int i = 0; i < M / 2; ++i) {
        const float keep = up ? v[M / 2 + i] : v[i];
        const float send = up ? v[i] : v[M / 2 + i];
        v[i] = __fadd_rn(keep, __shfl_xor_sync(kFull, send, bit));
    }
}

// Packed f32x2 arithmetic (FADD2 / FFMA2 on sm_100): each half is an IEEE round-to-nearest
// operation, so a pair of rows advances with one instruction and the same bits as two scalar ones.
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
template <int KIND>
__device__ __forceinline__ uint64_t step2(uint64_t acc, uint64_t x2, uint64_t y2) {
    if (KIND == KIND_L2) {
        uint64_t c2;
        asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(c2) : "l"(x2), "l"(y2));
        asm("fma.rn.f32x2 %0, %1, %1, %2;" : "=l"(acc) : "l"(c2), "l"(acc));
    } else {
        asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(acc) : "l"(x2), "l"(y2), "l"(acc));
    }
    return acc;
}

// distances of 8 staged rows (shared memory) against the query (shared memory, f32); returns on
// every lane the value of row u = ((lane>>3)&1)<<2 | ((lane>>4)&1)<<1 | ((lane>>2)&1)
template <typename TD, int KIND>
__device__ __forceinline__ float group_distance(const float* __restrict__ q, const uint8_t* __restrict__ rows,
                                                uint32_t row_slot, int dim, int lane) {
    const int full8 = dim & ~7, rem = dim & 7;
    float v[kGroup];
    uint64_t v2[kGroup / 2];
#pragma unroll
    for (int g = 0; g < kGroup / 2; ++g) v2[g] = 0ull;
    for (int e = lane; e < full8; e += 32) {
        const float x = q[e];
        const uint64_t x2 = pack2(x, x);
#pragma unroll
        for (int g = 0; g < kGroup / 2; ++g) {
            const float y0 = to_f32(reinterpret_cast<const TD*>(rows + (size_t)(2 * g) * row_slot)[e]);
            const float y1 = to_f32(reinterpret_cast<const TD*>(rows + (size_t)(2 * g + 1) * row_slot)[e]);
            v2[g] = step2<KIND>(v2[g], x2, pack2(y0, y1));
        }
    }
#pragma unroll
    for (int g = 0; g < kGroup / 2; ++g) unpack2(v2[g], v[2 * g], v[2 * g + 1]);
    bfly8<8>(v, lane, 8);
    bfly8<4>(v, lane, 16);
    if (rem) {
        // two live values: index i | b4 << 1 | b3 << 2 (b3 = lane bit 3, b4 = lane bit 4)
        const int hi = (((lane >> 4) & 1) << 1) | (((lane >> 3) & 1) << 2);
        const int l = lane & 7;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int g = i | hi;
            const float x = l < rem ? q[full8 + l] : 0.0f;
            const float y = l < rem ? to_f32(reinterpret_cast<const TD*>(rows + (size_t)g * row_slot)[full8 + l]) : 0.0f;
            if (KIND == KIND_L2) {
                const float c = __fsub_rn(x, y);
                v[i] = __fmaf_rn(c, c, v[i]);
            } else {
                v[i] = __fmaf_rn(x, y, v[i]);
            }
        }
    }
    bfly8<2>(v, lane, 4);
    float a = v[0];
    a = __fadd_rn(a, __shfl_xor_sync(kFull, a, 2));
    a = __fadd_rn(a, __shfl_xor_sync(kFull, a, 1));
    return a;
}

// i8 / u8 rows through the same hop structure.  Integer distances are exact in i32
// (Sum(x-y)^2 = Sum x^2 + Sum y^2 - 2 Sum xy in wrapping arithmetic, as warp_int_multi), so any
// summation order gives the reference's value: lane w owns 4-byte word w of all 8 staged rows.
template <typename T>
struct V2Int {
    static constexpr bool value = false, is_signed = false;
};
template <>
struct V2Int<int8_t> {
    static constexpr bool value = true, is_signed = true;
};
template <>
struct V2Int<uint8_t> {
    static constexpr bool value = true, is_signed = false;
};

// value (before the post-op) of staged row u on every lane, for u = 0..7
template <bool SIGNED, int KIND>
__device__ __forceinline__ void group_distance_int(const uint8_t* __restrict__ q, const uint8_t* __restrict__ rows, uint32_t row_slot, int dim,
                                                   int lane, int qq, float (&out)[kGroup]) {
    int xy[kGroup], yy[kGroup];
#pragma unroll
    for (int g = 0; g < kGroup; ++g) xy[g] = yy[g] = 0;
    const int nwords = dim >> 2;
    for (int w = lane; w < nwords; w += 32) {
        const int x = reinterpret_cast<const int*>(q)[w];
#pragma unroll
        for (int g = 0; g < kGroup; ++g) {
            const int y = reinterpret_cast<const int*>(rows + (size_t)g * row_slot)[w];
            xy[g] = dp4<SIGNED>(x, y, xy[g]);
            if (KIND != KIND_IP) yy[g] = dp4<SIGNED>(y, y, yy[g]);
        }
    }
    const int tail = dim & 3;
    if (lane < tail) {
        const int i = (nwords << 2) + lane;
        const int x = byte_at<SIGNED>(q, i);
#pragma unroll
        for (int g = 0; g < kGroup; ++g) {
            const int y = byte_at<SIGNED>(rows + (size_t)g * row_slot, i);
            xy[g] += x * y;
            if (KIND != KIND_IP) yy[g] += y * y;
        }
    }
#pragma unroll
    for (int g = 0; g < kGroup; ++g) {
        const int sxy = __reduce_add_sync(kFull, xy[g]);
        if (KIND == KIND_IP) {
            out[g] = (float)sxy;
        } else {
            const int syy = __reduce_add_sync(kFull, yy[g]);
            if (KIND == KIND_L2) out[g] = (float)(int)((unsigned)qq + (unsigned)syy - 2u * (unsigned)sxy);
            else out[g] = cosine_finish((float)qq, (float)syy, (float)sxy);
        }
    }
}

// Rare paths of the two-level visited set: clearing the warp's global table when its first id arrives, and the
// atomic insert.  (The kernel is sensitive to its code size — at ~100 KB of SASS every phase ran ~20 % slower than at
// 60 KB — so the hot loop is kept compact: one rolled loop over a row's chunks, no unrolled copies of these.)
__device__ __forceinline__ void clear_global_table(uint32_t* table, uint32_t nbk, int lane) {
#pragma unroll 1
    for (uint32_t i = lane; i < nbk; i += 32) store_empty_bucket(table + (size_t)i * 8);
    __syncwarp();
}
__device__ __forceinline__ bool global_table_insert(uint32_t* table, uint32_t nbk, uint32_t id) {
    uint32_t bs[8];
    const uint32_t b = bucket_of(id, nbk);
    load_bucket(table + (size_t)b * 8, bs);
    return bucket_insert(table, nbk, b, bs, id);
}

// L1 = true: two-level visited set.  Level 1 is a table of 16-bit quotient tags in the warp's own shared memory
// (tag16_probe, search_common.cuh); an id lives in exactly one level: level 1 while it has room for it (its three
// buckets not full, table not closed at 87.5 % load), otherwise level 2, this warp's global table.  A probe asks level 1
// first and only an id that is neither found nor placed there goes on to the global table — for most queries never,
// so their visited set costs no global traffic at all; the global table is cleared when its first id arrives.
// L1 = false: the global table alone (ids too wide for 14-bit tags at the table size, or level 1 disabled).
template <typename TD, int KIND, int POST, int QT, bool L1>
__global__ void __launch_bounds__(kV2Warps * 32, kV2MinCtas) search_kernel_v2(const SearchParamsV2 p) {
    extern __shared__ __align__(128) uint8_t smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    uint8_t* base = smem + (size_t)wib * p.warp_smem;
    float* qf = reinterpret_cast<float*>(base + p.off_q);
    float* qd = reinterpret_cast<float*>(base + p.off_qd);
    uint32_t* qi = reinterpret_cast<uint32_t*>(base + p.off_qi);
    uint32_t* cid = reinterpret_cast<uint32_t*>(base + p.off_cid);
    float* cd = reinterpret_cast<float*>(base + p.off_cd);
    uint32_t* beam_ids = reinterpret_cast<uint32_t*>(base + p.off_beam);
    uint8_t* rows = base + p.off_rows;
    const uint32_t rows_a = smem_u32(rows);
    uint32_t* adjbuf = reinterpret_cast<uint32_t*>(base + p.off_adj);
    const uint32_t adjbuf_a = smem_u32(adjbuf);

    uint32_t* t1 = reinterpret_cast<uint32_t*>(base + p.off_t1);
    const uint32_t nb1 = p.t1_buckets;
    const Tag16Map tmap{p.tag_kmask, nb1, p.tag_magic, p.tag_shift};

    const uint32_t warp_slot = blockIdx.x * kV2Warps + wib;
    const uint32_t nbk = p.n_buckets;
    uint32_t* table = p.tables + (size_t)warp_slot * nbk * 8;
    const uint32_t hlimit = nbk * 7;  // 87.5 % load: 8-way buckets stay short
    const uint64_t n_total = p.n_points + p.n_start;
    const int dim = (int)p.dim;
    // vector rows stream through L2 (a row is read once per query): evict them first so the
    // visited tables, which are re-probed every hop, stay resident
    uint64_t row_policy;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(row_policy));

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
            if constexpr (V2Int<TD>::value) {
                uint8_t* qb = reinterpret_cast<uint8_t*>(qf);
                const int qbytes = (dim + 3) & ~3;
                for (int e = lane; e < qbytes; e += 32) qb[e] = e < dim ? reinterpret_cast<const uint8_t*>(s)[e] : 0;
            } else {
                for (int e = lane; e < dim; e += 32) qf[e] = to_f32(s[e]);
            }
            if constexpr (L1) {
                const uint4 e4 = make_uint4(kEmptyV2, kEmptyV2, kEmptyV2, kEmptyV2);
                for (uint32_t i = lane; i < nb1 * 2; i += 32) reinterpret_cast<uint4*>(t1)[i] = e4;
            } else {
                for (uint32_t i = lane; i < nbk; i += 32) store_empty_bucket(table + (size_t)i * 8);
            }
        }
        __syncwarp();
        int qq = 0;  // Sum x^2 of the query (unused by inner product)
        if constexpr (V2Int<TD>::value) {
            if (KIND != KIND_IP) qq = warp_int_self<V2Int<TD>::is_signed>(reinterpret_cast<const uint8_t*>(qf), dim, lane);
        }

        uint32_t size = 0, cursor_lo = 0, cmps = 0, hops = 0, nvisited = 0, nrec = 0;
        uint32_t n1 = 0;          // ids held by level 1 (nvisited counts those of the global table when L1 is on)
        bool closed = false;      // level 1 takes no more ids
        bool l2_used = false;     // the global table has been cleared for this query and may hold ids
        uint32_t pred = kEmptyV2;  // node whose adjacency row sits in adjbuf
        bool overflow = false;

        // HashSet::insert of one id per lane through both levels (`ok`: this lane has an id); whole warp calls
        auto visit_l1 = [&](uint32_t id, bool ok) -> bool {
            bool ins = false, need = false;
            if (ok) {
                uint32_t b1, tg;
                tag16_of(id, tmap, b1, tg);
                const int r = tag16_probe(t1, nb1, b1, tg, !closed);
                ins = r == 1;
                need = r == 2;
            }
            n1 += __popc(__ballot_sync(kFull, ins));
            if (__any_sync(kFull, need)) {  // rare
                if (!l2_used) {
                    clear_global_table(table, nbk, lane);
                    l2_used = true;
                }
                bool ins2 = false;
                if (need) ins2 = global_table_insert(table, nbk, id);
                nvisited += __popc(__ballot_sync(kFull, ins2));
                ins |= ins2;
            }
            return ins;
        };


        // stage `n` candidate rows (ids cid[c0..)) with per-lane 16 B async copies and compute
        // their distances into cd[]
        auto distances = [&](uint32_t c0, uint32_t n) {
            // eight lanes per row, 16 B each: one warp instruction moves 128 B of four different
            // rows, and every lane forms its own source address (no cross-lane traffic)
            const uint32_t sub = (uint32_t)lane >> 3, nsub = 4, off0 = ((uint32_t)lane & 7u) * 16u, offs = 128;
            auto copy16 = [&](uint32_t dst, const uint8_t* src) {
                asm volatile("cp.async.cg.shared.global.L2::cache_hint [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "l"(row_policy) : "memory");
            };
            // copies of rows [lo, hi) as one cp.async group
            auto issue = [&](uint32_t lo, uint32_t hi) {
                if (p.row_bytes == 4 * offs) {  // 128-d f32 / 256-d f16 rows: fixed trip count, immediate offsets
                    for (uint32_t j = lo + sub; j < hi; j += nsub) {
                        const uint8_t* src = p.vectors + (size_t)cid[c0 + j] * p.row_stride + off0;
                        const uint32_t dst = rows_a + j * p.row_slot + off0;
#pragma unroll
                        for (uint32_t k = 0; k < 4; ++k) copy16(dst + k * offs, src + k * offs);
                    }
                } else {
                    for (uint32_t j = lo + sub; j < hi; j += nsub) {
                        const uint8_t* src = p.vectors + (size_t)cid[c0 + j] * p.row_stride;
                        const uint32_t dst = rows_a + j * p.row_slot;
                        for (uint32_t off = off0; off < p.row_bytes; off += offs) copy16(dst + off, src + off);
                    }
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
            };
            auto compute = [&](uint32_t g0) {
                if constexpr (V2Int<TD>::value) {
                    float vals[kGroup];
                    group_distance_int<V2Int<TD>::is_signed, KIND>(reinterpret_cast<const uint8_t*>(qf), rows + (size_t)g0 * p.row_slot,
                                                                  p.row_slot, dim, lane, qq, vals);
#pragma unroll
                    for (int u = 0; u < kGroup; ++u)
                        if (lane == u && g0 + u < n) cd[c0 + g0 + u] = post_op<POST>(vals[u]);
                } else {
                    const float r = group_distance<TD, KIND>(qf, rows + (size_t)g0 * p.row_slot, p.row_slot, dim, lane);
                    const uint32_t u = (((lane >> 3) & 1) << 2) | (((lane >> 4) & 1) << 1) | ((lane >> 2) & 1);
                    if ((lane & 3) == 0 && g0 + u < n) cd[c0 + g0 + u] = post_op<POST>(r);
                }
            };
            issue(0, n);
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            __syncwarp();
            for (uint32_t g0 = 0; g0 < n; g0 += kGroup) compute(g0);
            __syncwarp();
        };

        // ---- start points (SearchAccessor::start_point_distances, provider.rs:406-433)
        for (uint32_t s0 = 0; s0 < p.n_start; s0 += 32) {
            const uint32_t n = min(32u, p.n_start - s0);
            if constexpr (L1) {
                const uint32_t id = (uint32_t)p.n_points + s0 + lane;
                if ((uint32_t)lane < n) cid[lane] = id;
                visit_l1(id, (uint32_t)lane < n);
            } else if ((uint32_t)lane < n) {
                const uint32_t id = (uint32_t)p.n_points + s0 + lane;
                cid[lane] = id;
                uint32_t bs[8];
                const uint32_t b = bucket_of(id, nbk);
                load_bucket(table + (size_t)b * 8, bs);
                bucket_insert(table, nbk, b, bs, id);
            }
            __syncwarp();
            for (uint32_t c0 = 0; c0 < n; c0 += p.stage_rows) distances(c0, min(p.stage_rows, n - c0));
            merge_round<QT>(qd, qi, p.cap, size, cursor_lo, cid, cd, 0, n, lane);
            if constexpr (!L1) nvisited += n;
            cmps += n;
        }

        // ---- greedy loop (index.rs:1961-1992)
        for (;;) {
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
                    // the speculative copy of the previous hop has long landed; it must be
                    // drained before the buffer is read or re-targeted
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
                    // speculative: the next hop most likely expands the now-first unvisited entry;
                    // fetch its adjacency row into shared memory (or at least into L2) while
                    // this hop runs
                    const uint32_t nxt = first_unvisited(qi, cursor_lo, lim, lane);
                    pred = kEmptyV2;
                    if (nxt < lim) {
                        const uint32_t nid = qi[nxt] & ~kFlagV2;
                        const uint32_t* nrow = p.adj + (size_t)nid * p.adj_stride;
                        if (p.adj_words) {
                            pred = nid;
                            if ((uint32_t)lane * 4 < p.adj_words)
                                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(adjbuf_a + lane * 16), "l"(nrow + lane * 4)
                                             : "memory");
                            asm volatile("cp.async.commit_group;" ::: "memory");
                        } else if (lane < 3) {
                            prefetch_l2(nrow + lane * 32);
                        }
                    }
                }
                const uint32_t deg = min(__shfl_sync(kFull, wd[0], 0), p.max_degree);
                if constexpr (L1) {
                    // one compact loop over the row's chunks of 32 neighbours (the first three sit in registers)
#pragma unroll 1
                    for (uint32_t c0 = 0; c0 <= deg; c0 += 32) {
                        const uint32_t j = c0 + lane;
                        uint32_t word = c0 == 0 ? wd[0] : (c0 == 32 ? wd[1] : wd[2]);
                        if (c0 >= 96) word = j < p.adj_stride ? __ldg(row + j) : kEmptyV2;
                        const bool ins = visit_l1(word, j >= 1 && j <= deg);
                        const bool isnew = ins && word < n_total;  // is_in_bounds
                        const unsigned mn = __ballot_sync(kFull, isnew);
                        if (isnew) cid[ncand + __popc(mn & ((1u << lane) - 1u))] = word;
                        ncand += __popc(mn);
                    }
                    if (!closed && n1 + p.max_degree > p.t1_limit) closed = true;
                } else {
                // bucket probes of all three chunks in flight together
                    bool valid[3];
                    uint32_t bk[3];
                    uint32_t bs[3][8];
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        const uint32_t j = c * 32 + lane;
                        valid[c] = j >= 1 && j <= deg;
                        bk[c] = bucket_of(wd[c], nbk);
                        if (valid[c]) load_bucket(table + (size_t)bk[c] * 8, bs[c]);
                    }
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        bool inserted = false;
                        if (valid[c]) inserted = bucket_insert(table, nbk, bk[c], bs[c], wd[c]);
                        const bool isnew = inserted && wd[c] < n_total;  // is_in_bounds
                        const unsigned mi = __ballot_sync(kFull, inserted);
                        const unsigned mn = __ballot_sync(kFull, isnew);
                        if (isnew) cid[ncand + __popc(mn & ((1u << lane) - 1u))] = wd[c];
                        ncand += __popc(mn);
                        nvisited += __popc(mi);
                    }
                    // adjacency rows longer than 95 neighbours: remaining chunks
                    for (uint32_t c0 = 96; c0 < deg + 1; c0 += 32) {
                        const uint32_t j = c0 + lane;
                        const uint32_t word = j < p.adj_stride ? __ldg(row + j) : kEmptyV2;
                        bool inserted = false;
                        if (j <= deg) {
                            const uint32_t b2 = bucket_of(word, nbk);
                            uint32_t bs2[8];
                            load_bucket(table + (size_t)b2 * 8, bs2);
                            inserted = bucket_insert(table, nbk, b2, bs2, word);
                        }
                        const bool isnew = inserted && word < n_total;
                        const unsigned mi = __ballot_sync(kFull, inserted);
                        const unsigned mn = __ballot_sync(kFull, isnew);
                        if (isnew) cid[ncand + __popc(mn & ((1u << lane) - 1u))] = word;
                        ncand += __popc(mn);
                        nvisited += __popc(mi);
                    }
                }
                if (nvisited + p.max_degree > hlimit) {  // the next node could pass the load limit: stop expanding now
                    overflow = true;
                    break;
                }
            }
            if (overflow) break;
            __syncwarp();

            for (uint32_t c0 = 0; c0 < ncand; c0 += p.stage_rows) distances(c0, min(p.stage_rows, ncand - c0));

            // best.insert for every neighbour in adjacency order (index.rs:1986-1988)
            for (uint32_t c0 = 0; c0 < ncand; c0 += 32)
                merge_round<QT>(qd, qi, p.cap, size, cursor_lo, cid, cd, c0, min(32u, ncand - c0), lane);
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
                atomicMax(p.counters + 2, n1 + nvisited);
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
// Returns 1 when this configuration is not covered by v2 (caller falls back to v1), 0 on
// success with `out` filled, or a negative DAB error code.
int v2_prepare(const dab_index* idx, uint32_t l_search, uint32_t beam, bool level1, SearchParamsV2& p, V2Launch& out) {
    const bool v2_int = idx->dtype == DAB_I8 || idx->dtype == DAB_U8;
    const MetricPlan plan = plan_for(idx->metric, v2_int);
    if (plan.kind == KIND_COS && !v2_int) return 1;
    const uint32_t cap = l_search + idx->n_start;
    if (cap > 256 || idx->max_degree > 1000) return 1;
    const uint32_t row_bytes = (uint32_t)round_up((size_t)idx->dim * elem_size(idx->dtype), 16);
    if (row_bytes > idx->row_stride) return 1;
    const uint32_t row_slot = row_bytes;
    size_t off = 0;
    p.off_q = (uint32_t)off;
    off += v2_int ? round_up(round_up((size_t)idx->dim, 4), 16) : round_up((size_t)idx->dim * 4, 16);
    const size_t ncand_max = (size_t)beam * idx->max_degree;
    p.off_cid = (uint32_t)off;
    off += round_up(std::max<size_t>(ncand_max, idx->n_start) * 4, 16);
    p.off_cd = (uint32_t)off;
    off += round_up(std::max<size_t>(ncand_max, idx->n_start) * 4, 16);
    p.off_beam = (uint32_t)off;
    off += round_up((size_t)beam * 4, 16);
    // speculative adjacency buffer: the first <= 96 words of a row, 16-byte granules
    p.adj_words = idx->adj_stride % 4 == 0 ? (uint32_t)std::min<size_t>(idx->adj_stride, 96) : 0;
    p.off_adj = (uint32_t)off;
    off += (size_t)p.adj_words * 4;
    const size_t cap_pad = round_up(cap, 4);
    p.off_qd = (uint32_t)off;
    off += cap_pad * 4;
    p.off_qi = (uint32_t)off;
    off += cap_pad * 4;
    off = round_up(off, 128);
    p.off_rows = (uint32_t)off;
    const size_t fixed = off;
    // rows staged per round: as many as fit ~6 KB per warp, a multiple of the reduce group
    const size_t stage_bytes = 6144;
    uint32_t stage = (uint32_t)std::max<size_t>(kGroup, (stage_bytes / row_slot) / kGroup * kGroup);
    stage = std::min<uint32_t>(stage, 32);
    p.stage_rows = stage;
    p.row_bytes = row_bytes;
    p.row_slot = row_slot;
    // level-1 visited table: 4 KB of 16-bit tags per warp (2048 slots; the mean visited set of the headline
    // workload is ~1200 ids) when the ids fit 14-bit quotient tags, i.e. n_total <= 16384 * buckets
    size_t t1_bytes = idx->hooks.test_visited_log2 ? 512 : 4096;  // tests: a level 1 that fills at once
    p.t1_buckets = 0;
    if (t1_bytes >= 512) {
        uint32_t K = 8;
        while (((uint64_t)1 << K) < idx->n_total()) ++K;
        const uint64_t nb1 = t1_bytes / 32;
        uint32_t sbits = 0;
        while (((uint64_t)1 << sbits) < nb1) ++sbits;
        if ((((uint64_t)1 << K) + 16383) >> 14 <= nb1 && K + sbits <= 32) {
            p.t1_buckets = (uint32_t)nb1;
            p.t1_limit = (uint32_t)(nb1 * 14);
            p.tag_kmask = (uint32_t)(((uint64_t)1 << K) - 1);
            p.tag_shift = K + sbits;
            p.tag_magic = (uint32_t)((((uint64_t)1 << (K + sbits)) + nb1 - 1) / nb1);
        }
    }
    p.off_t1 = (uint32_t)round_up(fixed + (size_t)stage * row_slot, 32);
    // level 1 pays for itself only while enough warps stay resident: at C2 (24 -> 20 one-warp CTAs per SM) it removes
    // the table traffic (8.8 -> 5.3 GB of DRAM traffic per 10K queries) and is 2 % faster, at C3 (12 -> 10) it is 11 % slower
    // ... and while batches overlap: one batch at a time is dominated by its tail, where the 4 resident warps fewer
    // cost more (2.96 vs 2.67 ms) than the traffic saves
    if (p.t1_buckets && !level1) p.t1_buckets = 0;
    if (p.t1_buckets && (227 * 1024) / (round_up((size_t)p.off_t1 + t1_bytes, 128) * kV2Warps + 1024) * kV2Warps < 16)
        p.t1_buckets = 0;
    if (!p.t1_buckets) t1_bytes = 0;
    p.warp_smem = (uint32_t)round_up((size_t)p.off_t1 + t1_bytes, 128);
    out.smem_block = (size_t)p.warp_smem * kV2Warps;
    if (out.smem_block > 200 * 1024) return 1;

#define PICK2(TD, K, P, Q)                                              \
    do {                                                                \
        if (p.t1_buckets) out.kern = search_kernel_v2<TD, K, P, Q, true>; \
        else out.kern = search_kernel_v2<TD, K, P, Q, false>;           \
    } while (0)
#define PICK_Q(TD, K, P)                 \
    do {                                 \
        if (cap <= 128) PICK2(TD, K, P, 4); \
        else PICK2(TD, K, P, 8);         \
    } while (0)
#define PICK_T(TD)                                                       \
    do {                                                                 \
        if (plan.kind == KIND_L2) PICK_Q(TD, KIND_L2, POST_ID);           \
        else if (plan.post == POST_NEG) PICK_Q(TD, KIND_IP, POST_NEG);    \
        else PICK_Q(TD, KIND_IP, POST_ONE_MINUS);                         \
    } while (0)
#define PICK_I(TD)                                                     \
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
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, out.kern, kV2Warps * 32, out.smem_block) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        return 1;
    }
    out.grid = per_sm * idx->sm_count;
    return 0;
}

}  // namespace dab
