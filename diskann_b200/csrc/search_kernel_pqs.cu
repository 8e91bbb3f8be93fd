// search_kernel_pqs.cu — PQ traversal with the pivot table resident in shared memory.
//
// Same search as search_kernel_pq.cu MODE 0 (providers' quant accessor, product.rs:311-340, around
// search_internal, diskann/src/graph/index.rs:1933-2000; QueryComputer::{TableL2, TableIP},
// pq/distance/dynamic.rs:63-87), same results bit for bit, different placement of the table:
//
//   * the reference builds one table of n_chunks x n_centers f32 per query (fixed_chunk_pq_table.rs:152-187) and
//     sums one entry per chunk (pq_dist_lookup_single, :82-98).  Held per resident warp that table is 32 KB: in
//     global memory (search_kernel_pq.cu) every ADC term is a 32-byte sector from L2 or DRAM — 33 GB of sector
//     traffic per 10K-query batch at the C4 shape against 3.7 GB of algorithmic bytes;
//   * here the CTA of an SM stages the PIVOTS once (n_centers x dim f32, 132 KB at 256 x 128, rows padded so
//     that different centres start in different 16-byte bank groups) and every warp of the CTA — one query per
//     warp, up to 16 per SM — computes the table entry it needs on the fly from shared memory: the entry of
//     (chunk, centre) is the same arithmetic whether it is stored first or not (thread_simd_l2ip over the chunk in
//     the reference's SIMD order), so the chunk-order sum from 0.0 has the reference's bits;
//   * a team of four lanes owns one candidate (eight chunks per lane, one 8-byte load of its code bytes); the
//     sequential chunk-order sum walks the team with three shuffles, so a hop with <= 8 new candidates is one pass;
//   * a hop's global round trips are issued together: all adjacency words of the row, then all visited-set
//     buckets, then all CAS inserts, while the code rows of the probable new candidates are prefetched into L2;
//   * one hop ahead: the adjacency row of the node the NEXT hop will most likely expand (the closest unvisited
//     entry after this hop's node) is copied into the warp's shared memory with cp.async while this hop runs, and
//     once it has landed the visited-set buckets of its neighbours are prefetched into L2 — when the guess holds
//     (a candidate of this hop rarely lands in front of it at large L) the next hop starts with its row in
//     shared memory and its buckets in L2 instead of two dependent DRAM round trips.
// No tensor cores: byte gathers + short FMA chains; HBM traffic is n_chunks code bytes per candidate + the adjacency.
#include "dab_common.cuh"
#include "quant_device.cuh"
#include "search_common.cuh"
#include "search_pq.cuh"

#include <algorithm>

namespace dab {

constexpr int kPqsMaxWarps = 16;
constexpr size_t kPqsSmemLimit = 227 * 1024;  // opt-in dynamic shared memory of one CTA on sm_100

template <int QT, int CL>
__global__ void __launch_bounds__(kPqsMaxWarps * 32, 1) search_kernel_pqs(const SearchParamsPq p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    float* spiv = reinterpret_cast<float*>(smem);
    {
        const uint32_t total = p.n_centers * p.dim;
        for (uint32_t e = threadIdx.x; e < total; e += blockDim.x) {
            const uint32_t c = e / p.dim, d = e - c * p.dim;
            spiv[(size_t)c * p.piv_stride + d] = __ldg(p.pivots + e);
        }
    }
    __syncthreads();  // the only CTA-wide barrier: from here on every warp runs its own queries

    uint8_t* base = smem + p.piv_bytes + (size_t)wib * p.warp_smem;
    float* qf = reinterpret_cast<float*>(base + p.off_q);
    float* qd = reinterpret_cast<float*>(base + p.off_qd);
    uint32_t* qi = reinterpret_cast<uint32_t*>(base + p.off_qi);
    uint32_t* cid = reinterpret_cast<uint32_t*>(base + p.off_cid);
    float* cd = reinterpret_cast<float*>(base + p.off_cd);
    uint32_t* beam_ids = reinterpret_cast<uint32_t*>(base + p.off_beam);
    uint32_t* nrow = reinterpret_cast<uint32_t*>(base + p.off_nrow);  // adjacency row copied one hop ahead (<= 96 words)
    const bool spec_ok = p.adj_stride <= 96;

    const uint32_t warp_slot = blockIdx.x * (blockDim.x >> 5) + wib;
    const uint32_t nbk = p.n_buckets;
    uint32_t* table = p.tables + (size_t)warp_slot * nbk * 8;
    const uint32_t hlimit = nbk * 7;
    const uint64_t n_total = p.n_points + p.n_start;
    const int dim = (int)p.dim;
    const bool ip = p.ip_table != 0;
    const uint32_t pstride = p.piv_stride;
    const bool codes8 = (p.n_chunks & 7u) == 0;  // code rows are 8-byte aligned and every lane's share is whole

    // ADC distances of candidates cid[0..n) -> cd[]: four lanes per candidate, lane g owns chunks [8g, 8g + 8)
    auto adc = [&](uint32_t n) {
        const int g = lane & 3;
        const uint32_t ch0 = (uint32_t)g * 8;
        for (uint32_t c0 = 0; c0 < n; c0 += 8) {
            const uint32_t c = c0 + (uint32_t)(lane >> 2);
            const bool live = c < n && ch0 < p.n_chunks;
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = 0.0f;
            if (live) {
                const uint8_t* code = p.codes + (size_t)cid[c] * p.n_chunks + ch0;
                uint32_t w0 = 0, w1 = 0;
                if (codes8) {
                    const uint2 w = __ldg(reinterpret_cast<const uint2*>(code));
                    w0 = w.x, w1 = w.y;
                } else {
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        if (ch0 + i < p.n_chunks) {
                            const uint32_t b = __ldg(code + i);
                            if (i < 4) w0 |= b << (i * 8);
                            else w1 |= b << ((i - 4) * 8);
                        }
                    }
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    if (ch0 + i < p.n_chunks) {
                        const uint32_t center = ((i < 4 ? w0 : w1) >> ((i & 3) * 8)) & 0xFFu;
                        v[i] = pqs_term<CL>(qf, spiv, pstride, p.offsets, ch0 + i, center, ip);
                    }
                }
            }
            // pq_dist_lookup_single (fixed_chunk_pq_table.rs:82-98): one accumulator from 0.0, chunks in order.  Lane s of
            // the team continues the sum lane s - 1 left; a lane's missing chunks are +0.0 terms, which change nothing
            // (the accumulator is never -0.0: it starts at +0.0 and (+0.0) + (-0.0) = +0.0)
            float acc = 0.0f;
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                if (g == s) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) acc = __fadd_rn(acc, v[i]);
                }
                acc = __shfl_sync(kFull, acc, (lane & ~3) | s);
            }
            if (c < n && g == 0) cd[c] = acc;
        }
        __syncwarp();
    };

    for (;;) {
        uint32_t w = 0;
        if (lane == 0) w = atomicAdd(p.counters, 1u);
        w = __shfl_sync(kFull, w, 0);
        if (w >= p.n_work) break;
        const uint32_t qidx = p.query_list ? p.query_list[w] : w;

        // ---- query -> f32 (T: Into<f32>), visited clear
        __syncwarp();
        for (int e = lane; e < dim; e += 32) {
            float v;
            switch (p.dtype) {
                case DAB_F32: v = reinterpret_cast<const float*>(p.queries)[(size_t)qidx * dim + e]; break;
                case DAB_F16: v = __half2float(reinterpret_cast<const __half*>(p.queries)[(size_t)qidx * dim + e]); break;
                case DAB_I8: v = (float)reinterpret_cast<const int8_t*>(p.queries)[(size_t)qidx * dim + e]; break;
                default: v = (float)reinterpret_cast<const uint8_t*>(p.queries)[(size_t)qidx * dim + e]; break;
            }
            qf[e] = v;
        }
        for (uint32_t i = lane; i < nbk; i += 32) store_empty_bucket(table + (size_t)i * 8);
        __syncwarp();

        uint32_t size = 0, cursor_lo = 0, cmps = 0, hops = 0, nvisited = 0;
        bool overflow = false;
        uint32_t spec_id = kEmptyV2;  // the node whose adjacency row is in (or on its way to) nrow

        // ---- start points first (groups of <= 32), then the greedy loop; both feed the one ADC + merge below
        uint32_t s0 = 0;
        for (;;) {
            uint32_t ncand = 0, nb = 0;
            if (s0 < p.n_start) {
                const uint32_t n = min(32u, p.n_start - s0);
                if ((uint32_t)lane < n) {
                    const uint32_t id = (uint32_t)p.n_points + s0 + lane;
                    cid[lane] = id;
                    const uint32_t b = bucket_of(id, nbk);
                    uint32_t bs[8];
                    load_bucket(table + (size_t)b * 8, bs);
                    bucket_insert(table, nbk, b, bs, id);
                }
                s0 += 32;
                ncand = n;
                nvisited += n;
            } else {
                const uint32_t lim = min(p.cap, size);
                while (nb < p.beam) {
                    const uint32_t idx = first_unvisited(qi, cursor_lo, lim, lane);
                    if (idx >= lim) break;
                    const uint32_t id = qi[idx];
                    __syncwarp();
                    if (lane == 0) {
                        qi[idx] = id | kFlagV2;
                        beam_ids[nb] = id;
                    }
                    cursor_lo = idx + 1;
                    ++nb;
                    __syncwarp();
                }
                if (nb == 0) break;
                // the row copied one hop ahead, if the guess was right
                uint32_t w0[3] = {kEmptyV2, kEmptyV2, kEmptyV2};
                bool have_row = false;
                if (spec_ok) {
                    asm volatile("cp.async.wait_group 0;" ::: "memory");
                    __syncwarp();
                    have_row = spec_id == beam_ids[0];
                    if (have_row) {
#pragma unroll
                        for (int t = 0; t < 3; ++t) {
                            const uint32_t j = (uint32_t)t * 32 + lane;
                            if (j < p.adj_stride) w0[t] = nrow[j];
                        }
                    }
                    __syncwarp();  // nrow has been read before the next copy is issued
                }
                {
                    // the node the next hop will most likely expand (unless a candidate of this hop lands in front of it)
                    const uint32_t nx = first_unvisited(qi, cursor_lo, lim, lane);
                    spec_id = kEmptyV2;
                    if (nx < lim) {
                        const uint32_t nid = qi[nx];
                        const uint32_t* r = p.adj + (size_t)nid * p.adj_stride;
                        if (spec_ok) {
                            if ((uint32_t)lane * 4u < p.adj_stride)
                                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(nrow + lane * 4)),
                                             "l"(r + lane * 4)
                                             : "memory");
                            asm volatile("cp.async.commit_group;" ::: "memory");
                            spec_id = nid;
                        } else {
                            const uint32_t bytes = p.adj_stride * 4;
                            for (uint32_t o = (uint32_t)lane * 128u; o < bytes; o += 32 * 128u) prefetch_l2(reinterpret_cast<const uint8_t*>(r) + o);
                        }
                    }
                }
                for (uint32_t b = 0; b < nb; ++b) {
                    const uint32_t node = beam_ids[b];
                    const uint32_t* row = p.adj + (size_t)node * p.adj_stride;
                    uint32_t deg = 0;
                    for (uint32_t g0 = 0; g0 == 0 || g0 <= deg; g0 += 96) {
                        // every word of (this part of) the row in one round trip; word 0 is the length
                        uint32_t wd[3];
#pragma unroll
                        for (int t = 0; t < 3; ++t) {
                            const uint32_t j = g0 + (uint32_t)t * 32 + lane;
                            if (b == 0 && have_row) wd[t] = w0[t];  // (adj_stride <= 96: one pass covers the row)
                            else wd[t] = j < p.adj_stride ? __ldg(row + j) : kEmptyV2;
                        }
                        if (g0 == 0) deg = min(__shfl_sync(kFull, wd[0], 0), p.max_degree);
                        // every bucket in one round trip
                        uint32_t bs[3][8], bk[3];
                        bool act[3];
#pragma unroll
                        for (int t = 0; t < 3; ++t) {
                            const uint32_t j = g0 + (uint32_t)t * 32 + lane;
                            act[t] = j >= 1 && j <= deg;
                            bk[t] = 0;
                            if (act[t]) {
                                bk[t] = bucket_of(wd[t], nbk);
                                load_bucket(table + (size_t)bk[t] * 8, bs[t]);
                            }
                        }
                        // every insert in one round trip (HashSet::insert: CAS into the first free slot of the home bucket);
                        // state 0: already in the set / inactive, 1: CAS issued, 2: needs the general probe loop
                        int state[3];
                        uint32_t old[3];
#pragma unroll
                        for (int t = 0; t < 3; ++t) {
                            state[t] = 0;
                            old[t] = 0;
                            if (act[t]) {
                                bool found = false;
                                int empty = -1;
#pragma unroll
                                for (int k2 = 7; k2 >= 0; --k2) {
                                    found |= bs[t][k2] == wd[t];
                                    if (bs[t][k2] == kEmptyV2) empty = k2;
                                }
                                if (!found) {
                                    if (empty >= 0) {
                                        if (wd[t] < n_total) prefetch_l2(p.codes + (size_t)wd[t] * p.n_chunks);
                                        old[t] = atomicCAS(table + (size_t)bk[t] * 8 + empty, kEmptyV2, wd[t]);
                                        state[t] = 1;
                                    } else {
                                        state[t] = 2;
                                    }
                                }
                            }
                        }
#pragma unroll
                        for (int t = 0; t < 3; ++t) {
                            bool inserted = false;
                            if (state[t] == 1) {
                                if (old[t] == kEmptyV2) inserted = true;
                                else if (old[t] != wd[t]) state[t] = 2;  // another lane took the slot for a different id
                            }
                            if (state[t] == 2) {
                                load_bucket(table + (size_t)bk[t] * 8, bs[t]);
                                inserted = bucket_insert(table, nbk, bk[t], bs[t], wd[t]);
                            }
                            const bool isnew = inserted && wd[t] < n_total;
                            const unsigned mi = __ballot_sync(kFull, inserted);
                            const unsigned mn = __ballot_sync(kFull, isnew);
                            if (isnew) cid[ncand + __popc(mn & ((1u << lane) - 1u))] = wd[t];
                            ncand += __popc(mn);
                            nvisited += __popc(mi);
                        }
                    }
                    if (nvisited + p.max_degree > hlimit) {
                        overflow = true;
                        break;
                    }
                }
                if (overflow) break;
            }
            __syncwarp();
            adc(ncand);
            if (spec_id != kEmptyV2) {
                // the next hop's row has landed by now: its neighbours' visited-set buckets go to L2 during the merge
                asm volatile("cp.async.wait_group 0;" ::: "memory");
                __syncwarp();
                const uint32_t d2 = min(nrow[0], p.max_degree);
#pragma unroll
                for (int t = 0; t < 3; ++t) {
                    const uint32_t j = (uint32_t)t * 32 + lane;
                    if (j >= 1 && j <= d2)
                        asm volatile("prefetch.global.L2::evict_last [%0];" ::"l"(table + (size_t)bucket_of(nrow[j], nbk) * 8));
                }
            }
            for (uint32_t c0 = 0; c0 < ncand; c0 += 32)
                merge_any<QT>(qd, qi, p.cap, size, cursor_lo, cid, cd, c0, min(32u, ncand - c0), lane);
            cmps += ncand;
            hops += nb;
        }

        if (overflow) {
            if (lane == 0) {
                const uint32_t o = atomicAdd(p.counters + 1, 1u);
                p.overflow_list[o] = qidx;
            }
            continue;
        }
        {
            const uint32_t n = min(p.cap, size);
            if (p.list_ids) {
                for (uint32_t i = lane; i < n; i += 32) p.list_ids[(size_t)qidx * p.list_cap + i] = qi[i] & ~kFlagV2;
                if (lane == 0) p.list_counts[qidx] = n;
            }
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
            }
        }
    }
}

bool pqs_plan(const dab_index* idx, uint32_t warp_smem, uint32_t nq, PqsPlan* out) {
    if (idx->hooks.pq_global_lut) return false;
    if (idx->pq_chunks == 0 || idx->pq_chunks > 32) return false;  // a team of four lanes covers 32 chunks
    // pivot rows padded to an odd multiple of four floats: 16-byte aligned chunk loads, and the rows of eight
    // consecutive centres start in eight different 16-byte bank groups
    uint32_t stride = (uint32_t)round_up(idx->dim, 4);
    if ((stride & 7u) == 0) stride += 4;
    const size_t piv_bytes = (size_t)idx->pq_centers * stride * 4;
    if (piv_bytes + 4 * (size_t)warp_smem > kPqsSmemLimit) return false;  // fewer than four warps would fit
    int warps = (int)std::min<size_t>(kPqsMaxWarps, (kPqsSmemLimit - piv_bytes) / warp_smem);
    // small batches: spread the queries over the SMs instead of filling a few CTAs
    const int need = (int)(((uint64_t)nq + idx->sm_count - 1) / idx->sm_count);
    warps = std::max(std::min(warps, std::max(need, 4)), 1);
    out->warps = warps;
    out->grid = (int)std::min<uint64_t>((uint64_t)idx->sm_count, ((uint64_t)nq + warps - 1) / warps);
    out->piv_stride = stride;
    out->piv_bytes = (uint32_t)piv_bytes;
    out->smem = piv_bytes + (size_t)warps * warp_smem;
    out->chunk_len = (idx->pq_uniform_len == 4 || idx->pq_uniform_len == 8) ? (int)idx->pq_uniform_len : 0;
    return true;
}

int pqs_launch(dab_index* idx, const SearchParamsPq& p, const PqsPlan& plan, uint32_t cap) {
    void (*kern)(const SearchParamsPq);
#define DAB_PQS_PICK(CL_)                                                                                        \
    kern = cap <= 128 ? search_kernel_pqs<4, CL_> : cap <= 256 ? search_kernel_pqs<8, CL_> : cap <= 512 ? search_kernel_pqs<16, CL_> : search_kernel_pqs<32, CL_>
    if (plan.chunk_len == 4) DAB_PQS_PICK(4);
    else if (plan.chunk_len == 8) DAB_PQS_PICK(8);
    else DAB_PQS_PICK(0);
#undef DAB_PQS_PICK
    DAB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem));
    kern<<<plan.grid, plan.warps * 32, plan.smem, idx->stream>>>(p);
    DAB_LAUNCHED();
    DAB_CUDA(cudaGetLastError());
    return DAB_OK;
}

}  // namespace dab
