// search_kernel_pq.cu — batched greedy search whose traversal distances come from a quantized store:
// PQ ADC lookups (MODE 0) or scalar-quantized codes (MODE 1, see the SQ notes below).
//
// Restates the providers' quant accessor (diskann-providers/src/model/graph/provider/async_/
// inmem/product.rs:311-340: expand_beam with `computer.evaluate_similarity(aux_vectors[i])`)
// around the same search_internal loop (diskann/src/graph/index.rs:1933-2000):
//   * QueryComputer::new (pq/distance/dynamic.rs:63-87): L2 and CosineNormalized -> TableL2,
//     InnerProduct -> TableIP (entries are -dot); the query is converted to f32 first;
//   * the warp builds its query's table once (n_chunks x n_centers f32, entries in the
//     reference's SIMD order for the chunk length, fixed_chunk_pq_table.rs:152-187) into a
//     per-warp global scratch that stays in L2;
//   * per hop every lane owns one surviving neighbour: coalesced 16 B code loads, one table
//     gather per chunk, and the sum is accumulated in chunk order from 0.0
//     (pq_dist_lookup_single, fixed_chunk_pq_table.rs:82-98) -> bit-identical ADC distances;
//   * visited set, sorted list and post-processing are the shared exact helpers.
// No tensor cores: LUT gather + byte loads, HBM traffic is n_chunks code bytes per candidate.
//
// MODE 1 — the scalar-quantized accessor (providers inmem/scalar.rs:449-570): the query is
// compressed once per search with the store's own quantizer (SQStore::query_computer, :227-253:
// as_f32, rescale to the mean norm for InnerProduct, ScalarQuantizer::compress) into the same
// dense N-bit layout as the rows (bits/slice.rs:261-323), and every candidate distance is
// Compensated{SquaredL2, IP, CosineNormalized} (scalar/vectors.rs:206-460): an exact integer core
// over the packed words (bits/distances.rs:397, 979 — here vabsdiffu4 + dp4a on masked fields,
// popc for 1 bit) and the reference's f32 epilogue.  One lane per candidate, 16 B code loads,
// the query words broadcast from shared memory; traffic is ceil(dim * N / 8) bytes per candidate
// (+ 4 B compensation for InnerProduct).
#include "dab_common.cuh"
#include "quant_device.cuh"
#include "search_common.cuh"
#include "search_pq.cuh"
#include "search_smem.cuh"

#include <algorithm>
#include <type_traits>

namespace dab {

template <int NBITS>
__device__ __forceinline__ void sq_row(const uint4* __restrict__ row, const uint4* qc, uint32_t vecs, bool want_ip, uint32_t& l2,
                                       uint32_t& ip) {
    for (uint32_t v = 0; v < vecs; ++v) {
        const uint4 a = __ldg(row + v);
        const uint4 b = qc[v];
        sq_word<NBITS>(a.x, b.x, want_ip, l2, ip);
        sq_word<NBITS>(a.y, b.y, want_ip, l2, ip);
        sq_word<NBITS>(a.z, b.z, want_ip, l2, ip);
        sq_word<NBITS>(a.w, b.w, want_ip, l2, ip);
    }
}

template <int QT, int MODE>
__global__ void __launch_bounds__(kPqWarps * 32) search_kernel_pq(const SearchParamsPq p) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    uint8_t* base = smem + (size_t)wib * p.warp_smem;
    float* qf = reinterpret_cast<float*>(base + p.off_q);
    float* qd = reinterpret_cast<float*>(base + p.off_qd);
    uint32_t* qi = reinterpret_cast<uint32_t*>(base + p.off_qi);
    uint32_t* cid = reinterpret_cast<uint32_t*>(base + p.off_cid);
    float* cd = reinterpret_cast<float*>(base + p.off_cd);
    uint32_t* beam_ids = reinterpret_cast<uint32_t*>(base + p.off_beam);
    uint32_t* qc = reinterpret_cast<uint32_t*>(base + p.off_qc);  // MODE 1: the query's packed codes
    float q_comp = 0.0f;

    const uint32_t warp_slot = blockIdx.x * kPqWarps + wib;
    const uint32_t nbk = p.n_buckets;
    uint32_t* table = p.tables + (size_t)warp_slot * nbk * 8;
    const uint32_t hlimit = nbk * 7;
    const uint64_t n_total = p.n_points + p.n_start;
    const uint32_t entries = p.n_chunks * p.n_centers;
    float* lut = p.luts + (size_t)warp_slot * entries;
    const int dim = (int)p.dim;

    // quantized distances of candidates cid[0..n) -> cd[]: one lane per candidate
    auto adc = [&](uint32_t n) {
        for (uint32_t c0 = 0; c0 < n; c0 += 32) {
            const uint32_t c = c0 + lane;
            if (MODE == 1) {
                if (c < n) {
                    const uint32_t id = cid[c];
                    const uint4* row = reinterpret_cast<const uint4*>(p.sq_codes + (size_t)id * p.sq_stride);
                    const uint4* q4 = reinterpret_cast<const uint4*>(qc);
                    const uint32_t vecs = p.sq_stride >> 4;
                    const bool want_ip = p.sq_metric == DAB_INNER_PRODUCT;
                    uint32_t l2 = 0, ip = 0;
                    switch (p.sq_nbits) {
                        case 8: sq_row<8>(row, q4, vecs, want_ip, l2, ip); break;
                        case 4: sq_row<4>(row, q4, vecs, want_ip, l2, ip); break;
                        case 2: sq_row<2>(row, q4, vecs, want_ip, l2, ip); break;
                        default: sq_row<1>(row, q4, vecs, want_ip, l2, ip); break;
                    }
                    // epilogues: scalar/vectors.rs:206-237 (L2), 310-376 (IP), 380-460 (CosineNormalized)
                    const float ibs = __fdiv_rn(1.0f, (float)((1u << p.sq_nbits) - 1u));
                    const float bit_scale = __fmul_rn(ibs, ibs);
                    const float mul = __fmul_rn(bit_scale, p.sq_scale_squared);
                    float r;
                    if (want_ip) {
                        const float m = __fadd_rn(__fmaf_rn(mul, (float)ip, p.sq_shift_square_norm), __fadd_rn(__ldg(p.sq_comp + id), q_comp));
                        r = -m;
                    } else if (p.sq_metric == DAB_L2) {
                        r = __fmul_rn(mul, (float)l2);
                    } else {
                        const float l = __fmul_rn(mul, (float)l2);
                        r = __fsub_rn(1.0f, __fsub_rn(1.0f, __fdiv_rn(l, 2.0f)));
                    }
                    cd[c] = r;
                }
            } else if (p.direct_cosine) {
                // DirectCosine (pq/distance/cosine.rs:16-70; direct_distance_impl, fixed_chunk_pq_table.rs:35-59): the
                // Resumable V3 cosine (Strategy2x4) accumulated chunk by chunk over the pivots the code selects, 1 - cos
                if (c < n) {
                    const uint8_t* code = p.codes + (size_t)cid[c] * p.n_chunks;
                    float nx[8], ny[8], xy[8];
#pragma unroll
                    for (int l = 0; l < 8; ++l) nx[l] = ny[l] = xy[l] = 0.0f;
                    for (uint32_t ch = 0; ch < p.n_chunks; ++ch) {
                        const uint32_t start = p.offsets[ch], stop = p.offsets[ch + 1];
                        const float* xc = qf + start;
                        const float* yc = p.pivots + (size_t)__ldg(code + ch) * dim + start;
                        float a[8], b[8], d[8];
                        thread_simd_combined<2, KIND_IP>(xc, xc, (int)(stop - start), a);
                        thread_simd_combined<2, KIND_IP>(yc, yc, (int)(stop - start), b);
                        thread_simd_combined<2, KIND_IP>(xc, yc, (int)(stop - start), d);
#pragma unroll
                        for (int l = 0; l < 8; ++l) {
                            nx[l] = __fadd_rn(nx[l], a[l]);
                            ny[l] = __fadd_rn(ny[l], b[l]);
                            xy[l] = __fadd_rn(xy[l], d[l]);
                        }
                    }
                    cd[c] = __fsub_rn(1.0f, cosine_finish(thread_tree8(nx), thread_tree8(ny), thread_tree8(xy)));
                }
            } else if (c < n) {
                const uint8_t* code = p.codes + (size_t)cid[c] * p.n_chunks;
                float accum = 0.0f;
                uint32_t ch = 0;
                if ((p.n_chunks & 15u) == 0) {
                    for (; ch < p.n_chunks; ch += 16) {
                        const uint4 w = __ldg(reinterpret_cast<const uint4*>(code + ch));
                        const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
                        float v[16];
#pragma unroll
                        for (int k2 = 0; k2 < 16; ++k2)
                            v[k2] = __ldcg(lut + (ch + k2) * p.n_centers + ((ws[k2 >> 2] >> ((k2 & 3) * 8)) & 0xFFu));
#pragma unroll
                        for (int k2 = 0; k2 < 16; ++k2) accum = __fadd_rn(accum, v[k2]);
                    }
                } else {
                    for (; ch < p.n_chunks; ++ch) accum = __fadd_rn(accum, __ldcg(lut + ch * p.n_centers + __ldg(code + ch)));
                }
                cd[c] = accum;
            }
        }
        __syncwarp();
    };

    for (;;) {
        uint32_t w = 0;
        if (lane == 0) w = atomicAdd(p.counters, 1u);
        w = __shfl_sync(kFull, w, 0);
        if (w >= p.n_work) break;
        const uint32_t qidx = p.query_list ? p.query_list[w] : w;

        // ---- query -> f32 (T: Into<f32>), table build, visited clear
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
        if (MODE == 1) {
            // rescale (scalar/quantizer.rs:300-310): InnerProduct::evaluate(x, x), sqrt, x *= to_norm / norm
            if (p.sq_metric == DAB_INNER_PRODUCT && p.sq_mean_norm != 0.0f) {
                float norm = 0.0f;
                if (lane == 0) norm = __fsqrt_rn(thread_simd_l2ip<KIND_IP>(qf, qf, dim));
                norm = __shfl_sync(kFull, norm, 0);
                if (norm != 0.0f) {
                    const float sc = __fdiv_rn(p.sq_mean_norm, norm);
                    for (int e = lane; e < dim; e += 32) qf[e] = __fmul_rn(qf[e], sc);
                }
                __syncwarp();
            }
            // ScalarQuantizer::compress (scalar/quantizer.rs:190-239): codes in parallel ...
            const float maxv = (float)((1u << p.sq_nbits) - 1u);
            const float inverse_scale = __fdiv_rn(maxv, p.sq_scale);
            for (int e = lane; e < dim; e += 32) {
                const float t = __fmul_rn(__fsub_rn(qf[e], __ldg(p.sq_shift + e)), inverse_scale);
                const float code = t != t ? t : (t < 0.0f ? 0.0f : (t > maxv ? maxv : t));
                qf[e] = roundf(code);
            }
            __syncwarp();
            // ... the compensation is one sequential FMA chain over the dimensions (:407-430)
            if (lane == 0) {
                float dot = 0.0f;
                for (int e = 0; e < dim; ++e) dot = __fmaf_rn(qf[e], __ldg(p.sq_shift + e), dot);
                q_comp = __fmul_rn(__fmul_rn(p.sq_scale, __fdiv_rn(1.0f, maxv)), dot);
            }
            q_comp = __shfl_sync(kFull, q_comp, 0);
            // dense packing, value i at bit i * nbits (bits/slice.rs:261-305); padding words are zero
            const uint32_t per_word = 32u / (uint32_t)p.sq_nbits;
            for (uint32_t wd = lane; wd < (p.sq_stride >> 2); wd += 32) {
                uint32_t acc = 0;
                for (uint32_t j = 0; j < per_word; ++j) {
                    const uint32_t e = wd * per_word + j;
                    if (e < (uint32_t)dim) {
                        const float c = qf[e];
                        acc |= (c != c ? 0u : (uint32_t)c) << (j * (uint32_t)p.sq_nbits);
                    }
                }
                qc[wd] = acc;
            }
            __syncwarp();
        }
        for (uint32_t t = lane; MODE == 0 && !p.direct_cosine && t < entries; t += 32) {
            const uint32_t chunk = t / p.n_centers, center = t % p.n_centers;
            const uint32_t start = p.offsets[chunk], stop = p.offsets[chunk + 1];
            const float* piv = p.pivots + (size_t)center * dim + start;
            float v;
            if (p.ip_table) v = -thread_simd_l2ip<KIND_IP>(qf + start, piv, (int)(stop - start));
            else v = thread_simd_l2ip<KIND_L2>(qf + start, piv, (int)(stop - start));
            __stcg(lut + t, v);
        }
        __syncwarp();

        uint32_t size = 0, cursor_lo = 0, cmps = 0, hops = 0, nvisited = 0;
        bool overflow = false;

        // ---- start points
        for (uint32_t s0 = 0; s0 < p.n_start; s0 += 32) {
            const uint32_t n = min(32u, p.n_start - s0);
            if ((uint32_t)lane < n) {
                const uint32_t id = (uint32_t)p.n_points + s0 + lane;
                cid[lane] = id;
                const uint32_t b = bucket_of(id, nbk);
                uint32_t bs[8];
                load_bucket(table + (size_t)b * 8, bs);
                bucket_insert(table, nbk, b, bs, id);
            }
            __syncwarp();
            adc(n);
            merge_any<QT>(qd, qi, p.cap, size, cursor_lo, cid, cd, 0, n, lane);
            nvisited += n;
            cmps += n;
        }

        // ---- greedy loop
        for (;;) {
            const uint32_t lim = min(p.cap, size);
            uint32_t nb = 0;
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
            uint32_t ncand = 0;
            for (uint32_t b = 0; b < nb; ++b) {
                const uint32_t node = beam_ids[b];
                const uint32_t* row = p.adj + (size_t)node * p.adj_stride;
                const uint32_t deg = min(__ldg(row), p.max_degree);
                for (uint32_t c0 = 0; c0 < deg + 1; c0 += 32) {
                    const uint32_t j = c0 + lane;
                    const uint32_t word = j < p.adj_stride ? __ldg(row + j) : kEmptyV2;
                    bool inserted = false;
                    if (j >= 1 && j <= deg) {
                        const uint32_t b2 = bucket_of(word, nbk);
                        uint32_t bs[8];
                        load_bucket(table + (size_t)b2 * 8, bs);
                        inserted = bucket_insert(table, nbk, b2, bs, word);
                    }
                    const bool isnew = inserted && word < n_total;
                    const unsigned mi = __ballot_sync(kFull, inserted);
                    const unsigned mn = __ballot_sync(kFull, isnew);
                    if (isnew) cid[ncand + __popc(mn & ((1u << lane) - 1u))] = word;
                    ncand += __popc(mn);
                    nvisited += __popc(mi);
                }
                if (nvisited + p.max_degree > hlimit) {
                    overflow = true;
                    break;
                }
            }
            if (overflow) break;
            __syncwarp();
            adc(ncand);
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

// ---- Rerank (diskann-providers/.../inmem/full_precision.rs:356-399 behind FilterStartPoints,
// product.rs:391-400): every candidate of best.iter() that is not a start point gets its
// full-precision Distance<T, T> to the query; the list is ordered by that distance (ties keep
// their traversal order: the reference's sort_unstable_by leaves them unspecified) and the
// first k are returned.  One warp per query; rows are gathered with the wide-load loops of
// search_smem.cuh (f32 x f32 has the query x row association; i8 / u8 are exact).
constexpr int kRerankWarps = 4;
struct RerankParams {
    const uint8_t* vectors;
    size_t row_stride;
    uint64_t n_points;
    uint32_t dim;
    const void* queries;  // index dtype
    uint32_t nq, k, list_cap;
    const uint32_t* list_ids;
    const uint32_t* list_counts;
    uint32_t* out_ids;
    float* out_dists;
    uint32_t* out_counts;
    uint32_t warp_smem, off_ids, off_d;
};

// NA = 4: the wide-load loops (f32 rows, L2 / InnerProduct / CosineNormalized; integers).  NA = 2: the schemas with two
// accumulators — f16 x f16 (Strategy2x4, simd.rs:424-483: both sides widened to f32 lanes, so the f32 copy of the query
// in shared memory is the same operand) and Metric::Cosine over float rows — one team of 16 lanes per row.
template <typename TD, int KIND, int POST, int NA = 4>
__global__ void __launch_bounds__(kRerankWarps * 32) rerank_kernel(const RerankParams p) {
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr bool kInt = std::is_same<TD, int8_t>::value || std::is_same<TD, uint8_t>::value;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    uint8_t* base = smem + (size_t)wib * p.warp_smem;
    float* qf = reinterpret_cast<float*>(base);
    uint32_t* cid = reinterpret_cast<uint32_t*>(base + p.off_ids);
    float* cd = reinterpret_cast<float*>(base + p.off_d);
    const int dim = (int)p.dim;
    for (uint32_t q = blockIdx.x * kRerankWarps + wib; q < p.nq; q += gridDim.x * kRerankWarps) {
        __syncwarp();
        const TD* s = reinterpret_cast<const TD*>(p.queries) + (size_t)q * dim;
        if constexpr (kInt) {
            uint8_t* qb = reinterpret_cast<uint8_t*>(qf);
            const int qbytes = (dim + 15) & ~15;
            for (int e = lane; e < qbytes; e += 32) qb[e] = e < dim ? reinterpret_cast<const uint8_t*>(s)[e] : 0;
        } else {
            for (int e = lane; e < dim; e += 32) qf[e] = to_f32(s[e]);
        }
        const uint32_t n = min(p.list_counts[q], p.list_cap);
        uint32_t m = 0;  // candidates that are not start points, traversal order kept
        for (uint32_t b = 0; b < n; b += 32) {
            const uint32_t i = b + lane;
            const uint32_t id = i < n ? p.list_ids[(size_t)q * p.list_cap + i] : kEmptyV2;
            const bool keep = i < n && id < p.n_points;
            const unsigned mk = __ballot_sync(kFull, keep);
            if (keep) cid[m + __popc(mk & ((1u << lane) - 1u))] = id;
            m += __popc(mk);
        }
        __syncwarp();
        if constexpr (kInt) {
            int qq = 0;
            if (KIND != KIND_IP) qq = warp_int_self<std::is_same<TD, int8_t>::value>(reinterpret_cast<const uint8_t*>(qf), dim, lane);
            wide_distances_int<std::is_same<TD, int8_t>::value, KIND, POST, 4>(reinterpret_cast<const uint8_t*>(qf), qq, p.vectors, p.row_stride,
                                                                             cid, m, cd, dim, lane);
        } else if constexpr (NA == 2) {
            constexpr int S = 16, U = 2;
            const int team = lane / S, slot = lane % S;
            for (uint32_t c0 = 0; c0 < m; c0 += 2 * U) {  // every lane takes part in the team shuffles: uniform trip count
                const TD* rows[U];
#pragma unroll
                for (int u = 0; u < U; ++u)
                    rows[u] = reinterpret_cast<const TD*>(p.vectors + (size_t)cid[min(c0 + team * U + u, m - 1)] * p.row_stride);
                float r[U];
                team_float_multi<2, KIND, U>(qf, rows, dim, slot, r);
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (slot == 0 && c0 + team * U + u < m) cd[c0 + team * U + u] = post_op<POST>(r[u]);
            }
        } else {
            wide_distances<TD, KIND, POST, 2, 4>(qf, p.vectors, p.row_stride, cid, m, cd, dim, lane);
        }
        __syncwarp();
        for (uint32_t i = lane; i < m; i += 32) {
            const float di = cd[i];
            uint32_t r = 0;
            for (uint32_t j = 0; j < m; ++j) {
                const float dj = cd[j];
                r += (dj < di || (dj == di && j < i)) ? 1u : 0u;
            }
            if (r < p.k) {
                p.out_ids[(size_t)q * p.k + r] = cid[i];
                p.out_dists[(size_t)q * p.k + r] = di;
            }
        }
        const uint32_t count = min(m, p.k);
        for (uint32_t i = count + lane; i < p.k; i += 32) {
            p.out_ids[(size_t)q * p.k + i] = kEmptyV2;
            p.out_dists[(size_t)q * p.k + i] = __int_as_float(0x7F800000);
        }
        if (lane == 0 && p.out_counts) p.out_counts[q] = count;
    }
}

static int launch_rerank(dab_index* idx, const void* d_queries, uint32_t nq, uint32_t k, uint32_t list_cap, const uint32_t* d_list,
                         const uint32_t* d_list_n, uint32_t* d_ids, float* d_dists, uint32_t* d_counts) {
    const bool is_int = idx->dtype == DAB_I8 || idx->dtype == DAB_U8;
    const MetricPlan plan = plan_for(idx->metric, is_int);
    RerankParams p;
    memset(&p, 0, sizeof(p));
    p.vectors = idx->d_vectors;
    p.row_stride = idx->row_stride;
    p.n_points = idx->n_points;
    p.dim = idx->dim;
    p.queries = d_queries;
    p.nq = nq;
    p.k = k;
    p.list_cap = list_cap;
    p.list_ids = d_list;
    p.list_counts = d_list_n;
    p.out_ids = d_ids;
    p.out_dists = d_dists;
    p.out_counts = d_counts;
    size_t off = is_int ? round_up((size_t)idx->dim, 16) : round_up((size_t)idx->dim * 4, 16);
    p.off_ids = (uint32_t)off;
    off += round_up((size_t)list_cap * 4, 16);
    p.off_d = (uint32_t)off;
    off += round_up((size_t)list_cap * 4, 16);
    p.warp_smem = (uint32_t)off;
    const size_t smem = off * kRerankWarps;
    if (smem > 200 * 1024) return fail(DAB_ERR_INVALID_ARGUMENT, "rerank: configuration needs %zu B shared memory per CTA", smem);
    const int grid = (int)std::min<uint64_t>(((uint64_t)nq + kRerankWarps - 1) / kRerankWarps, (uint64_t)idx->sm_count * 8);
#define DAB_RERANK(TD, K_, P_, ...)                                                                          \
    do {                                                                                                     \
        auto kern = rerank_kernel<TD, K_, P_, ##__VA_ARGS__>;                                                \
        DAB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));        \
        kern<<<grid, kRerankWarps * 32, smem, idx->stream>>>(p);                                             \
    } while (0)
    if (idx->dtype == DAB_F32) {
        if (plan.kind == KIND_L2) DAB_RERANK(float, KIND_L2, POST_ID);
        else if (plan.kind == KIND_COS) DAB_RERANK(float, KIND_COS, POST_ONE_MINUS, 2);
        else if (plan.post == POST_NEG) DAB_RERANK(float, KIND_IP, POST_NEG);
        else DAB_RERANK(float, KIND_IP, POST_ONE_MINUS);
    } else if (idx->dtype == DAB_F16) {
        if (plan.kind == KIND_L2) DAB_RERANK(__half, KIND_L2, POST_ID, 2);
        else if (plan.kind == KIND_COS) DAB_RERANK(__half, KIND_COS, POST_ONE_MINUS, 2);
        else if (plan.post == POST_NEG) DAB_RERANK(__half, KIND_IP, POST_NEG, 2);
        else DAB_RERANK(__half, KIND_IP, POST_ONE_MINUS, 2);
    } else if (idx->dtype == DAB_I8) {
        if (plan.kind == KIND_L2) DAB_RERANK(int8_t, KIND_L2, POST_ID);
        else if (plan.kind == KIND_IP) DAB_RERANK(int8_t, KIND_IP, POST_NEG);
        else DAB_RERANK(int8_t, KIND_COS, POST_ONE_MINUS);
    } else {
        if (plan.kind == KIND_L2) DAB_RERANK(uint8_t, KIND_L2, POST_ID);
        else if (plan.kind == KIND_IP) DAB_RERANK(uint8_t, KIND_IP, POST_NEG);
        else DAB_RERANK(uint8_t, KIND_COS, POST_ONE_MINUS);
    }
#undef DAB_RERANK
    DAB_LAUNCHED();
    DAB_CUDA(cudaGetLastError());
    return DAB_OK;
}

static int run_search_pq(dab_index* idx, const void* d_queries, uint32_t nq, uint32_t k, uint32_t l_search, uint32_t beam,
                         uint32_t* d_ids, float* d_dists, uint32_t* d_counts, uint32_t* d_cmps, uint32_t* d_hops, bool rerank,
                         int mode = 0) {
    if (!idx->graph_ready) return fail(DAB_ERR_NOT_READY, "dab_search_batch_pq: graph must be uploaded first");
    if (mode == 0 && (!idx->d_pivots || !idx->d_codes || !idx->pq_codes_ready))
        return fail(DAB_ERR_NOT_READY, "dab_search_batch_pq: no PQ codes (dab_upload_pq with codes, or dab_pq_encode_all)");
    if (mode == 1 && (!idx->d_sq_codes || !idx->sq_codes_ready))
        return fail(DAB_ERR_NOT_READY, "dab_search_batch_sq: no scalar-quantized rows (dab_upload_sq with rows, or dab_sq_encode_all)");
    if (k == 0 || l_search == 0 || beam == 0 || beam > 64) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_pq: bad k / l_search / beam_width");
    // SQStore::distance_computer (providers inmem/scalar.rs:214-226): UnsupportedDistanceMetric
    if (mode == 1 && idx->metric == DAB_COSINE)
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_sq: the scalar-quantized store supports L2, InnerProduct and CosineNormalized");
    const uint32_t cap = l_search + idx->n_start;
    if (cap > 1024) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_pq: L + #start must be <= 1024");
    SearchParamsPq p;
    memset(&p, 0, sizeof(p));
    p.adj = idx->d_adj;
    p.adj_stride = idx->adj_stride;
    p.n_points = idx->n_points;
    p.n_start = idx->n_start;
    p.dim = idx->dim;
    p.max_degree = idx->max_degree;
    p.dtype = idx->dtype;
    p.queries = d_queries;
    p.k = k;
    p.cap = cap;
    p.beam = beam;
    p.pivots = idx->d_pivots;
    p.offsets = idx->d_offsets;
    p.codes = idx->d_codes;
    p.n_chunks = idx->pq_chunks;
    p.n_centers = idx->pq_centers;
    p.ip_table = idx->metric == DAB_INNER_PRODUCT ? 1 : 0;  // L2 and CosineNormalized use TableL2 (dynamic.rs:80-85)
    p.direct_cosine = mode == 0 && idx->metric == DAB_COSINE ? 1 : 0;
    if (mode == 1) {
        p.sq_codes = idx->d_sq_codes;
        p.sq_comp = idx->d_sq_comp;
        p.sq_shift = idx->d_sq_shift;
        p.sq_stride = idx->sq_stride;
        p.sq_nbits = idx->sq_nbits;
        p.sq_metric = idx->metric;
        p.sq_scale = idx->sq_scale;
        p.sq_scale_squared = idx->sq_scale * idx->sq_scale;  // AsFunctor (scalar/quantizer.rs:316-335)
        p.sq_shift_square_norm = idx->sq_shift_square_norm;
        p.sq_mean_norm = idx->sq_mean_norm;
        p.n_chunks = 0;
    }
    p.out_ids = d_ids;
    p.out_dists = d_dists;
    p.out_counts = d_counts;
    p.out_cmps = d_cmps;
    p.out_hops = d_hops;

    size_t off = 0;
    p.off_q = 0;
    off += round_up((size_t)idx->dim * 4, 16);
    const size_t cap_pad = round_up(cap, 32) + 32;
    p.off_qd = (uint32_t)off;
    off += cap_pad * 4;
    p.off_qi = (uint32_t)off;
    off += cap_pad * 4;
    const size_t ncand_max = std::max<size_t>((size_t)beam * idx->max_degree, idx->n_start);
    p.off_cid = (uint32_t)off;
    off += round_up(ncand_max * 4, 16);
    p.off_cd = (uint32_t)off;
    off += round_up(ncand_max * 4, 16);
    p.off_beam = (uint32_t)off;
    off += round_up((size_t)beam * 4, 16);
    p.off_qc = (uint32_t)off;
    if (mode == 1) off += idx->sq_stride;
    off = round_up(off, 16);
    p.off_nrow = (uint32_t)off;  // search_kernel_pqs: the adjacency row copied one hop ahead
    if (mode == 0) off += 96 * 4;
    p.warp_smem = (uint32_t)round_up(off, 16);
    // table metrics with a pivot table that fits shared memory: search_kernel_pqs (pivots resident per SM, entries
    // computed on the fly); everything else — SQ, DirectCosine, wide pivots, > 32 chunks — the per-warp kernel below
    PqsPlan plan;
    memset(&plan, 0, sizeof(plan));
    const bool use_pqs = mode == 0 && !p.direct_cosine && pqs_plan(idx, p.warp_smem, nq, &plan);
    const size_t smem_block = (size_t)p.warp_smem * kPqWarps;
    void (*kern)(const SearchParamsPq) = nullptr;
    int grid;
    uint32_t warps;
    if (use_pqs) {
        p.piv_stride = plan.piv_stride;
        p.piv_bytes = plan.piv_bytes;
        grid = plan.grid;
        warps = (uint32_t)plan.grid * (uint32_t)plan.warps;
    } else {
        if (smem_block > 200 * 1024) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_pq: configuration needs %zu B shared memory per CTA", smem_block);
        if (mode == 1) kern = cap <= 128 ? search_kernel_pq<4, 1> : cap <= 256 ? search_kernel_pq<8, 1> : cap <= 512 ? search_kernel_pq<16, 1> : search_kernel_pq<32, 1>;
        else kern = cap <= 128 ? search_kernel_pq<4, 0> : cap <= 256 ? search_kernel_pq<8, 0> : cap <= 512 ? search_kernel_pq<16, 0> : search_kernel_pq<32, 0>;
        DAB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_block));
        int per_sm = 0;
        DAB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kPqWarps * 32, smem_block));
        if (per_sm < 1) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_pq: kernel does not fit");
        // every resident warp owns a LUT (n_chunks x n_centers f32: 32 KB at 32 x 256) and a visited table in
        // global memory; ADC terms and probes are L2 hits only while all of them stay L2-resident
        // (the SQ kernel has no LUT: it keeps the occupancy the shared memory allows)
        if (mode == 0) per_sm = std::min(per_sm, 6);
        grid = (int)std::min<uint64_t>((uint64_t)per_sm * idx->sm_count, ((uint64_t)nq + kPqWarps - 1) / kPqWarps);
        warps = (uint32_t)grid * kPqWarps;
    }

    // visited-table capacity: the reference's estimate (scratch.rs:186-192) on the first call, then 1.15x the
    // largest visited set seen at this (or a larger) L at 87.5 % load — the estimate is ~10x what a search
    // touches, and every query clears its table; queries that still overflow are re-run below
    uint64_t slots = std::max<uint64_t>(256, (uint64_t)(1.1 * idx->max_degree * 1.3 * (double)l_search) + 1);
    if (idx->pq_hint_visited > 0 && l_search <= idx->pq_hint_l && beam <= idx->pq_hint_beam && mode == idx->pq_hint_mode &&
        !idx->hooks.test_visited_log2) {
        const uint64_t seen = (uint64_t)(((double)idx->pq_hint_visited * 1.15 + idx->max_degree) / 0.875) + 8;
        slots = std::min(slots, std::max<uint64_t>(256, seen));
    }
    if (slots > 2 * idx->n_total() + 2048) slots = 2 * idx->n_total() + 2048;
    if (idx->hooks.test_visited_log2) slots = 1ull << idx->hooks.test_visited_log2;  // tests force the overflow re-runs
    int rc;
    if ((rc = idx->s_counters.reserve(16 + (size_t)nq * 4))) return rc;
    uint32_t* d_counters = (uint32_t*)idx->s_counters.p;
    p.counters = d_counters;
    p.overflow_list = d_counters + 4;
    const size_t lut_bytes = mode == 0 && !use_pqs ? (size_t)warps * idx->pq_chunks * idx->pq_centers * 4 : 16;
    if ((rc = idx->s_out2.reserve(lut_bytes))) return rc;
    p.luts = (float*)idx->s_out2.p;
    p.n_work = nq;
    if (rerank) {
        if (!idx->vectors_ready) return fail(DAB_ERR_NOT_READY, "dab_search_batch_pq: rerank needs the full-precision vectors");
        if ((rc = idx->s_ids.reserve(((size_t)nq * cap + nq) * 4))) return rc;
        p.list_ids = (uint32_t*)idx->s_ids.p;
        p.list_counts = p.list_ids + (size_t)nq * cap;
        p.list_cap = cap;
    }
    Scratch retry;
    for (int pass = 0; pass < 6; ++pass) {
        p.n_buckets = (uint32_t)((slots + 7) / 8);
        if ((rc = idx->s_tables.reserve((size_t)warps * p.n_buckets * 32))) {
            retry.release();
            return rc;
        }
        p.tables = (uint32_t*)idx->s_tables.p;
        DAB_CUDA(cudaMemsetAsync(d_counters, 0, 16, idx->stream));
        if (use_pqs) {
            if ((rc = pqs_launch(idx, p, plan, cap))) {
                retry.release();
                return rc;
            }
        } else {
            kern<<<grid, kPqWarps * 32, smem_block, idx->stream>>>(p);
            DAB_LAUNCHED();
            DAB_CUDA(cudaGetLastError());
        }
        uint32_t h[3] = {0, 0, 0};
        DAB_CUDA(cudaMemcpyAsync(h, d_counters, 12, cudaMemcpyDeviceToHost, idx->stream));
        DAB_CUDA(cudaStreamSynchronize(idx->stream));
        if (l_search != idx->pq_hint_l || beam != idx->pq_hint_beam || mode != idx->pq_hint_mode) {
            idx->pq_hint_l = l_search;
            idx->pq_hint_beam = beam;
            idx->pq_hint_mode = mode;
            idx->pq_hint_visited = 0;
        }
        idx->pq_hint_visited = std::max(idx->pq_hint_visited, h[2]);
        if (h[1] == 0) {
            retry.release();
            if (rerank) return launch_rerank(idx, d_queries, nq, k, cap, p.list_ids, p.list_counts, d_ids, d_dists, d_counts);
            return DAB_OK;
        }
        Scratch next;
        if ((rc = next.reserve((size_t)h[1] * 4))) {
            retry.release();
            return rc;
        }
        DAB_CUDA(cudaMemcpy(next.p, d_counters + 4, (size_t)h[1] * 4, cudaMemcpyDeviceToDevice));
        retry.release();
        retry = next;
        p.query_list = (const uint32_t*)retry.p;
        p.n_work = h[1];
        slots *= 4;
    }
    retry.release();
    return fail(DAB_ERR_VISITED_OVERFLOW, "dab_search_batch_pq: visited set still overflowing after 6 passes");
}

}  // namespace dab

using namespace dab;

static int search_pq_host(dab_index* idx, const void* queries, uint32_t nq, uint32_t k, uint32_t l_search, uint32_t beam_width,
                          uint32_t* out_ids, float* out_dists, uint32_t* out_counts, uint32_t* out_cmps, uint32_t* out_hops, bool rerank,
                          int mode = 0) {
    if (!idx) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_pq: idx is NULL");
    if (nq == 0) return DAB_OK;
    if (!queries || !out_ids || !out_dists) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_pq: NULL argument");
    if (k == 0) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_pq: k must be > 0");
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
    if ((rc = run_search_pq(idx, idx->s_queries.p, nq, k, l_search, beam_width, d_ids, d_dists, d_counts, d_cmps, d_hops, rerank, mode))) return rc;
    DAB_CUDA(cudaMemcpyAsync(out_ids, d_ids, rbytes, cudaMemcpyDeviceToHost, idx->stream));
    DAB_CUDA(cudaMemcpyAsync(out_dists, d_dists, rbytes, cudaMemcpyDeviceToHost, idx->stream));
    if (out_counts) DAB_CUDA(cudaMemcpyAsync(out_counts, d_counts, (size_t)nq * 4, cudaMemcpyDeviceToHost, idx->stream));
    if (out_cmps) DAB_CUDA(cudaMemcpyAsync(out_cmps, d_cmps, (size_t)nq * 4, cudaMemcpyDeviceToHost, idx->stream));
    if (out_hops) DAB_CUDA(cudaMemcpyAsync(out_hops, d_hops, (size_t)nq * 4, cudaMemcpyDeviceToHost, idx->stream));
    DAB_CUDA(cudaStreamSynchronize(idx->stream));
    return DAB_OK;
}

extern "C" {

int dab_search_batch_pq(dab_index* idx, const void* queries, uint32_t nq, uint32_t k, uint32_t l_search, uint32_t beam_width,
                        uint32_t* out_ids, float* out_dists, uint32_t* out_counts, uint32_t* out_cmps, uint32_t* out_hops) {
    return search_pq_host(idx, queries, nq, k, l_search, beam_width, out_ids, out_dists, out_counts, out_cmps, out_hops, false);
}

int dab_search_batch_pq_rerank(dab_index* idx, const void* queries, uint32_t nq, uint32_t k, uint32_t l_search, uint32_t beam_width,
                               uint32_t* out_ids, float* out_dists, uint32_t* out_counts, uint32_t* out_cmps, uint32_t* out_hops) {
    return search_pq_host(idx, queries, nq, k, l_search, beam_width, out_ids, out_dists, out_counts, out_cmps, out_hops, true);
}

int dab_search_batch_pq_device(dab_index* idx, const void* d_queries, uint32_t nq, uint32_t k, uint32_t l_search, uint32_t beam_width,
                               int rerank, uint32_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts, uint32_t* d_out_cmps,
                               uint32_t* d_out_hops) {
    if (!idx) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_pq_device: idx is NULL");
    if (nq == 0) return DAB_OK;
    if (!d_queries || !d_out_ids || !d_out_dists) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_pq_device: NULL argument");
    DAB_CUDA(cudaSetDevice(idx->device));
    return run_search_pq(idx, d_queries, nq, k, l_search, beam_width, d_out_ids, d_out_dists, d_out_counts, d_out_cmps, d_out_hops, rerank != 0);
}

int dab_search_batch_sq(dab_index* idx, const void* queries, uint32_t nq, uint32_t k, uint32_t l_search, uint32_t beam_width,
                        int rerank, uint32_t* out_ids, float* out_dists, uint32_t* out_counts, uint32_t* out_cmps, uint32_t* out_hops) {
    return search_pq_host(idx, queries, nq, k, l_search, beam_width, out_ids, out_dists, out_counts, out_cmps, out_hops, rerank != 0, 1);
}

int dab_search_batch_sq_device(dab_index* idx, const void* d_queries, uint32_t nq, uint32_t k, uint32_t l_search, uint32_t beam_width,
                               int rerank, uint32_t* d_out_ids, float* d_out_dists, uint32_t* d_out_counts, uint32_t* d_out_cmps,
                               uint32_t* d_out_hops) {
    if (!idx) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_sq_device: idx is NULL");
    if (nq == 0) return DAB_OK;
    if (!d_queries || !d_out_ids || !d_out_dists) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_search_batch_sq_device: NULL argument");
    DAB_CUDA(cudaSetDevice(idx->device));
    return run_search_pq(idx, d_queries, nq, k, l_search, beam_width, d_out_ids, d_out_dists, d_out_counts, d_out_cmps, d_out_hops, rerank != 0, 1);
}

}  // extern "C"
