// quant_kernels.cu — product-quantization (LUT build, ADC gather, encode) and
// scalar-quantization (compress, compensated distances) kernels.
//
// PQ ADC is a shared-memory LUT gather with coalesced code loads and *sequential chunk-order*
// f32 accumulation (fixed_chunk_pq_table.rs:82-98), so sums are bit-identical to the
// reference; no tensor cores.  LUT entries are computed in the reference's SIMD order for the
// (short) chunk length, one thread per (chunk, pivot) entry.
#include "dab_common.cuh"
#include "distance_device.cuh"
#include "quant_device.cuh"

#include <vector>

namespace dab {

// ------------------------------------------------------------------ LUT build (K6)
// lut[q][chunk][center] = SquaredL2 / InnerProduct(query chunk, pivot chunk)
// (fixed_chunk_pq_table.rs:152-187; IP entries are -dot, implementations.rs:309-314).
template <int KIND>
__global__ void __launch_bounds__(256)
pq_lut_kernel(const float* __restrict__ queries, uint32_t nq, const float* __restrict__ pivots, uint32_t n_centers,
              const uint32_t* __restrict__ offsets, uint32_t n_chunks, uint32_t dim, float* __restrict__ lut) {
    extern __shared__ float sq[];  // the query
    const uint32_t q = blockIdx.x;
    for (uint32_t e = threadIdx.x; e < dim; e += blockDim.x) sq[e] = queries[(size_t)q * dim + e];
    __syncthreads();
    const uint32_t entries = n_chunks * n_centers;
    for (uint32_t t = threadIdx.x; t < entries; t += blockDim.x) {
        const uint32_t chunk = t / n_centers, center = t % n_centers;
        const uint32_t start = offsets[chunk], stop = offsets[chunk + 1];
        float v = thread_simd_l2ip<KIND>(sq + start, pivots + (size_t)center * dim + start, (int)(stop - start));
        lut[((size_t)q * n_chunks + chunk) * n_centers + center] = KIND == KIND_IP ? -v : v;
    }
}

// ------------------------------------------------------------------ ADC gather (K7)
// One CTA per (query, tile of candidates): the query's LUT (n_chunks x n_centers f32) is staged
// in shared memory, each thread owns one candidate and adds lut[c][code[c]] in chunk order.
__global__ void __launch_bounds__(256)
pq_adc_kernel(const float* __restrict__ lut, uint32_t nq, const uint32_t* __restrict__ ids, uint32_t c,
              const uint8_t* __restrict__ codes, uint32_t n_chunks, uint32_t n_centers, uint64_t n_total,
              float* __restrict__ out, uint32_t tiles_per_q) {
    extern __shared__ float slut[];
    const uint32_t q = blockIdx.x / tiles_per_q, tile = blockIdx.x % tiles_per_q;
    const uint32_t entries = n_chunks * n_centers;
    const float4* src = reinterpret_cast<const float4*>(lut + (size_t)q * entries);
    for (uint32_t e = threadIdx.x; e < entries / 4; e += blockDim.x) reinterpret_cast<float4*>(slut)[e] = src[e];
    for (uint32_t e = (entries & ~3u) + threadIdx.x; e < entries; e += blockDim.x) slut[e] = lut[(size_t)q * entries + e];
    __syncthreads();
    const uint32_t per_tile = (c + tiles_per_q - 1) / tiles_per_q;
    const uint32_t j0 = tile * per_tile, j1 = min(c, j0 + per_tile);
    for (uint32_t j = j0 + threadIdx.x; j < j1; j += blockDim.x) {
        const uint32_t id = ids[(size_t)q * c + j];
        if (id == kNoId || id >= n_total) {
            out[(size_t)q * c + j] = __int_as_float(0x7FC00000);
            continue;
        }
        const uint8_t* code = codes + (size_t)id * n_chunks;
        float accum = 0.0f;
        uint32_t ch = 0;
        if ((n_chunks & 15u) == 0) {
            for (; ch < n_chunks; ch += 16) {
                const uint4 w = __ldg(reinterpret_cast<const uint4*>(code + ch));
                const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const uint32_t b = (ws[k >> 2] >> ((k & 3) * 8)) & 0xFFu;
                    accum = __fadd_rn(accum, slut[(ch + k) * n_centers + b]);
                }
            }
        } else {
            for (; ch < n_chunks; ++ch) accum = __fadd_rn(accum, slut[ch * n_centers + __ldg(code + ch)]);
        }
        out[(size_t)q * c + j] = accum;
    }
}

// ------------------------------------------------------------------ fused LUT build + ADC (K6 + K7)
// pq_lut_kernel + pq_adc_kernel spend their time moving tables: every query re-reads the 128 KB pivot table from L2
// to build its LUT, writes the 32 KB LUT to global memory and reads it back.  Here a persistent CTA per SM stages the
// pivots in shared memory ONCE (rows padded to an odd multiple of four floats), then per query: stage the query,
// build the LUT shared-to-shared (same entry arithmetic, quant_device.cuh pqs_term), optionally write it out
// (dab_pq_populate_lut), and sum one entry per chunk for every candidate in chunk order from 0.0.  While the LUT is
// being built the code rows of the query's candidates and the ids of the CTA's next query are on their way to L2.
struct PqFusedParams {
    const float* queries;
    uint32_t nq;
    const float* pivots;
    const uint32_t* offsets;
    uint32_t n_centers, n_chunks, dim;
    uint32_t piv_stride, piv_bytes;
    int ip;
    float* lut_out;        // [nq][n_chunks][n_centers] or NULL
    const uint32_t* ids;   // [nq][c] or NULL (LUT only)
    uint32_t c;
    const uint8_t* codes;
    uint64_t n_total;
    float* out;            // [nq][c]
    uint32_t groups;       // thread groups of the CTA, each with its own table + query (1 or 2)
    uint32_t group_floats; // floats of shared memory per group (table + query)
};

// The CTA is split into `groups` equal thread groups (1 or 2), each with its own table and query in shared memory and
// its own named barrier, so two queries are in flight per SM: one group builds while the other waits for its codes.
template <int CL>
__global__ void __launch_bounds__(512, 1) pq_fused_kernel(const PqFusedParams p) {
    extern __shared__ __align__(16) uint8_t fsm[];
    float* spiv = reinterpret_cast<float*>(fsm);
    const uint32_t entries = p.n_chunks * p.n_centers;
    const uint32_t gsize = blockDim.x / p.groups, grp = threadIdx.x / gsize, tid = threadIdx.x - grp * gsize;
    float* slut = reinterpret_cast<float*>(fsm + p.piv_bytes) + (size_t)grp * p.group_floats;
    float* sq = slut + ((entries + 3u) & ~3u);
    {
        const uint32_t total = p.n_centers * p.dim;
        for (uint32_t e = threadIdx.x; e < total; e += blockDim.x) {
            const uint32_t c = e / p.dim, d = e - c * p.dim;
            spiv[(size_t)c * p.piv_stride + d] = __ldg(p.pivots + e);
        }
    }
    __syncthreads();  // pivots staged; from here on the groups synchronise on their own barriers (ids 1, 2)
    auto group_sync = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "r"(gsize) : "memory"); };
    const bool ip = p.ip != 0;
    const uint32_t qstep = gridDim.x * p.groups;
    for (uint32_t q = blockIdx.x * p.groups + grp; q < p.nq; q += qstep) {
        group_sync();  // the previous query's table is no longer read
        for (uint32_t e = tid; e < p.dim; e += gsize) sq[e] = __ldg(p.queries + (size_t)q * p.dim + e);
        if (p.ids) {
            for (uint32_t j = tid; j < p.c; j += gsize) {
                const uint32_t id = __ldg(p.ids + (size_t)q * p.c + j);
                if (id != kNoId && id < p.n_total) prefetch_l2(p.codes + (size_t)id * p.n_chunks);
            }
            const uint32_t qn = q + qstep;  // the ids of this group's next query: one 128-byte line per thread
            for (uint32_t o = tid * 32u; qn < p.nq && o < p.c; o += gsize * 32u) prefetch_l2(p.ids + (size_t)qn * p.c + o);
        }
        group_sync();
        {   // entry t = chunk * n_centers + center, walked without a division per entry
            uint32_t chunk = tid / p.n_centers, center = tid - chunk * p.n_centers;
            const uint32_t dchunk = gsize / p.n_centers, dcenter = gsize - dchunk * p.n_centers;
            for (uint32_t t = tid; t < entries; t += gsize) {
                const float v = pqs_term<CL>(sq, spiv, p.piv_stride, p.offsets, chunk, center, ip);
                slut[t] = v;
                if (p.lut_out) p.lut_out[(size_t)q * entries + t] = v;
                chunk += dchunk;
                center += dcenter;
                if (center >= p.n_centers) {
                    center -= p.n_centers;
                    ++chunk;
                }
            }
        }
        group_sync();
        if (!p.ids) continue;
        for (uint32_t j = tid; j < p.c; j += gsize) {
            const uint32_t id = __ldg(p.ids + (size_t)q * p.c + j);
            if (id == kNoId || id >= p.n_total) {
                p.out[(size_t)q * p.c + j] = __int_as_float(0x7FC00000);
                continue;
            }
            const uint8_t* code = p.codes + (size_t)id * p.n_chunks;
            float accum = 0.0f;
            uint32_t ch = 0;
            if ((p.n_chunks & 15u) == 0) {
                for (; ch < p.n_chunks; ch += 16) {
                    const uint4 w = __ldg(reinterpret_cast<const uint4*>(code + ch));
                    const uint32_t ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                    for (int k = 0; k < 16; ++k) {
                        const uint32_t b = (ws[k >> 2] >> ((k & 3) * 8)) & 0xFFu;
                        accum = __fadd_rn(accum, slut[(ch + k) * p.n_centers + b]);
                    }
                }
            } else {
                for (; ch < p.n_chunks; ++ch) accum = __fadd_rn(accum, slut[ch * p.n_centers + __ldg(code + ch)]);
            }
            p.out[(size_t)q * p.c + j] = accum;
        }
    }
}

// DirectCosine (pq/distance/cosine.rs:16-70; direct_distance_impl,
// fixed_chunk_pq_table.rs:35-59): resumable V3 cosine (Strategy2x4) over gathered pivot
// chunks, 1 - cos.  One thread per candidate (rare path).
__global__ void __launch_bounds__(128)
pq_direct_cosine_kernel(const float* __restrict__ queries, uint32_t nq, const uint32_t* __restrict__ ids, uint32_t c,
                        const uint8_t* __restrict__ codes, const float* __restrict__ pivots,
                        const uint32_t* __restrict__ offsets, uint32_t n_chunks, uint32_t dim, uint64_t n_total,
                        float* __restrict__ out) {
    const uint64_t total = (uint64_t)nq * c;
    for (uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; t < total; t += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t q = (uint32_t)(t / c);
        const uint32_t id = ids[t];
        if (id == kNoId || id >= n_total) {
            out[t] = __int_as_float(0x7FC00000);
            continue;
        }
        const float* x = queries + (size_t)q * dim;
        const uint8_t* code = codes + (size_t)id * n_chunks;
        float nx[8], ny[8], xy[8];
#pragma unroll
        for (int l = 0; l < 8; ++l) nx[l] = ny[l] = xy[l] = 0.0f;
        for (uint32_t ch = 0; ch < n_chunks; ++ch) {
            const uint32_t start = offsets[ch], stop = offsets[ch + 1];
            const float* xc = x + start;
            const float* yc = pivots + (size_t)code[ch] * dim + start;
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
        out[t] = __fsub_rn(1.0f, cosine_finish(thread_tree8(nx), thread_tree8(ny), thread_tree8(xy)));
    }
}

// DistanceComputer (pq/distance/dynamic.rs:101-140, VTable :117-131) over two CODES:
// FixedChunkPQTable::{qq_l2_distance, qq_inner_product, qq_cosine_distance}
// (fixed_chunk_pq_table.rs:285-361) = direct_distance_impl (:35-59) with both sides gathered from
// the pivots: one Resumable accumulator across the chunks (simd.rs:1515-1547, 2240-2272,
// 3163-3199: the combined 8-lane accumulator of every chunk is added lane-wise), sum_tree at the
// end.  L2 -> value, InnerProduct -> -value, Cosine / CosineNormalized -> 1 - cos.
// kind: 0 L2, 1 IP, 2 cosine.  One thread per pair.
__global__ void __launch_bounds__(128)
pq_self_distance_kernel(const uint32_t* __restrict__ ids_a, const uint32_t* __restrict__ ids_b, uint64_t n, int kind,
                        const uint8_t* __restrict__ codes, const float* __restrict__ pivots, const uint32_t* __restrict__ offsets,
                        uint32_t n_chunks, uint32_t dim, uint64_t n_total, float* __restrict__ out) {
    for (uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; t < n; t += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t ia = ids_a[t], ib = ids_b[t];
        if (ia >= n_total || ib >= n_total) {
            out[t] = __int_as_float(0x7FC00000);
            continue;
        }
        const uint8_t* ca = codes + (size_t)ia * n_chunks;
        const uint8_t* cb = codes + (size_t)ib * n_chunks;
        float nx[8], ny[8], xy[8];
#pragma unroll
        for (int l = 0; l < 8; ++l) nx[l] = ny[l] = xy[l] = 0.0f;
        for (uint32_t ch = 0; ch < n_chunks; ++ch) {
            const uint32_t start = offsets[ch], stop = offsets[ch + 1];
            const float* xc = pivots + (size_t)ca[ch] * dim + start;
            const float* yc = pivots + (size_t)cb[ch] * dim + start;
            const int len = (int)(stop - start);
            float d[8];
            if (kind == 0) {
                thread_simd_combined<4, KIND_L2>(xc, yc, len, d);
            } else if (kind == 1) {
                thread_simd_combined<4, KIND_IP>(xc, yc, len, d);
            } else {
                float a[8], b[8];
                thread_simd_combined<2, KIND_IP>(xc, xc, len, a);
                thread_simd_combined<2, KIND_IP>(yc, yc, len, b);
                thread_simd_combined<2, KIND_IP>(xc, yc, len, d);
#pragma unroll
                for (int l = 0; l < 8; ++l) {
                    nx[l] = __fadd_rn(nx[l], a[l]);
                    ny[l] = __fadd_rn(ny[l], b[l]);
                }
            }
#pragma unroll
            for (int l = 0; l < 8; ++l) xy[l] = __fadd_rn(xy[l], d[l]);
        }
        float v;
        if (kind == 0) v = thread_tree8(xy);
        else if (kind == 1) v = -thread_tree8(xy);
        else v = __fsub_rn(1.0f, cosine_finish(thread_tree8(nx), thread_tree8(ny), thread_tree8(xy)));
        out[t] = v;
    }
}

// ------------------------------------------------------------------ encode
// BasicTable::compress_into (product/tables/basic.rs:161-194): one warp per (vector, chunk),
// lanes stride the pivots, strict `<` so the lowest pivot index among ties wins.
__global__ void __launch_bounds__(256)
pq_encode_kernel(const float* __restrict__ vectors, uint64_t n, const float* __restrict__ pivots, uint32_t n_centers,
                 const uint32_t* __restrict__ offsets, uint32_t n_chunks, uint32_t dim, uint8_t* __restrict__ out_codes,
                 unsigned long long* __restrict__ first_bad) {
    const int lane = threadIdx.x & 31;
    const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t total = n * n_chunks;
    for (uint64_t t = warp; t < total; t += nwarps) {
        const uint64_t v = t / n_chunks;
        const uint32_t chunk = (uint32_t)(t % n_chunks);
        const uint32_t start = offsets[chunk], stop = offsets[chunk + 1];
        const float* x = vectors + v * dim + start;
        float best = __int_as_float(0x7F800000);
        uint32_t best_idx = 0xFFFFFFFFu;
        for (uint32_t p = lane; p < n_centers; p += 32) {
            float d = thread_simd_l2ip<KIND_L2>(x, pivots + (size_t)p * dim + start, (int)(stop - start));
            if (d < best) {
                best = d;
                best_idx = p;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            float ob = __shfl_xor_sync(kFull, best, o);
            uint32_t oi = __shfl_xor_sync(kFull, best_idx, o);
            if (ob < best || (ob == best && oi < best_idx)) {
                best = ob;
                best_idx = oi;
            }
        }
        if (lane == 0) {
            if (isinf(best) || best_idx == 0xFFFFFFFFu) {
                atomicMin(first_bad, (unsigned long long)t);
                out_codes[t] = 0;
            } else {
                out_codes[t] = (uint8_t)best_idx;
            }
        }
    }
}

// ------------------------------------------------------------------ scalar quantization
// ScalarQuantizer::compress (+ compensation): scalar/quantizer.rs:190-239, 407-430.  The
// compensation dot product is a sequential FMA chain over the dimensions, so one thread owns
// one vector.
__global__ void __launch_bounds__(128)
sq_compress_kernel(const float* __restrict__ shift, float scale, uint32_t dim, int nbits,
                   const float* __restrict__ vectors, uint64_t n, uint8_t* __restrict__ codes, float* __restrict__ comp) {
    const float maxv = (float)((1u << nbits) - 1u);
    const float inverse_scale = __fdiv_rn(maxv, scale);
    const float inverse_bit_scale = __fdiv_rn(1.0f, maxv);
    for (uint64_t v = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; v < n; v += (uint64_t)gridDim.x * blockDim.x) {
        float dot = 0.0f;
        for (uint32_t i = 0; i < dim; ++i) {
            const float f = vectors[v * dim + i], s = shift[i];
            float t = __fmul_rn(__fsub_rn(f, s), inverse_scale);
            float code = t != t ? t : (t < 0.0f ? 0.0f : (t > maxv ? maxv : t));  // f32::clamp keeps NaN
            code = roundf(code);                                                  // half away from zero
            dot = __fmaf_rn(code, s, dot);
            codes[v * dim + i] = code != code ? (uint8_t)0 : (uint8_t)code;
        }
        comp[v] = __fmul_rn(__fmul_rn(scale, inverse_bit_scale), dot);
    }
}

// Compensated{SquaredL2, IP, CosineNormalized}: scalar/vectors.rs:206-237, 310-376, 380-460.
// Integer cores exact (bits/distances.rs:397, 979); one warp per pair.
__global__ void __launch_bounds__(256)
sq_distance_kernel(int metric, int nbits, float scale_squared, float shift_square_norm, uint32_t dim,
                   const uint8_t* __restrict__ x, const float* __restrict__ comp_x, const uint8_t* __restrict__ y,
                   const float* __restrict__ comp_y, uint64_t n, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const float ibs = __fdiv_rn(1.0f, (float)((1u << nbits) - 1u));
    const float bit_scale = __fmul_rn(ibs, ibs);
    for (uint64_t i = warp; i < n; i += nwarps) {
        const uint8_t* a = x + i * dim;
        const uint8_t* b = y + i * dim;
        uint32_t l2 = 0, ip = 0;
        for (uint32_t e = lane; e < dim; e += 32) {
            int av = a[e], bv = b[e];
            l2 += (uint32_t)((av - bv) * (av - bv));
            ip += (uint32_t)(av * bv);
        }
        l2 = __reduce_add_sync(kFull, l2);
        ip = __reduce_add_sync(kFull, ip);
        if (lane == 0) {
            float r;
            if (metric == DAB_L2) {
                r = __fmul_rn(__fmul_rn(bit_scale, scale_squared), (float)l2);
            } else if (metric == DAB_INNER_PRODUCT) {
                float m = __fadd_rn(__fmaf_rn(__fmul_rn(bit_scale, scale_squared), (float)ip, shift_square_norm),
                                    __fadd_rn(comp_y[i], comp_x[i]));
                r = -m;
            } else {
                float l = __fmul_rn(__fmul_rn(bit_scale, scale_squared), (float)l2);
                float mathematical = __fsub_rn(1.0f, __fdiv_rn(l, 2.0f));
                r = __fsub_rn(1.0f, mathematical);
            }
            out[i] = r;
        }
    }
}

static int require_pq(const dab_index* idx, const char* who) {
    if (!idx) return fail(DAB_ERR_INVALID_ARGUMENT, "%s: idx is NULL", who);
    if (!idx->d_pivots) return fail(DAB_ERR_NOT_READY, "%s: dab_upload_pq has not been called", who);
    return DAB_OK;
}

// true when the pivot table + one table + one query fit the shared memory of a CTA: launches pq_fused_kernel.
// d_lut / d_ids may be NULL (ADC only / LUT only).
static bool fused_fits(const dab_index* idx, uint32_t* stride_out, size_t* piv_bytes_out, size_t* smem_out, uint32_t* groups_out = nullptr,
                       uint32_t* group_floats_out = nullptr) {
    uint32_t stride = (uint32_t)round_up(idx->dim, 4);
    if ((stride & 7u) == 0) stride += 4;
    const size_t piv_bytes = (size_t)idx->pq_centers * stride * 4;
    const size_t entries = (size_t)idx->pq_chunks * idx->pq_centers;
    const size_t group_floats = round_up(entries, 4) + round_up(idx->dim, 4);  // one table + one query
    const uint32_t groups = piv_bytes + 2 * group_floats * 4 <= 227 * 1024 ? 2 : 1;  // two queries in flight per SM when both tables fit
    *stride_out = stride;
    *piv_bytes_out = piv_bytes;
    *smem_out = piv_bytes + groups * group_floats * 4;
    if (groups_out) *groups_out = groups;
    if (group_floats_out) *group_floats_out = (uint32_t)group_floats;
    return piv_bytes + group_floats * 4 <= 227 * 1024 && !idx->hooks.pq_global_lut;
}

static int launch_fused(const dab_index* idx, const float* d_queries, uint32_t nq, int lut_metric, float* d_lut, const uint32_t* d_ids,
                        uint32_t c, float* d_out) {
    PqFusedParams p;
    memset(&p, 0, sizeof(p));
    uint32_t stride;
    size_t piv_bytes, smem;
    fused_fits(idx, &stride, &piv_bytes, &smem, &p.groups, &p.group_floats);
    p.queries = d_queries;
    p.nq = nq;
    p.pivots = idx->d_pivots;
    p.offsets = idx->d_offsets;
    p.n_centers = idx->pq_centers;
    p.n_chunks = idx->pq_chunks;
    p.dim = idx->dim;
    p.piv_stride = stride;
    p.piv_bytes = (uint32_t)piv_bytes;
    p.ip = lut_metric == DAB_INNER_PRODUCT ? 1 : 0;
    p.lut_out = d_lut;
    p.ids = d_ids;
    p.c = c;
    p.codes = idx->d_codes;
    p.n_total = idx->n_total();
    p.out = d_out;
    void (*kern)(const PqFusedParams) = idx->pq_uniform_len == 4 ? pq_fused_kernel<4> : idx->pq_uniform_len == 8 ? pq_fused_kernel<8> : pq_fused_kernel<0>;
    DAB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int grid = (int)std::min<uint32_t>((nq + p.groups - 1) / p.groups, (uint32_t)idx->sm_count);
    kern<<<grid, 512, smem, idx->stream>>>(p);
    DAB_LAUNCHED();
    DAB_CUDA(cudaGetLastError());
    return DAB_OK;
}

static int launch_lut(const dab_index* idx, const float* d_queries, uint32_t nq, int metric, float* d_lut) {
    {
        uint32_t stride;
        size_t piv_bytes, smem;
        if (fused_fits(idx, &stride, &piv_bytes, &smem)) return launch_fused(idx, d_queries, nq, metric, d_lut, nullptr, 0, nullptr);
    }
    const size_t smem = (size_t)idx->dim * 4;
    if (metric == DAB_INNER_PRODUCT)
        pq_lut_kernel<KIND_IP><<<nq, 256, smem, idx->stream>>>(d_queries, nq, idx->d_pivots, idx->pq_centers, idx->d_offsets,
                                                               idx->pq_chunks, idx->dim, d_lut);
    else
        pq_lut_kernel<KIND_L2><<<nq, 256, smem, idx->stream>>>(d_queries, nq, idx->d_pivots, idx->pq_centers, idx->d_offsets,
                                                               idx->pq_chunks, idx->dim, d_lut);
    DAB_LAUNCHED();
    DAB_CUDA(cudaGetLastError());
    return DAB_OK;
}

}  // namespace dab

using namespace dab;

namespace dab {
// pq_encode_kernel over n f32 vectors already on the device; codes written to d_codes_out (device).
// Used by dab_pq_encode_all (pq_train.cu).  Rows that are infinitely far from every centre
// (inf / NaN input) are reported like BasicTable::compress_into does.
int pq_encode_device(dab_index* idx, const float* d_vectors, uint64_t n, uint8_t* d_codes_out) {
    int rc;
    if ((rc = idx->s_counters.reserve(16))) return rc;
    unsigned long long* d_bad = (unsigned long long*)idx->s_counters.p;
    DAB_CUDA(cudaMemsetAsync(d_bad, 0xFF, 8, idx->stream));
    const uint64_t warps = n * idx->pq_chunks;
    const int grid = (int)std::min<uint64_t>((warps + 7) / 8, (uint64_t)idx->sm_count * 8);
    pq_encode_kernel<<<grid, 256, 0, idx->stream>>>(d_vectors, n, idx->d_pivots, idx->pq_centers, idx->d_offsets, idx->pq_chunks, idx->dim,
                                                    d_codes_out, d_bad);
    DAB_LAUNCHED();
    DAB_CUDA(cudaGetLastError());
    unsigned long long bad = 0;
    DAB_CUDA(cudaMemcpyAsync(&bad, d_bad, 8, cudaMemcpyDeviceToHost, idx->stream));
    DAB_CUDA(cudaStreamSynchronize(idx->stream));
    if (bad != ~0ull)
        return fail(DAB_ERR_INVALID_ARGUMENT, "pq encode: vector %llu chunk %llu is infinitely far from every center (inf/NaN input)",
                    bad / idx->pq_chunks, bad % idx->pq_chunks);
    return DAB_OK;
}
}  // namespace dab

extern "C" {

int dab_pq_populate_lut(dab_index* idx, const float* queries, uint32_t nq, int metric, float* out_lut) {
    int rc = require_pq(idx, "dab_pq_populate_lut");
    if (rc) return rc;
    if (nq == 0) return DAB_OK;
    if (!queries || !out_lut) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_pq_populate_lut: NULL argument");
    if (metric != DAB_L2 && metric != DAB_INNER_PRODUCT && metric != DAB_COSINE_NORMALIZED)
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_pq_populate_lut: tables exist for L2 / InnerProduct only (Cosine is direct)");
    DAB_CUDA(cudaSetDevice(idx->device));
    const size_t qbytes = (size_t)nq * idx->dim * 4;
    const size_t lbytes = (size_t)nq * idx->pq_chunks * idx->pq_centers * 4;
    if ((rc = idx->s_queries.reserve(qbytes))) return rc;
    if ((rc = idx->s_out2.reserve(lbytes))) return rc;
    DAB_CUDA(cudaMemcpyAsync(idx->s_queries.p, queries, qbytes, cudaMemcpyHostToDevice, idx->stream));
    if ((rc = launch_lut(idx, (const float*)idx->s_queries.p, nq, metric, (float*)idx->s_out2.p))) return rc;
    DAB_CUDA(cudaMemcpyAsync(out_lut, idx->s_out2.p, lbytes, cudaMemcpyDeviceToHost, idx->stream));
    DAB_CUDA(cudaStreamSynchronize(idx->stream));
    return DAB_OK;
}

int dab_pq_distances(dab_index* idx, const float* queries, uint32_t nq, const uint32_t* ids, uint32_t c, float* out) {
    int rc = require_pq(idx, "dab_pq_distances");
    if (rc) return rc;
    if (nq == 0 || c == 0) return DAB_OK;
    if (!queries || !ids || !out) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_pq_distances: NULL argument");
    DAB_CUDA(cudaSetDevice(idx->device));
    const size_t qbytes = (size_t)nq * idx->dim * 4;
    const size_t ibytes = (size_t)nq * c * 4;
    const size_t entries = (size_t)idx->pq_chunks * idx->pq_centers;
    if ((rc = idx->s_queries.reserve(qbytes))) return rc;
    if ((rc = idx->s_ids.reserve(ibytes))) return rc;
    if ((rc = idx->s_out.reserve(ibytes))) return rc;
    DAB_CUDA(cudaMemcpyAsync(idx->s_queries.p, queries, qbytes, cudaMemcpyHostToDevice, idx->stream));
    DAB_CUDA(cudaMemcpyAsync(idx->s_ids.p, ids, ibytes, cudaMemcpyHostToDevice, idx->stream));
    if (idx->metric == DAB_COSINE) {
        // QueryComputer::Cosine -> DirectCosine (pq/distance/dynamic.rs:83)
        const uint64_t total = (uint64_t)nq * c;
        int grid = (int)std::min<uint64_t>((total + 127) / 128, (uint64_t)idx->sm_count * 16);
        pq_direct_cosine_kernel<<<grid, 128, 0, idx->stream>>>((const float*)idx->s_queries.p, nq, (const uint32_t*)idx->s_ids.p, c,
                                                               idx->d_codes, idx->d_pivots, idx->d_offsets, idx->pq_chunks,
                                                               idx->dim, idx->n_total(), (float*)idx->s_out.p);
        DAB_LAUNCHED();
        DAB_CUDA(cudaGetLastError());
    } else {
        // L2 and CosineNormalized -> TableL2, InnerProduct -> TableIP (dynamic.rs:80-85)
        const int lut_metric = idx->metric == DAB_INNER_PRODUCT ? DAB_INNER_PRODUCT : DAB_L2;
        uint32_t stride;
        size_t piv_bytes, fsmem;
        if (fused_fits(idx, &stride, &piv_bytes, &fsmem)) {
            // pivots resident in shared memory, LUT built and consumed there: no table ever leaves the SM
            if ((rc = launch_fused(idx, (const float*)idx->s_queries.p, nq, lut_metric, nullptr, (const uint32_t*)idx->s_ids.p, c,
                                   (float*)idx->s_out.p)))
                return rc;
            DAB_CUDA(cudaMemcpyAsync(out, idx->s_out.p, ibytes, cudaMemcpyDeviceToHost, idx->stream));
            DAB_CUDA(cudaStreamSynchronize(idx->stream));
            return DAB_OK;
        }
        if ((rc = idx->s_out2.reserve((size_t)nq * entries * 4))) return rc;
        if ((rc = launch_lut(idx, (const float*)idx->s_queries.p, nq, lut_metric, (float*)idx->s_out2.p))) return rc;
        const size_t smem = entries * 4;
        if (smem > 200 * 1024) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_pq_distances: LUT of %zu B does not fit shared memory", smem);
        DAB_CUDA(cudaFuncSetAttribute(pq_adc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        // enough CTAs per query to fill the machine, at least 256 candidates per CTA
        uint32_t tiles = std::max<uint32_t>(1, std::min<uint32_t>((c + 255) / 256, (uint32_t)((idx->sm_count * 4 + nq - 1) / nq)));
        pq_adc_kernel<<<nq * tiles, 256, smem, idx->stream>>>((const float*)idx->s_out2.p, nq, (const uint32_t*)idx->s_ids.p, c,
                                                              idx->d_codes, idx->pq_chunks, idx->pq_centers, idx->n_total(),
                                                              (float*)idx->s_out.p, tiles);
        DAB_LAUNCHED();
        DAB_CUDA(cudaGetLastError());
    }
    DAB_CUDA(cudaMemcpyAsync(out, idx->s_out.p, ibytes, cudaMemcpyDeviceToHost, idx->stream));
    DAB_CUDA(cudaStreamSynchronize(idx->stream));
    return DAB_OK;
}

int dab_pq_encode(dab_index* idx, const float* vectors, uint64_t n, uint8_t* out_codes) {
    int rc = require_pq(idx, "dab_pq_encode");
    if (rc) return rc;
    if (n == 0) return DAB_OK;
    if (!vectors || !out_codes) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_pq_encode: NULL argument");
    DAB_CUDA(cudaSetDevice(idx->device));
    const size_t vbytes = n * idx->dim * 4, cbytes = n * idx->pq_chunks;
    if ((rc = idx->s_queries.reserve(vbytes))) return rc;
    if ((rc = idx->s_out.reserve(cbytes + 16))) return rc;
    unsigned long long* d_bad = (unsigned long long*)idx->s_out.p;
    uint8_t* d_codes = (uint8_t*)idx->s_out.p + 16;
    DAB_CUDA(cudaMemcpyAsync(idx->s_queries.p, vectors, vbytes, cudaMemcpyHostToDevice, idx->stream));
    DAB_CUDA(cudaMemsetAsync(d_bad, 0xFF, 8, idx->stream));
    const uint64_t warps = n * idx->pq_chunks;
    int grid = (int)std::min<uint64_t>((warps + 7) / 8, (uint64_t)idx->sm_count * 8);
    pq_encode_kernel<<<grid, 256, 0, idx->stream>>>((const float*)idx->s_queries.p, n, idx->d_pivots, idx->pq_centers,
                                                    idx->d_offsets, idx->pq_chunks, idx->dim, d_codes, d_bad);
    DAB_LAUNCHED();
    DAB_CUDA(cudaGetLastError());
    unsigned long long bad = 0;
    DAB_CUDA(cudaMemcpyAsync(&bad, d_bad, 8, cudaMemcpyDeviceToHost, idx->stream));
    DAB_CUDA(cudaMemcpyAsync(out_codes, d_codes, cbytes, cudaMemcpyDeviceToHost, idx->stream));
    DAB_CUDA(cudaStreamSynchronize(idx->stream));
    if (bad != ~0ull)
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_pq_encode: vector %llu chunk %llu is infinitely far from every center (inf/NaN input)",
                    bad / idx->pq_chunks, bad % idx->pq_chunks);
    return DAB_OK;
}

int dab_pq_self_distances(dab_index* idx, const uint32_t* ids_a, const uint32_t* ids_b, uint64_t n, float* out) {
    int rc = require_pq(idx, "dab_pq_self_distances");
    if (rc) return rc;
    if (!idx->pq_codes_ready) return fail(DAB_ERR_NOT_READY, "dab_pq_self_distances: no PQ codes (dab_upload_pq with codes, or dab_pq_encode_all)");
    if (n == 0) return DAB_OK;
    if (!ids_a || !ids_b || !out) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_pq_self_distances: NULL argument");
    DAB_CUDA(cudaSetDevice(idx->device));
    if ((rc = idx->s_ids.reserve(n * 8))) return rc;
    if ((rc = idx->s_out.reserve(n * 4))) return rc;
    uint32_t* d_a = (uint32_t*)idx->s_ids.p;
    uint32_t* d_b = d_a + n;
    DAB_CUDA(cudaMemcpyAsync(d_a, ids_a, n * 4, cudaMemcpyHostToDevice, idx->stream));
    DAB_CUDA(cudaMemcpyAsync(d_b, ids_b, n * 4, cudaMemcpyHostToDevice, idx->stream));
    const int kind = idx->metric == DAB_L2 ? 0 : idx->metric == DAB_INNER_PRODUCT ? 1 : 2;  // VTable, dynamic.rs:117-131
    const int grid = (int)std::min<uint64_t>((n + 127) / 128, (uint64_t)idx->sm_count * 16);
    pq_self_distance_kernel<<<grid, 128, 0, idx->stream>>>(d_a, d_b, n, kind, idx->d_codes, idx->d_pivots, idx->d_offsets, idx->pq_chunks, idx->dim,
                                                          idx->n_total(), (float*)idx->s_out.p);
    DAB_LAUNCHED();
    DAB_CUDA(cudaGetLastError());
    DAB_CUDA(cudaMemcpyAsync(out, idx->s_out.p, n * 4, cudaMemcpyDeviceToHost, idx->stream));
    DAB_CUDA(cudaStreamSynchronize(idx->stream));
    return DAB_OK;
}

int dab_sq_compress(int device, const float* shift, float scale, uint32_t dim, int nbits, const float* vectors,
                    uint64_t n, uint8_t* out_codes, float* out_comp) {
    if (nbits != 1 && nbits != 2 && nbits != 4 && nbits != 8)
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_sq_compress: nbits must be 1, 2, 4 or 8");
    if (n == 0) return DAB_OK;
    if (!shift || !vectors || !out_codes || !out_comp || dim == 0) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_sq_compress: NULL argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(DAB_ERR_NO_DEVICE, "dab_sq_compress: no CUDA device visible");
    DAB_CUDA(cudaSetDevice(device));
    float *d_shift = nullptr, *d_vec = nullptr, *d_comp = nullptr;
    uint8_t* d_codes = nullptr;
    cudaError_t e = cudaMalloc(&d_shift, (size_t)dim * 4);
    if (e == cudaSuccess) e = cudaMalloc(&d_vec, n * dim * 4);
    if (e == cudaSuccess) e = cudaMalloc(&d_comp, n * 4);
    if (e == cudaSuccess) e = cudaMalloc(&d_codes, n * dim);
    if (e == cudaSuccess) e = cudaMemcpy(d_shift, shift, (size_t)dim * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d_vec, vectors, n * dim * 4, cudaMemcpyHostToDevice);
    int rc = DAB_OK;
    if (e == cudaSuccess) {
        int grid = (int)std::min<uint64_t>((n + 127) / 128, 148ull * 16);
        sq_compress_kernel<<<grid, 128>>>(d_shift, scale, dim, nbits, d_vec, n, d_codes, d_comp);
        DAB_LAUNCHED();
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(out_codes, d_codes, n * dim, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(out_comp, d_comp, n * 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) rc = fail(DAB_ERR_CUDA, "dab_sq_compress: %s", cudaGetErrorString(e));
    cudaFree(d_shift);
    cudaFree(d_vec);
    cudaFree(d_comp);
    cudaFree(d_codes);
    return rc;
}

int dab_sq_distances(int device, int metric, int nbits, float scale_squared, float shift_square_norm, uint32_t dim,
                     const uint8_t* x, const float* comp_x, const uint8_t* y, const float* comp_y, uint64_t n, float* out) {
    if (nbits != 1 && nbits != 2 && nbits != 4 && nbits != 8)
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_sq_distances: nbits must be 1, 2, 4 or 8");
    if (metric != DAB_L2 && metric != DAB_INNER_PRODUCT && metric != DAB_COSINE_NORMALIZED)
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_sq_distances: metric must be L2, InnerProduct or CosineNormalized");
    if (n == 0) return DAB_OK;
    if (!x || !y || !comp_x || !comp_y || !out || dim == 0) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_sq_distances: NULL argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(DAB_ERR_NO_DEVICE, "dab_sq_distances: no CUDA device visible");
    DAB_CUDA(cudaSetDevice(device));
    uint8_t *dx = nullptr, *dy = nullptr;
    float *dcx = nullptr, *dcy = nullptr, *dout = nullptr;
    cudaError_t e = cudaMalloc(&dx, n * dim);
    if (e == cudaSuccess) e = cudaMalloc(&dy, n * dim);
    if (e == cudaSuccess) e = cudaMalloc(&dcx, n * 4);
    if (e == cudaSuccess) e = cudaMalloc(&dcy, n * 4);
    if (e == cudaSuccess) e = cudaMalloc(&dout, n * 4);
    if (e == cudaSuccess) e = cudaMemcpy(dx, x, n * dim, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(dy, y, n * dim, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(dcx, comp_x, n * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(dcy, comp_y, n * 4, cudaMemcpyHostToDevice);
    int rc = DAB_OK;
    if (e == cudaSuccess) {
        int grid = (int)std::min<uint64_t>((n + 7) / 8, 148ull * 8);
        sq_distance_kernel<<<grid, 256>>>(metric, nbits, scale_squared, shift_square_norm, dim, dx, dcx, dy, dcy, n, dout);
        DAB_LAUNCHED();
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(out, dout, n * 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) rc = fail(DAB_ERR_CUDA, "dab_sq_distances: %s", cudaGetErrorString(e));
    cudaFree(dx);
    cudaFree(dy);
    cudaFree(dcx);
    cudaFree(dcy);
    cudaFree(dout);
    return rc;
}

}  // extern "C"
