// search_smem.cuh — device helpers shared by the search kernels that keep the visited set in
// shared memory (search_kernel_v3.cu) and by the rerank kernel (search_kernel_pq.cu): the tag tables
// and the wide-load row-gather distance loops.
#pragma once

#include "distance_device.cuh"
#include "search_common.cuh"

namespace dab {
namespace {

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- shared-memory visited set: 16 tags of 16 bits per 32-byte bucket -----------------------
// Entries fill a bucket from slot 0 upwards and are never removed, so an id that is absent
// from its home bucket while that bucket has a free slot is new; an id displaced to the d-th
// following bucket (d <= 2) carries d in its top two bits.  0xFFFF marks an empty slot.
__device__ __forceinline__ void load_bucket_smem(const uint32_t* bp, uint32_t (&s)[8]) {
    const uint4 lo = reinterpret_cast<const uint4*>(bp)[0];
    const uint4 hi = reinterpret_cast<const uint4*>(bp)[1];
    s[0] = lo.x, s[1] = lo.y, s[2] = lo.z, s[3] = lo.w, s[4] = hi.x, s[5] = hi.y, s[6] = hi.z, s[7] = hi.w;
}

// true when the id was newly inserted (HashSet::insert); `ovf` is raised when the home bucket
// and the two after it are full
__device__ __forceinline__ bool smem16_insert(uint32_t* table, uint32_t n_buckets, uint32_t b, uint32_t tag, bool& ovf) {
    uint32_t d = 0;
    for (;;) {
        uint32_t* bp = table + (size_t)b * 8;
        uint32_t s[8];
        load_bucket_smem(bp, s);
        const uint32_t want = (d << 14) | tag, want2 = want * 0x10001u;
        // "some 16-bit half of x is zero" <=> ((x - 0x00010001) & ~x & 0x80008000) != 0
        uint32_t hit = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const uint32_t x = s[k] ^ want2;
            hit |= (x - 0x00010001u) & ~x & 0x80008000u;
        }
        if (hit) return false;
        // first free slot: slots fill in order, so it is the number of occupied halves
        int ew = -1;
        uint32_t old = 0;
#pragma unroll
        for (int k = 7; k >= 0; --k) {
            if ((s[k] >> 16) == 0xFFFFu) {
                ew = k;
                old = s[k];
            }
        }
        if (ew >= 0) {
            const uint32_t neu = (old & 0xFFFFu) == 0xFFFFu ? (0xFFFF0000u | want) : ((old & 0xFFFFu) | (want << 16));
            if (atomicCAS(bp + ew, old, neu) == old) return true;
            continue;  // another lane of this warp changed the word: look at the bucket again
        }
        if (++d > 2) {
            ovf = true;
            return false;
        }
        b = b + 1 == n_buckets ? 0 : b + 1;
    }
}

// Packed f32x2 arithmetic (FADD2 / FFMA2): each half is an IEEE round-to-nearest operation.
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

__device__ __forceinline__ uint4 ldg16(const uint8_t* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }

// All candidate rows of a hop are requested from HBM at once with one bulk L2 prefetch per row
// (no registers, no shared memory); the register passes below then overlap with the fills and
// find all but the first rows in L2.
__device__ __forceinline__ void prefetch_rows(const uint8_t* __restrict__ vectors, size_t row_stride, const uint32_t* __restrict__ cid,
                                              uint32_t n, uint32_t row_bytes16, int lane) {
    for (uint32_t j = lane; j < n; j += 32) {
        const uint8_t* src = vectors + (size_t)cid[j] * row_stride;
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(row_bytes16) : "memory");
    }
}


// ---- float rows: distances of candidates cid[0..n) into cd[0..n) ----------------------------
// Lane mapping of frontier_wide_kernel (distance_kernels.cu): a 16-byte load carries EPL
// elements of one 8-element SIMD block; block k belongs to accumulator k mod 4, so the lane
// with (a, h) = (accumulator, half of the block) loads blocks a, a+4, a+8, ... and runs the FMA
// chains of its EPL slots itself.  LPR lanes cover a row, a pass covers ROWS rows, P passes of U
// loads each are in flight together.  Association as distance_device.cuh: (s0+s1)+(s2+s3),
// zero-filled remainder on the combined vector, sum_tree.
template <typename TD, int KIND, int POST, int P, int U>
__device__ __forceinline__ void wide_distances(const float* __restrict__ q, const uint8_t* __restrict__ vectors, size_t row_stride,
                                               const uint32_t* __restrict__ cid, uint32_t n, float* __restrict__ cd, int dim, int lane) {
    constexpr int EPL = 16 / (int)sizeof(TD), LPR = 32 / EPL, ROWS = EPL, HALVES = 8 / EPL;
    const int team = lane / LPR, tl = lane % LPR;
    const int a = tl / HALVES, h = tl % HALVES;
    const int nb8 = dim >> 3, full8 = dim & ~7, rem = dim & 7;
    const int nm = (nb8 + 3) >> 2;  // 16-byte loads per lane per row (the last may be predicated off)
    if (n > P * ROWS) prefetch_rows(vectors, row_stride, cid, n, (uint32_t)((dim * (int)sizeof(TD) + 15) & ~15), lane);
    for (uint32_t j0 = 0; j0 < n; j0 += P * ROWS) {
        const uint8_t* row[P];
        bool act[P];
#pragma unroll
        for (int pp = 0; pp < P; ++pp) {
            act[pp] = j0 + pp * ROWS < n;  // warp-uniform
            const uint32_t jj = min(j0 + pp * ROWS + team, n - 1);
            row[pp] = vectors + (size_t)cid[jj] * row_stride + 16 * tl;
        }
        uint64_t acc2[P][EPL / 2];
#pragma unroll
        for (int pp = 0; pp < P; ++pp)
#pragma unroll
            for (int i = 0; i < EPL / 2; ++i) acc2[pp][i] = 0ull;
        for (int m0 = 0; m0 < nm; m0 += U) {
            uint4 v[P][U];
#pragma unroll
            for (int pp = 0; pp < P; ++pp) {
                if (act[pp]) {
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        if (a + 4 * (m0 + u) < nb8) v[pp][u] = ldg16(row[pp] + (size_t)(m0 + u) * (LPR * 16));
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (a + 4 * (m0 + u) < nb8) {
                    const float* qx = q + ((m0 + u) * (LPR * 16) + 16 * tl) / (int)sizeof(TD);
                    float4 x[EPL / 4];
#pragma unroll
                    for (int i = 0; i < EPL / 4; ++i) x[i] = reinterpret_cast<const float4*>(qx)[i];
#pragma unroll
                    for (int pp = 0; pp < P; ++pp) {
                        if (act[pp]) {
                            if constexpr (sizeof(TD) == 2) {
                                const __half2* hp = reinterpret_cast<const __half2*>(&v[pp][u]);
                                const float2 f0 = __half22float2(hp[0]), f1 = __half22float2(hp[1]);
                                const float2 f2 = __half22float2(hp[2]), f3 = __half22float2(hp[3]);
                                acc2[pp][0] = step2<KIND>(acc2[pp][0], pack2(x[0].x, x[0].y), pack2(f0.x, f0.y));
                                acc2[pp][1] = step2<KIND>(acc2[pp][1], pack2(x[0].z, x[0].w), pack2(f1.x, f1.y));
                                acc2[pp][2] = step2<KIND>(acc2[pp][2], pack2(x[1].x, x[1].y), pack2(f2.x, f2.y));
                                acc2[pp][3] = step2<KIND>(acc2[pp][3], pack2(x[1].z, x[1].w), pack2(f3.x, f3.y));
                            } else {
                                const uint4 w = v[pp][u];
                                acc2[pp][0] = step2<KIND>(acc2[pp][0], pack2(x[0].x, x[0].y),
                                                          pack2(__uint_as_float(w.x), __uint_as_float(w.y)));
                                acc2[pp][1] = step2<KIND>(acc2[pp][1], pack2(x[0].z, x[0].w),
                                                          pack2(__uint_as_float(w.z), __uint_as_float(w.w)));
                            }
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int pp = 0; pp < P; ++pp) {
            if (!act[pp]) continue;
            float acc[EPL];
#pragma unroll
            for (int i = 0; i < EPL / 2; ++i) unpack2(acc2[pp][i], acc[2 * i], acc[2 * i + 1]);
            // (s0 + s1) + (s2 + s3), slot-wise
#pragma unroll
            for (int i = 0; i < EPL; ++i) {
                acc[i] = __fadd_rn(acc[i], __shfl_xor_sync(kFull, acc[i], HALVES));
                acc[i] = __fadd_rn(acc[i], __shfl_xor_sync(kFull, acc[i], 2 * HALVES));
            }
            if (rem) {  // zero-filled tail on the combined vector (simd.rs:733-744)
                const TD* tail = reinterpret_cast<const TD*>(row[pp] - 16 * tl) + full8;
#pragma unroll
                for (int i = 0; i < EPL; ++i) {
                    const int l = EPL * h + i;
                    const float x = l < rem ? q[full8 + l] : 0.0f;
                    const float yv = l < rem ? ldg_elem(tail + l) : 0.0f;
                    if (KIND == KIND_L2) {
                        const float dd = __fsub_rn(x, yv);
                        acc[i] = __fmaf_rn(dd, dd, acc[i]);
                    } else {
                        acc[i] = __fmaf_rn(x, yv, acc[i]);
                    }
                }
            }
            float r;
            if constexpr (HALVES == 1) {
                r = __fadd_rn(__fadd_rn(__fadd_rn(acc[0], acc[4]), __fadd_rn(acc[2], acc[6])),
                              __fadd_rn(__fadd_rn(acc[1], acc[5]), __fadd_rn(acc[3], acc[7])));
            } else {
                float ts[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) ts[i] = __fadd_rn(acc[i], __shfl_xor_sync(kFull, acc[i], 1));  // x_i + x_{i+4}
                r = __fadd_rn(__fadd_rn(ts[0], ts[2]), __fadd_rn(ts[1], ts[3]));
            }
            const uint32_t jj = j0 + pp * ROWS + team;
            if (tl == 0 && jj < n) cd[jj] = post_op<POST>(r);
        }
    }
}

// ---- i8 / u8 rows: exact i32 arithmetic, so any summation order gives the reference's value --
// 8 lanes per row, 16 bytes per lane per load, 4 rows per pass, P passes in flight.
// q: query bytes in shared memory, zero-padded to a multiple of 16; qq = sum q*q.
template <bool SIGNED, int KIND, int POST, int P>
__device__ __forceinline__ void wide_distances_int(const uint8_t* __restrict__ q, int qq, const uint8_t* __restrict__ vectors,
                                                   size_t row_stride, const uint32_t* __restrict__ cid, uint32_t n,
                                                   float* __restrict__ cd, int dim, int lane) {
    constexpr int ROWS = 4;
    const int team = lane >> 3, tl = lane & 7;
    const int nfull = dim >> 4, tail = dim & 15;
    const int nm = (nfull + 7) >> 3;
    if (n > P * ROWS) prefetch_rows(vectors, row_stride, cid, n, (uint32_t)((dim + 15) & ~15), lane);
    for (uint32_t j0 = 0; j0 < n; j0 += P * ROWS) {
        const uint8_t* row[P];
        bool act[P];
        int xy[P], yy[P];
#pragma unroll
        for (int pp = 0; pp < P; ++pp) {
            act[pp] = j0 + pp * ROWS < n;
            const uint32_t jj = min(j0 + pp * ROWS + team, n - 1);
            row[pp] = vectors + (size_t)cid[jj] * row_stride;
            xy[pp] = yy[pp] = 0;
        }
        for (int m = 0; m < nm; ++m) {
            const int c = m * 8 + tl;
            if (c < nfull) {
                uint4 v[P];
#pragma unroll
                for (int pp = 0; pp < P; ++pp)
                    if (act[pp]) v[pp] = ldg16(row[pp] + (size_t)c * 16);
                const uint4 x = reinterpret_cast<const uint4*>(q)[c];
#pragma unroll
                for (int pp = 0; pp < P; ++pp) {
                    if (act[pp]) {
                        xy[pp] = dp4<SIGNED>((int)x.x, (int)v[pp].x, xy[pp]);
                        xy[pp] = dp4<SIGNED>((int)x.y, (int)v[pp].y, xy[pp]);
                        xy[pp] = dp4<SIGNED>((int)x.z, (int)v[pp].z, xy[pp]);
                        xy[pp] = dp4<SIGNED>((int)x.w, (int)v[pp].w, xy[pp]);
                        if (KIND != KIND_IP) {
                            yy[pp] = dp4<SIGNED>((int)v[pp].x, (int)v[pp].x, yy[pp]);
                            yy[pp] = dp4<SIGNED>((int)v[pp].y, (int)v[pp].y, yy[pp]);
                            yy[pp] = dp4<SIGNED>((int)v[pp].z, (int)v[pp].z, yy[pp]);
                            yy[pp] = dp4<SIGNED>((int)v[pp].w, (int)v[pp].w, yy[pp]);
                        }
                    }
                }
            }
        }
        if (tail) {
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                const int i = (nfull << 4) + tl * 2 + t;
                if (tl * 2 + t < tail) {
                    const int x = byte_at<SIGNED>(q, i);
#pragma unroll
                    for (int pp = 0; pp < P; ++pp) {
                        if (act[pp]) {
                            const int y = SIGNED ? (int)(int8_t)__ldg(row[pp] + i) : (int)__ldg(row[pp] + i);
                            xy[pp] += x * y;
                            if (KIND != KIND_IP) yy[pp] += y * y;
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int pp = 0; pp < P; ++pp) {
            if (!act[pp]) continue;
            int sxy = xy[pp], syy = yy[pp];
#pragma unroll
            for (int o = 4; o >= 1; o >>= 1) {
                sxy += __shfl_xor_sync(kFull, sxy, o);
                if (KIND != KIND_IP) syy += __shfl_xor_sync(kFull, syy, o);
            }
            float r;
            if (KIND == KIND_IP) r = (float)sxy;
            else if (KIND == KIND_L2) r = (float)(int)((unsigned)qq + (unsigned)syy - 2u * (unsigned)sxy);
            else r = cosine_finish((float)qq, (float)syy, (float)sxy);
            const uint32_t jj = j0 + pp * ROWS + team;
            if (tl == 0 && jj < n) cd[jj] = post_op<POST>(r);
        }
    }
}

}  // namespace
}  // namespace dab
