// distance_kernels.cu — batched distance kernels behind the per-pair / per-query boundary
// (SURVEY.md §8b.1): dab_pair_distances, dab_distances (frontier gather), data x data pairs
// and the prune candidate block.  HBM-gather bound: one team of lanes per row, coalesced
// element loads, no tensor cores (arithmetic intensity ~0.5 flop/B).
#include "dab_common.cuh"
#include "distance_device.cuh"

namespace dab {

constexpr int kWarpsPerBlock = 8;

template <typename T>
struct IsInt {
    static constexpr bool value = false;
};
template <>
struct IsInt<int8_t> {
    static constexpr bool value = true;
};
template <>
struct IsInt<uint8_t> {
    static constexpr bool value = true;
};

// ------------------------------------------------------------------ n independent pairs
// x[i] (dense rows of TX), y[i] (dense rows of TY) -> out[i]
template <typename TX, typename TY, int NA, int KIND, int POST>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
pair_float_kernel(const TX* __restrict__ x, size_t x_stride, const TY* __restrict__ y, size_t y_stride,
                  uint64_t n, int dim, float* __restrict__ out) {
    constexpr int S = 8 * NA, TEAMS = 32 / S;
    const int lane = threadIdx.x & 31;
    const int team = lane / S, slot = lane % S;
    const uint64_t warp = (uint64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const uint64_t nwarps = (uint64_t)gridDim.x * kWarpsPerBlock;
    for (uint64_t base = warp * TEAMS; base < n; base += nwarps * TEAMS) {
        uint64_t i = base + team;
        const bool valid = i < n;
        if (!valid) i = n - 1;
        const TY* rows[1] = {reinterpret_cast<const TY*>(reinterpret_cast<const uint8_t*>(y) + i * y_stride)};
        const TX* q = reinterpret_cast<const TX*>(reinterpret_cast<const uint8_t*>(x) + i * x_stride);
        float r[1];
        team_float_multi<NA, KIND, 1>(q, rows, dim, slot, r);
        if (valid && slot == 0) out[i] = post_op<POST>(r[0]);
    }
}

template <bool SIGNED, int KIND, int POST>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
pair_int_kernel(const uint8_t* __restrict__ x, size_t x_stride, const uint8_t* __restrict__ y, size_t y_stride,
                uint64_t n, int dim, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const uint64_t warp = (uint64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const uint64_t nwarps = (uint64_t)gridDim.x * kWarpsPerBlock;
    for (uint64_t i = warp; i < n; i += nwarps) {
        const uint8_t* q = x + i * x_stride;
        const uint8_t* rows[1] = {y + i * y_stride};
        int qq = KIND == KIND_IP ? 0 : warp_int_self<SIGNED>(q, dim, lane);
        float r[1];
        warp_int_multi<SIGNED, KIND, 1>(q, rows, dim, lane, qq, r);
        if (lane == 0) out[i] = post_op<POST>(r[0]);
    }
}

// ------------------------------------------------------------------ frontier distances
// out[q][j] = dist(query q, row ids[q][j]); one warp per (query, 32*U-candidate tile).
// The query is staged once per warp in shared memory (f16 queries widened to f32,
// diskann-inmem/src/layers/full.rs:421-423).
template <typename TQS /*smem query type*/, typename TQG /*global query type*/, typename TD, int NA, int KIND,
          int POST, int U>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
frontier_float_kernel(const TQG* __restrict__ queries, uint32_t nq, const uint32_t* __restrict__ ids, uint32_t c,
                      const uint8_t* __restrict__ vectors, size_t row_stride, uint64_t n_total, int dim,
                      float* __restrict__ out) {
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr int S = 8 * NA, TEAMS = 32 / S;
    constexpr int TILE = 32;  // candidates per warp tile
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int team = lane / S, slot = lane % S;
    TQS* q = reinterpret_cast<TQS*>(smem) + (size_t)wib * dim;
    const uint32_t tiles_per_q = (c + TILE - 1) / TILE;
    const uint64_t total_tiles = (uint64_t)nq * tiles_per_q;
    const uint64_t nwarps = (uint64_t)gridDim.x * kWarpsPerBlock;
    for (uint64_t t = (uint64_t)blockIdx.x * kWarpsPerBlock + wib; t < total_tiles; t += nwarps) {
        const uint32_t qi = (uint32_t)(t / tiles_per_q);
        const uint32_t j0 = (uint32_t)(t % tiles_per_q) * TILE;
        __syncwarp();
        for (int e = lane; e < dim; e += 32) q[e] = (TQS)to_f32(queries[(size_t)qi * dim + e]);
        __syncwarp();
        const uint32_t jend = min(j0 + TILE, c);
        for (uint32_t j = j0; j < jend; j += TEAMS * U) {
            const TD* rows[U];
            uint32_t jj[U];
            bool ok[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                jj[u] = j + u * TEAMS + team;
                uint32_t id = jj[u] < jend ? ids[(size_t)qi * c + jj[u]] : kNoId;
                ok[u] = id != kNoId && id < n_total;
                rows[u] = reinterpret_cast<const TD*>(vectors + (size_t)(ok[u] ? id : 0) * row_stride);
            }
            float r[U];
            team_float_multi<NA, KIND, U, 4>(q, rows, dim, slot, r);
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (slot == 0 && jj[u] < jend) out[(size_t)qi * c + jj[u]] = ok[u] ? post_op<POST>(r[u]) : __int_as_float(0x7FC00000);
        }
    }
}

// Wide-load variant for the NA = 4 schemas (L2 / InnerProduct / CosineNormalized over f32 or
// f16 rows against an f32 query): every lane reads 16 contiguous bytes of its row per step
// (8 f16 = all eight slots of one accumulator; 4 f32 = half of them) and runs those slots'
// sequential FMA chains itself, so a row needs only 4 (f16) or 8 (f32) lanes and a warp works on
// 8 or 4 rows at once with LDG.128 instead of 2- / 4-byte loads.  Same association as
// team_float_multi: block k of 8 elements goes to accumulator k mod 4, accumulators are combined
// (s0+s1)+(s2+s3) with xor-shuffles, the zero-filled remainder is applied to the combined
// vector, then sum_tree ((x0+x4)+(x2+x6))+((x1+x5)+(x3+x7)).
template <typename TQG, typename TD, int KIND, int POST>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
frontier_wide_kernel(const TQG* __restrict__ queries, uint32_t nq, const uint32_t* __restrict__ ids, uint32_t c,
                     const uint8_t* __restrict__ vectors, size_t row_stride, uint64_t n_total, int dim, int qstride,
                     float* __restrict__ out) {
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr int EPL = 16 / (int)sizeof(TD);  // elements per 16-byte load: 8 (f16) or 4 (f32)
    constexpr int LPR = 32 / EPL;              // lanes per row: 4 or 8
    constexpr int ROWS = EPL;                  // rows per warp pass: 8 or 4
    constexpr int HALVES = 8 / EPL;            // lanes sharing one accumulator: 1 or 2
    constexpr int TILE = 32;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int team = lane / LPR, tl = lane % LPR;
    const int a = tl / HALVES, h = tl % HALVES;
    float* q = reinterpret_cast<float*>(smem) + (size_t)wib * qstride;
    const int nb8 = dim >> 3, full8 = dim & ~7, rem = dim & 7;
    const uint32_t tiles_per_q = (c + TILE - 1) / TILE;
    const uint64_t total_tiles = (uint64_t)nq * tiles_per_q;
    const uint64_t nwarps = (uint64_t)gridDim.x * kWarpsPerBlock;
    for (uint64_t t = (uint64_t)blockIdx.x * kWarpsPerBlock + wib; t < total_tiles; t += nwarps) {
        const uint32_t qi = (uint32_t)(t / tiles_per_q);
        const uint32_t j0 = (uint32_t)(t % tiles_per_q) * TILE;
        __syncwarp();
        for (int e = lane; e < qstride; e += 32) q[e] = e < dim ? to_f32(queries[(size_t)qi * dim + e]) : 0.0f;
        __syncwarp();
        const uint32_t jend = min(j0 + TILE, c);
        for (uint32_t j = j0; j < jend; j += ROWS) {
            const uint32_t jj = j + team;
            const uint32_t id = jj < jend ? ids[(size_t)qi * c + jj] : kNoId;
            const bool ok = id != kNoId && id < n_total;
            const uint8_t* row = vectors + (size_t)(ok ? id : 0) * row_stride;
            float acc[EPL];
#pragma unroll
            for (int i = 0; i < EPL; ++i) acc[i] = 0.0f;
#pragma unroll 4
            for (int k = a; k < nb8; k += 4) {
                const int e0 = 8 * k + EPL * h;
                const uint4 v = __ldg(reinterpret_cast<const uint4*>(row + (size_t)e0 * sizeof(TD)));
                float y[EPL];
                if constexpr (sizeof(TD) == 2) {
                    const __half2* hp = reinterpret_cast<const __half2*>(&v);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float2 f = __half22float2(hp[i]);
                        y[2 * i] = f.x;
                        y[2 * i + 1] = f.y;
                    }
                } else {
                    y[0] = __uint_as_float(v.x), y[1] = __uint_as_float(v.y), y[2] = __uint_as_float(v.z), y[3] = __uint_as_float(v.w);
                }
#pragma unroll
                for (int i = 0; i < EPL; i += 4) {
                    const float4 x = *reinterpret_cast<const float4*>(q + e0 + i);
                    const float xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        if (KIND == KIND_L2) {
                            const float d = __fsub_rn(xs[u], y[i + u]);
                            acc[i + u] = __fmaf_rn(d, d, acc[i + u]);
                        } else {
                            acc[i + u] = __fmaf_rn(xs[u], y[i + u], acc[i + u]);
                        }
                    }
                }
            }
            // (s0 + s1) + (s2 + s3), slot-wise
#pragma unroll
            for (int i = 0; i < EPL; ++i) {
                acc[i] = __fadd_rn(acc[i], __shfl_xor_sync(kFull, acc[i], HALVES));
                acc[i] = __fadd_rn(acc[i], __shfl_xor_sync(kFull, acc[i], 2 * HALVES));
            }
            if (rem) {  // zero-filled tail on the combined vector (simd.rs:733-744)
                const TD* tail = reinterpret_cast<const TD*>(row) + full8;
#pragma unroll
                for (int i = 0; i < EPL; ++i) {
                    const int l = EPL * h + i;
                    const float x = l < rem ? q[full8 + l] : 0.0f;
                    const float yv = l < rem ? ldg_elem(tail + l) : 0.0f;
                    if (KIND == KIND_L2) {
                        const float d = __fsub_rn(x, yv);
                        acc[i] = __fmaf_rn(d, d, acc[i]);
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
                float tsum[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    // x_i + x_{i+4}: the partner lane holds the other half of the slots
                    const float other = __shfl_xor_sync(kFull, acc[i], 1);
                    tsum[i] = h == 0 ? __fadd_rn(acc[i], other) : __fadd_rn(other, acc[i]);
                }
                r = __fadd_rn(__fadd_rn(tsum[0], tsum[2]), __fadd_rn(tsum[1], tsum[3]));
            }
            if (tl == 0 && jj < jend) out[(size_t)qi * c + jj] = ok ? post_op<POST>(r) : __int_as_float(0x7FC00000);
        }
    }
}

template <bool SIGNED, int KIND, int POST, int U>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
frontier_int_kernel(const uint8_t* __restrict__ queries, uint32_t nq, const uint32_t* __restrict__ ids, uint32_t c,
                    const uint8_t* __restrict__ vectors, size_t row_stride, uint64_t n_total, int dim,
                    float* __restrict__ out) {
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr int TILE = 32;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int qbytes = (dim + 3) & ~3;
    uint8_t* q = smem + (size_t)wib * qbytes;
    const uint32_t tiles_per_q = (c + TILE - 1) / TILE;
    const uint64_t total_tiles = (uint64_t)nq * tiles_per_q;
    const uint64_t nwarps = (uint64_t)gridDim.x * kWarpsPerBlock;
    for (uint64_t t = (uint64_t)blockIdx.x * kWarpsPerBlock + wib; t < total_tiles; t += nwarps) {
        const uint32_t qi = (uint32_t)(t / tiles_per_q);
        const uint32_t j0 = (uint32_t)(t % tiles_per_q) * TILE;
        __syncwarp();
        for (int e = lane; e < qbytes; e += 32) q[e] = e < dim ? queries[(size_t)qi * dim + e] : 0;
        __syncwarp();
        const int qq = KIND == KIND_IP ? 0 : warp_int_self<SIGNED>(q, dim, lane);
        const uint32_t jend = min(j0 + TILE, c);
        for (uint32_t j = j0; j < jend; j += U) {
            const uint8_t* rows[U];
            bool ok[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                uint32_t id = j + u < jend ? ids[(size_t)qi * c + j + u] : kNoId;
                ok[u] = id != kNoId && id < n_total;
                rows[u] = vectors + (size_t)(ok[u] ? id : 0) * row_stride;
            }
            float r[U];
            warp_int_multi<SIGNED, KIND, U>(q, rows, dim, lane, qq, r);
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (lane == 0 && j + u < jend) out[(size_t)qi * c + j + u] = ok[u] ? post_op<POST>(r[u]) : __int_as_float(0x7FC00000);
        }
    }
}

// Integer rows, wide loads: eight lanes own one row (16 B each per 128-byte step), so one warp instruction
// requests four rows and eight rows are in flight per pass (a 128-byte i8 row is ONE request of the warp instead of
// a quarter of four).  Integer sums are exact in any order (wrapping i32, as warp_int_multi), so the lane split
// is free; the three xor-shuffles reduce within the team.  Needs dim % 16 == 0 (rows are 32-byte aligned).
template <bool SIGNED, int KIND, int POST>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
frontier_int_wide_kernel(const uint8_t* __restrict__ queries, uint32_t nq, const uint32_t* __restrict__ ids, uint32_t c,
                         const uint8_t* __restrict__ vectors, size_t row_stride, uint64_t n_total, int dim,
                         float* __restrict__ out) {
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr int TILE = 32, ROWS = 4, PASS = 2;  // rows per load instruction, load instructions in flight
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int team = lane >> 3, tl = lane & 7;
    uint8_t* q = smem + (size_t)wib * dim;
    const uint32_t tiles_per_q = (c + TILE - 1) / TILE;
    const uint64_t total_tiles = (uint64_t)nq * tiles_per_q;
    const uint64_t nwarps = (uint64_t)gridDim.x * kWarpsPerBlock;
    for (uint64_t t = (uint64_t)blockIdx.x * kWarpsPerBlock + wib; t < total_tiles; t += nwarps) {
        const uint32_t qi = (uint32_t)(t / tiles_per_q);
        const uint32_t j0 = (uint32_t)(t % tiles_per_q) * TILE;
        __syncwarp();
        for (int e = lane * 16; e < dim; e += 512)
            *reinterpret_cast<uint4*>(q + e) = __ldg(reinterpret_cast<const uint4*>(queries + (size_t)qi * dim + e));
        __syncwarp();
        const int qq = KIND == KIND_IP ? 0 : warp_int_self<SIGNED>(q, dim, lane);
        const uint32_t jend = min(j0 + TILE, c);
        for (uint32_t j = j0; j < jend; j += ROWS * PASS) {
            uint32_t id[PASS];
            bool ok[PASS];
            const uint8_t* row[PASS];
            int xy[PASS], yy[PASS];
#pragma unroll
            for (int u = 0; u < PASS; ++u) {
                const uint32_t jj = j + u * ROWS + team;
                id[u] = jj < jend ? ids[(size_t)qi * c + jj] : kNoId;
                ok[u] = id[u] != kNoId && id[u] < n_total;
                row[u] = vectors + (size_t)(ok[u] ? id[u] : 0) * row_stride;
                xy[u] = yy[u] = 0;
            }
            for (int e = tl * 16; e < dim; e += 128) {
                const uint4 x = *reinterpret_cast<const uint4*>(q + e);
                uint4 y[PASS];
#pragma unroll
                for (int u = 0; u < PASS; ++u) y[u] = __ldg(reinterpret_cast<const uint4*>(row[u] + e));
#pragma unroll
                for (int u = 0; u < PASS; ++u) {
                    xy[u] = dp4<SIGNED>((int)x.x, (int)y[u].x, xy[u]);
                    xy[u] = dp4<SIGNED>((int)x.y, (int)y[u].y, xy[u]);
                    xy[u] = dp4<SIGNED>((int)x.z, (int)y[u].z, xy[u]);
                    xy[u] = dp4<SIGNED>((int)x.w, (int)y[u].w, xy[u]);
                    if (KIND != KIND_IP) {
                        yy[u] = dp4<SIGNED>((int)y[u].x, (int)y[u].x, yy[u]);
                        yy[u] = dp4<SIGNED>((int)y[u].y, (int)y[u].y, yy[u]);
                        yy[u] = dp4<SIGNED>((int)y[u].z, (int)y[u].z, yy[u]);
                        yy[u] = dp4<SIGNED>((int)y[u].w, (int)y[u].w, yy[u]);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < PASS; ++u) {
#pragma unroll
                for (int m = 1; m < 8; m <<= 1) {
                    xy[u] += __shfl_xor_sync(kFull, xy[u], m);
                    if (KIND != KIND_IP) yy[u] += __shfl_xor_sync(kFull, yy[u], m);
                }
                const uint32_t jj = j + u * ROWS + team;
                if (tl == 0 && jj < jend) {
                    float r;
                    if (KIND == KIND_IP) r = (float)xy[u];
                    else if (KIND == KIND_L2) r = (float)(int)((unsigned)qq + (unsigned)yy[u] - 2u * (unsigned)xy[u]);
                    else r = cosine_finish((float)qq, (float)yy[u], (float)xy[u]);
                    out[(size_t)qi * c + jj] = ok[u] ? post_op<POST>(r) : __int_as_float(0x7FC00000);
                }
            }
        }
    }
}

// ------------------------------------------------------------------ data x data pairs by id
template <typename T, int NA, int KIND, int POST>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
rowpair_float_kernel(const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, uint64_t n,
                     const uint8_t* __restrict__ vectors, size_t row_stride, uint64_t n_total, int dim,
                     float* __restrict__ out) {
    constexpr int S = 8 * NA, TEAMS = 32 / S;
    const int lane = threadIdx.x & 31;
    const int team = lane / S, slot = lane % S;
    const uint64_t warp = (uint64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const uint64_t nwarps = (uint64_t)gridDim.x * kWarpsPerBlock;
    for (uint64_t base = warp * TEAMS; base < n; base += nwarps * TEAMS) {
        uint64_t i = base + team;
        const bool in = i < n;
        uint32_t ia = in ? a[i] : 0, ib = in ? b[i] : 0;
        const bool ok = in && ia < n_total && ib < n_total;
        if (!ok) ia = ib = 0;
        const T* q = reinterpret_cast<const T*>(vectors + (size_t)ia * row_stride);
        const T* rows[1] = {reinterpret_cast<const T*>(vectors + (size_t)ib * row_stride)};
        float r[1];
        team_float_multi<NA, KIND, 1>(q, rows, dim, slot, r);
        if (in && slot == 0) out[i] = ok ? post_op<POST>(r[0]) : __int_as_float(0x7FC00000);
    }
}

template <bool SIGNED, int KIND, int POST>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
rowpair_int_kernel(const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, uint64_t n,
                   const uint8_t* __restrict__ vectors, size_t row_stride, uint64_t n_total, int dim,
                   float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const uint64_t warp = (uint64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    const uint64_t nwarps = (uint64_t)gridDim.x * kWarpsPerBlock;
    for (uint64_t i = warp; i < n; i += nwarps) {
        uint32_t ia = a[i], ib = b[i];
        const bool ok = ia < n_total && ib < n_total;
        if (!ok) ia = ib = 0;
        const uint8_t* q = vectors + (size_t)ia * row_stride;
        const uint8_t* rows[1] = {vectors + (size_t)ib * row_stride};
        int qq = KIND == KIND_IP ? 0 : warp_int_self<SIGNED>(q, dim, lane);
        float r[1];
        warp_int_multi<SIGNED, KIND, 1>(q, rows, dim, lane, qq, r);
        if (lane == 0) out[i] = ok ? post_op<POST>(r[0]) : __int_as_float(0x7FC00000);
    }
}

__global__ void expand_pairs_kernel(const uint32_t* __restrict__ ids, uint32_t n, uint32_t* __restrict__ a,
                                    uint32_t* __restrict__ b) {
    const uint64_t total = (uint64_t)n * n;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        a[i] = ids[i / n];
        b[i] = ids[i % n];
    }
}

// ------------------------------------------------------------------ host-side dispatch
static int grid_for(uint64_t work_warps, int sm_count) {
    uint64_t blocks = (work_warps + kWarpsPerBlock - 1) / kWarpsPerBlock;
    uint64_t cap = (uint64_t)sm_count * 8;  // 8 blocks of 8 warps = 64 warps per SM
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

#define DAB_KIND_POST_SWITCH(plan, MACRO)                                                       \
    do {                                                                                        \
        if ((plan).kind == KIND_L2) { MACRO(KIND_L2, POST_ID); }                                \
        else if ((plan).kind == KIND_IP && (plan).post == POST_NEG) { MACRO(KIND_IP, POST_NEG); } \
        else if ((plan).kind == KIND_IP) { MACRO(KIND_IP, POST_ONE_MINUS); }                    \
        else { MACRO(KIND_COS, POST_ONE_MINUS); }                                               \
    } while (0)

int launch_pairs(int dx, int dy, int metric, int dim, const void* x, size_t xs, const void* y, size_t ys, uint64_t n,
                 float* out, int sm_count, cudaStream_t stream) {
    const bool is_int = dx == DAB_I8 || dx == DAB_U8;
    const MetricPlan plan = plan_for(metric, is_int);
    const int grid = grid_for(n, sm_count);
    const int block = kWarpsPerBlock * 32;
    if (dx == DAB_F32 && dy == DAB_F32) {
#define L(K, P)                                                                                       \
    if (K == KIND_COS)                                                                                \
        pair_float_kernel<float, float, 2, K, P><<<grid, block, 0, stream>>>((const float*)x, xs, (const float*)y, ys, n, dim, out); \
    else                                                                                              \
        pair_float_kernel<float, float, 4, K, P><<<grid, block, 0, stream>>>((const float*)x, xs, (const float*)y, ys, n, dim, out)
        DAB_KIND_POST_SWITCH(plan, L);
#undef L
    } else if (dx == DAB_F16 && dy == DAB_F16) {
#define L(K, P) pair_float_kernel<__half, __half, 2, K, P><<<grid, block, 0, stream>>>((const __half*)x, xs, (const __half*)y, ys, n, dim, out)
        DAB_KIND_POST_SWITCH(plan, L);
#undef L
    } else if (dx == DAB_F32 && dy == DAB_F16) {
#define L(K, P)                                                                                       \
    if (K == KIND_COS)                                                                                \
        pair_float_kernel<float, __half, 2, K, P><<<grid, block, 0, stream>>>((const float*)x, xs, (const __half*)y, ys, n, dim, out); \
    else                                                                                              \
        pair_float_kernel<float, __half, 4, K, P><<<grid, block, 0, stream>>>((const float*)x, xs, (const __half*)y, ys, n, dim, out)
        DAB_KIND_POST_SWITCH(plan, L);
#undef L
    } else if (dx == DAB_I8 && dy == DAB_I8) {
#define L(K, P) pair_int_kernel<true, K, P><<<grid, block, 0, stream>>>((const uint8_t*)x, xs, (const uint8_t*)y, ys, n, dim, out)
        DAB_KIND_POST_SWITCH(plan, L);
#undef L
    } else if (dx == DAB_U8 && dy == DAB_U8) {
#define L(K, P) pair_int_kernel<false, K, P><<<grid, block, 0, stream>>>((const uint8_t*)x, xs, (const uint8_t*)y, ys, n, dim, out)
        DAB_KIND_POST_SWITCH(plan, L);
#undef L
    } else {
        return fail(DAB_ERR_INVALID_ARGUMENT, "unsupported dtype pair (%d, %d)", dx, dy);
    }
    DAB_LAUNCHED();
    DAB_CUDA(cudaGetLastError());
    return DAB_OK;
}

int launch_frontier(const dab_index* idx, const void* d_queries, uint32_t nq, const uint32_t* d_ids, uint32_t c,
                    float* d_out) {
    const bool is_int = idx->dtype == DAB_I8 || idx->dtype == DAB_U8;
    const MetricPlan plan = plan_for(idx->metric, is_int);
    const uint64_t tiles = (uint64_t)nq * ((c + 31) / 32);
    const int grid = grid_for(tiles, idx->sm_count);
    const int block = kWarpsPerBlock * 32;
    const int dim = (int)idx->dim;
    const size_t smem = (size_t)kWarpsPerBlock * (is_int ? ((dim + 3) & ~3) : dim * 4);
    if (smem > 200 * 1024) return fail(DAB_ERR_INVALID_ARGUMENT, "dim %d too large for the frontier kernel", dim);
    cudaStream_t st = idx->stream;
    constexpr int U = 4;
    // NA = 4 schemas over f32 / f16 rows: the wide-load kernel (16 B per lane; rows start on 32 B bounds)
    if (plan.kind != KIND_COS && (idx->dtype == DAB_F32 || idx->dtype == DAB_F16)) {
        const int qstride = (dim + 3) & ~3;
        const size_t wsmem = (size_t)kWarpsPerBlock * qstride * 4;
#define LW(TQ, TDD, K, P)                                                                                          \
    do {                                                                                                          \
        auto kern = frontier_wide_kernel<TQ, TDD, K, P>;                                                          \
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem);                      \
        kern<<<grid, block, wsmem, st>>>((const TQ*)d_queries, nq, d_ids, c, idx->d_vectors, idx->row_stride,      \
                                         idx->n_total(), dim, qstride, d_out);                                    \
    } while (0)
        if (idx->dtype == DAB_F32) {
            if (plan.kind == KIND_L2) LW(float, float, KIND_L2, POST_ID);
            else if (plan.post == POST_NEG) LW(float, float, KIND_IP, POST_NEG);
            else LW(float, float, KIND_IP, POST_ONE_MINUS);
        } else {
            if (plan.kind == KIND_L2) LW(__half, __half, KIND_L2, POST_ID);
            else if (plan.post == POST_NEG) LW(__half, __half, KIND_IP, POST_NEG);
            else LW(__half, __half, KIND_IP, POST_ONE_MINUS);
        }
#undef LW
        DAB_LAUNCHED();
        DAB_CUDA(cudaGetLastError());
        return DAB_OK;
    }
#define ARGS nq, d_ids, c, idx->d_vectors, idx->row_stride, idx->n_total(), dim, d_out
    // float cosine (NA = 2): the 4-byte-load kernel
    if (idx->dtype == DAB_F32) {
        auto kern = frontier_float_kernel<float, float, float, 2, KIND_COS, POST_ONE_MINUS, U>;
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        kern<<<grid, block, smem, st>>>((const float*)d_queries, ARGS);
    } else if (idx->dtype == DAB_F16) {
        auto kern = frontier_float_kernel<float, __half, __half, 2, KIND_COS, POST_ONE_MINUS, U>;
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        kern<<<grid, block, smem, st>>>((const __half*)d_queries, ARGS);
    } else if (is_int && dim % 16 == 0 && ((uintptr_t)d_queries & 15) == 0) {
        const size_t ismem = (size_t)kWarpsPerBlock * dim;
#define L(K, P)                                                                                   \
    do {                                                                                          \
        if (idx->dtype == DAB_I8) {                                                               \
            auto kern = frontier_int_wide_kernel<true, K, P>;                                     \
            cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ismem);  \
            kern<<<grid, block, ismem, st>>>((const uint8_t*)d_queries, ARGS);                    \
        } else {                                                                                  \
            auto kern = frontier_int_wide_kernel<false, K, P>;                                    \
            cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ismem);  \
            kern<<<grid, block, ismem, st>>>((const uint8_t*)d_queries, ARGS);                    \
        }                                                                                         \
    } while (0)
        DAB_KIND_POST_SWITCH(plan, L);
#undef L
    } else if (idx->dtype == DAB_I8) {
#define L(K, P)                                                                                   \
    do {                                                                                          \
        auto kern = frontier_int_kernel<true, K, P, U>;                                           \
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);       \
        kern<<<grid, block, smem, st>>>((const uint8_t*)d_queries, ARGS);                         \
    } while (0)
        DAB_KIND_POST_SWITCH(plan, L);
#undef L
    } else {
#define L(K, P)                                                                                   \
    do {                                                                                          \
        auto kern = frontier_int_kernel<false, K, P, U>;                                          \
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);       \
        kern<<<grid, block, smem, st>>>((const uint8_t*)d_queries, ARGS);                         \
    } while (0)
        DAB_KIND_POST_SWITCH(plan, L);
#undef L
    }
#undef ARGS
    DAB_LAUNCHED();
    DAB_CUDA(cudaGetLastError());
    return DAB_OK;
}

int launch_rowpairs(const dab_index* idx, const uint32_t* d_a, const uint32_t* d_b, uint64_t n, float* d_out) {
    const bool is_int = idx->dtype == DAB_I8 || idx->dtype == DAB_U8;
    const MetricPlan plan = plan_for(idx->metric, is_int);
    const int grid = grid_for(n, idx->sm_count);
    const int block = kWarpsPerBlock * 32;
    const int dim = (int)idx->dim;
    cudaStream_t st = idx->stream;
#define ARGS d_a, d_b, n, idx->d_vectors, idx->row_stride, idx->n_total(), dim, d_out
    if (idx->dtype == DAB_F32) {
#define L(K, P)                                                             \
    if (K == KIND_COS)                                                      \
        rowpair_float_kernel<float, 2, K, P><<<grid, block, 0, st>>>(ARGS); \
    else                                                                    \
        rowpair_float_kernel<float, 4, K, P><<<grid, block, 0, st>>>(ARGS)
        DAB_KIND_POST_SWITCH(plan, L);
#undef L
    } else if (idx->dtype == DAB_F16) {
        // data x data for f16 is the f16 x f16 schema (Strategy2x4), simd.rs:989, 1752, 2591
#define L(K, P) rowpair_float_kernel<__half, 2, K, P><<<grid, block, 0, st>>>(ARGS)
        DAB_KIND_POST_SWITCH(plan, L);
#undef L
    } else if (idx->dtype == DAB_I8) {
#define L(K, P) rowpair_int_kernel<true, K, P><<<grid, block, 0, st>>>(ARGS)
        DAB_KIND_POST_SWITCH(plan, L);
#undef L
    } else {
#define L(K, P) rowpair_int_kernel<false, K, P><<<grid, block, 0, st>>>(ARGS)
        DAB_KIND_POST_SWITCH(plan, L);
#undef L
    }
#undef ARGS
    DAB_LAUNCHED();
    DAB_CUDA(cudaGetLastError());
    return DAB_OK;
}

}  // namespace dab

using namespace dab;

extern "C" {

int dab_pair_distances(int dtype_x, int dtype_y, int metric, uint32_t dim, const void* x, const void* y, uint64_t n,
                       float* out, int device) {
    if ((!x || !y || !out) && n) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_pair_distances: NULL argument");
    if (metric < DAB_COSINE || metric > DAB_COSINE_NORMALIZED)
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_pair_distances: unknown metric %d", metric);
    if (dtype_x < 0 || dtype_x > 3 || dtype_y < 0 || dtype_y > 3)
        return fail(DAB_ERR_INVALID_ARGUMENT, "dab_pair_distances: unknown dtype");
    if (n == 0) return DAB_OK;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(DAB_ERR_NO_DEVICE, "dab_pair_distances: no CUDA device visible (no CPU fallback)");
    DAB_CUDA(cudaSetDevice(device));
    int sm = 148;
    cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, device);
    // rows are padded to 4 bytes on the device so the integer kernels can use word loads
    const size_t xb = (size_t)dim * elem_size(dtype_x), yb = (size_t)dim * elem_size(dtype_y);
    const size_t xs = round_up(xb ? xb : 1, 4), ys = round_up(yb ? yb : 1, 4);
    uint8_t *dx = nullptr, *dy = nullptr;
    float* dout = nullptr;
    int rc = DAB_OK;
    cudaError_t e = cudaMalloc(&dx, xs * n);
    if (e == cudaSuccess) e = cudaMalloc(&dy, ys * n);
    if (e == cudaSuccess) e = cudaMalloc(&dout, n * 4);
    if (e == cudaSuccess) e = cudaMemset(dx, 0, xs * n);
    if (e == cudaSuccess) e = cudaMemset(dy, 0, ys * n);
    if (e == cudaSuccess && xb) e = cudaMemcpy2D(dx, xs, x, xb, xb, n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && yb) e = cudaMemcpy2D(dy, ys, y, yb, yb, n, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        rc = fail(DAB_ERR_CUDA, "dab_pair_distances: staging failed: %s", cudaGetErrorString(e));
    } else {
        rc = launch_pairs(dtype_x, dtype_y, metric, (int)dim, dx, xs, dy, ys, n, dout, sm, 0);
        if (rc == DAB_OK) {
            e = cudaMemcpy(out, dout, n * 4, cudaMemcpyDeviceToHost);
            if (e != cudaSuccess) rc = fail(DAB_ERR_CUDA, "dab_pair_distances: kernel/copy failed: %s", cudaGetErrorString(e));
        }
    }
    cudaFree(dx);
    cudaFree(dy);
    cudaFree(dout);
    return rc;
}

int dab_distances_device(dab_index* idx, const void* d_queries, uint32_t nq, const uint32_t* d_ids, uint32_t c,
                         float* d_out) {
    if (!idx) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_distances: idx is NULL");
    if (!idx->vectors_ready) return fail(DAB_ERR_NOT_READY, "dab_distances: vectors not uploaded");
    if (nq == 0 || c == 0) return DAB_OK;
    if (!d_queries || !d_ids || !d_out) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_distances: NULL argument");
    DAB_CUDA(cudaSetDevice(idx->device));
    return launch_frontier(idx, d_queries, nq, d_ids, c, d_out);
}

int dab_distances(dab_index* idx, const void* queries, uint32_t nq, const uint32_t* ids, uint32_t c, float* out) {
    if (!idx) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_distances: idx is NULL");
    if (!idx->vectors_ready) return fail(DAB_ERR_NOT_READY, "dab_distances: vectors not uploaded");
    if (nq == 0 || c == 0) return DAB_OK;
    if (!queries || !ids || !out) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_distances: NULL argument");
    DAB_CUDA(cudaSetDevice(idx->device));
    const size_t qbytes = (size_t)nq * idx->dim * elem_size(idx->dtype);
    const size_t ibytes = (size_t)nq * c * 4;
    int rc;
    if ((rc = idx->s_queries.reserve(qbytes))) return rc;
    if ((rc = idx->s_ids.reserve(ibytes))) return rc;
    if ((rc = idx->s_out.reserve(ibytes))) return rc;
    DAB_CUDA(cudaMemcpyAsync(idx->s_queries.p, queries, qbytes, cudaMemcpyHostToDevice, idx->stream));
    DAB_CUDA(cudaMemcpyAsync(idx->s_ids.p, ids, ibytes, cudaMemcpyHostToDevice, idx->stream));
    if ((rc = launch_frontier(idx, idx->s_queries.p, nq, (const uint32_t*)idx->s_ids.p, c, (float*)idx->s_out.p))) return rc;
    DAB_CUDA(cudaMemcpyAsync(out, idx->s_out.p, ibytes, cudaMemcpyDeviceToHost, idx->stream));
    DAB_CUDA(cudaStreamSynchronize(idx->stream));
    return DAB_OK;
}

int dab_row_pair_distances(dab_index* idx, const uint32_t* a, const uint32_t* b, uint64_t n, float* out) {
    if (!idx) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_row_pair_distances: idx is NULL");
    if (!idx->vectors_ready) return fail(DAB_ERR_NOT_READY, "dab_row_pair_distances: vectors not uploaded");
    if (n == 0) return DAB_OK;
    if (!a || !b || !out) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_row_pair_distances: NULL argument");
    DAB_CUDA(cudaSetDevice(idx->device));
    int rc;
    if ((rc = idx->s_ids.reserve(n * 8))) return rc;
    if ((rc = idx->s_out.reserve(n * 4))) return rc;
    uint32_t* da = (uint32_t*)idx->s_ids.p;
    uint32_t* db = da + n;
    DAB_CUDA(cudaMemcpyAsync(da, a, n * 4, cudaMemcpyHostToDevice, idx->stream));
    DAB_CUDA(cudaMemcpyAsync(db, b, n * 4, cudaMemcpyHostToDevice, idx->stream));
    if ((rc = launch_rowpairs(idx, da, db, n, (float*)idx->s_out.p))) return rc;
    DAB_CUDA(cudaMemcpyAsync(out, idx->s_out.p, n * 4, cudaMemcpyDeviceToHost, idx->stream));
    DAB_CUDA(cudaStreamSynchronize(idx->stream));
    return DAB_OK;
}

int dab_pairwise(dab_index* idx, const uint32_t* ids, uint32_t n, float* out) {
    if (!idx) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_pairwise: idx is NULL");
    if (!idx->vectors_ready) return fail(DAB_ERR_NOT_READY, "dab_pairwise: vectors not uploaded");
    if (n == 0) return DAB_OK;
    if (!ids || !out) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_pairwise: NULL argument");
    DAB_CUDA(cudaSetDevice(idx->device));
    const uint64_t total = (uint64_t)n * n;
    int rc;
    if ((rc = idx->s_ids.reserve(total * 8 + (size_t)n * 4))) return rc;
    if ((rc = idx->s_out.reserve(total * 4))) return rc;
    uint32_t* da = (uint32_t*)idx->s_ids.p;
    uint32_t* db = da + total;
    uint32_t* dids = db + total;
    DAB_CUDA(cudaMemcpyAsync(dids, ids, (size_t)n * 4, cudaMemcpyHostToDevice, idx->stream));
    expand_pairs_kernel<<<idx->sm_count * 4, 256, 0, idx->stream>>>(dids, n, da, db);
    DAB_LAUNCHED();
    if ((rc = launch_rowpairs(idx, da, db, total, (float*)idx->s_out.p))) return rc;
    DAB_CUDA(cudaMemcpyAsync(out, idx->s_out.p, total * 4, cudaMemcpyDeviceToHost, idx->stream));
    DAB_CUDA(cudaStreamSynchronize(idx->stream));
    return DAB_OK;
}

}  // extern "C"
