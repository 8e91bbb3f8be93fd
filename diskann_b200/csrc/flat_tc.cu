// flat_tc.cu — exhaustive scan (diskann/src/flat, ground truth for recall) on the 5th-generation
// tensor cores: the query x base distance block is a dense contraction, so it runs as a
// tcgen05.mma GEMM with TMA-staged tiles and a fused norm expansion + per-row candidate selection
// (BASELINE.json north_star; SURVEY.md §8f.3).
//
//   * operands are bf16.  f32 / f16 rows are split x = hi + lo (hi = bf16(x), lo = bf16(x - hi)) and
//     the three significant products are obtained from ONE GEMM over a 3x longer K:
//     A' = [q_hi | q_hi | q_lo], B' = [b_hi | b_lo | b_hi]  =>  A'.B' = hi.hi + hi.lo + lo.hi
//     (relative error of the dot product ~2^-16; fp32 accumulation in TMEM).  i8 / u8 rows are exact
//     in bf16 and their products / sums are exact in fp32 (128 * 127^2 < 2^24): one segment.
//   * one CTA = 128 query rows x a range of base rows; per 128-column tile: K' / 64 pipeline stages
//     of (A k-block, B k-block) 128 x 64 bf16 tiles loaded by TMA (128-byte swizzle) into shared
//     memory, 4 x tcgen05.mma (M 128, N 128, K 16, cta_group::1) per stage issued by one thread,
//     accumulators double-buffered in TMEM (2 x 128 columns) so the epilogue of tile t overlaps the
//     MMAs of tile t + 1;
//   * epilogue (4 warps = the 4 TMEM lane quarters, one query row per thread): tcgen05.ld the 128
//     accumulators of the row, score = alpha[col] * dot + beta[col] (L2: ||b||^2 - 2 q.b, the ||q||^2
//     term is constant per row; inner product: -q.b; cosine: -q.b / ||b||), keep the KP best columns of
//     the row in a small per-thread set;
//   * the KP candidates of every (query, base range) are then re-scored with the exact, reference-order
//     distance kernel (launch_frontier) and the final top-k is taken by (distance, id) — so the
//     returned distances are bit-identical to the exact scan and the ids are the exact scan's as long
//     as the approximate scores (error ~1e-5 relative) do not push a true neighbour below KP - k others.
#include "dab_common.cuh"
#include "distance_device.cuh"

#include <cuda.h>
#include <cuda_bf16.h>

#include <algorithm>
#include <vector>

namespace dab {

int launch_frontier(const dab_index* idx, const void* d_queries, uint32_t nq, const uint32_t* d_ids, uint32_t c, float* d_out);

namespace {

constexpr int kBM = 128, kBN = 128, kBK = 64;  // CTA tile; one k-block = 64 bf16 = one 128-byte swizzle row
constexpr int kStages = 5;                    // stages of (A k-block, B k-block)
constexpr int kTcThreads = 192;                // warp 0: TMA, warp 1: MMA + TMEM owner, warps 2-5: epilogue
constexpr int kKP = 32;                        // largest candidate set per (query row, base range); k <= 10 uses 16
constexpr uint32_t kTileBytes = kBM * kBK * 2; // 16 KB per operand tile

// ---- PTX wrappers ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int32_t x, int32_t y) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
                 "l"(map), "r"(smem_u32(bar)), "r"(x), "r"(y)
                 : "memory");
}
// K-major operand tile [rows][64 bf16] written by TMA with the 128-byte swizzle: 8-row groups of
// 1024 bytes (SBO = 64 x 16 B), LBO = 1, descriptor version 1, layout SWIZZLE_128B
// (cute/arch/mma_sm100_desc.hpp SmemDescriptor; cute/atom/mma_traits_sm100.hpp make_umma_desc<Major::K>)
__device__ __forceinline__ uint64_t umma_desc(const void* tile, uint32_t k_byte_offset) {
    const uint32_t addr = smem_u32(tile) + k_byte_offset;
    return (uint64_t)((addr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// kind::f16, A = B = bf16 (format 1), D = f32 (format 1), both K-major, M = 128, N = 128
__device__ __forceinline__ uint32_t umma_idesc() {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kBN >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {  // arrives on `bar` when every MMA issued so far has completed
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
          "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
          "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- operand preparation --------------------------------------------------------------------
// rows of the index dtype -> bf16 [n][kp]: f32 / f16: (hi, hi, lo) for queries, (hi, lo, hi) for base
// rows; i8 / u8: one exact segment.  Base rows also get their score coefficients.
template <typename T>
__device__ __forceinline__ float elem_f32(const T* p, uint32_t i) {
    if constexpr (sizeof(T) == 2) return __half2float(p[i]);
    else return (float)p[i];
}
template <typename T>
__global__ void prep_bf16_kernel(const uint8_t* __restrict__ rows, size_t row_stride, uint64_t n, uint32_t dim, uint32_t kp, int is_query,
                                 int score_kind /*0 L2, 1 IP, 2 cosine*/, __nv_bfloat16* __restrict__ out, float* __restrict__ alpha,
                                 float* __restrict__ beta) {
    constexpr bool kInt = sizeof(T) == 1;
    const int lane = threadIdx.x & 31;
    const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5, nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t r = warp; r < n; r += nwarps) {
        const T* row = reinterpret_cast<const T*>(rows + r * row_stride);
        __nv_bfloat16* o = out + r * kp;
        float nn = 0.0f;
        for (uint32_t d = lane; d < dim; d += 32) {
            const float x = elem_f32(row, d);
            nn = fmaf(x, x, nn);
            const __nv_bfloat16 hi = __float2bfloat16_rn(x);
            if constexpr (kInt) {
                o[d] = hi;
            } else {
                const __nv_bfloat16 lo = __float2bfloat16_rn(x - __bfloat162float(hi));
                o[d] = hi;
                o[dim + d] = is_query ? hi : lo;
                o[2 * dim + d] = is_query ? lo : hi;
            }
        }
        for (uint32_t d = (kInt ? dim : 3 * dim) + lane; d < kp; d += 32) o[d] = __float2bfloat16_rn(0.0f);
        if (!is_query) {
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) nn += __shfl_xor_sync(0xFFFFFFFFu, nn, s);
            if (lane == 0) {
                if (score_kind == 0) {
                    alpha[r] = -2.0f;
                    beta[r] = nn;
                } else if (score_kind == 1) {
                    alpha[r] = -1.0f;
                    beta[r] = 0.0f;
                } else {
                    alpha[r] = nn > 0.0f ? -rsqrtf(nn) : 0.0f;
                    beta[r] = 0.0f;
                }
            }
        }
    }
}

struct TcParams {
    uint32_t nq, n_base, kp;
    uint32_t tiles_per_split;  // 128-column tiles per base range
    uint32_t n_splits;
    const float* alpha;
    const float* beta;
    uint32_t* cand;            // [nq][n_splits][kKP]
};

template <int KP>
__global__ void __launch_bounds__(kTcThreads, 1)
flat_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const TcParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* sa = smem;                                                   // kStages x 16 KB
    uint8_t* sb = smem + kStages * kTileBytes;                            // kStages x 16 KB
    float* s_coef = reinterpret_cast<float*>(sb + kStages * kTileBytes);  // [2 accumulators][alpha 128 | beta 128]
    float* s_scores = s_coef + 2 * 2 * kBN;                                      // [128 epilogue threads][33]: private scratch rows
    float* s_cd = s_scores + 128 * 33;                                           // [KP][128]: candidate scores, entry-major (conflict-free)
    uint32_t* s_ci = reinterpret_cast<uint32_t*>(s_cd + KP * 128);               // [KP][128]: candidate ids
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_ci + KP * 128);               // offsets stay 8-byte aligned
    uint64_t* full = bars;                 // [kStages] TMA -> MMA
    uint64_t* empty = bars + kStages;      // [kStages] MMA -> TMA
    uint64_t* tfull = bars + 2 * kStages;  // [2] MMA -> epilogue
    uint64_t* tempty = tfull + 2;          // [2] epilogue -> MMA
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t m0 = blockIdx.y * kBM;
    const uint32_t split = blockIdx.x;
    const uint32_t n_tiles_total = (p.n_base + kBN - 1) / kBN;
    const uint32_t t0 = split * p.tiles_per_split, t1 = min(n_tiles_total, t0 + p.tiles_per_split);
    const uint32_t kblocks = p.kp / kBK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) {
            mbar_init(full + s, 1);
            mbar_init(empty + s, 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(tfull + a, 1);
            mbar_init(tempty + a, 4);  // one arrival per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    }
    if (warp == 1) {  // TMEM: 256 columns = two 128-column f32 accumulators
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(256u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *s_tmem;

    if (warp == 0) {
        // ===== TMA producer (one lane) =====
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (uint32_t t = t0; t < t1; ++t) {
                for (uint32_t kb = 0; kb < kblocks; ++kb) {
                    mbar_wait(empty + stage, phase ^ 1);
                    mbar_expect_tx(full + stage, 2 * kTileBytes);
                    tma_load_2d(&map_a, full + stage, sa + stage * kTileBytes, (int32_t)(kb * kBK), (int32_t)m0);
                    tma_load_2d(&map_b, full + stage, sb + stage * kTileBytes, (int32_t)(kb * kBK), (int32_t)(t * kBN));
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (one lane) =====
        if (lane == 0) {
            const uint32_t idesc = umma_idesc();
            uint32_t stage = 0, phase = 0;
            for (uint32_t t = t0; t < t1; ++t) {
                const uint32_t acc = (t - t0) & 1, use = (t - t0) >> 1;
                mbar_wait(tempty + acc, (use & 1) ^ 1);  // the epilogue has drained this accumulator
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t tmem_d = tmem_base + acc * kBN;
                for (uint32_t kb = 0; kb < kblocks; ++kb) {
                    mbar_wait(full + stage, phase);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                    for (int k = 0; k < kBK / 16; ++k) {
                        const uint64_t da = umma_desc(sa + stage * kTileBytes, k * 32);
                        const uint64_t db = umma_desc(sb + stage * kTileBytes, k * 32);
                        umma_f16(tmem_d, da, db, idesc, (kb | (uint32_t)k) != 0 ? 1u : 0u);
                    }
                    umma_commit(empty + stage);  // frees the stage once these MMAs have read it
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                umma_commit(tfull + acc);  // accumulator complete
            }
        }
    } else {
        // ===== epilogue: warps 2..5 own TMEM lane quarters (warp % 4), one query row per thread =====
        const uint32_t quarter = (uint32_t)warp & 3u;
        const uint32_t row = quarter * 32 + lane;  // row of the 128-row tile == TMEM lane
        const uint32_t q = m0 + row;
        const int et = (warp - 2) * 32 + lane;     // 0..127 among the epilogue threads
        float* my_scores = s_scores + et * 33;      // stride 33: conflict-free rows
        float* cd = s_cd + et;        // entry e of this thread: cd[e * 128]
        uint32_t* ci = s_ci + et;
        uint32_t cn = 0;
        float worst = -1.0f;   // largest kept score (valid when cn == KP)
        int worst_at = 0;
        // per-column score coefficients (alpha, beta): tile t's are in s_coef[t & 1]; the next tile's are
        // fetched from global memory while this tile is processed
        auto load_coef = [&](uint32_t t, float& a, float& b) {
            const uint32_t col = t * kBN + et;
            a = col < p.n_base ? p.alpha[col] : 0.0f;
            b = col < p.n_base ? p.beta[col] : __int_as_float(0x7F800000);
        };
        {
            float a, b;
            load_coef(t0, a, b);
            s_coef[et] = a;
            s_coef[kBN + et] = b;
        }
        for (uint32_t t = t0; t < t1; ++t) {
            const uint32_t acc = (t - t0) & 1, use = (t - t0) >> 1;
            float* coef = s_coef + acc * 2 * kBN;
            float a_next = 0.0f, b_next = 0.0f;
            if (t + 1 < t1) load_coef(t + 1, a_next, b_next);
            asm volatile("bar.sync 1, 128;" ::: "memory");  // coef[acc] written by everyone; coef[acc ^ 1] no longer read
            mbar_wait(tfull + acc, use & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t taddr = tmem_base + acc * kBN + ((quarter * 32u) << 16);
            uint32_t rbuf[2][32];
            tmem_ld32(taddr, rbuf[0]);
#pragma unroll
            for (int cc = 0; cc < kBN / 32; ++cc) {
                const int c0 = cc * 32;
                uint32_t (&r)[32] = rbuf[cc & 1];
                tmem_ld_wait();
                if (cc + 1 < kBN / 32) tmem_ld32(taddr + c0 + 32, rbuf[(cc + 1) & 1]);  // next chunk in flight during this one
                // fast path, branch-free: the 32 scores go to this thread's scratch row and a bit mask
                // marks the ones that beat the current threshold (all of them while the set fills)
                uint32_t mask = 0;
                const float thr = cn < (uint32_t)KP ? __int_as_float(0x7F800000) : worst;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float sc = fmaf(__uint_as_float(r[j]), coef[c0 + j], coef[kBN + c0 + j]);
                    my_scores[j] = sc;
                    mask |= sc < thr ? (1u << j) : 0u;
                }
                // slow path (rare once the threshold has settled): one candidate at a time
                while (mask) {
                    const int j = __ffs(mask) - 1;
                    mask &= mask - 1;
                    const float sc = my_scores[j];
                    const uint32_t id = t * kBN + c0 + j;
                    if (cn < (uint32_t)KP) {
                        cd[cn * 128] = sc;
                        ci[cn * 128] = id;
                        if (++cn < (uint32_t)KP) continue;
                    } else if (sc < worst) {
                        cd[worst_at * 128] = sc;
                        ci[worst_at * 128] = id;
                    } else {
                        continue;
                    }
                    // new threshold: the largest kept score (independent loads, then a max tree)
                    float v[KP];
#pragma unroll
                    for (int e = 0; e < KP; ++e) v[e] = cd[e * 128];
                    worst = v[0];
                    worst_at = 0;
#pragma unroll
                    for (int e = 1; e < KP; ++e)
                        if (v[e] > worst) worst = v[e], worst_at = e;
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty + acc);
            if (t + 1 < t1) {
                float* nxt = s_coef + (acc ^ 1u) * 2 * kBN;
                nxt[et] = a_next;
                nxt[kBN + et] = b_next;
            }
        }
        if (q < p.nq) {
            uint32_t* out = p.cand + ((size_t)q * p.n_splits + split) * KP;
            for (uint32_t e = 0; e < (uint32_t)KP; ++e) out[e] = e < cn ? ci[e * 128] : kNoId;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256u) : "memory");
}

// exact distances of the candidates -> top-k by (distance, id); one warp per query
__global__ void __launch_bounds__(128) cand_topk_kernel(const uint32_t* __restrict__ cand, const float* __restrict__ dist, uint32_t nq, uint32_t c,
                                                        uint32_t k, uint32_t* __restrict__ out_ids, float* __restrict__ out_d) {
    extern __shared__ uint8_t sm[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    float* sd = reinterpret_cast<float*>(sm) + (size_t)wib * c;
    uint32_t* si = reinterpret_cast<uint32_t*>(reinterpret_cast<float*>(sm) + (size_t)(blockDim.x >> 5) * c) + (size_t)wib * c;
    const uint32_t q = blockIdx.x * (blockDim.x >> 5) + wib;
    if (q >= nq) return;
    for (uint32_t i = lane; i < c; i += 32) {
        const uint32_t id = cand[(size_t)q * c + i];
        const float d = dist[(size_t)q * c + i];
        si[i] = id;
        sd[i] = (id == kNoId || d != d) ? __int_as_float(0x7F800000) : d;  // NaN never enters (flat_topk_kernel)
        if (id != kNoId && d != d) si[i] = kNoId;
    }
    __syncwarp();
    for (uint32_t r = 0; r < k; ++r) {
        float bd = __int_as_float(0x7F800000);
        uint32_t bi = kNoId, bp = 0xFFFFFFFFu;
        for (uint32_t i = lane; i < c; i += 32) {
            const float d = sd[i];
            const uint32_t id = si[i];
            if (id != kNoId && (d < bd || (d == bd && id < bi))) bd = d, bi = id, bp = i;
        }
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) {
            const float od = __shfl_xor_sync(0xFFFFFFFFu, bd, s);
            const uint32_t oi = __shfl_xor_sync(0xFFFFFFFFu, bi, s), op = __shfl_xor_sync(0xFFFFFFFFu, bp, s);
            if (oi != kNoId && (bi == kNoId || od < bd || (od == bd && oi < bi))) bd = od, bi = oi, bp = op;
        }
        if (lane == 0) {
            out_ids[(size_t)q * k + r] = bi;
            out_d[(size_t)q * k + r] = bi == kNoId ? __int_as_float(0x7F800000) : bd;
            if (bp != 0xFFFFFFFFu) si[bp] = kNoId;
        }
        __syncwarp();
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int make_map(CUtensorMap* map, void* base, uint64_t rows, uint32_t kp) {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess || !p)
            return fail(DAB_ERR_CUDA, "flat_tc: cuTensorMapEncodeTiled is not available from this driver");
        fn = (EncodeTiledFn)p;
    }
    const cuuint64_t dims[2] = {kp, rows};
    const cuuint64_t strides[1] = {(cuuint64_t)kp * 2};
    const cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)kBM};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(DAB_ERR_CUDA, "flat_tc: cuTensorMapEncodeTiled failed (%d)", (int)r);
    return DAB_OK;
}

template <typename... A>
void launch_prep(int dtype, int grid, cudaStream_t st, A... a) {
    switch (dtype) {
        case DAB_F32: prep_bf16_kernel<float><<<grid, 256, 0, st>>>(a...); break;
        case DAB_F16: prep_bf16_kernel<__half><<<grid, 256, 0, st>>>(a...); break;
        case DAB_I8: prep_bf16_kernel<int8_t><<<grid, 256, 0, st>>>(a...); break;
        default: prep_bf16_kernel<uint8_t><<<grid, 256, 0, st>>>(a...); break;
    }
}

}  // namespace

void tc_release(dab_index* idx) {
    cudaFree(idx->d_tc_base);
    cudaFree(idx->d_tc_coef);
    idx->d_tc_base = nullptr;
    idx->d_tc_coef = nullptr;
}

}  // namespace dab

using namespace dab;

extern "C" {

int dab_flat_knn_tc(dab_index* idx, const void* queries, uint32_t nq, uint32_t k, uint32_t* out_ids, float* out_dists) {
    if (!idx) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_flat_knn_tc: idx is NULL");
    if (!idx->vectors_ready) return fail(DAB_ERR_NOT_READY, "dab_flat_knn_tc: vectors not uploaded");
    if (nq == 0) return DAB_OK;
    if (!queries || !out_ids || !out_dists) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_flat_knn_tc: NULL argument");
    if (k == 0 || k + 8 > (uint32_t)kKP) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_flat_knn_tc: k must be in [1, %d] (use dab_flat_knn beyond)", kKP - 8);
    DAB_CUDA(cudaSetDevice(idx->device));
    cudaStream_t st = idx->stream;
    const bool is_int = idx->dtype == DAB_I8 || idx->dtype == DAB_U8;
    const uint32_t dim = idx->dim;
    const uint32_t kp = (uint32_t)round_up((size_t)(is_int ? dim : 3 * dim), kBK);
    const uint64_t n = idx->n_points;  // start points are not data
    const int score_kind = idx->metric == DAB_L2 ? 0 : idx->metric == DAB_COSINE ? 2 : (is_int && idx->metric == DAB_COSINE_NORMALIZED) ? 2 : 1;
    int rc;
    // base operand (bf16 split rows + score coefficients): built once per uploaded snapshot
    if (!idx->d_tc_base || idx->tc_version != idx->vectors_version) {
        tc_release(idx);
        DAB_CUDA(cudaMalloc(&idx->d_tc_base, n * (size_t)kp * 2));
        DAB_CUDA(cudaMalloc(&idx->d_tc_coef, n * 2 * sizeof(float)));
        launch_prep(idx->dtype, idx->sm_count * 8, st, (const uint8_t*)idx->d_vectors, idx->row_stride, n, dim, kp, 0, score_kind,
                    (__nv_bfloat16*)idx->d_tc_base, (float*)idx->d_tc_coef, (float*)idx->d_tc_coef + n);
        DAB_LAUNCHED();
        DAB_CUDA(cudaGetLastError());
        idx->tc_version = idx->vectors_version;
    }
    // queries: raw copy (exact re-scoring) + bf16 operand, padded to whole 128-row tiles
    const uint32_t m_tiles = (nq + kBM - 1) / kBM;
    const size_t qraw = (size_t)nq * dim * elem_size(idx->dtype);
    const size_t qop = (size_t)m_tiles * kBM * kp * 2;
    if ((rc = idx->s_queries.reserve(round_up(qraw, 256) + qop))) return rc;
    uint8_t* d_qraw = (uint8_t*)idx->s_queries.p;
    __nv_bfloat16* d_qop = (__nv_bfloat16*)(d_qraw + round_up(qraw, 256));
    DAB_CUDA(cudaMemcpyAsync(d_qraw, queries, qraw, cudaMemcpyHostToDevice, st));
    DAB_CUDA(cudaMemsetAsync(d_qop, 0, qop, st));
    launch_prep(idx->dtype, idx->sm_count * 4, st, (const uint8_t*)d_qraw, (size_t)dim * elem_size(idx->dtype), (uint64_t)nq, dim, kp, 1, score_kind,
                d_qop, (float*)nullptr, (float*)nullptr);
    DAB_LAUNCHED();
    // base ranges: enough CTAs to fill the machine, whole 128-column tiles each
    const uint32_t n_tiles = (uint32_t)((n + kBN - 1) / kBN);
    // (at most 48 ranges: the exact re-scoring handles splits x kKP candidates per query)
    uint32_t splits = std::max<uint32_t>(1, std::min<uint32_t>(std::min<uint32_t>(n_tiles, 48), (uint32_t)(idx->sm_count * 2 + m_tiles - 1) / m_tiles));
    const uint32_t tiles_per_split = (n_tiles + splits - 1) / splits;
    splits = (n_tiles + tiles_per_split - 1) / tiles_per_split;
    const uint32_t kp_sel = k <= 10 ? 16u : (uint32_t)kKP;  // per-range candidates: k plus slack for the approximate scores
    const uint32_t c = splits * kp_sel;
    if ((rc = idx->s_ids.reserve((size_t)nq * c * 4))) return rc;
    if ((rc = idx->s_out2.reserve((size_t)nq * c * 4))) return rc;
    if ((rc = idx->s_out.reserve((size_t)nq * k * 8))) return rc;
    CUtensorMap map_a, map_b;
    if ((rc = make_map(&map_a, d_qop, (uint64_t)m_tiles * kBM, kp))) return rc;
    if ((rc = make_map(&map_b, idx->d_tc_base, n, kp))) return rc;
    TcParams p;
    p.nq = nq;
    p.n_base = (uint32_t)n;
    p.kp = kp;
    p.tiles_per_split = tiles_per_split;
    p.n_splits = splits;
    p.alpha = (const float*)idx->d_tc_coef;
    p.beta = (const float*)idx->d_tc_coef + n;
    p.cand = (uint32_t*)idx->s_ids.p;
    const size_t tiles_smem = 2 * (size_t)kStages * kTileBytes;
    const size_t smem = 1024 + tiles_smem + 2 * 2 * kBN * 4 + 128 * 33 * 4 + 2 * (size_t)kp_sel * 128 * 4 + (2 * (size_t)kStages + 4) * 8 + 16;
#define DAB_TC_LAUNCH(KP_)                                                                                        \
    do {                                                                                                          \
        DAB_CUDA(cudaFuncSetAttribute(flat_tc_kernel<KP_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        flat_tc_kernel<KP_><<<dim3(splits, m_tiles), kTcThreads, smem, st>>>(map_a, map_b, p);                    \
    } while (0)
    if (kp_sel == 16) DAB_TC_LAUNCH(16);
    else DAB_TC_LAUNCH(32);
#undef DAB_TC_LAUNCH
    DAB_LAUNCHED();
    DAB_CUDA(cudaGetLastError());
    // exact distances of the candidates in the reference's SIMD order, then the final top-k
    if ((rc = launch_frontier(idx, d_qraw, nq, (const uint32_t*)idx->s_ids.p, c, (float*)idx->s_out2.p))) return rc;
    uint32_t* d_top_ids = (uint32_t*)idx->s_out.p;
    float* d_top_d = (float*)(d_top_ids + (size_t)nq * k);
    const size_t tsmem = (size_t)4 * c * 8;
    if (tsmem > 200 * 1024) return fail(DAB_ERR_INVALID_ARGUMENT, "dab_flat_knn_tc: %u candidates per query do not fit the selection kernel", c);
    DAB_CUDA(cudaFuncSetAttribute(cand_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsmem));
    cand_topk_kernel<<<(nq + 3) / 4, 128, tsmem, st>>>((const uint32_t*)idx->s_ids.p, (const float*)idx->s_out2.p, nq, c, k, d_top_ids, d_top_d);
    DAB_LAUNCHED();
    DAB_CUDA(cudaGetLastError());
    DAB_CUDA(cudaMemcpyAsync(out_ids, d_top_ids, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, st));
    DAB_CUDA(cudaMemcpyAsync(out_dists, d_top_d, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, st));
    DAB_CUDA(cudaStreamSynchronize(st));
    return DAB_OK;
}

}  // extern "C"
