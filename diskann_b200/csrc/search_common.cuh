// search_common.cuh — device helpers shared by the warp-per-query search kernels: the exact
// bucketed visited set and the batched rank-merge of the sorted candidate list.
#pragma once

#include "distance_device.cuh"

namespace dab {

constexpr uint32_t kEmptyV2 = 0xFFFFFFFFu;
constexpr uint32_t kFlagV2 = 0x80000000u;

__device__ __forceinline__ uint32_t bucket_of(uint32_t id, uint32_t n_buckets) { return __umulhi(id * 0x9E3779B1u, n_buckets); }

// ---- shared-memory sorted list with batched, rank-based merges ------------------------------
// NeighborPriorityQueue::insert (queue.rs:130-171) applied to a whole round of candidates at
// once.  Sequential lower-bound insertion with eviction of the tail is the same as keeping the
// `cap` smallest elements under the total order (distance ascending, later-inserted first among
// equal distances): a rejected / evicted element had >= cap elements ahead of it and can never
// re-enter.  So each candidate's final index is
//     #old(d < x) + #new((d_i < x) or (d_i == x and i later)),
// each old entry moves right by #new(d_i <= d_old), and everything landing at >= cap is dropped.
// NaN candidates are ignored; a full list pre-rejects `worst < x` exactly like the reference.

// first unvisited index in [from, lim), or lim
__device__ __forceinline__ uint32_t first_unvisited(const uint32_t* qi, uint32_t from, uint32_t lim, int lane) {
    for (uint32_t b = from & ~31u; b < lim; b += 32) {
        const uint32_t i = b + lane;
        const bool u = i >= from && i < lim && !(qi[i] & kFlagV2);
        const unsigned m = __ballot_sync(kFull, u);
        if (m) return b + __ffs(m) - 1;
    }
    return lim;
}

// merge candidates c0 .. c0+m-1 (m <= 32; lane j owns candidate j) into the list
template <int QT>
__device__ __forceinline__ void merge_round(float* qd, uint32_t* qi, uint32_t cap, uint32_t& size, uint32_t& cursor_lo,
                                            const uint32_t* cid, const float* cd, uint32_t c0, uint32_t m, int lane) {
    const uint32_t j = (uint32_t)lane;
    const float dj = j < m ? cd[c0 + j] : __int_as_float(0x7FC00000);
    const uint32_t idj = j < m ? cid[c0 + j] : 0;
    const float worst = size == cap ? qd[cap - 1] : __int_as_float(0x7F800000);
    const bool valid = j < m && dj == dj && !(worst < dj);
    const unsigned vm = __ballot_sync(kFull, valid);
    if (!vm) return;
    // lower bound among the old entries
    uint32_t lo = 0, hi = size;
    while (__any_sync(kFull, lo < hi)) {
        const uint32_t mid = (lo + hi) >> 1;
        if (lo < hi) {
            if (qd[mid] < dj) lo = mid + 1;
            else hi = mid;
        }
    }
    // old entries into registers (striped: entry t*32 + lane)
    float od[QT];
    uint32_t oi[QT], sh[QT];
#pragma unroll
    for (int t = 0; t < QT; ++t) {
        const uint32_t e = (uint32_t)t * 32 + lane;
        od[t] = e < size ? qd[e] : __int_as_float(0x7F800000);
        oi[t] = e < size ? qi[e] : kEmptyV2;
        sh[t] = 0;
    }
    uint32_t rn = 0;
    unsigned it = vm;
    while (it) {
        const int i = __ffs(it) - 1;
        it &= it - 1;
        const float di = __shfl_sync(kFull, dj, i);
        rn += (di < dj || (di == dj && (uint32_t)i > j)) ? 1u : 0u;
#pragma unroll
        for (int t = 0; t < QT; ++t) sh[t] += di <= od[t] ? 1u : 0u;
    }
    const uint32_t pos = lo + rn;
    const bool keep_new = valid && pos < cap;
    __syncwarp();
#pragma unroll
    for (int t = 0; t < QT; ++t) {
        const uint32_t e = (uint32_t)t * 32 + lane;
        const uint32_t ne = e + sh[t];
        if (e < size && sh[t] != 0 && ne < cap) {
            qd[ne] = od[t];
            qi[ne] = oi[t];
        }
    }
    if (keep_new) {
        qd[pos] = dj;
        qi[pos] = idj;
    }
    size = min(cap, size + (uint32_t)__popc(vm));
    cursor_lo = min(cursor_lo, __reduce_min_sync(kFull, keep_new ? pos : 0xFFFFFFFFu));
    __syncwarp();
}

// The same merge for lists longer than one register tile (QT * 32 entries): the list is walked in CH tiles from the top
// one down.  Entries only move right, by sh = #new(d_i <= d_old), which does not decrease along the sorted list, and
// final positions are unique — so a tile's writes (all at or above its own first entry) never touch an entry a lower
// tile still has to read, and what a lower tile writes above its own range are final positions no upper entry owns.
template <int QT, int CH>
__device__ __forceinline__ void merge_round_chunked(float* qd, uint32_t* qi, uint32_t cap, uint32_t& size, uint32_t& cursor_lo,
                                                    const uint32_t* cid, const float* cd, uint32_t c0, uint32_t m, int lane) {
    const uint32_t j = (uint32_t)lane;
    const float dj = j < m ? cd[c0 + j] : __int_as_float(0x7FC00000);
    const uint32_t idj = j < m ? cid[c0 + j] : 0;
    const float worst = size == cap ? qd[cap - 1] : __int_as_float(0x7F800000);
    const bool valid = j < m && dj == dj && !(worst < dj);
    const unsigned vm = __ballot_sync(kFull, valid);
    if (!vm) return;
    uint32_t lo = 0, hi = size;
    while (__any_sync(kFull, lo < hi)) {
        const uint32_t mid = (lo + hi) >> 1;
        if (lo < hi) {
            if (qd[mid] < dj) lo = mid + 1;
            else hi = mid;
        }
    }
    uint32_t rn = 0;
    for (unsigned it = vm; it;) {
        const int i = __ffs(it) - 1;
        it &= it - 1;
        const float di = __shfl_sync(kFull, dj, i);
        rn += (di < dj || (di == dj && (uint32_t)i > j)) ? 1u : 0u;
    }
    const uint32_t pos = lo + rn;
    const bool keep_new = valid && pos < cap;
    __syncwarp();
#pragma unroll 1
    for (int c = CH - 1; c >= 0; --c) {
        const uint32_t e0 = (uint32_t)c * QT * 32;
        if (e0 >= size) continue;  // nothing stored in this tile yet (warp-uniform)
        float od[QT];
        uint32_t oi[QT], sh[QT];
#pragma unroll
        for (int t = 0; t < QT; ++t) {
            const uint32_t e = e0 + (uint32_t)t * 32 + lane;
            od[t] = e < size ? qd[e] : __int_as_float(0x7F800000);
            oi[t] = e < size ? qi[e] : kEmptyV2;
            sh[t] = 0;
        }
        for (unsigned it = vm; it;) {
            const int i = __ffs(it) - 1;
            it &= it - 1;
            const float di = __shfl_sync(kFull, dj, i);
#pragma unroll
            for (int t = 0; t < QT; ++t) sh[t] += di <= od[t] ? 1u : 0u;
        }
        __syncwarp();  // every lane holds its entries of the tile before any of them is overwritten
#pragma unroll
        for (int t = 0; t < QT; ++t) {
            const uint32_t e = e0 + (uint32_t)t * 32 + lane;
            const uint32_t ne = e + sh[t];
            if (e < size && sh[t] != 0 && ne < cap) {
                qd[ne] = od[t];
                qi[ne] = oi[t];
            }
        }
        __syncwarp();
    }
    if (keep_new) {
        qd[pos] = dj;
        qi[pos] = idj;
    }
    size = min(cap, size + (uint32_t)__popc(vm));
    cursor_lo = min(cursor_lo, __reduce_min_sync(kFull, keep_new ? pos : 0xFFFFFFFFu));
    __syncwarp();
}

// QT = 4 / 8 / 16: one register tile covers the list (<= 128 / 256 / 512 entries); QT = 32: two tiles of 16 (<= 1024)
template <int QT>
__device__ __forceinline__ void merge_any(float* qd, uint32_t* qi, uint32_t cap, uint32_t& size, uint32_t& cursor_lo, const uint32_t* cid,
                                          const float* cd, uint32_t c0, uint32_t m, int lane) {
    if constexpr (QT == 32) merge_round_chunked<16, 2>(qd, qi, cap, size, cursor_lo, cid, cd, c0, m, lane);
    else merge_round<QT>(qd, qi, cap, size, cursor_lo, cid, cd, c0, m, lane);
}

// ---- exact visited set: bucketed open addressing, 8 ids per 32-byte bucket ------------------
// The tables are the only data of a search that is re-read (every hop probes ~R buckets of the
// same 10-20 KB per-query table) while ~0.6 MB of vector rows stream past per query.  Bucket
// loads therefore carry the L2 evict_last priority (one 256-bit coherent load per bucket) and
// the row copies evict_first (search_kernel_v2.cu), so the streaming rows do not push the
// tables out of L2 and every probe is an L2 hit instead of a DRAM sector.
__device__ __forceinline__ void load_bucket(const uint32_t* bp, uint32_t (&s)[8]) {
    asm volatile("ld.relaxed.gpu.global.L2::evict_last.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(s[0]), "=r"(s[1]), "=r"(s[2]), "=r"(s[3]), "=r"(s[4]), "=r"(s[5]), "=r"(s[6]), "=r"(s[7])
                 : "l"(bp));
}

// table-clear store of one 32-byte bucket, same priority as the probes
__device__ __forceinline__ void store_empty_bucket(uint32_t* bp) {
    asm volatile("st.global.L2::evict_last.v8.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1};" ::"l"(bp), "r"(kEmptyV2) : "memory");
}

// One probe = one 32 B sector: returns true when `id` was newly inserted (HashSet::insert).
// `s` holds the bucket's words as loaded by load_bucket(table + b * 8).
__device__ __forceinline__ bool bucket_insert(uint32_t* table, uint32_t n_buckets, uint32_t b, uint32_t (&s)[8], uint32_t id) {
    // (the callers stop inserting at 87.5 % load, so a free slot always exists; the probe bound only
    // guarantees that a completely full table can never hang the device)
    for (uint32_t advanced = 0;;) {
        bool found = false;
        int empty = -1;
#pragma unroll
        for (int k = 7; k >= 0; --k) {
            found |= s[k] == id;
            if (s[k] == kEmptyV2) empty = k;
        }
        if (found) return false;
        uint32_t* bp = table + (size_t)b * 8;
        if (empty >= 0) {
            const uint32_t old = atomicCAS(bp + empty, kEmptyV2, id);
            if (old == kEmptyV2) return true;
            if (old == id) return false;
            // another lane of this warp took the slot: re-read the bucket
        } else {
            if (++advanced > n_buckets) return false;
            b = b + 1 == n_buckets ? 0 : b + 1;
            bp = table + (size_t)b * 8;
        }
        load_bucket(bp, s);
    }
}

// ---- 16-bit quotient tags (the shared-memory visited tables of search_kernel_v3, search_smem.cuh) ----
// A table of 16-bit entries holds twice the ids per byte without giving up exactness.  Ids < 2^K are hashed with an odd
// multiplier modulo 2^K (a bijection), h = tag * n_buckets + bucket, so (bucket, tag) identifies
// the id and only the tag (< 2^K / n_buckets + 1 <= 2^14) is stored: 16 entries per 32-byte
// bucket.  An entry displaced to the d-th following bucket (d <= 2) carries d in its top two
// bits, which keeps it distinct from the entries at home there; 0xFFFF is the empty marker.
struct Tag16Map {
    uint32_t kmask;   // 2^K - 1, K = bits of the largest id
    uint32_t nbk;     // buckets per table
    uint32_t magic;   // ceil(2^(K+s) / nbk), s = ceil(log2 nbk): exact h / nbk for h < 2^K
    uint32_t shift;   // K + s
};

__device__ __forceinline__ void tag16_of(uint32_t id, const Tag16Map& m, uint32_t& bucket, uint32_t& tag) {
    const uint32_t h = (id * 0x9E3779B1u) & m.kmask;
    tag = (uint32_t)(((uint64_t)h * m.magic) >> m.shift);  // h / nbk
    bucket = h - tag * m.nbk;                              // h % nbk
}


// Probe of a shared-memory tag table (same layout and rules as smem16_insert, search_smem.cuh: 16 tags per
// 32-byte bucket, slots fill upwards, an entry displaced to the d-th following bucket (d <= 2) carries d in
// its top two bits, 0xFFFF = empty).  Returns 0: the id is in the table; 1: it was absent and has been
// inserted; 2: it is absent and was not inserted (`allow_insert` false, or its three buckets are full).
__device__ __forceinline__ int tag16_probe(uint32_t* table, uint32_t n_buckets, uint32_t b, uint32_t tag, bool allow_insert) {
    uint32_t d = 0;
    for (;;) {
        uint32_t* bp = table + (size_t)b * 8;
        const uint4 lo = reinterpret_cast<const uint4*>(bp)[0];
        const uint4 hi = reinterpret_cast<const uint4*>(bp)[1];
        const uint32_t s[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
        const uint32_t want = (d << 14) | tag, want2 = want * 0x10001u;
        // "some 16-bit half of x is zero" <=> ((x - 0x00010001) & ~x & 0x80008000) != 0
        uint32_t hit = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const uint32_t x = s[k] ^ want2;
            hit |= (x - 0x00010001u) & ~x & 0x80008000u;
        }
        if (hit) return 0;
        // first word with a free (upper) half: slots fill in order
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
            if (!allow_insert) return 2;
            const uint32_t neu = (old & 0xFFFFu) == 0xFFFFu ? (0xFFFF0000u | want) : ((old & 0xFFFFu) | (want << 16));
            if (atomicCAS(bp + ew, old, neu) == old) return 1;
            continue;  // another lane of this warp changed the word: look at the bucket again
        }
        if (++d > 2) return 2;
        b = b + 1 == n_buckets ? 0 : b + 1;
    }
}

}  // namespace dab
