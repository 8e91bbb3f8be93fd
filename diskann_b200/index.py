"""Host-side mirror of the reference interface for the distance hot path, over the C ABI.

Names follow the reference: `Metric` (diskann-vector/src/distance/metric.rs:8-20),
`distance_comparer` (distance_provider.rs:44-46), the provider-level snapshot
(`diskann_inmem::Provider`, diskann-inmem/src/provider.rs:71-131) and the batched
`KNN::search` (diskann-benchmark-core/src/search/graph/knn.rs:208-238).  All compute happens
in libdiskann_b200.so on the GPU; numpy is only the host container.
"""
import ctypes as C
import enum

import numpy as np

from . import _lib
from ._lib import DabError, check

__all__ = ["Metric", "DType", "GpuIndex", "distance_comparer", "pair_distances", "DabError", "launch_count"]


class Metric(enum.IntEnum):
    """#[repr(C)] values of diskann_vector::distance::Metric."""
    Cosine = 0
    InnerProduct = 1
    L2 = 2
    CosineNormalized = 3


class DType(enum.IntEnum):
    f32 = 0
    f16 = 1
    i8 = 2
    u8 = 3


_NP = {DType.f32: np.float32, DType.f16: np.float16, DType.i8: np.int8, DType.u8: np.uint8}


def dtype_of(arr):
    try:
        return {np.dtype(np.float32): DType.f32, np.dtype(np.float16): DType.f16,
                np.dtype(np.int8): DType.i8, np.dtype(np.uint8): DType.u8}[arr.dtype]
    except KeyError:
        raise DabError(1, f"unsupported element type {arr.dtype}") from None


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def launch_count():
    return int(_lib.lib().dab_launch_count())


def pair_distances(x, y, metric, device=0):
    """n independent distances x[i] . y[i] (Distance<T, U>::call for each pair)."""
    x = np.ascontiguousarray(x)
    y = np.ascontiguousarray(y)
    if x.ndim != 2 or y.ndim != 2 or x.shape != y.shape:
        raise DabError(1, f"expected two [n, dim] arrays of equal shape, got {x.shape} and {y.shape}")
    out = np.empty(x.shape[0], np.float32)
    check(_lib.lib().dab_pair_distances(int(dtype_of(x)), int(dtype_of(y)), int(metric), x.shape[1], _ptr(x), _ptr(y),
                                        x.shape[0], _ptr(out), device))
    return out


def distance_comparer(metric, dim=None, device=0):
    """T::distance_comparer(metric, Some(dim)) -> callable(x, y) -> f32.

    Length mismatches raise (the providers' DistanceFunction panics, implementations.rs:105-130;
    the inmem layer returns Err, layers/full.rs:203-213)."""

    def call(x, y):
        x = np.ascontiguousarray(x)
        y = np.ascontiguousarray(y)
        if x.ndim != 1 or x.shape != y.shape or (dim is not None and x.shape[0] != dim):
            raise DabError(1, f"expected slices of length {dim} - instead got {x.shape} and {y.shape}")
        return pair_distances(x[None, :], y[None, :], metric, device)[0]

    return call


def minmax_compress(vectors, nbits, grid_scale=1.0, device=0):
    """MinMaxQuantizer (Transform::Null) over the rows of `vectors` [n, dim] f32: (rows u8 [n, 20 + ceil(dim * nbits / 8)]
    in the reference's canonical-front Data<NBITS> layout, loss f32 [n]).  Raises DabError when a vector contains NaN."""
    vectors = np.ascontiguousarray(vectors, np.float32)
    if vectors.ndim != 2:
        raise DabError(1, "minmax_compress: vectors must be [n, dim] f32")
    n, dim = vectors.shape
    rb = _lib.lib().dab_minmax_row_bytes(dim, nbits)
    rows = np.zeros((n, rb), np.uint8)
    loss = np.zeros(n, np.float32)
    check(_lib.lib().dab_minmax_compress(device, grid_scale, dim, nbits, _ptr(vectors), n, _ptr(rows), _ptr(loss)))
    return rows, loss


def minmax_distances(metric, nbits_x, nbits_y, dim, x_rows, y_rows, device=0):
    """MinMax{L2Squared, IP, Cosine, CosineNormalized} between compressed rows: out[i] = d(x_rows[i], y_rows[i])."""
    x_rows = np.ascontiguousarray(x_rows, np.uint8)
    y_rows = np.ascontiguousarray(y_rows, np.uint8)
    n = x_rows.shape[0]
    out = np.empty(n, np.float32)
    check(_lib.lib().dab_minmax_distances(device, int(metric), nbits_x, nbits_y, dim, _ptr(x_rows), _ptr(y_rows), n, _ptr(out)))
    return out


def minmax_query_distances(metric, nbits, queries, rows, device=0):
    """Full-precision queries [nq, dim] f32 against MinMax-compressed rows [n, row_bytes]: out [nq, n]
    (MinMax{L2Squared, IP, Cosine, CosineNormalized}::evaluate(FullQueryRef, DataRef<NBITS>))."""
    queries = np.ascontiguousarray(queries, np.float32)
    rows = np.ascontiguousarray(rows, np.uint8)
    nq, dim = queries.shape
    out = np.empty((nq, rows.shape[0]), np.float32)
    check(_lib.lib().dab_minmax_query_distances(device, int(metric), nbits, dim, _ptr(queries), nq, _ptr(rows), rows.shape[0], _ptr(out)))
    return out


class GpuIndex:
    """Device-resident snapshot of an in-memory index: vectors + adjacency (+ PQ)."""

    def __init__(self, dtype, metric, dim, n_points, n_start=1, max_degree=83, device=0):
        self._h = C.c_void_p()
        self._inflight = {}  # slot -> (queries, outputs) kept alive while a batch is in flight
        self.dtype, self.metric, self.dim = DType(dtype), Metric(metric), int(dim)
        self.n_points, self.n_start, self.max_degree, self.device = int(n_points), int(n_start), int(max_degree), device
        check(_lib.lib().dab_create(C.byref(self._h), int(dtype), int(metric), dim, n_points, n_start, max_degree, device))

    # -- lifecycle
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            _lib.lib().dab_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def n_total(self):
        return self.n_points + self.n_start

    def set_stream(self, cuda_stream_ptr):
        check(_lib.lib().dab_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    # -- replication (one process per GPU): NCCL inside the library
    @staticmethod
    def comm_unique_id():
        buf = C.create_string_buffer(128)
        check(_lib.lib().dab_comm_unique_id(buf))
        return buf.raw

    def comm_init(self, unique_id, n_ranks, rank):
        check(_lib.lib().dab_comm_init(self._h, C.c_char_p(unique_id), n_ranks, rank))

    def broadcast_index(self, root=0):
        """One NCCL broadcast per resident buffer (vectors, adjacency, PQ) from `root` to every rank."""
        check(_lib.lib().dab_broadcast_index(self._h, root))

    # -- uploads
    def _rows(self, rows):
        rows = np.ascontiguousarray(rows)
        if rows.ndim != 2 or rows.shape[1] != self.dim or dtype_of(rows) != self.dtype:
            raise DabError(1, f"expected [n, {self.dim}] rows of {self.dtype.name}, got {rows.shape} {rows.dtype}")
        return rows

    def upload_vectors(self, rows, first=0):
        rows = self._rows(rows)
        check(_lib.lib().dab_upload_vectors(self._h, _ptr(rows), first, rows.shape[0]))

    def upload_vectors_device(self, dev_ptr, count, first=0):
        check(_lib.lib().dab_upload_vectors_device(self._h, C.c_void_p(dev_ptr), first, count))

    def upload_graph(self, adj, first=0):
        adj = np.ascontiguousarray(adj, dtype=np.uint32)
        if adj.ndim != 2:
            raise DabError(1, "adjacency must be [n, stride] u32 with row[0] = degree")
        check(_lib.lib().dab_upload_graph(self._h, _ptr(adj), adj.shape[1], first, adj.shape[0]))

    def upload_graph_device(self, dev_ptr, src_stride, count, first=0):
        check(_lib.lib().dab_upload_graph_device(self._h, C.c_void_p(dev_ptr), src_stride, first, count))

    def download_graph(self, first=0, count=None):
        count = self.n_total - first if count is None else count
        adj = np.zeros((count, self.max_degree + 1), np.uint32)
        check(_lib.lib().dab_download_graph(self._h, _ptr(adj), adj.shape[1], first, count))
        return adj

    def upload_pq(self, pivots, offsets, codes=None):
        pivots = np.ascontiguousarray(pivots, np.float32)
        offsets = np.ascontiguousarray(offsets, np.uint64)
        if pivots.ndim != 2 or pivots.shape[1] != self.dim:
            raise DabError(1, f"pivots must be [n_centers, {self.dim}] f32")
        if codes is not None:
            codes = np.ascontiguousarray(codes, np.uint8)
            if codes.shape != (self.n_total, len(offsets) - 1):
                raise DabError(1, f"codes must be [{self.n_total}, {len(offsets) - 1}] u8, got {codes.shape}")
        self.pq_chunks, self.pq_centers = len(offsets) - 1, pivots.shape[0]
        check(_lib.lib().dab_upload_pq(self._h, _ptr(pivots), pivots.shape[0], _ptr(offsets), len(offsets) - 1, _ptr(codes)))

    def pq_train(self, train, n_chunks, n_centers=256, lloyds_reps=5, seed=0):
        """train_pq on the device: k-means++ + Lloyd per chunk over host training rows [n, dim] f32."""
        train = np.ascontiguousarray(train, np.float32)
        if train.ndim != 2 or train.shape[1] != self.dim:
            raise DabError(1, f"training rows must be [n, {self.dim}] f32")
        check(_lib.lib().dab_pq_train(self._h, _ptr(train), train.shape[0], n_chunks, n_centers, lloyds_reps, seed))
        self.pq_chunks, self.pq_centers = n_chunks, n_centers

    def pq_encode_all(self):
        check(_lib.lib().dab_pq_encode_all(self._h))

    def download_pq(self, codes=True):
        """(pivots [n_centers, dim] f32, offsets u64 [n_chunks + 1], codes u8 [n_total, n_chunks] or None)."""
        pivots = np.empty((self.pq_centers, self.dim), np.float32)
        offsets = np.empty(self.pq_chunks + 1, np.uint64)
        c = np.empty((self.n_total, self.pq_chunks), np.uint8) if codes else None
        check(_lib.lib().dab_pq_download(self._h, _ptr(pivots), _ptr(offsets), _ptr(c)))
        return pivots, offsets, c

    # -- distances
    def _queries(self, queries):
        queries = np.ascontiguousarray(queries)
        if queries.ndim != 2 or queries.shape[1] != self.dim or dtype_of(queries) != self.dtype:
            raise DabError(1, f"expected [nq, {self.dim}] queries of {self.dtype.name}, got {queries.shape} {queries.dtype}")
        return queries

    def distances(self, queries, ids):
        """out[q][j] = QueryDistance(queries[q]).evaluate(row ids[q][j]) (expand_beam's distance stage)."""
        queries = self._queries(queries)
        ids = np.ascontiguousarray(ids, np.uint32)
        if ids.ndim != 2 or ids.shape[0] != queries.shape[0]:
            raise DabError(1, "ids must be [nq, c] u32")
        out = np.empty(ids.shape, np.float32)
        check(_lib.lib().dab_distances(self._h, _ptr(queries), queries.shape[0], _ptr(ids), ids.shape[1], _ptr(out)))
        return out

    def row_pair_distances(self, a, b):
        a = np.ascontiguousarray(a, np.uint32)
        b = np.ascontiguousarray(b, np.uint32)
        if a.shape != b.shape or a.ndim != 1:
            raise DabError(1, "a and b must be 1-d u32 arrays of equal length")
        out = np.empty(a.shape[0], np.float32)
        check(_lib.lib().dab_row_pair_distances(self._h, _ptr(a), _ptr(b), a.shape[0], _ptr(out)))
        return out

    def pairwise(self, ids):
        ids = np.ascontiguousarray(ids, np.uint32)
        out = np.empty((ids.shape[0], ids.shape[0]), np.float32)
        check(_lib.lib().dab_pairwise(self._h, _ptr(ids), ids.shape[0], _ptr(out)))
        return out

    # -- search
    def search_batch(self, queries, k, l_search, beam_width=1):
        """KNN::search for the whole batch: (ids [nq,k], dists [nq,k], counts, cmps, hops)."""
        queries = self._queries(queries)
        nq = queries.shape[0]
        ids = np.empty((nq, k), np.uint32)
        dists = np.empty((nq, k), np.float32)
        counts = np.empty(nq, np.uint32)
        cmps = np.empty(nq, np.uint32)
        hops = np.empty(nq, np.uint32)
        check(_lib.lib().dab_search_batch(self._h, _ptr(queries), nq, k, l_search, beam_width, _ptr(ids), _ptr(dists),
                                          _ptr(counts), _ptr(cmps), _ptr(hops)))
        return ids, dists, counts, cmps, hops

    def search_batch_device(self, d_queries, nq, k, l_search, beam_width, d_ids, d_dists, d_counts=0, d_cmps=0, d_hops=0):
        """Same with device pointers (integers); results stay in HBM."""
        check(_lib.lib().dab_search_batch_device(self._h, C.c_void_p(d_queries), nq, k, l_search, beam_width,
                                                 C.c_void_p(d_ids), C.c_void_p(d_dists), C.c_void_p(d_counts or None),
                                                 C.c_void_p(d_cmps or None), C.c_void_p(d_hops or None)))

    def search_batch_async(self, slot, queries, k, l_search, beam_width=1, out=None):
        """Queue a batch on `slot` (host buffers) and return its output arrays without waiting; they are
        valid after wait(slot).  `queries` is used as passed (it must stay alive and unchanged until then);
        `out` = (ids, dists, counts, cmps, hops) re-uses caller-owned (e.g. pinned) arrays."""
        nq = queries.shape[0]
        if out is None:
            out = (np.empty((nq, k), np.uint32), np.empty((nq, k), np.float32), np.empty(nq, np.uint32),
                   np.empty(nq, np.uint32), np.empty(nq, np.uint32))
        ids, dists, counts, cmps, hops = out
        check(_lib.lib().dab_search_batch_async(self._h, slot, _ptr(queries), nq, k, l_search, beam_width, _ptr(ids), _ptr(dists),
                                                _ptr(counts), _ptr(cmps), _ptr(hops)))
        self._inflight[slot] = (queries, out)
        return out

    def search_batch_device_async(self, slot, d_queries, nq, k, l_search, beam_width, d_ids, d_dists, d_counts=0, d_cmps=0, d_hops=0):
        """Device-pointer flavour of search_batch_async; results stay in HBM."""
        check(_lib.lib().dab_search_batch_device_async(self._h, slot, C.c_void_p(d_queries), nq, k, l_search, beam_width,
                                                       C.c_void_p(d_ids), C.c_void_p(d_dists), C.c_void_p(d_counts or None),
                                                       C.c_void_p(d_cmps or None), C.c_void_p(d_hops or None)))

    def wait(self, slot):
        """Join the batch in flight on `slot` (no-op when idle)."""
        check(_lib.lib().dab_wait(self._h, slot))
        return self._inflight.pop(slot, (None, None))[1]

    # -- PQ
    def pq_populate_lut(self, queries, metric=None):
        queries = np.ascontiguousarray(queries, np.float32)
        out = np.empty((queries.shape[0], self.pq_chunks, self.pq_centers), np.float32)
        check(_lib.lib().dab_pq_populate_lut(self._h, _ptr(queries), queries.shape[0],
                                             int(self.metric if metric is None else metric), _ptr(out)))
        return out

    def pq_distances(self, queries, ids):
        queries = np.ascontiguousarray(queries, np.float32)
        ids = np.ascontiguousarray(ids, np.uint32)
        out = np.empty(ids.shape, np.float32)
        check(_lib.lib().dab_pq_distances(self._h, _ptr(queries), queries.shape[0], _ptr(ids), ids.shape[1], _ptr(out)))
        return out

    def search_batch_pq(self, queries, k, l_search, beam_width=1, rerank=False):
        """KNN::search with PQ ADC traversal distances (providers' QuantAccessor); rerank=True adds the
        providers' full-precision Rerank post-processing."""
        queries = self._queries(queries)
        nq = queries.shape[0]
        ids = np.empty((nq, k), np.uint32)
        dists = np.empty((nq, k), np.float32)
        counts = np.empty(nq, np.uint32)
        cmps = np.empty(nq, np.uint32)
        hops = np.empty(nq, np.uint32)
        fn = _lib.lib().dab_search_batch_pq_rerank if rerank else _lib.lib().dab_search_batch_pq
        check(fn(self._h, _ptr(queries), nq, k, l_search, beam_width, _ptr(ids), _ptr(dists), _ptr(counts), _ptr(cmps), _ptr(hops)))
        return ids, dists, counts, cmps, hops

    def search_batch_pq_device(self, d_queries, nq, k, l_search, beam_width, d_ids, d_dists, d_counts=0, d_cmps=0, d_hops=0,
                               rerank=True):
        """Same with device pointers (integers); results stay in HBM."""
        check(_lib.lib().dab_search_batch_pq_device(self._h, C.c_void_p(d_queries), nq, k, l_search, beam_width, int(bool(rerank)),
                                                    C.c_void_p(d_ids), C.c_void_p(d_dists), C.c_void_p(d_counts or None),
                                                    C.c_void_p(d_cmps or None), C.c_void_p(d_hops or None)))

    def pq_self_distances(self, a, b):
        """DistanceComputer over two stored codes (the PQ prune path): out[i] = d(code[a[i]], code[b[i]])."""
        a = np.ascontiguousarray(a, np.uint32)
        b = np.ascontiguousarray(b, np.uint32)
        if a.shape != b.shape or a.ndim != 1:
            raise DabError(1, "a and b must be 1-d u32 arrays of equal length")
        out = np.empty(a.shape[0], np.float32)
        check(_lib.lib().dab_pq_self_distances(self._h, _ptr(a), _ptr(b), a.shape[0], _ptr(out)))
        return out

    # -- scalar-quantized store
    def upload_sq(self, nbits, shift, scale, shift_square_norm, mean_norm=0.0, rows=None):
        """SQStore<NBITS>: the quantizer and (optionally) the canonical-front rows
        (f32 compensation | dense N-bit codes) of every point including the start points."""
        shift = np.ascontiguousarray(shift, np.float32)
        if shift.shape != (self.dim,):
            raise DabError(1, "shift must have dim entries")
        row_bytes = 4 + (self.dim * nbits + 7) // 8
        if rows is not None:
            rows = np.ascontiguousarray(rows, np.uint8)
            if rows.shape != (self.n_points + self.n_start, row_bytes):
                raise DabError(1, "rows must be (n_points + n_start) x (4 + ceil(dim * nbits / 8)) bytes")
        check(_lib.lib().dab_upload_sq(self._h, int(nbits), _ptr(shift), float(scale), float(shift_square_norm),
                                       float(mean_norm), _ptr(rows) if rows is not None else None))
        self.sq_nbits = int(nbits)

    def sq_encode_all(self):
        check(_lib.lib().dab_sq_encode_all(self._h))

    def download_sq(self):
        rows = np.empty((self.n_points + self.n_start, 4 + (self.dim * self.sq_nbits + 7) // 8), np.uint8)
        check(_lib.lib().dab_sq_download(self._h, _ptr(rows)))
        return rows

    def search_batch_sq(self, queries, k, l_search, beam_width=1, rerank=False):
        """KNN::search through the scalar-quantized accessor; rerank=True adds the full-precision Rerank."""
        queries = self._queries(queries)
        nq = queries.shape[0]
        ids = np.empty((nq, k), np.uint32)
        dists = np.empty((nq, k), np.float32)
        counts = np.empty(nq, np.uint32)
        cmps = np.empty(nq, np.uint32)
        hops = np.empty(nq, np.uint32)
        check(_lib.lib().dab_search_batch_sq(self._h, _ptr(queries), nq, k, l_search, beam_width, int(bool(rerank)),
                                             _ptr(ids), _ptr(dists), _ptr(counts), _ptr(cmps), _ptr(hops)))
        return ids, dists, counts, cmps, hops

    def search_batch_sq_device(self, d_queries, nq, k, l_search, beam_width, d_ids, d_dists, d_counts=0, d_cmps=0, d_hops=0,
                               rerank=True):
        check(_lib.lib().dab_search_batch_sq_device(self._h, C.c_void_p(d_queries), nq, k, l_search, beam_width, int(bool(rerank)),
                                                    C.c_void_p(d_ids), C.c_void_p(d_dists), C.c_void_p(d_counts or None),
                                                    C.c_void_p(d_cmps or None), C.c_void_p(d_hops or None)))

    def pq_encode(self, vectors):
        vectors = np.ascontiguousarray(vectors, np.float32)
        out = np.empty((vectors.shape[0], self.pq_chunks), np.uint8)
        check(_lib.lib().dab_pq_encode(self._h, _ptr(vectors), vectors.shape[0], _ptr(out)))
        return out

    # -- build-side reuse / ground truth
    def robust_prune(self, pool_ids, pool_dists, pool_lens, locations, degree, alpha=1.2):
        """robust_prune for a batch of pools -> (ids [n_pools, degree] padded UINT32_MAX, counts)."""
        pool_ids = np.ascontiguousarray(pool_ids, np.uint32)
        pool_dists = np.ascontiguousarray(pool_dists, np.float32)
        pool_lens = np.ascontiguousarray(pool_lens, np.uint32)
        locations = np.ascontiguousarray(locations, np.uint32)
        if pool_ids.ndim != 2 or pool_ids.shape != pool_dists.shape or pool_lens.shape != (pool_ids.shape[0],) \
                or locations.shape != pool_lens.shape:
            raise DabError(1, "robust_prune: expected pool_ids/pool_dists [n_pools, cap], pool_lens/locations [n_pools]")
        out = np.empty((pool_ids.shape[0], degree), np.uint32)
        counts = np.empty(pool_ids.shape[0], np.uint32)
        check(_lib.lib().dab_robust_prune(self._h, _ptr(pool_ids), _ptr(pool_dists), _ptr(pool_lens), _ptr(locations),
                                          pool_ids.shape[0], pool_ids.shape[1], degree, alpha, _ptr(out), _ptr(counts)))
        return out, counts

    def build(self, pruned_degree, l_build, alpha=1.2, batch_size=0):
        check(_lib.lib().dab_build(self._h, pruned_degree, l_build, alpha, batch_size))

    def flat_knn(self, queries, k):
        queries = self._queries(queries)
        ids = np.empty((queries.shape[0], k), np.uint32)
        dists = np.empty((queries.shape[0], k), np.float32)
        check(_lib.lib().dab_flat_knn(self._h, _ptr(queries), queries.shape[0], k, _ptr(ids), _ptr(dists)))
        return ids, dists

    def flat_knn_tc(self, queries, k):
        """The exhaustive scan as a tcgen05 GEMM with fused candidate selection + exact re-scoring."""
        queries = self._queries(queries)
        ids = np.empty((queries.shape[0], k), np.uint32)
        dists = np.empty((queries.shape[0], k), np.float32)
        check(_lib.lib().dab_flat_knn_tc(self._h, _ptr(queries), queries.shape[0], k, _ptr(ids), _ptr(dists)))
        return ids, dists
