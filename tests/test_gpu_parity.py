"""GPU parity tests: the CUDA path through the C ABI against the CPU oracle on the same seeded
inputs.  Bar: bit-exact for every path (integer, PQ, and — because the kernels reproduce the
reference's SIMD summation order — floating point too)."""
import json
import math
import os

import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
METRICS = [O.L2, O.INNER_PRODUCT, O.COSINE, O.COSINE_NORMALIZED]
PAIRS = [(np.float32, np.float32), (np.float16, np.float16), (np.float32, np.float16),
         (np.int8, np.int8), (np.uint8, np.uint8)]


@pytest.fixture(scope="module")
def dab():
    import diskann_b200
    diskann_b200.lib()
    return diskann_b200


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def same_bits(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return np.array_equal(bits(a)[~(np.isnan(a) & np.isnan(b))], bits(b)[~(np.isnan(a) & np.isnan(b))]) and \
        np.array_equal(np.isnan(a), np.isnan(b))


def fuzz(rng, dt, shape):
    if dt in (np.float32, np.float16):
        return rng.normal(0.0, 1.0, shape).astype(dt)
    info = np.iinfo(dt)
    return rng.integers(info.min, info.max + 1, shape).astype(dt)


def corner(dt):
    if dt in (np.float32, np.float16):
        return [0.0, -5.0, 5.0, 10.0]
    return [-128, 127, 0] if dt == np.int8 else [0, 255, 0]


def clustered(rng, n, d, n_centers=32, spread=0.3):
    centers = rng.normal(size=(n_centers, d)).astype(np.float32)
    return (centers[rng.integers(0, n_centers, n)] + spread * rng.normal(size=(n, d))).astype(np.float32)


# ---------------------------------------------------------------- per-pair distances

def test_kat_l2_through_the_c_abi(dab):
    g = json.load(open(os.path.join(GOLDEN, "kat_l2_f32_256.json")))
    v = np.array(g["values"], np.float32)
    out = dab.pair_distances(v[None, :256], v[None, 256:], dab.Metric.L2)
    assert out[0] == np.float32(g["expected"])  # 429141.2 exactly, distance_provider.rs:744-828
    f = dab.distance_comparer(dab.Metric.L2, 256)
    assert f(v[:256], v[256:]) == np.float32(g["expected"])


@pytest.mark.parametrize("dl,dr", PAIRS)
def test_pair_distances_bit_exact_all_dims(dab, dl, dr):
    """The reference's sweep (distance_provider.rs:551-606): every dim 0..64 + the specialised
    and ragged sizes, corner broadcasts + fuzz, 4 metrics."""
    rng = np.random.default_rng(1234)
    for dim in list(range(1, 66)) + [95, 96, 97, 100, 127, 128, 129, 160, 255, 256, 384, 768, 1000]:
        xs = [np.full(dim, a, dl) for a in corner(dl) for _ in corner(dr)]
        ys = [np.full(dim, b, dr) for _ in corner(dl) for b in corner(dr)]
        xs += [fuzz(rng, dl, dim) for _ in range(7)]
        ys += [fuzz(rng, dr, dim) for _ in range(7)]
        x, y = np.stack(xs), np.stack(ys)
        for metric in METRICS:
            got = dab.pair_distances(x, y, metric)
            want = np.array([O.distance(a, b, metric, O.SIMD) for a, b in zip(x, y)], np.float32)
            assert same_bits(got, want), (dim, metric, got, want)


def test_pair_distances_special_values(dab):
    a = np.full((1, 384), np.inf, np.float16)
    assert math.isnan(dab.pair_distances(a, a, dab.Metric.L2)[0])  # distance_provider.rs:970-977
    z = np.zeros((1, 37), np.float32)
    o = np.ones((1, 37), np.float32)
    assert dab.pair_distances(z, o, dab.Metric.Cosine)[0] == np.float32(1.0)  # zero norm -> similarity 0
    # i32 accumulators hold the extreme broadcasts exactly
    x = np.full((1, 256), -128, np.int8)
    y = np.full((1, 256), 127, np.int8)
    assert dab.pair_distances(x, y, dab.Metric.L2)[0] == np.float32(255 * 255 * 256)
    u = np.full((1, 256), 255, np.uint8)
    assert dab.pair_distances(u, u, dab.Metric.InnerProduct)[0] == np.float32(-255 * 255 * 256)


def test_error_behaviour_matches_the_layer(dab):
    # layers/full.rs:203-213, 306-314: length / type mismatch is an error, never a crash
    with pytest.raises(dab.DabError):
        dab.pair_distances(np.zeros((2, 4), np.float32), np.zeros((2, 5), np.float32), dab.Metric.L2)
    with pytest.raises(dab.DabError):
        dab.pair_distances(np.zeros((2, 4), np.int8), np.zeros((2, 4), np.uint8), dab.Metric.L2)
    with pytest.raises(dab.DabError):
        dab.pair_distances(np.zeros((2, 4), np.float64), np.zeros((2, 4), np.float64), dab.Metric.L2)
    assert dab.pair_distances(np.zeros((0, 4), np.float32), np.zeros((0, 4), np.float32), dab.Metric.L2).shape == (0,)
    with dab.GpuIndex(dab.DType.f32, dab.Metric.L2, 8, 10, 1, 4) as g:
        with pytest.raises(dab.DabError):
            g.upload_vectors(np.zeros((3, 7), np.float32))
        with pytest.raises(dab.DabError):
            g.upload_vectors(np.zeros((12, 8), np.float32))  # more rows than the index holds
        with pytest.raises(dab.DabError) as e:
            g.search_batch(np.zeros((1, 8), np.float32), 1, 4)
        assert e.value.code == 5  # DAB_ERR_NOT_READY
        bad = np.zeros((11, 5), np.uint32)
        bad[0, 0] = 9  # degree > max_degree
        with pytest.raises(dab.DabError):
            g.upload_graph(bad)


# ---------------------------------------------------------------- frontier distances (K1/K5 + K10)

@pytest.mark.parametrize("dt,metric,dim", [
    (np.float32, O.L2, 128), (np.float32, O.L2, 100), (np.float32, O.L2, 96), (np.float32, O.COSINE, 37),
    (np.float16, O.INNER_PRODUCT, 768), (np.float16, O.L2, 100), (np.float16, O.COSINE_NORMALIZED, 64),
    (np.int8, O.L2, 128), (np.int8, O.INNER_PRODUCT, 100), (np.uint8, O.L2, 128), (np.uint8, O.COSINE, 33),
    # wide-load kernel corners: fewer than four 8-blocks, no full block at all, leftover blocks + tail
    (np.float32, O.INNER_PRODUCT, 17), (np.float16, O.L2, 7), (np.float32, O.COSINE_NORMALIZED, 43), (np.float16, O.INNER_PRODUCT, 61),
])
def test_frontier_distances_bit_exact(dab, dt, metric, dim):
    rng = np.random.default_rng(dim * 7 + metric)
    n, nq, c = 3000, 40, 83
    base = fuzz(rng, dt, (n + 1, dim))
    queries = fuzz(rng, dt, (nq, dim))
    ids = rng.integers(0, n + 1, (nq, c)).astype(np.uint32)
    ids[0, 3] = 0xFFFFFFFF          # skipped slot
    ids[1, :] = 0xFFFFFFFF          # empty (ragged) list
    ids[2, 5] = n + 5               # out of bounds
    with dab.GpuIndex(O.dtype_code(base), metric, dim, n, 1, 8) as g:
        g.upload_vectors(base)
        got = g.distances(queries, ids)
        pa = rng.integers(0, n, 500).astype(np.uint32)
        pb = rng.integers(0, n, 500).astype(np.uint32)
        got_pairs = g.row_pair_distances(pa, pb)
        sub = rng.integers(0, n, 17).astype(np.uint32)
        got_block = g.pairwise(sub)
    for qi in range(nq):
        q = queries[qi].astype(np.float32) if dt == np.float16 else queries[qi]  # layers/full.rs:421-423
        valid = ids[qi] <= n
        want = O.distance_rows(q, base[np.where(valid, ids[qi], 0)], metric)
        assert same_bits(got[qi][valid], want[valid]), (qi,)
        assert np.isnan(got[qi][~valid]).all()
    want_pairs = np.array([O.distance(base[a], base[b], metric) for a, b in zip(pa, pb)], np.float32)
    assert same_bits(got_pairs, want_pairs)
    want_block = np.array([[O.distance(base[a], base[b], metric) for b in sub] for a in sub], np.float32)
    assert same_bits(got_block, want_block)


# ---------------------------------------------------------------- greedy search

def test_grid_search_baselines_on_gpu(dab):
    """The reference's checked-in greedy-search baselines
    (diskann/test/generated/graph/test/cases/grid_search/*.json) through dab_search_batch."""
    from test_oracle_golden import grid
    g = json.load(open(os.path.join(GOLDEN, "grid_search.json")))
    for case in g["cases"]:
        data, adj, n = grid(case["grid_dims"], case["grid_size"])
        with dab.GpuIndex(dab.DType.f32, dab.Metric.L2, data.shape[1], n, 1, adj.shape[1] - 1) as gi:
            gi.upload_vectors(data)
            gi.upload_graph(adj)
            ids, dists, counts, cmps, hops = gi.search_batch(np.array([case["query"]], np.float32), 10, 10,
                                                             case["beam_width"])
        assert counts[0] == case["num_results"] and cmps[0] == case["comparisons"] and hops[0] == case["hops"], case
        want = case["results"][:case["num_results"]]
        assert [int(i) for i in ids[0][:counts[0]]] == [r[0] for r in want], case
        assert [float(d) for d in dists[0][:counts[0]]] == [r[1] for r in want], case


def make_index(rng, dt, metric, n, d, R, L_build):
    base = clustered(rng, n, d)
    if dt == np.float16:
        base = (base / np.linalg.norm(base, axis=1, keepdims=True)).astype(np.float16)
    elif dt == np.int8:
        base = np.clip(np.round(base * 40), -127, 127).astype(np.int8)
    elif dt == np.uint8:
        base = np.clip(np.round(base * 40 + 128), 0, 255).astype(np.uint8)
    mean = base.astype(np.float32).mean(0)
    medoid = base[np.argmin(((base.astype(np.float32) - mean) ** 2).sum(1))]
    vecs = np.concatenate([base, medoid[None]])
    maxdeg = int(R * 1.3)
    adj = O.build_graph(vecs, n, 1, metric, R, maxdeg, L_build)
    return vecs, adj, maxdeg


SEARCH_CASES = [
    (np.float32, O.L2, 128, 6000, 32, 50),
    (np.float32, O.L2, 100, 3000, 16, 30),
    (np.float32, O.COSINE, 48, 3000, 16, 30),
    (np.float16, O.INNER_PRODUCT, 96, 3000, 16, 30),
    (np.float16, O.L2, 64, 3000, 16, 30),
    (np.int8, O.L2, 128, 4000, 24, 40),
    (np.uint8, O.L2, 128, 3000, 16, 30),
    (np.uint8, O.COSINE, 40, 2000, 16, 30),
]


@pytest.mark.parametrize("dt,metric,d,n,R,Lb", SEARCH_CASES)
def test_search_batch_identical_to_oracle(dab, dt, metric, d, n, R, Lb):
    """Same graph, same queries: ids, distances (bitwise), result counts, cmps and hops are all
    identical to the oracle's search_internal for several (L, beam, k)."""
    rng = np.random.default_rng(d * 31 + n)
    vecs, adj, maxdeg = make_index(rng, dt, metric, n, d, R, Lb)
    nq = 300
    queries = vecs[rng.integers(0, n, nq)].astype(np.float32) + 0.1 * rng.normal(size=(nq, d)).astype(np.float32)
    if dt in (np.int8, np.uint8):
        info = np.iinfo(dt)
        queries = np.clip(np.round(queries), info.min, info.max)
    queries = queries.astype(dt)
    oidx = O.Index(vecs, adj, n, 1, metric)
    with dab.GpuIndex(O.dtype_code(vecs), metric, d, n, 1, maxdeg) as g:
        g.upload_vectors(vecs)
        g.upload_graph(adj)
        assert np.array_equal(g.download_graph()[:, :adj.shape[1]], adj)
        for (k, L, beam) in [(10, 10, 1), (10, 40, 1), (5, 100, 1), (10, 32, 2), (20, 33, 4), (1, 1, 1), (64, 20, 1)]:
            got = g.search_batch(queries, k, L, beam)
            want = oidx.search_batch(queries, k, L, beam=beam, threads=4)
            for a, b, name in zip(got, want, ("ids", "dists", "counts", "cmps", "hops")):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), (name, k, L, beam)
            # batches in flight run the two-level visited set (shared-memory tags first): same answer
            out = g.search_batch_async(1, queries, k, L, beam)
            g.wait(1)
            for a, b, name in zip(out, want, ("ids", "dists", "counts", "cmps", "hops")):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), ("in flight", name, k, L, beam)


def test_search_edge_cases(dab):
    rng = np.random.default_rng(99)
    n, d = 500, 16
    vecs, adj, maxdeg = make_index(rng, np.float32, O.L2, n, d, 8, 20)
    oidx = O.Index(vecs, adj, n, 1, O.L2)
    with dab.GpuIndex(dab.DType.f32, dab.Metric.L2, d, n, 1, maxdeg) as g:
        g.upload_vectors(vecs)
        g.upload_graph(adj)
        # empty batch
        ids, dists, counts, cmps, hops = g.search_batch(np.zeros((0, d), np.float32), 10, 10)
        assert ids.shape == (0, 10)
        # k larger than anything reachable with L: padded with UINT32_MAX / +inf
        q = vecs[:7]
        got = g.search_batch(q, 50, 5)
        want = oidx.search_batch(q, 50, 5)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[2], want[2]) and (got[2] <= 6).all()  # cap = L + #start
        assert (got[0][:, 6:] == 0xFFFFFFFF).all() and np.isinf(got[1][:, 6:]).all()
        # a query with NaNs: every insert is ignored except ... all distances NaN -> no results
        qn = np.full((1, d), np.nan, np.float32)
        got = g.search_batch(qn, 10, 10)
        want = oidx.search_batch(qn, 10, 10)
        assert np.array_equal(got[0], want[0]) and got[2][0] == want[2][0] == 0
        with pytest.raises(dab.DabError):
            g.search_batch(q, 0, 10)
        with pytest.raises(dab.DabError):
            g.search_batch(q.astype(np.float16), 10, 10)


def test_graph_upload_from_device_memory_is_validated(dab):
    """dab_upload_graph_device: rows already in HBM get the same degree check as the host path (a kernel instead of a
    host loop); a valid upload searches like the host upload."""
    import torch
    rng = np.random.default_rng(17)
    n, d = 800, 24
    vecs, adj, maxdeg = make_index(rng, np.float32, O.L2, n, d, 8, 20)
    oidx = O.Index(vecs, adj, n, 1, O.L2)
    q = clustered(rng, 40, d)
    want = oidx.search_batch(q, 10, 20)
    with dab.GpuIndex(dab.DType.f32, dab.Metric.L2, d, n, 1, maxdeg) as g:
        g.upload_vectors(vecs)
        d_adj = torch.from_numpy(adj.view(np.int32).copy()).cuda()
        g.upload_graph_device(d_adj.data_ptr(), adj.shape[1], n + 1)
        got = g.search_batch(q, 10, 20)
        for a, b in zip(got, want):
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
        bad = adj.copy()
        bad[123, 0] = maxdeg + 1
        d_bad = torch.from_numpy(bad.view(np.int32).copy()).cuda()
        with pytest.raises(dab.DabError, match="row 123"):
            g.upload_graph_device(d_bad.data_ptr(), bad.shape[1], n + 1)


def test_visited_table_overflow_is_retried_exactly(dab, monkeypatch):
    """Force a tiny visited table: overflowing queries are re-run with a larger table and the
    results stay identical to the oracle."""
    rng = np.random.default_rng(5)
    n, d = 5000, 32
    vecs, adj, maxdeg = make_index(rng, np.float32, O.L2, n, d, 24, 40)
    queries = clustered(rng, 200, d)
    oidx = O.Index(vecs, adj, n, 1, O.L2)
    want = oidx.search_batch(queries, 10, 60, threads=4)
    monkeypatch.setenv("DAB_TEST_VISITED_LOG2", "8")
    with dab.GpuIndex(dab.DType.f32, dab.Metric.L2, d, n, 1, maxdeg) as g:
        g.upload_vectors(vecs)
        g.upload_graph(adj)
        got = g.search_batch(queries, 10, 60)
    assert (want[3] > 192).all(), "every query must actually overflow a 256-slot table (75 % load limit)"
    for a, b in zip(got, want):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.parametrize("force_overflow", [False, True])
def test_batches_in_flight_match_the_oracle(dab, monkeypatch, force_overflow):
    """dab_search_batch_async / dab_wait: several batches queued on different slots before any is joined
    return what the synchronous call (and the oracle) returns — also when every query of a batch outgrows
    its visited table and is re-run inside dab_wait — and the slot rules hold (one batch per slot, idle wait)."""
    rng = np.random.default_rng(15)
    n, d = 5000, 32
    vecs, adj, maxdeg = make_index(rng, np.float32, O.L2, n, d, 24, 40)
    oidx = O.Index(vecs, adj, n, 1, O.L2)
    batches = [clustered(rng, m, d) for m in (200, 64, 333, 1)]
    want = [oidx.search_batch(q, 10, 60, threads=4) for q in batches]
    if force_overflow:
        monkeypatch.setenv("DAB_TEST_VISITED_LOG2", "8")
    with dab.GpuIndex(dab.DType.f32, dab.Metric.L2, d, n, 1, maxdeg) as g:
        g.upload_vectors(vecs)
        g.upload_graph(adj)
        g.wait(2)  # idle slot: no-op
        for rounds in range(2):  # slots are reusable
            outs = [g.search_batch_async(s, q, 10, 60) for s, q in enumerate(batches)]
            with pytest.raises(dab.DabError):
                g.search_batch_async(1, batches[1], 10, 60)  # slot 1 still has a batch in flight
            for s in (2, 0, 3, 1):
                g.wait(s)
            for got, w in zip(outs, want):
                for a, b in zip(got, w):
                    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
        with pytest.raises(dab.DabError):
            g.search_batch_async(dab.MAX_SLOTS, batches[0], 10, 60)
        # interleaved with the synchronous call on the handle's own stream
        out = g.search_batch_async(0, batches[0], 10, 60)
        sync = g.search_batch(batches[2], 10, 60)
        g.wait(0)
        for a, b in zip(out, want[0]):
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
        for a, b in zip(sync, want[2]):
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


# ---------------------------------------------------------------- product quantization

def trained_pq(rng, base, chunks, centers=256):
    """A quick k-means-free codebook: sampled rows as pivots (codebook quality is irrelevant
    for arithmetic parity)."""
    piv = base[rng.choice(base.shape[0], centers, replace=False)].astype(np.float32)
    off = O.pq_offsets(base.shape[1], chunks)
    return piv, off


@pytest.mark.parametrize("metric,dim,chunks", [(O.L2, 128, 32), (O.INNER_PRODUCT, 128, 32), (O.COSINE_NORMALIZED, 96, 12),
                                               (O.COSINE, 64, 8), (O.L2, 100, 7), (O.L2, 17, 17)])
@pytest.mark.parametrize("path", ["fused", "separate_kernels"])
def test_pq_lut_adc_encode_bit_exact(dab, monkeypatch, metric, dim, chunks, path):
    """K6 / K7 through dab_pq_populate_lut / dab_pq_distances: pq_fused_kernel (pivots and the query's table in shared
    memory, the default where they fit) and the pq_lut_kernel + pq_adc_kernel pair (DAB_TEST_PQ_GLOBAL_LUT)."""
    if path == "separate_kernels":
        monkeypatch.setenv("DAB_TEST_PQ_GLOBAL_LUT", "1")
    rng = np.random.default_rng(dim + chunks)
    n, nq, c = 2000, (300 if chunks == 32 else 16), (700 if chunks == 32 else 200)  # > one CTA per SM, > one pass of candidates
    base = clustered(rng, n + 1, dim)
    piv, off = trained_pq(rng, base, chunks)
    L = O.lib()
    with dab.GpuIndex(dab.DType.f32, metric, dim, n, 1, 8) as g:
        g.upload_vectors(base)
        g.upload_pq(piv, off)
        codes = g.pq_encode(base)
        want_codes = np.zeros_like(codes)
        for i in range(n + 1):
            assert L.orc_pq_encode(O.ptr(piv), 256, dim, O.ptr(off), chunks, O.ptr(base[i]), O.ptr(want_codes[i])) == 0
        assert np.array_equal(codes, want_codes)
        g.upload_pq(piv, off, codes)
        queries = clustered(rng, nq, dim)
        ids = rng.integers(0, n + 1, (nq, c)).astype(np.uint32)
        ids[0, 0] = 0xFFFFFFFF
        got = g.pq_distances(queries, ids)
        if metric != O.COSINE:
            lut = g.pq_populate_lut(queries)
            want_lut = np.zeros((chunks, 256), np.float32)
            for qi in range(nq):
                L.orc_pq_populate_lut(O.ptr(piv), 256, dim, O.ptr(off), chunks,
                                      O.INNER_PRODUCT if metric == O.INNER_PRODUCT else O.L2, O.ptr(queries[qi]), O.ptr(want_lut))
                assert np.array_equal(bits(lut[qi]), bits(want_lut)), qi
        for qi in range(nq):
            valid = ids[qi] != 0xFFFFFFFF
            sel = np.ascontiguousarray(codes[np.where(valid, ids[qi], 0)])
            want = np.zeros(c, np.float32)
            L.orc_pq_query_distances(O.ptr(piv), 256, dim, O.ptr(off), chunks, metric, O.ptr(queries[qi]), O.ptr(sel), c, O.ptr(want))
            assert same_bits(got[qi][valid], want[valid]), qi
            assert np.isnan(got[qi][~valid]).all()
        # DistanceComputer (code x code, the PQ prune path): Resumable L2 / IP / cosine across chunks
        a = rng.integers(0, n + 1, 300).astype(np.uint32)
        b2 = rng.integers(0, n + 1, 300).astype(np.uint32)
        got_self = g.pq_self_distances(a, b2)
        want_self = np.array([L.orc_pq_self_distance(O.ptr(piv), dim, O.ptr(off), chunks, metric, O.ptr(codes[i]), O.ptr(codes[j]))
                              for i, j in zip(a, b2)], np.float32)
        assert same_bits(got_self, want_self)
        # inf input -> error naming the row/chunk (basic.rs:187-189)
        bad = base[:3].copy()
        bad[1, 0] = np.inf
        with pytest.raises(dab.DabError):
            g.pq_encode(bad)


# ---------------------------------------------------------------- MinMax quantization

@pytest.mark.parametrize("nbits", [8, 4, 2, 1])
def test_minmax_compress_and_distances_bit_exact(dab, nbits):
    """dab_minmax_compress / dab_minmax_distances == the oracle's restatement of MinMaxQuantizer::compress and
    MinMax{L2Squared, IP, Cosine, CosineNormalized} (diskann-quantization/src/minmax), byte for byte and bit for bit:
    every dimension 1..70 plus wide rows (row lengths that are and are not multiples of four bytes), three grid scales,
    constant vectors, the N x N and 8 x N pairings, NaN input."""
    rng = np.random.default_rng(40 + nbits)
    for dim, n, scale in [(d, 70, 1.0) for d in range(1, 71)] + [(128, 3000, 1.0), (100, 1000, 0.9), (257, 300, 1.1), (768, 200, 1.0)]:
        v = rng.uniform(-1.0, 1.0, (n, dim)).astype(np.float32)
        v[0] = 42.5                       # min == max (quantizer.rs:632)
        if n > 3:
            v[1] = 0.0
            v[2, ::2] = -10.0             # two distinct values
            v[2, 1::2] = 15.0
        want_rows, want_loss, want_nan = O.minmax_compress(v, nbits, scale)
        assert not want_nan.any()
        rows, loss = dab.minmax_compress(v, nbits, scale)
        assert rows.shape == want_rows.shape and np.array_equal(rows, want_rows), (dim, nbits)
        assert same_bits(loss, want_loss), (dim, nbits)
        perm = rng.permutation(n)
        for metric in METRICS:
            got = dab.minmax_distances(metric, nbits, nbits, dim, rows, rows[perm])
            want = O.minmax_distances(metric, nbits, nbits, want_rows, want_rows[perm])
            assert same_bits(got, want), (dim, nbits, metric)
        if nbits != 8 and dim in (17, 64, 100, 128):
            rows8, _ = dab.minmax_compress(v, 8, scale)
            want8, _, _ = O.minmax_compress(v, 8, scale)
            assert np.array_equal(rows8, want8)
            for metric in METRICS:
                got = dab.minmax_distances(metric, 8, nbits, dim, rows8, rows[perm])
                want = O.minmax_distances(metric, 8, nbits, want8, want_rows[perm])
                assert same_bits(got, want), ("8 x N", dim, nbits, metric)
    # InputContainsNaN: the call fails, naming the vector (quantizer.rs:728-750)
    bad = rng.uniform(-1.0, 1.0, (40, 100)).astype(np.float32)
    bad[33, 7] = np.nan
    with pytest.raises(dab.DabError, match="vector 33"):
        dab.minmax_compress(bad, nbits)
    with pytest.raises(dab.DabError):
        dab.minmax_compress(bad[:2], 3)                      # no Representation<3>
    with pytest.raises(dab.DabError):
        dab.minmax_distances(O.L2, 4, 8, 100, np.zeros((1, 70), np.uint8), np.zeros((1, 120), np.uint8))  # only N x N and 8 x N


@pytest.mark.parametrize("nbits", [8, 4, 2, 1])
def test_minmax_full_query_distances_bit_exact(dab, nbits):
    """dab_minmax_query_distances == the oracle's restatement of MinMax*::evaluate(FullQueryRef, DataRef<NBITS>): the f32 x N-bit
    inner product in the reference's x86-64-v3 lane order (every remainder length: dims 1..100 and wide rows), the
    FullQueryMeta sums and the four epilogues, bit for bit."""
    rng = np.random.default_rng(60 + nbits)
    for dim in list(range(1, 101)) + [128, 250, 257, 768]:
        n, nq = (300, 5) if dim > 100 else (37, 3)
        v = rng.uniform(-1.0, 1.0, (n, dim)).astype(np.float32)
        q = rng.uniform(-1.0, 1.0, (nq, dim)).astype(np.float32)
        rows, _, _ = O.minmax_compress(v, nbits, 1.0)
        for metric in METRICS:
            got = dab.minmax_query_distances(metric, nbits, q, rows)
            want = O.minmax_query_distances(metric, nbits, q, rows)
            assert same_bits(got, want), (dim, nbits, metric)
    bad = rng.uniform(-1.0, 1.0, (4, 64)).astype(np.float32)
    bad[2, 5] = np.nan
    rows, _, _ = O.minmax_compress(rng.uniform(-1.0, 1.0, (10, 64)).astype(np.float32), nbits, 1.0)
    with pytest.raises(dab.DabError, match="query 2"):
        dab.minmax_query_distances(O.L2, nbits, bad, rows)


# ---------------------------------------------------------------- scalar quantization

@pytest.mark.parametrize("nbits", [8, 4, 2, 1])
def test_sq_compress_and_distances_bit_exact(dab, nbits):
    import ctypes as C
    from diskann_b200 import _lib
    rng = np.random.default_rng(nbits)
    n, dim = 300, 100
    vecs = clustered(rng, 2 * n, dim)
    vecs[5, 7] = np.nan
    shift = vecs[np.isfinite(vecs).all(1)].mean(0).astype(np.float32)
    scale = np.float32(4.2)
    codes = np.zeros((2 * n, dim), np.uint8)
    comp = np.zeros(2 * n, np.float32)
    _lib.check(_lib.lib().dab_sq_compress(0, O.ptr(shift), scale, dim, nbits, O.ptr(vecs), 2 * n, O.ptr(codes), O.ptr(comp)))
    L = O.lib()
    for i in range(2 * n):
        wc = np.zeros(dim, np.uint8)
        w = L.orc_sq_compress(O.ptr(shift), scale, dim, nbits, O.ptr(vecs[i]), O.ptr(wc), None)
        assert np.array_equal(wc, codes[i]) and same_bits([w], [comp[i]]), i
    ss = float(np.float32(scale) * np.float32(scale))
    ssn = float(np.float32((shift.astype(np.float64) ** 2).sum()))
    for metric in (O.L2, O.INNER_PRODUCT, O.COSINE_NORMALIZED):
        out = np.zeros(n, np.float32)
        x, y = np.ascontiguousarray(codes[:n]), np.ascontiguousarray(codes[n:])
        cx, cy = np.ascontiguousarray(comp[:n]), np.ascontiguousarray(comp[n:])
        _lib.check(_lib.lib().dab_sq_distances(0, metric, nbits, ss, ssn, dim, O.ptr(x), O.ptr(cx), O.ptr(y), O.ptr(cy), n, O.ptr(out)))
        want = np.array([L.orc_sq_distance(metric, nbits, ss, ssn, O.ptr(x[i]), float(cx[i]), O.ptr(y[i]), float(cy[i]), dim)
                         for i in range(n)], np.float32)
        assert same_bits(out, want), metric


# ---------------------------------------------------------------- flat scan (ground truth)

@pytest.mark.parametrize("dt,metric,dim,n", [
    (np.float32, O.L2, 128, 5000), (np.float32, O.L2, 100, 3001), (np.float32, O.INNER_PRODUCT, 37, 2000),
    (np.float32, O.COSINE, 48, 1500), (np.float16, O.INNER_PRODUCT, 96, 3000), (np.float16, O.L2, 768, 700),
    (np.int8, O.L2, 128, 3000), (np.uint8, O.COSINE, 40, 1000),
])
def test_flat_knn_bit_exact(dab, dt, metric, dim, n):
    rng = np.random.default_rng(dim + n)
    base = fuzz(rng, dt, (n + 1, dim))
    base[7] = base[3]  # exact ties: lower id first
    queries = fuzz(rng, dt, (70, dim))
    queries[0] = base[3]
    with dab.GpuIndex(O.dtype_code(base), metric, dim, n, 1, 4) as g:
        g.upload_vectors(base)
        ids, dists = g.flat_knn(queries, 10)
        ids1, dists1 = g.flat_knn(queries[:3], 1)
    want_ids, want_d = O.bruteforce_knn(base[:n], queries, metric, 10)
    assert np.array_equal(ids, want_ids)
    assert same_bits(dists, want_d)
    assert np.array_equal(ids1[:, 0], want_ids[:3, 0])


# ---------------------------------------------------------------- robust_prune

@pytest.mark.parametrize("dt,metric,dim", [(np.float32, O.L2, 64), (np.float32, O.INNER_PRODUCT, 32), (np.float32, O.COSINE, 24),
                                           (np.float16, O.L2, 48), (np.int8, O.L2, 128), (np.uint8, O.INNER_PRODUCT, 16)])
def test_robust_prune_selects_the_same_neighbours(dab, dt, metric, dim):
    """prune.rs:106-259 on the device vs the oracle: same pools -> same selected ids in the same
    order (candidate x candidate distances are Distance<T,T>, bit-exact)."""
    import ctypes as C
    rng = np.random.default_rng(dim)
    n, n_pools, cap, degree = 3000, 150, 200, 24
    base = clustered(rng, n + 1, dim)
    if dt == np.float16:
        base = base.astype(np.float16)
    elif dt == np.int8:
        base = np.clip(np.round(base * 40), -127, 127).astype(np.int8)
    elif dt == np.uint8:
        base = np.clip(np.round(base * 40 + 128), 0, 255).astype(np.uint8)
    base[11] = base[10]  # zero candidate-candidate distance -> f32::MAX occlude factor
    oidx = O.Index(base, np.zeros((n + 1, 2), np.uint32), n, 1, metric)
    pool_ids = np.full((n_pools, cap), 0xFFFFFFFF, np.uint32)
    pool_d = np.zeros((n_pools, cap), np.float32)
    lens = rng.integers(0, cap + 1, n_pools).astype(np.uint32)
    lens[0], lens[1] = 0, 1
    locs = rng.integers(0, n, n_pools).astype(np.uint32)
    for p in range(n_pools):
        ids = rng.choice(n, lens[p], replace=False).astype(np.uint32)
        if lens[p] > 3:
            ids[2] = locs[p]  # the location itself appears in its pool and must be excluded
            if 10 not in ids and 11 not in ids:
                ids[0], ids[1] = 10, 11
        q = base[locs[p]].astype(np.float32) if dt == np.float16 else base[locs[p]]
        pool_ids[p, :lens[p]] = ids
        pool_d[p, :lens[p]] = O.distance_rows(q, base[ids], metric) if lens[p] else []
    for alpha in (1.2, 1.0):
        with dab.GpuIndex(O.dtype_code(base), metric, dim, n, 1, 4) as g:
            g.upload_vectors(base)
            got, counts = g.robust_prune(pool_ids, pool_d, lens, locs, degree, alpha)
        L = O.lib()
        for p in range(n_pools):
            m = int(lens[p])
            order = np.argsort(pool_d[p, :m], kind="stable")
            sid = np.ascontiguousarray(pool_ids[p, :m][order])
            sd = np.ascontiguousarray(pool_d[p, :m][order])
            excl = np.ascontiguousarray((sid == locs[p]).astype(np.uint8))
            pos = np.zeros(degree, np.uint32)
            found = L.orc_robust_prune(C.byref(oidx.c), O.ptr(sid), O.ptr(sd), O.ptr(excl), m, degree, alpha, O.SIMD, O.ptr(pos), None)
            assert counts[p] == found, (p, alpha)
            assert list(got[p, :found]) == list(sid[pos[:found]]), (p, alpha)
            assert (got[p, found:] == 0xFFFFFFFF).all()


# ---------------------------------------------------------------- device build

@pytest.mark.parametrize("dt,metric,dim,n", [(np.float32, O.L2, 64, 20000), (np.float16, O.INNER_PRODUCT, 48, 8000),
                                             (np.int8, O.L2, 64, 8000)])
def test_device_build_graph_is_valid_and_searchable(dab, dt, metric, dim, n):
    rng = np.random.default_rng(n)
    base = clustered(rng, n, dim, n_centers=64)
    if dt == np.float16:
        base = (base / np.linalg.norm(base, axis=1, keepdims=True)).astype(np.float16)
    elif dt == np.int8:
        base = np.clip(np.round(base * 40), -127, 127).astype(np.int8)
    mean = base.astype(np.float32).mean(0)
    medoid = base[np.argmin(((base.astype(np.float32) - mean) ** 2).sum(1))]
    vecs = np.concatenate([base, medoid[None]])
    R, maxdeg, Lb = 32, 41, 64
    queries = base[rng.integers(0, n, 400)].astype(np.float32) + 0.05 * rng.normal(size=(400, dim)).astype(np.float32)
    if dt == np.int8:
        queries = np.clip(np.round(queries), -127, 127)
    queries = queries.astype(dt)
    with dab.GpuIndex(O.dtype_code(vecs), metric, dim, n, 1, maxdeg) as g:
        g.upload_vectors(vecs)
        g.build(R, Lb, 1.2)
        adj = g.download_graph()
        got = g.search_batch(queries, 10, 64)
        gt_ids, _ = g.flat_knn(queries, 10)
    deg = adj[:, 0]
    assert deg.max() <= maxdeg and deg[:n].min() >= 1
    for i in rng.integers(0, n + 1, 500):
        row = adj[i, 1:1 + deg[i]]
        assert (row <= n).all() and i not in row and len(set(row.tolist())) == len(row)
    # the device-built graph searched by the oracle gives the identical answer (graph is data)
    oidx = O.Index(vecs, adj, n, 1, metric)
    want = oidx.search_batch(queries, 10, 64, threads=4)
    for a, b in zip(got, want):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    rec = O.recall(gt_ids, got[0], got[2], 10, 10)
    # reference-quality graph: compare with the oracle's sequential build on a subset size
    assert rec > 0.95, rec


@pytest.mark.parametrize("dt,metric,d,n,R,Lb", [(np.float32, O.L2, 32, 1500, 16, 30), (np.int8, O.L2, 64, 1200, 12, 24),
                                                (np.float32, O.INNER_PRODUCT, 24, 1000, 8, 20)])
def test_device_build_one_insert_at_a_time_reproduces_the_sequential_reference_build(dab, dt, metric, d, n, R, Lb):
    """dab_build with batch_size = 1 is DiskANNIndex::insert for i = 0..n (index.rs:226-341: search with
    a VisitedSearchRecord, robust_prune, set_neighbors, add_edge_and_prune per out-edge): the adjacency
    must equal the oracle's sequential build (which the single-insert grid baselines pin) bit for bit."""
    rng = np.random.default_rng(n + d)
    vecs, want, maxdeg = make_index(rng, dt, metric, n, d, R, Lb)
    with dab.GpuIndex(O.dtype_code(vecs), metric, d, n, 1, maxdeg) as g:
        g.upload_vectors(vecs)
        g.build(R, Lb, 1.2, batch_size=1)
        got = g.download_graph()
    assert np.array_equal(got[:, 0], want[:, 0]), "degrees differ"
    for i in range(n + 1):
        assert np.array_equal(got[i, 1:1 + got[i, 0]], want[i, 1:1 + want[i, 0]]), i


@pytest.mark.parametrize("dt,metric,d,n,R,Lb,bs", [(np.float32, O.L2, 32, 4000, 16, 30, 64), (np.float32, O.L2, 48, 6000, 16, 32, 0),
                                                   (np.int8, O.L2, 64, 3000, 12, 24, 100), (np.float16, O.INNER_PRODUCT, 32, 2500, 12, 24, 50)])
def test_device_batched_build_is_the_reference_multi_insert(dab, dt, metric, d, n, R, Lb, bs):
    """dab_build == DiskANNIndex::multi_insert (index.rs:815-1050; intra_batch_candidates = None, bootstrap
    branch not taken) over the same batch schedule: candidate generation against the graph as it was
    before the batch, aggregated and sorted back-edges, one add_edge_and_prune per target — the
    adjacency equals the oracle's restatement bit for bit."""
    rng = np.random.default_rng(n + d + bs)
    base = clustered(rng, n, d)
    if dt == np.float16:
        base = (base / np.linalg.norm(base, axis=1, keepdims=True)).astype(np.float16)
    elif dt == np.int8:
        base = np.clip(np.round(base * 40), -127, 127).astype(np.int8)
    mean = base.astype(np.float32).mean(0)
    vecs = np.concatenate([base, base[np.argmin(((base.astype(np.float32) - mean) ** 2).sum(1))][None]])
    maxdeg = int(R * 1.3)
    want = O.build_graph_batched(vecs, n, 1, metric, R, maxdeg, Lb, batch_size=bs)
    with dab.GpuIndex(O.dtype_code(vecs), metric, d, n, 1, maxdeg) as g:
        g.upload_vectors(vecs)
        g.build(R, Lb, 1.2, batch_size=bs)
        got = g.download_graph()
    assert np.array_equal(got[:, 0], want[:, 0]), "degrees differ"
    for i in range(n + 1):
        assert np.array_equal(got[i, 1:1 + got[i, 0]], want[i, 1:1 + want[i, 0]]), i


# ---------------------------------------------------------------- PQ traversal (C4 shape) and C3 shape

@pytest.mark.parametrize("path", ["smem_pivots", "global_lut", "smem_pivots_overflow"])
@pytest.mark.parametrize("dt,metric,d,chunks", [(np.int8, O.L2, 128, 32), (np.float32, O.L2, 96, 12), (np.float32, O.INNER_PRODUCT, 64, 16),
                                                (np.uint8, O.COSINE_NORMALIZED, 40, 7), (np.float32, O.INNER_PRODUCT, 100, 25),
                                                (np.float16, O.L2, 64, 16)])
def test_pq_traversal_search_identical_to_oracle(dab, monkeypatch, dt, metric, d, chunks, path):
    """dab_search_batch_pq: greedy search whose traversal distances are ADC lookups over the codes
    (providers' QuantAccessor, product.rs:311-340) == the oracle's search with pq_codes set.
    Both kernels are covered: search_kernel_pqs (pivots in shared memory, the default where they fit: chunk
    lengths 4 / 8 / mixed, 32 / 25 / 16 / 12 / 7 chunks) and search_kernel_pq (per-warp table in global memory),
    and the overflow re-run of the former (a 256-slot visited table)."""
    if path == "global_lut":
        monkeypatch.setenv("DAB_TEST_PQ_GLOBAL_LUT", "1")
    if path == "smem_pivots_overflow":
        monkeypatch.setenv("DAB_TEST_VISITED_LOG2", "8")
    rng = np.random.default_rng(d + chunks)
    n = 4000
    vecs, adj, maxdeg = make_index(rng, dt, O.L2 if metric == O.COSINE_NORMALIZED else metric, n, d, 24, 40)
    f32 = vecs.astype(np.float32)
    piv = f32[rng.choice(n, 256, replace=False)]
    off = O.pq_offsets(d, chunks)
    L = O.lib()
    codes = np.zeros((n + 1, chunks), np.uint8)
    for i in range(n + 1):
        assert L.orc_pq_encode(O.ptr(piv), 256, d, O.ptr(off), chunks, O.ptr(f32[i]), O.ptr(codes[i])) == 0
    nq = 200
    queries = vecs[rng.integers(0, n, nq)].copy()
    oidx = O.Index(vecs, adj, n, 1, metric, pq=(piv, off, codes))
    with dab.GpuIndex(O.dtype_code(vecs), metric, d, n, 1, maxdeg) as g:
        g.upload_vectors(vecs)
        g.upload_graph(adj)
        g.upload_pq(piv, off, codes)
        # (the last case: a list longer than one register tile of the merge, two tiles of 512 entries)
        for (k, Ls, beam) in [(10, 30, 1), (5, 64, 2), (10, 150, 1)] + ([(10, 700, 1)] if chunks in (32, 7) else []):
            got = g.search_batch_pq(queries, k, Ls, beam)
            want = oidx.search_batch(queries, k, Ls, beam=beam, threads=4)
            for a, b, name in zip(got, want, ("ids", "dists", "counts", "cmps", "hops")):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), (name, k, Ls, beam)
            # + Pipeline<FilterStartPoints, Rerank>: the candidate list re-scored with Distance<T, T>
            # (f16 rows: the f16 x f16 schema with two accumulators)
            got = g.search_batch_pq(queries, k, Ls, beam, rerank=True)
            want = oidx.search_batch_rerank(queries, k, Ls, beam=beam, threads=4)
            for a, b, name in zip(got, want, ("ids", "dists", "counts", "cmps", "hops")):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), ("rerank", name, k, Ls, beam)
    with dab.GpuIndex(dab.DType.f32, dab.Metric.Cosine, d, n, 1, maxdeg) as g:
        g.upload_vectors(f32)
        g.upload_graph(adj)
        g.upload_pq(piv, off, codes)
        # Metric::Cosine traverses with QueryComputer::DirectCosine (no table): resumable cosine over the gathered pivots
        ocos = O.Index(np.ascontiguousarray(f32), adj, n, 1, O.COSINE, pq=(piv, off, codes))
        qf = np.ascontiguousarray(f32[rng.integers(0, n, 100)])
        for (k, Ls, beam) in [(10, 30, 1), (5, 64, 2)]:
            got = g.search_batch_pq(qf, k, Ls, beam)
            want = ocos.search_batch(qf, k, Ls, beam=beam, threads=4)
            for a, b, name in zip(got, want, ("ids", "dists", "counts", "cmps", "hops")):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), ("direct cosine", name, k, Ls, beam)
            # rerank with the float cosine schema (two accumulators, FullCosineAccumulator)
            got = g.search_batch_pq(qf, k, Ls, beam, rerank=True)
            want = ocos.search_batch_rerank(qf, k, Ls, beam=beam, threads=4)
            for a, b, name in zip(got, want, ("ids", "dists", "counts", "cmps", "hops")):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), ("direct cosine + rerank", name, k, Ls, beam)


def test_pq_traversal_wide_adjacency_rows(dab):
    """Adjacency rows longer than the 96 words search_kernel_pqs copies one hop ahead (max_degree 110): the kernel reads them in
    two passes and falls back to the L2 prefetch of the next row; every node of this random graph has 100 neighbours."""
    rng = np.random.default_rng(7)
    n, d, chunks, maxdeg = 3000, 32, 8, 110
    base = clustered(rng, n + 1, d)
    adj = np.zeros((n + 1, maxdeg + 1), np.uint32)
    adj[:, 0] = 100
    adj[:, 1:101] = rng.integers(0, n, (n + 1, 100))
    piv = base[rng.choice(n, 256, replace=False)]
    off = O.pq_offsets(d, chunks)
    L = O.lib()
    codes = np.zeros((n + 1, chunks), np.uint8)
    for i in range(n + 1):
        assert L.orc_pq_encode(O.ptr(piv), 256, d, O.ptr(off), chunks, O.ptr(base[i]), O.ptr(codes[i])) == 0
    queries = clustered(rng, 100, d)
    oidx = O.Index(base, adj, n, 1, O.L2, pq=(piv, off, codes))
    with dab.GpuIndex(dab.DType.f32, dab.Metric.L2, d, n, 1, maxdeg) as g:
        g.upload_vectors(base)
        g.upload_graph(adj)
        g.upload_pq(piv, off, codes)
        for (k, Ls, beam) in [(10, 40, 1), (10, 300, 1), (5, 64, 2)]:
            got = g.search_batch_pq(queries, k, Ls, beam, rerank=True)
            want = oidx.search_batch_rerank(queries, k, Ls, beam=beam, threads=4)
            for a, b, name in zip(got, want, ("ids", "dists", "counts", "cmps", "hops")):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), (name, k, Ls, beam)


def sq_quantizer(f32, metric):
    """A ScalarQuantizer in the shape of scalar/train.rs: shift below the per-dimension mean, one scale."""
    mean = f32.mean(0).astype(np.float32)
    std = float(f32.std())
    shift = (mean - np.float32(2.5 * std)).astype(np.float32)
    scale = np.float32(5.0 * std)
    ssn = np.float32(-O.distance(shift, shift, O.INNER_PRODUCT))  # InnerProduct::evaluate(shift, shift)
    mean_norm = np.float32(np.linalg.norm(f32, axis=1).mean()) if metric == O.INNER_PRODUCT else np.float32(0)
    return shift, float(scale), float(ssn), float(mean_norm)


@pytest.mark.parametrize("dt,metric,d,nbits", [(np.float32, O.L2, 128, 8), (np.float32, O.L2, 100, 4), (np.float32, O.INNER_PRODUCT, 64, 8),
                                               (np.float32, O.INNER_PRODUCT, 96, 4), (np.float16, O.COSINE_NORMALIZED, 48, 2),
                                               (np.uint8, O.L2, 128, 1), (np.int8, O.L2, 72, 2), (np.float32, O.L2, 37, 4)])
def test_sq_traversal_search_identical_to_oracle(dab, dt, metric, d, nbits):
    """dab_search_batch_sq: greedy search through the scalar-quantized accessor (providers inmem/scalar.rs:449-570):
    rows encoded on the device == SQStore::set_vector restated on the CPU (canonical-front layout, dense N-bit codes),
    and ids / distance bits / cmps / hops == the oracle's search with sq_rows set, with and without Rerank."""
    rng = np.random.default_rng(d * 10 + nbits)
    n = 4000
    vecs, adj, maxdeg = make_index(rng, dt, O.L2 if metric == O.COSINE_NORMALIZED else metric, n, d, 24, 40)
    f32 = vecs.astype(np.float32)
    shift, scale, ssn, mean_norm = sq_quantizer(f32, metric)
    rows = O.sq_encode_rows(f32, shift, scale, nbits)
    nq = 200
    queries = vecs[rng.integers(0, n, nq)].copy()
    if metric == O.INNER_PRODUCT:
        queries = (queries.astype(np.float32) * rng.uniform(0.3, 3.0, (nq, 1))).astype(vecs.dtype)  # exercise the rescale
    oidx = O.Index(vecs, adj, n, 1, metric, sq=(rows, nbits, shift, scale, ssn, mean_norm))
    with dab.GpuIndex(O.dtype_code(vecs), metric, d, n, 1, maxdeg) as g:
        g.upload_vectors(vecs)
        g.upload_graph(adj)
        g.upload_sq(nbits, shift, scale, ssn, mean_norm)
        with pytest.raises(dab.DabError):
            g.search_batch_sq(queries[:2], 5, 10)  # no rows yet
        g.sq_encode_all()
        assert np.array_equal(g.download_sq(), rows)
        for (k, Ls, beam) in [(10, 30, 1), (5, 64, 2), (10, 150, 1)]:
            got = g.search_batch_sq(queries, k, Ls, beam)
            want = oidx.search_batch(queries, k, Ls, beam=beam, threads=4)
            for a, b, name in zip(got, want, ("ids", "dists", "counts", "cmps", "hops")):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), (name, k, Ls, beam)
            got = g.search_batch_sq(queries, k, Ls, beam, rerank=True)
            want = oidx.search_batch_rerank(queries, k, Ls, beam=beam, threads=4)
            for a, b, name in zip(got, want, ("ids", "dists", "counts", "cmps", "hops")):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), ("rerank", name, k, Ls, beam)
        # rows handed over by the host (set_quant_vector) give the same searches
        g.upload_sq(nbits, shift, scale, ssn, mean_norm, rows=rows)
        assert np.array_equal(g.download_sq(), rows)
        got = g.search_batch_sq(queries, 10, 50, 1)
        want = oidx.search_batch(queries, 10, 50, beam=1, threads=4)
        for a, b in zip(got, want):
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    with dab.GpuIndex(dab.DType.f32, dab.Metric.Cosine, d, n, 1, maxdeg) as g:
        g.upload_vectors(f32)
        g.upload_graph(adj)
        g.upload_sq(nbits, shift, scale, ssn, mean_norm, rows=rows)
        with pytest.raises(dab.DabError):
            g.search_batch_sq(f32[:2], 5, 10)  # SQStore::distance_computer: UnsupportedDistanceMetric


@pytest.mark.parametrize("dim,chunks,centers,n", [(24, 5, 32, 3000), (128, 32, 256, 6000), (40, 1, 16, 1500)])
def test_pq_training_on_the_device_is_bit_identical_to_the_cpu_restatement(dab, dim, chunks, centers, n):
    """train_pq (k-means++ + 5 Lloyd iterations per chunk) and the encoding of every stored row:
    same pivots (bits), offsets and codes as oracle/kmeans.cpp + BasicTable::compress_into."""
    rng = np.random.default_rng(dim * 1000 + chunks)
    base = clustered(rng, n + 1, dim, n_centers=64)
    train = base[rng.choice(n, n // 2, replace=False)]
    want_piv, want_off, st = O.pq_train(train, chunks, centers, 5, 12345)
    assert st == 0
    with dab.GpuIndex(dab.DType.f32, dab.Metric.L2, dim, n, 1, 8) as g:
        g.upload_vectors(base)
        g.pq_train(train, chunks, centers, 5, 12345)
        with pytest.raises(dab.DabError):
            g.search_batch_pq(base[:2], 5, 10)  # no codes yet: NOT_READY, never distances to centre 0
        g.pq_encode_all()
        piv, off, codes = g.download_pq()
    assert np.array_equal(off, want_off)
    assert np.array_equal(bits(piv), bits(want_piv))
    want_codes = np.zeros_like(codes)
    L = O.lib()
    for i in range(n + 1):
        assert L.orc_pq_encode(O.ptr(want_piv), centers, dim, O.ptr(want_off), chunks, O.ptr(base[i]), O.ptr(want_codes[i])) == 0
    assert np.array_equal(codes, want_codes)


def test_search_c3_shape_f16_768_inner_product(dab):
    """BASELINE config C3 shape (768-d f16, inner product) at test size through the v2 kernel."""
    rng = np.random.default_rng(768)
    n, d = 3000, 768
    vecs, adj, maxdeg = make_index(rng, np.float16, O.INNER_PRODUCT, n, d, 32, 50)
    queries = vecs[rng.integers(0, n, 64)].copy()
    oidx = O.Index(vecs, adj, n, 1, O.INNER_PRODUCT)
    with dab.GpuIndex(dab.DType.f16, dab.Metric.InnerProduct, d, n, 1, maxdeg) as g:
        g.upload_vectors(vecs)
        g.upload_graph(adj)
        for (k, Ls) in [(10, 100), (10, 200)]:
            got = g.search_batch(queries, k, Ls, 1)
            want = oidx.search_batch(queries, k, Ls, threads=4)
            for a, b in zip(got, want):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


# ---------------------------------------------------------------- tensor-core exhaustive scan

@pytest.mark.timeout(180)
@pytest.mark.parametrize("dt,metric,n,d,nq", [(np.float32, O.L2, 20000, 128, 300), (np.float32, O.INNER_PRODUCT, 5000, 96, 129),
                                               (np.int8, O.L2, 30000, 128, 200), (np.float16, O.INNER_PRODUCT, 9000, 100, 64),
                                               (np.uint8, O.COSINE, 7000, 40, 50), (np.float32, O.COSINE_NORMALIZED, 3001, 33, 17)])
def test_tensor_core_flat_scan_equals_the_exact_scan(dab, dt, metric, n, d, nq):
    """dab_flat_knn_tc (tcgen05 GEMM over bf16 hi/lo splits, fused candidate selection, exact
    re-scoring) returns the exact scan's ids and bit-identical distances."""
    rng = np.random.default_rng(n + d)
    if dt in (np.float32, np.float16):
        base = clustered(rng, n + 1, d, n_centers=50).astype(dt)
        queries = clustered(rng, nq, d, n_centers=50).astype(dt)
        if metric == O.COSINE_NORMALIZED:
            base = (base / np.linalg.norm(base.astype(np.float32), axis=1, keepdims=True)).astype(dt)
            queries = (queries / np.linalg.norm(queries.astype(np.float32), axis=1, keepdims=True)).astype(dt)
    else:
        base, queries = fuzz(rng, dt, (n + 1, d)), fuzz(rng, dt, (nq, d))
    with dab.GpuIndex(O.dtype_code(base), metric, d, n, 1, 8) as g:
        g.upload_vectors(base)
        want_ids, want_d = g.flat_knn(queries, 10)
        got_ids, got_d = g.flat_knn_tc(queries, 10)
    assert np.array_equal(bits(got_d), bits(want_d))
    assert np.array_equal(got_ids, want_ids)
