"""debug aid: one small pass over every kernel family, sized to run under
`compute-sanitizer --tool memcheck` (or racecheck / initcheck) in about a minute."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import diskann_b200 as dab

rng = np.random.default_rng(0)
if len(sys.argv) > 1 and sys.argv[1] == "pq":
    # only the product-quantization kernels (search_kernel_pqs with its cp.async row hand-off and the two-tile merge,
    # pq_fused_kernel, the global-table kernel, rerank): `compute-sanitizer --tool racecheck python tools/sanitize_check.py pq`
    for dt, ddt, d, chunks in ((np.float32, dab.DType.f32, 100, 25), (np.int8, dab.DType.i8, 32, 4), (np.float32, dab.DType.f32, 40, 7)):
        n = 1500
        base = (rng.normal(size=(n + 1, d)) * (30 if dt == np.int8 else 1)).astype(dt)
        with dab.GpuIndex(ddt, dab.Metric.L2, d, n, 1, 41) as g:
            g.upload_vectors(base)
            adj = np.zeros((n + 1, 42), np.uint32)             # a random 24-regular graph: traversal only, no build kernels here
            adj[:, 0] = 24
            adj[:, 1:25] = rng.integers(0, n, (n + 1, 24))
            g.upload_graph(adj)
            g.pq_train(base[:1200].astype(np.float32), chunks, 64, 2, 7)
            g.pq_encode_all()
            a = g.search_batch_pq(base[:48], 5, 40, 1, rerank=True)
            b = g.search_batch_pq(base[:48], 5, 600, 1, rerank=True)   # list longer than one merge tile
            c = g.search_batch_pq(base[:48], 5, 64, 2)
            ids = rng.integers(0, n + 1, (20, 300)).astype(np.uint32)
            lut = g.pq_populate_lut(base[:20].astype(np.float32))
            dd = g.pq_distances(base[:20].astype(np.float32), ids)
            # the same index with the per-query tables in global memory (search_kernel_pq, pq_lut_kernel + pq_adc_kernel)
            os.environ["DAB_TEST_PQ_GLOBAL_LUT"] = "1"
            with dab.GpuIndex(ddt, dab.Metric.L2, d, n, 1, 41) as g2:
                g2.upload_vectors(base)
                g2.upload_graph(adj)
                g2.upload_pq(*g.download_pq())
                a2 = g2.search_batch_pq(base[:48], 5, 40, 1, rerank=True)
                dd2 = g2.pq_distances(base[:20].astype(np.float32), ids)
            del os.environ["DAB_TEST_PQ_GLOBAL_LUT"]
            assert np.array_equal(a[0], a2[0]) and np.array_equal(dd.view(np.uint32), dd2.view(np.uint32))
            print(dt.__name__, d, chunks, "pq ok", int(a[2].min()), int(b[2].min()), int(c[2].min()), lut.shape)
    for nb in (8, 4, 1):                                                       # MinMax quantizer: compress + distances
        v = rng.uniform(-1, 1, (200, 77)).astype(np.float32)
        rows, loss = dab.minmax_compress(v, nb, 0.9)
        dmm = dab.minmax_distances(dab.Metric.L2, nb, nb, 77, rows, rows[::-1].copy())
        r8, _ = dab.minmax_compress(v, 8)
        dmx = dab.minmax_distances(dab.Metric.Cosine, 8, nb, 77, r8, rows)
        dq = dab.minmax_query_distances(dab.Metric.L2, nb, v[:9], rows)           # full-precision queries x compressed rows
        print("minmax", nb, rows.shape, bool(np.isfinite(dmm).all() and np.isfinite(dmx).all() and np.isfinite(dq).all()))
    print("sanitize_check pq done")
    sys.exit(0)
for dt, ddt, metric, d in ((np.float32, dab.DType.f32, dab.Metric.L2, 100), (np.float16, dab.DType.f16, dab.Metric.InnerProduct, 61),
                           (np.int8, dab.DType.i8, dab.Metric.L2, 33)):
    n = 3000
    base = (rng.normal(size=(n + 1, d)) * (30 if dt == np.int8 else 1)).astype(dt)
    with dab.GpuIndex(ddt, metric, d, n, 1, 41) as g:
        g.upload_vectors(base)
        g.build(32, 64, 1.2)                                     # search (records) + prune + back-edge kernels
        adj = g.download_graph()
        ids = rng.integers(0, n + 1, (50, 83)).astype(np.uint32)
        ids[0, :5] = 0xFFFFFFFF
        out = g.distances(base[:50], ids)                        # frontier kernels (wide for f32 / f16)
        pairs = g.row_pair_distances(ids[1, :40], ids[2, :40])
        block = g.pairwise(ids[3, :17])
        got = g.search_batch(base[:64], 5, 64, 1)                # search_kernel_v2 / generic
        got4 = g.search_batch(base[:64], 5, 40, 4)
        knn = g.flat_knn(base[:16], 5)
        knn_tc = g.flat_knn_tc(base[:16], 5)                     # tcgen05 + TMA + TMEM path
        assert np.array_equal(knn[0], knn_tc[0])
        if dt != np.float16:
            g.pq_train(base[:1500].astype(np.float32), 4, 32, 2, 7)  # k-means++ / Lloyd kernels
            g.pq_encode_all()
            pq = g.search_batch_pq(base[:32], 5, 40, 1, rerank=True)  # PQ traversal + rerank kernel
            g.pq_self_distances(ids[4, :20], ids[5, :20])
        print(dt.__name__, "deg max", int(adj[:, 0].max()), "search ok", int(got[2].min()), int(got4[2].min()),
              "finite", bool(np.isfinite(out[1:]).all() and np.isfinite(pairs).all() and np.isfinite(block).all()), knn[0].shape)
print("sanitize_check done")
