#!/usr/bin/env python3
"""bench.py — benchmark of the B200-native DiskANN distance hot path (greedy search over a Vamana graph).

Headline metric (BASELINE.json): QPS at recall@10 >= 0.95 on synthetic 1M x 128 f32 L2 (R=64, max
degree 83, L_build=100, alpha=1.2, L_search=100, batches of 10K queries, beam 1), plus the achieved
fraction of the HBM roofline of the search kernel.  A "step" is one pass of the hot path over one
batch of 10K queries; consecutive steps rotate over NB distinct query batches.

    python bench.py --gpus N --steps K --warmup W             # this repo (GPU), default workload C2
    python bench.py --workload c3_1Mx768_f16_ip               # BASELINE configs[2]
    python bench.py --workload c4_10Mx128_i8_pq32             # BASELINE configs[3] (PQ traversal + rerank)
    python bench.py --impl reference --steps K --warmup W     # CPU restatement of the reference path

value : device-timed QPS with the queries already resident in HBM (dab_search_batch*_device)
e2e   : the same through the reference-facing C-ABI call with pinned HOST buffers
        (H2D of the queries and D2H of ids/distances inside the timed region)
Every GPU arm ends with a parity gate outside the timed region: >= 1024 queries of the timed
batches are re-run by the CPU oracle on the same index and must match bit for bit (ids, distance
bits, result counts, cmps, hops).
Multi-GPU: one process per GPU (torchrun); rank 0 builds the index, vectors and adjacency are
replicated with NCCL broadcasts at load, every rank searches its own query shard with no
collective on the search path.  --scaling weak: 10K queries per GPU; --scaling strong: 10K in total.
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1]
    "c2_1Mx128_f32_l2": dict(n=1_000_000, dim=128, dtype="f32", metric="l2", nq=10_000, centers=1024, R=64, l_build=100,
                             l_search=100, path="fp"),
    # configs[2]: text-embedding shape, unit-normalised rows cast to f16, inner product
    "c3_1Mx768_f16_ip": dict(n=1_000_000, dim=768, dtype="f16", metric="ip", nq=10_000, centers=1024, R=64, l_build=100,
                             l_search=100, path="fp", normalize=True),
    # configs[3]: i8 rows, PQ 32 x 256 traversal (codes are the only rows read per candidate) + full-precision rerank
    "c4_10Mx128_i8_pq32": dict(n=10_000_000, dim=128, dtype="i8", metric="l2", nq=10_000, centers=4096, R=64, l_build=100,
                               l_search=100, path="pq", pq_chunks=32, pq_train=256_000, int_scale=25.0),
    # configs[4] shape (index replicated per GPU); --n-points scales it to what the run window allows
    "c5_100Mx96_f32_l2": dict(n=100_000_000, dim=96, dtype="f32", metric="l2", nq=10_000, centers=16384, R=64, l_build=100,
                              l_search=100, path="fp"),
    "small_100Kx128_f32_l2": dict(n=100_000, dim=128, dtype="f32", metric="l2", nq=10_000, centers=256, R=64, l_build=100,
                                  l_search=100, path="fp"),
    "small_200Kx128_i8_pq32": dict(n=200_000, dim=128, dtype="i8", metric="l2", nq=10_000, centers=256, R=64, l_build=100,
                                   l_search=100, path="pq", pq_chunks=32, pq_train=50_000, int_scale=25.0),
}
ALPHA = 1.2
K = 10
TARGET_RECALL = 0.95
NB = 4            # distinct query batches rotated through the timed loop
PARITY_PER_BATCH = 256
L_SWEEP = [10, 15, 20, 25, 30, 40, 50, 60, 70, 80, 90, 100, 120, 140, 160, 200, 250]
L_SWEEP_PQ = L_SWEEP + [300, 350, 400, 450, 500, 600, 700, 800, 900, 1000]  # the PQ traversal kernels hold lists of up to 1024 entries
SEED_BASE, SEED_QUERY, SEED_PQ = 0xD15C0003, 0xD15C0004, 13076402859301299683  # PQ seed of example/product.json
NP_DTYPE = {"f32": np.float32, "f16": np.float16, "i8": np.int8}
ELEM = {"f32": 4, "f16": 2, "i8": 1}


def max_degree(R):
    return int(R * 1.3)  # graph slack factor, diskann/src/graph/config/defaults.rs:26


def make_centers(cfg):
    return np.random.default_rng(SEED_BASE ^ 0xC0FFEE).standard_normal((cfg["centers"], cfg["dim"]), dtype=np.float32)


def make_data(cfg, seed, count, centers):
    """Clustered Gaussians (SURVEY.md §8d): centre ~ N(0, I), point = centre + 0.3 N(0, I); C3: rows
    normalised to unit length and cast to f16; C4: scaled by `int_scale`, rounded, clamped to [-127, 127]."""
    rng = np.random.default_rng(seed)
    out = np.empty((count, cfg["dim"]), NP_DTYPE[cfg["dtype"]])
    step = 1 << 17
    for i in range(0, count, step):
        m = min(step, count - i)
        which = rng.integers(0, centers.shape[0], m)
        x = centers[which] + np.float32(0.3) * rng.standard_normal((m, cfg["dim"]), dtype=np.float32)
        if cfg.get("normalize"):
            x /= np.maximum(np.sqrt((x * x).sum(1, dtype=np.float32, keepdims=True)), np.float32(1e-12))
        if cfg["dtype"] == "i8":
            x = np.clip(np.rint(x * np.float32(cfg["int_scale"])), -127, 127)
        out[i:i + m] = x
    return out


def find_medoid(base):
    """Start point = copy of the data point closest (squared L2) to the mean (start_point_strategy: medoid)."""
    mean = np.zeros(base.shape[1], np.float64)
    step = 1 << 18
    for i in range(0, base.shape[0], step):
        mean += base[i:i + step].astype(np.float32).sum(0, dtype=np.float64)
    mean = (mean / base.shape[0]).astype(np.float32)
    best, best_i = np.inf, 0
    for i in range(0, base.shape[0], step):
        d = ((base[i:i + step].astype(np.float32) - mean) ** 2).sum(1)
        j = int(np.argmin(d))
        if d[j] < best:
            best, best_i = float(d[j]), i + j
    return base[best_i].copy()


def host_cores():
    """Threads the CPU arm may really use: scheduler affinity capped by the cgroup CPU quota."""
    hw = os.cpu_count() or 1
    try:
        aff = len(os.sched_getaffinity(0))
    except AttributeError:
        aff = hw
    quota = None
    try:
        txt = open("/sys/fs/cgroup/cpu.max").read().split()
        if txt[0] != "max":
            quota = float(txt[0]) / float(txt[1])
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    use = aff if quota is None else max(1, min(aff, int(math.ceil(quota))))
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return {"threads": use, "cores_affinity": aff, "cores_hw": hw, "cgroup_cpu_quota": quota, "cpu_model": model}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 8 for n, v in zip(names, r[4:8]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def unit_bytes(cfg):
    """SURVEY.md §8d: algorithmic bytes of one (query, candidate) distance."""
    if cfg["path"] == "pq":
        return cfg["pq_chunks"] + 8                       # code bytes + id + output (C4-pq: 40 B)
    return cfg["dim"] * ELEM[cfg["dtype"]] + 8            # row bytes + id + output (C2 520, C3 1544, C5 392)


def algorithmic_bytes(cfg, cmps, hops, nq, md, rerank_rows=0):
    """per query: cmps * unit + hops * (max_degree + 1) * 4 + query bytes + k * 8 (+ rerank rows)."""
    qbytes = cfg["dim"] * ELEM[cfg["dtype"]]
    return float(cmps * unit_bytes(cfg) + hops * (md + 1) * 4 + nq * (qbytes + K * 8) + rerank_rows * (qbytes + 8))


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload):
    """DRAM bytes (read + write) of one launch of the workload's search kernel from the committed `ncu --set full`
    capture (profiles/traffic.json: {workload: {search_kernel_dram_bytes_per_launch, source, kernel}}), else None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        t = json.load(open(p))
    except Exception:
        return None
    if "search_kernel_dram_bytes_per_launch" in t:  # round-1 layout: one entry, the C2 kernel
        t = {t.get("workload", "c2_1Mx128_f32_l2"): t}
    e = t.get(workload)
    return e.get("search_kernel_dram_bytes_per_launch") if isinstance(e, dict) else None


def metric_name(cfg):
    if cfg["path"] == "pq":
        return (f"QPS @ recall@10>=0.95, {cfg['n'] // 1_000_000}Mx{cfg['dim']} {cfg['dtype']} + PQ-{cfg['pq_chunks']}x8 "
                f"(Vamana R={cfg['R']} greedy search over ADC distances + full-precision rerank, batch 10K)")
    n = cfg["n"]
    ns = f"{n // 1_000_000}M" if n >= 1_000_000 else f"{n // 1000}K"
    return (f"QPS @ recall@10>=0.95, {ns}x{cfg['dim']} {cfg['dtype']} {cfg['metric'].upper()} "
            f"(Vamana R={cfg['R']} greedy search, batch 10K)")


def common_config(cfg, args, l_search, recall, cmps_mean, hops_mean, min_l, nq_step):
    """Keys shared verbatim by both arms (the driver compares the two dicts)."""
    md = max_degree(cfg["R"])
    return {"workload": args.workload, "n_points": cfg["n"], "dim": cfg["dim"], "elem": cfg["dtype"], "metric": cfg["metric"].upper(),
            "queries_per_step": nq_step, "query_batches_rotated": NB, "pruned_degree": cfg["R"], "max_degree": md,
            "l_build": cfg["l_build"], "alpha": ALPHA, "k": K, "l_search": l_search, "beam_width": 1,
            "search_path": "pq_adc_traversal+fp_rerank" if cfg["path"] == "pq" else "full_precision",
            "recall_at_10": round(recall, 5), "mean_cmps": cmps_mean, "mean_hops": hops_mean, "min_l_for_target_recall": min_l}


def dab_enums(dab, cfg):
    dt = {"f32": dab.DType.f32, "f16": dab.DType.f16, "i8": dab.DType.i8}[cfg["dtype"]]
    mt = {"l2": dab.Metric.L2, "ip": dab.Metric.InnerProduct}[cfg["metric"]]
    return dt, mt


def recall_of(gt_ids, ids, counts):
    hits = 0
    for i in range(ids.shape[0]):
        hits += len(set(gt_ids[i].tolist()) & set(ids[i, :counts[i]].tolist()))
    return hits / (ids.shape[0] * K)


def dump_outputs(out_dir, ids, dists, counts, cmps, hops):
    """--dump-outputs: the arrays one search step returns to its caller, as out_dir/<name>.npy, so that two builds
    run with the same arguments (hence the same seeded inputs) can be compared output for output.  ids and the
    per-query counters are uint32 and stored as float64 (exact); distances stay float32.  A step is at most
    10K queries x k=10, about 1.4 MB in all."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("ids", ids), ("counts", counts), ("cmps", cmps), ("hops", hops)):
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a).view(np.uint32).astype(np.float64))
    np.save(os.path.join(out_dir, "dists.npy"), np.ascontiguousarray(dists, np.float32))


# ------------------------------------------------------------------------------------------ index preparation (GPU)

def prepare_index(g, cfg, base, medoid, rank, world, dist, torch, log):
    """Rank 0: upload, device build (+ PQ training / encoding).  Then ONE NCCL broadcast per resident
    buffer (vectors, adjacency, PQ table + codes) from rank 0, issued inside the library
    (dab_comm_init / dab_broadcast_index); torch.distributed only ships the 128-byte NCCL id."""
    n = cfg["n"]
    t = {}
    t0 = time.time()
    if rank == 0:
        g.upload_vectors(base)
        g.upload_vectors(medoid[None, :], first=n)
    t["upload_s"] = round(time.time() - t0, 2)
    t0 = time.time()
    if rank == 0:
        g.build(cfg["R"], cfg["l_build"], ALPHA)
    t["build_s"] = round(time.time() - t0, 2)
    if cfg["path"] == "pq" and rank == 0:
        t0 = time.time()
        rng = np.random.default_rng(SEED_PQ & 0xFFFFFFFF)
        sample = np.sort(rng.choice(n, size=min(cfg["pq_train"], n), replace=False))
        g.pq_train(base[sample].astype(np.float32), cfg["pq_chunks"], 256, 5, SEED_PQ)
        t["pq_train_s"] = round(time.time() - t0, 2)
        t0 = time.time()
        g.pq_encode_all()
        t["pq_encode_s"] = round(time.time() - t0, 2)
    if world > 1:
        t0 = time.time()
        ident = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            ident.copy_(torch.frombuffer(bytearray(g.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(ident, src=0)
        g.comm_init(bytes(ident.cpu().numpy().tobytes()), world, rank)
        g.broadcast_index(0)
        if cfg["path"] == "pq":
            g.pq_chunks, g.pq_centers = cfg["pq_chunks"], 256
        t["replicate_s"] = round(time.time() - t0, 2)
    adj_host = g.download_graph() if rank == 0 else None
    pq = g.download_pq() if (cfg["path"] == "pq" and rank == 0) else None
    return adj_host, pq, t


# ------------------------------------------------------------------------------------------ GPU arm

def run_gpu(args):
    import torch
    import torch.distributed as dist

    import diskann_b200 as dab

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # whatever NCCL logs, stdout stays the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cfg = dict(WORKLOADS[args.workload])
    if args.n_points:
        cfg["n"] = args.n_points
    n, dim, R = cfg["n"], cfg["dim"], cfg["R"]
    md = max_degree(R)
    strong = args.scaling == "strong"
    nq_total = cfg["nq"] if strong else cfg["nq"] * world
    from diskann_b200.sharding import partition, max_over_ranks
    lo_hi = partition(nq_total, world)  # PartitionIter (benchmark-core/src/search/api.rs:410-419): contiguous ranges
    bounds = [lo for lo, _ in lo_hi] + [lo_hi[-1][1]]
    nq = bounds[rank + 1] - bounds[rank]
    log = (lambda *a: print(*a, file=sys.stderr, flush=True)) if rank == 0 else (lambda *a: None)

    t0 = time.time()
    centers = make_centers(cfg)
    base = make_data(cfg, SEED_BASE, n, centers) if rank == 0 else None  # other ranks receive the rows by broadcast
    medoid = find_medoid(base) if base is not None else None
    # NB distinct global batches; this rank owns rows [bounds[rank], bounds[rank+1]) of each
    batches = [make_data(cfg, SEED_QUERY + 97 * b, nq_total, centers)[bounds[rank]:bounds[rank + 1]] for b in range(NB)]
    t_data = time.time() - t0
    log(f"[bench] data {t_data:.1f}s")

    dt, mt = dab_enums(dab, cfg)
    g = dab.GpuIndex(dt, mt, dim, n, 1, md, device=local)
    # a real (non-default) stream shared by torch and the library, so the CUDA events below are
    # recorded on the stream the kernels are launched on
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    g.set_stream(stream.cuda_stream)
    adj_host, pq, t_prep = prepare_index(g, cfg, base, medoid, rank, world, dist, torch, log)
    log(f"[bench] index {t_prep}")
    is_pq = cfg["path"] == "pq"

    def search_host(q, L):
        return g.search_batch_pq(q, K, L, 1, rerank=True) if is_pq else g.search_batch(q, K, L, 1)

    # ground truth: exhaustive scan on the device (bit-identical distances), cross-checked below
    t0 = time.time()
    # (large indexes: the tcgen05 scan — tensor-core candidate selection + exact re-scoring, same answer)
    flat = g.flat_knn_tc if n >= 2_000_000 else g.flat_knn
    gts = [flat(q, K)[0] for q in batches]
    t_gt = time.time() - t0

    # BASELINE.json names L_search=100; the sweep records the smallest L that already reaches the
    # recall target (reported, and used instead only if L=100 itself misses it)
    sweep, min_l = [], None
    l_search = args.l_search or cfg["l_search"]
    if rank == 0 and not args.l_search:
        for L in (L_SWEEP_PQ if is_pq else L_SWEEP):
            ids, _, counts, cmps, hops = search_host(batches[0], L)
            r = recall_of(gts[0], ids, counts)
            sweep.append({"l": L, "recall": round(r, 5), "mean_cmps": float(cmps.mean()), "mean_hops": float(hops.mean())})
            if r >= TARGET_RECALL:
                min_l = L
                break
        if min_l is None:
            min_l = (L_SWEEP_PQ if is_pq else L_SWEEP)[-1]
        if min_l > l_search:
            l_search = min_l
    if world > 1:
        t = torch.tensor([l_search, min_l or 0], device="cuda")
        dist.broadcast(t, src=0)
        l_search, min_l = int(t[0].item()), int(t[1].item()) or None

    # resident inputs / outputs for `value`
    d_q = [torch.from_numpy(q).cuda() for q in batches]
    d_ids = torch.empty((nq, K), dtype=torch.int32, device="cuda")
    d_dists = torch.empty((nq, K), dtype=torch.float32, device="cuda")
    d_counts = torch.empty(nq, dtype=torch.int32, device="cuda")
    d_cmps = torch.empty(nq, dtype=torch.int32, device="cuda")
    d_hops = torch.empty(nq, dtype=torch.int32, device="cuda")
    # pinned host buffers for `e2e` (the C-ABI call a Rust caller makes)
    h_q = [torch.from_numpy(q).pin_memory() for q in batches]
    h_ids = torch.empty((nq, K), dtype=torch.int32).pin_memory()
    h_dists = torch.empty((nq, K), dtype=torch.float32).pin_memory()
    lib = dab.lib()
    step_no = [0]

    def step_device(L=None):
        b = step_no[0] % NB
        step_no[0] += 1
        fn = g.search_batch_pq_device if is_pq else g.search_batch_device
        fn(d_q[b].data_ptr(), nq, K, L or l_search, 1, d_ids.data_ptr(), d_dists.data_ptr(), d_counts.data_ptr(),
           d_cmps.data_ptr(), d_hops.data_ptr())

    def step_e2e():
        b = step_no[0] % NB
        step_no[0] += 1
        if is_pq:
            dab._lib.check(lib.dab_search_batch_pq_rerank(g._h, C.c_void_p(h_q[b].data_ptr()), nq, K, l_search, 1,
                                                          C.c_void_p(h_ids.data_ptr()), C.c_void_p(h_dists.data_ptr()), None, None, None))
        else:
            dab._lib.check(lib.dab_search_batch(g._h, C.c_void_p(h_q[b].data_ptr()), nq, K, l_search, 1, C.c_void_p(h_ids.data_ptr()),
                                                C.c_void_p(h_dists.data_ptr()), None, None, None))

    # ---- batches in flight (dab_search_batch_async / dab_wait): SLOTS consecutive steps overlap, each on its own
    # slot (stream + visited tables + result buffers), so the draining tail of one batch is filled by the CTAs of
    # the next and, end to end, the copies of one batch run under the kernel of another
    # default: two batches in flight; a strong-scaled shard smaller than half the resident workers (~3400 one-warp
    # CTAs) keeps four, so that consecutive 10K-query steps still fill the GPU (profiles/r02_nq_sweep_strong_scaling_shares.txt)
    in_flight = args.in_flight or (4 if nq < 5000 else 2)
    slots = 1 if is_pq else max(1, min(in_flight, dab.MAX_SLOTS))
    sd = [dict(ids=torch.empty((nq, K), dtype=torch.int32, device="cuda"), dists=torch.empty((nq, K), dtype=torch.float32, device="cuda"),
               counts=torch.empty(nq, dtype=torch.int32, device="cuda"), cmps=torch.empty(nq, dtype=torch.int32, device="cuda"),
               hops=torch.empty(nq, dtype=torch.int32, device="cuda"),
               h_ids=torch.empty((nq, K), dtype=torch.int32).pin_memory(), h_dists=torch.empty((nq, K), dtype=torch.float32).pin_memory())
          for _ in range(slots)] if slots > 1 else []

    def step_device_async():
        i = step_no[0]
        step_no[0] += 1
        s, b = i % slots, i % NB
        g.wait(s)
        o = sd[s]
        g.search_batch_device_async(s, d_q[b].data_ptr(), nq, K, l_search, 1, o["ids"].data_ptr(), o["dists"].data_ptr(),
                                    o["counts"].data_ptr(), o["cmps"].data_ptr(), o["hops"].data_ptr())

    def step_e2e_async():
        i = step_no[0]
        step_no[0] += 1
        s, b = i % slots, i % NB
        g.wait(s)
        o = sd[s]
        dab._lib.check(lib.dab_search_batch_async(g._h, s, C.c_void_p(h_q[b].data_ptr()), nq, K, l_search, 1,
                                                  C.c_void_p(o["h_ids"].data_ptr()), C.c_void_p(o["h_dists"].data_ptr()), None, None, None))

    def drain():
        for s in range(slots):
            g.wait(s)

    def timed(fn, steps, warmup, drain=lambda: None):
        for _ in range(warmup):
            fn()
        drain()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = dab.launch_count()
        e0.record(stream)
        for _ in range(steps):
            fn()
        drain()  # joins every batch in flight (host-side wait), so e1 is recorded after the last kernel has finished
        e1.record(stream)
        torch.cuda.synchronize()
        timed.launches = dab.launch_count() - l0
        ms = e0.elapsed_time(e1)
        if world > 1:
            dist.barrier()
            ms = max_over_ranks(ms, device="cuda")
        return ms

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if args.profile_range:  # ncu --profile-from-start off: only the timed region is captured
        torch.cuda.profiler.start()
    step_no[0] = 0
    ms_dev_serial = timed(step_device, args.steps, args.warmup)
    launches = timed.launches
    # the last step of the loop that `value` times: its buffers are overwritten by the loops and checks that follow
    last_out = [t.cpu().numpy() for t in (d_ids, d_dists, d_counts, d_cmps, d_hops)] if args.dump_outputs else None
    step_no[0] = 0
    ms_e2e_serial = timed(step_e2e, args.steps, args.warmup)
    ms_dev, ms_e2e = ms_dev_serial, ms_e2e_serial
    if slots > 1:
        step_no[0] = 0
        ms_dev = timed(step_device_async, args.steps, args.warmup, drain)
        launches = timed.launches
        if args.dump_outputs:
            o = sd[(args.warmup + args.steps - 1) % slots]
            last_out = [o[f].cpu().numpy() for f in ("ids", "dists", "counts", "cmps", "hops")]
        step_no[0] = 0
        ms_e2e = timed(step_e2e_async, args.steps, args.warmup, drain)
    if args.profile_range:
        torch.cuda.profiler.stop()
    clocks = sampler.stop() if rank == 0 else None

    # ---- what was timed is correct: statistics + recall over all NB batches (host API), the
    # device-resident path agrees with it, and the parity gate against the CPU oracle
    res = [search_host(q, l_search) for q in batches]
    cmps_sum = float(sum(r[3].astype(np.float64).sum() for r in res))
    hops_sum = float(sum(r[4].astype(np.float64).sum() for r in res))
    recall = float(np.mean([recall_of(gts[b], res[b][0], res[b][2]) for b in range(NB)]))
    step_no[0] = 0
    step_device()
    torch.cuda.synchronize()
    assert np.array_equal(d_ids.cpu().numpy().view(np.uint32), res[0][0]), "device-resident and host C-ABI results differ"
    if slots > 1:  # what the pipelined loops left in their buffers is the answer of the batch each slot ran last
        for s_ in range(slots):
            last = max(i for i in range(args.warmup + args.steps) if i % slots == s_) % NB
            assert np.array_equal(sd[s_]["h_ids"].numpy().view(np.uint32), res[last][0]), "async host-buffer results differ"
            assert np.array_equal(sd[s_]["h_dists"].numpy().view(np.uint32), res[last][1].view(np.uint32)), "async host-buffer distances differ"
        step_no[0] = 0
        for _ in range(slots):
            step_device_async()
        drain()
        for s_ in range(slots):
            assert np.array_equal(sd[s_]["ids"].cpu().numpy().view(np.uint32), res[s_ % NB][0]), "async device-resident results differ"
            assert np.array_equal(sd[s_]["cmps"].cpu().numpy().view(np.uint32), res[s_ % NB][3]), "async device-resident cmps differ"
    if world > 1:  # recall is asserted on the worst rank
        t = torch.tensor([recall], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        recall_min = float(t.item())
        t = torch.tensor([cmps_sum, hops_sum], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        cmps_all, hops_all = float(t[0].item()), float(t[1].item())
    else:
        recall_min, cmps_all, hops_all = recall, cmps_sum, hops_sum

    parity = None
    if rank == 0 and not args.no_parity:
        parity = parity_gate(cfg, base, medoid, adj_host, pq, batches, gts, res, l_search)

    at_min_l = None
    if rank == 0 and min_l and min_l != l_search:  # informative only
        for _ in range(3):
            step_device(min_l)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            step_device(min_l)
        e1.record(stream)
        torch.cuda.synchronize()
        ms_min = e0.elapsed_time(e1) / args.steps
        at_min_l = {"l_search": min_l, "ms_per_step": ms_min, "queries_per_s_this_gpu": nq / (ms_min / 1e3)}

    ms_step = ms_dev / args.steps
    value = nq_total / (ms_step / 1e3)
    e2e_value = nq_total / ((ms_e2e / args.steps) / 1e3)
    # algorithmic bytes of ONE step on this rank = mean over the rotated batches
    rerank_rows = (l_search * nq) if is_pq else 0
    alg_bytes = algorithmic_bytes(cfg, cmps_sum / NB, hops_sum / NB, nq, md, rerank_rows)
    peak, peak_src = measured_peak_gbs()
    achieved = alg_bytes / (ms_step / 1e3) / 1e9

    result = None
    if rank == 0:
        conf = common_config(cfg, args, l_search, recall_min, cmps_all / (NB * nq_total), hops_all / (NB * nq_total), min_l, nq_total)
        conf.update({
            "queries_per_gpu": nq, "scaling_mode": args.scaling,
            "generator": f"{cfg['centers']} Gaussian centres N(0,I), point = centre + 0.3 N(0,I)"
                         + (", unit-normalised, cast to f16" if cfg.get("normalize") else "")
                         + (f", x{cfg['int_scale']} rounded and clamped to i8" if cfg["dtype"] == "i8" else "")
                         + f"; seeds base {SEED_BASE:#x} queries {SEED_QUERY:#x}+97*batch; start = copy of the medoid",
            "index": "built on rank 0 by dab_build (device); vectors, adjacency (and PQ) replicated by one NCCL broadcast each inside the library",
            "parallelism": f"replica x{world}, queries sharded ({args.scaling}), no collective on the search path",
            "l2_policy": f"no flush: index {(n * dim * ELEM[cfg['dtype']] + (n + 1) * 4 * (md + 1)) / 1e6:.0f} MB >> 126 MB L2, "
                         f"{NB} query batches rotate and each step gathers GBs of random rows",
            "batches_in_flight": slots,
            "serial": {"ms_per_step": ms_dev_serial / args.steps, "e2e_ms_per_step": ms_e2e_serial / args.steps,
                       "roofline_frac": alg_bytes / (ms_dev_serial / args.steps / 1e3) / 1e9 / peak,
                       "note": "one batch at a time (dab_search_batch_device / dab_search_batch): launch, wait, next"},
            "setup_s": dict(t_prep, data=round(t_data, 1), ground_truth=round(t_gt, 2)),
            "l_sweep": sweep, "at_min_l": at_min_l, "parity_gate": parity})
        kernel = ("search_kernel_pqs + rerank_kernel" if is_pq else "search_kernel_v3 / v2") + f"<{cfg['dtype']},{cfg['metric'].upper()}>"
        result = {
            "metric": metric_name(cfg), "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": cfg["dtype"], "data": "synthetic", "config": conf, "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": nq * dim * ELEM[cfg["dtype"]],
                    "d2h_bytes_per_step": nq * K * 8, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic(args.workload), "kernel": kernel, "algorithmic_bytes_per_launch": alg_bytes,
                         "peak_source": peak_src,
                         "note": f"achieved = algorithmic bytes (cmps*{unit_bytes(cfg)} + hops*{(md + 1) * 4} + query + k*8 per query"
                                 + (" + L rerank rows" if is_pq else "") + ", run's own counters, mean over the rotated batches) "
                                 "/ CUDA-event step time on this rank (timed region / steps; with batches_in_flight > 1 "
                                 "consecutive launches overlap, config.serial has the one-at-a-time figure)"},
        }
        if not args.no_cpu_baseline and world == 1:
            result["cpu_baseline"] = cpu_baseline(cfg, base, medoid, adj_host, pq, batches, gts, l_search)
    g.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        if args.dump_outputs:  # with several GPUs: rank 0's query shard
            dump_outputs(args.dump_outputs, *last_out)
        emit(result)


# ------------------------------------------------------------------------------------------ CPU oracle legs

def oracle_index(cfg, base, medoid, adj, pq):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O  # the CPU checker: only the parity gate and the CPU baseline legs use it
    vecs = np.concatenate([base, medoid[None, :]])
    mt = {"l2": O.L2, "ip": O.INNER_PRODUCT}[cfg["metric"]]
    return O, O.Index(vecs, adj, cfg["n"], 1, mt, pq=pq)


def oracle_search(cfg, oidx, q, l_search, threads):
    if cfg["path"] == "pq":
        return oidx.search_batch_rerank(q, K, l_search, threads=threads)
    return oidx.search_batch(q, K, l_search, threads=threads)


def parity_gate(cfg, base, medoid, adj, pq, batches, gts, res, l_search):
    """>= 1024 queries of the timed batches on the CPU oracle, same index, same L: bit-identical ids,
    distances, counts, cmps, hops.  Also cross-checks the device ground truth on a sample with the
    oracle's brute force."""
    O, oidx = oracle_index(cfg, base, medoid, adj, pq)
    threads = host_cores()["threads"]
    t0 = time.time()
    checked = 0
    for b, q in enumerate(batches):
        m = min(PARITY_PER_BATCH, q.shape[0])
        want = oracle_search(cfg, oidx, q[:m], l_search, threads)
        for name, a, w in zip(("ids", "dists", "counts", "cmps", "hops"), res[b], want):
            if not np.array_equal(np.ascontiguousarray(a[:m]).view(np.uint32), np.ascontiguousarray(w).view(np.uint32)):
                bad = int(np.argmax((np.ascontiguousarray(a[:m]).view(np.uint32) != np.ascontiguousarray(w).view(np.uint32)).reshape(m, -1).any(1)))
                raise SystemExit(f"bench.py: PARITY FAILED at full scale: batch {b} query {bad}: GPU {name} differ from the oracle")
        checked += m
    gt_n = min(8, batches[0].shape[0])
    mt = {"l2": O.L2, "ip": O.INNER_PRODUCT}[cfg["metric"]]
    want_gt, _ = O.bruteforce_knn(base, batches[0][:gt_n], mt, K, threads=threads)
    if not np.array_equal(want_gt, gts[0][:gt_n]):
        raise SystemExit("bench.py: device ground truth differs from the oracle's brute force")
    return {"queries_checked": checked, "fields": "ids,dists(bits),counts,cmps,hops", "result": "bit-identical",
            "ground_truth_cross_check": f"{gt_n} queries vs oracle brute force: identical", "seconds": round(time.time() - t0, 1)}


def cpu_baseline(cfg, base, medoid, adj, pq, batches, gts, l_search):
    """The CPU restatement of the reference path (AVX2, reference threading model: contiguous
    query partitions, one thread each) on the host cores this process may use."""
    O, oidx = oracle_index(cfg, base, medoid, adj, pq)
    hc = host_cores()
    threads = hc["threads"]
    q = batches[0]
    t0 = time.perf_counter()
    ids, _, counts, _, _ = oracle_search(cfg, oidx, q, l_search, threads)
    first = time.perf_counter() - t0
    best, reps = first, 1
    while reps < 3 and first * (reps + 1) < 25.0:
        t0 = time.perf_counter()
        oracle_search(cfg, oidx, batches[reps % NB], l_search, threads)
        best = min(best, time.perf_counter() - t0)
        reps += 1
    t0 = time.perf_counter()
    oracle_search(cfg, oidx, q[:200], l_search, 1)
    dt1 = time.perf_counter() - t0
    out = {"value": q.shape[0] / best, "unit": "queries/s", "cores": threads, "kind": "port",
           "sample": f"{reps} batch(es) of {q.shape[0]} queries (best), same graph / L as the GPU arm, AVX2 V3-order kernels, "
                     f"{threads} threads",
           "recall_at_10": round(recall_of(gts[0], ids, counts), 5), "single_thread_qps": 200 / dt1}
    out.update({k: hc[k] for k in ("cores_affinity", "cores_hw", "cgroup_cpu_quota", "cpu_model")})
    return out


# ------------------------------------------------------------------------------------------ reference arm

def prepare_only(args):
    """Child process of --impl reference: builds the graph (and PQ tables, ground truth, L sweep) on the
    GPU and leaves them as .npy files, so that the timed CPU process never maps the CUDA library."""
    import diskann_b200 as dab
    cfg = dict(WORKLOADS[args.workload])
    if args.n_points:
        cfg["n"] = args.n_points
    n, dim, md = cfg["n"], cfg["dim"], max_degree(cfg["R"])
    centers = make_centers(cfg)
    base = make_data(cfg, SEED_BASE, n, centers)
    medoid = find_medoid(base)
    queries = make_data(cfg, SEED_QUERY, cfg["nq"], centers)
    dt, mt = dab_enums(dab, cfg)
    g = dab.GpuIndex(dt, mt, dim, n, 1, md)
    adj, pq, _ = prepare_index(g, cfg, base, medoid, 0, 1, None, None, lambda *a: None)
    flat = g.flat_knn_tc if n >= 2_000_000 else g.flat_knn
    gt_all = [flat(make_data(cfg, SEED_QUERY + 97 * b, cfg["nq"], centers), K)[0] for b in range(NB)]
    l_search = args.l_search or cfg["l_search"]
    min_l = None
    if not args.l_search:
        for L in (L_SWEEP_PQ if cfg["path"] == "pq" else L_SWEEP):
            r = g.search_batch_pq(queries, K, L, 1, rerank=True) if cfg["path"] == "pq" else g.search_batch(queries, K, L, 1)
            min_l = L
            if recall_of(gt_all[0], r[0], r[2]) >= TARGET_RECALL:
                break
        if min_l > l_search:
            l_search = min_l
    g.close()
    np.save(os.path.join(args.prepare_only, "adj.npy"), adj)
    np.save(os.path.join(args.prepare_only, "gt.npy"), np.stack(gt_all))
    if pq is not None:
        for i, a in enumerate(pq):
            np.save(os.path.join(args.prepare_only, f"pq{i}.npy"), a)
    json.dump({"l_search": l_search, "min_l": min_l}, open(os.path.join(args.prepare_only, "meta.json"), "w"))


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle restatement; the Rust workspace cannot be
    compiled here) on the host cores.  The graph is input data: it is produced once by the device
    build in a CHILD process (untimed; a sequential CPU build of 1M points would take hours), so the
    timed process maps only the oracle."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = dict(WORKLOADS[args.workload])
    if args.n_points:
        cfg["n"] = args.n_points
    n, nq = cfg["n"], cfg["nq"]
    with tempfile.TemporaryDirectory(prefix="dab_bench_") as tmp:
        env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT")}
        cmd = [sys.executable, os.path.abspath(__file__), "--prepare-only", tmp, "--workload", args.workload]
        if args.n_points:
            cmd += ["--n-points", str(args.n_points)]
        if args.l_search:
            cmd += ["--l-search", str(args.l_search)]
        cp = subprocess.run(cmd, env=env, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True)
        if cp.returncode != 0:
            emit({"impl": "reference", "unavailable": "no GPU to prepare the graph input for the CPU arm: "
                  + (cp.stderr.strip().splitlines() or ["child failed"])[-1][:200]})
            return
        adj = np.load(os.path.join(tmp, "adj.npy"))
        gts = np.load(os.path.join(tmp, "gt.npy"))
        meta = json.load(open(os.path.join(tmp, "meta.json")))
        pq = tuple(np.load(os.path.join(tmp, f"pq{i}.npy")) for i in range(3)) if cfg["path"] == "pq" else None
    l_search, min_l = meta["l_search"], meta["min_l"]
    centers = make_centers(cfg)
    base = make_data(cfg, SEED_BASE, n, centers)
    medoid = find_medoid(base)
    batches = [make_data(cfg, SEED_QUERY + 97 * b, nq, centers) for b in range(NB)]
    O, oidx = oracle_index(cfg, base, medoid, adj, pq)
    hc = host_cores()
    threads = hc["threads"]
    # each step = a bounded sample of one batch, sized so that the whole run stays within minutes
    t0 = time.perf_counter()
    oracle_search(cfg, oidx, batches[0][:max(64, threads * 8)], l_search, threads)
    probe_qps = max(64, threads * 8) / (time.perf_counter() - t0)
    budget_s = 150.0 / max(1, args.steps + args.warmup)
    m = int(min(nq, max(threads * 16, probe_qps * budget_s)))
    step = [0]

    def one():
        b = step[0] % NB
        step[0] += 1
        return b, oracle_search(cfg, oidx, batches[b][:m], l_search, threads)

    for _ in range(args.warmup):
        one()
    step[0] = 0
    t0 = time.perf_counter()
    outs = [one() for _ in range(args.steps)]
    dt = (time.perf_counter() - t0) / args.steps
    qps = m / dt
    rec = float(np.mean([recall_of(gts[b][:m], r[0], r[2]) for b, r in outs[:NB]]))
    cm = float(np.mean([r[3].mean() for _, r in outs[:NB]]))
    hp = float(np.mean([r[4].mean() for _, r in outs[:NB]]))
    conf = common_config(cfg, args, l_search, rec, cm, hp, min_l, cfg["nq"])
    conf["sample_queries_per_step"] = m
    cb = {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port",
          "sample": f"each step = the first {m} queries of one of {NB} rotating 10K batches on {threads} threads (contiguous partitions)"}
    cb.update({k: hc[k] for k in ("cores_affinity", "cores_hw", "cgroup_cpu_quota", "cpu_model")})
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *outs[-1][1])
    emit({"impl": "reference", "metric": metric_name(cfg), "value": qps, "unit": "queries/s", "n_gpus": args.gpus,
          "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
          "scaling": args.scaling, "vs_baseline": None, "dtype": cfg["dtype"], "data": "synthetic", "config": conf,
          "cpu_baseline": cb, "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


_REAL_STDOUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries loaded later (NCCL prints its version
    banner there) write to file descriptor 1 directly, so fd 1 is pointed at stderr for the rest
    of the process and the JSON line goes to a private duplicate of the original stdout."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(obj):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2_1Mx128_f32_l2", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--n-points", type=int, default=0, help="override the workload's point count (C5-shaped runs)")
    ap.add_argument("--l-search", type=int, default=0, help="skip the sweep and use this L")
    ap.add_argument("--in-flight", type=int, default=0, help="batches kept in flight by the timed loops (1: one at a time; default 2, or 4 for shards of < 5000 queries)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle parity gate (tuning runs only)")
    ap.add_argument("--profile-range", action="store_true", help="cudaProfilerStart/Stop around the timed region (for ncu)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the result arrays of the last one as DIR/<name>.npy")
    ap.add_argument("--prepare-only", default="", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.prepare_only:
        prepare_only(args)
        return
    claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
