"""bench.py contract pieces that can be checked without a GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_algorithmic_bytes_follows_the_survey_formula():
    # SURVEY.md §8d: cmps*(d*sizeof(T)+8) + hops*(max_degree+1)*4 + d*sizeof(T) + k*8 per query
    c2 = bench.WORKLOADS["c2_1Mx128_f32_l2"]
    assert bench.unit_bytes(c2) == 520
    assert bench.algorithmic_bytes(c2, 3000, 210, 2, 83) == 3000 * 520 + 210 * 336 + 2 * (512 + 80)
    assert bench.unit_bytes(bench.WORKLOADS["c3_1Mx768_f16_ip"]) == 1544
    c4 = bench.WORKLOADS["c4_10Mx128_i8_pq32"]
    assert bench.unit_bytes(c4) == 40  # 32 code bytes + id + output
    # PQ traversal + rerank: L full-precision rows (136 B each) per query on top
    assert bench.algorithmic_bytes(c4, 1000, 100, 1, 83, rerank_rows=100) == 1000 * 40 + 100 * 336 + (128 + 80) + 100 * 136
    assert bench.unit_bytes(bench.WORKLOADS["c5_100Mx96_f32_l2"]) == 392


def test_host_cores_respects_affinity():
    hc = bench.host_cores()
    assert 1 <= hc["threads"] <= hc["cores_affinity"] <= hc["cores_hw"]


def test_data_generators():
    cfg = dict(bench.WORKLOADS["c3_1Mx768_f16_ip"], centers=8)
    x = bench.make_data(cfg, 1, 100, bench.make_centers(cfg))
    assert x.dtype == np.float16 and abs(float((x.astype(np.float32) ** 2).sum(1).mean()) - 1.0) < 1e-2
    cfg = dict(bench.WORKLOADS["c4_10Mx128_i8_pq32"], centers=8)
    y = bench.make_data(cfg, 1, 100, bench.make_centers(cfg))
    assert y.dtype == np.int8 and y.min() >= -127 and np.abs(y).max() > 40
    assert np.array_equal(bench.find_medoid(y), y[np.argmin(((y.astype(np.float32) - y.astype(np.float32).mean(0)) ** 2).sum(1))])


def test_max_degree_is_the_reference_slack():
    assert bench.max_degree(64) == 83 and bench.max_degree(32) == 41  # config/mod.rs:269-275


def test_stdout_carries_exactly_one_json_line():
    """Anything a library writes to file descriptor 1 after start-up must not reach stdout."""
    code = ("import os, sys; sys.path.insert(0, %r); import bench; bench.claim_stdout(); "
            "os.write(1, b'library banner\\n'); print('python noise'); bench.emit({'ok': 1})" % ROOT)
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert p.returncode == 0
    assert p.stdout.strip().splitlines() == ['{"ok": 1}']
    assert "library banner" in p.stderr and "python noise" in p.stderr


def test_reference_arm_prints_one_json_line_without_a_gpu():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--workload", "small_100Kx128_f32_l2"], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert p.returncode == 0
    lines = p.stdout.strip().splitlines()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference"


def test_dump_outputs_stores_exact_float_arrays(tmp_path):
    """ids and counters (uint32, the empty-slot id 0xFFFFFFFF included) round-trip exactly through float64."""
    ids = np.array([[3, 0xFFFFFFFF], [0xFFFFFFFE, 7]], np.uint32)
    dists = np.array([[0.5, np.inf], [1e-30, 2.0]], np.float32)
    counters = np.array([1, 2], np.uint32)
    bench.dump_outputs(str(tmp_path / "out"), ids.view(np.int32), dists, counters, counters + 10, counters + 20)
    got = {f[:-4]: np.load(tmp_path / "out" / f) for f in os.listdir(tmp_path / "out")}
    assert sorted(got) == ["cmps", "counts", "dists", "hops", "ids"]
    assert got["dists"].dtype == np.float32 and np.array_equal(got["dists"].view(np.uint32), dists.view(np.uint32))
    for name, want in (("ids", ids), ("counts", counters), ("cmps", counters + 10), ("hops", counters + 20)):
        assert got[name].dtype == np.float64 and np.array_equal(got[name].astype(np.uint32), want), name


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    """--dump-outputs writes one search step's results (k sorted neighbours per query of the timed batch), and a second
    run with the same arguments writes the same arrays."""
    runs = []
    for r in range(2):
        out = tmp_path / f"run{r}"
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "small_100Kx128_f32_l2", "--steps", "5",
                            "--warmup", "3", "--no-cpu-baseline", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stderr[-2000:]
        d = json.loads(p.stdout.strip().splitlines()[-1])
        assert d["steps"] == 5 and d["config"]["parity_gate"]["result"] == "bit-identical"
        runs.append({f: np.load(out / f"{f}.npy") for f in ("ids", "dists", "counts", "cmps", "hops")})
    nq, n = d["config"]["queries_per_step"], d["config"]["n_points"]
    a = runs[0]
    assert a["ids"].shape == (nq, bench.K) and a["dists"].shape == (nq, bench.K) and a["counts"].shape == (nq,)
    assert np.all(a["counts"] == bench.K) and np.all(a["ids"] < n) and np.all(np.diff(a["dists"], axis=1) >= 0)
    assert np.all(a["cmps"] > 0) and np.all(a["hops"] > 0)
    for f in a:
        assert np.array_equal(a[f], runs[1][f]), f


def test_traffic_json_is_keyed_by_workload(tmp_path, monkeypatch):
    """roofline.traffic comes from the committed ncu capture of the workload's own search kernel."""
    assert bench.ncu_traffic("c2_1Mx128_f32_l2") > 1e9 and bench.ncu_traffic("c4_10Mx128_i8_pq32") > 1e9
    assert bench.ncu_traffic("c3_1Mx768_f16_ip") is None  # no capture committed under that key
    t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    for entry in t.values():
        assert os.path.exists(os.path.join(ROOT, entry["source"].split(", ")[1])), entry["source"]
    # round-1 layout (one entry, no key) still reads as the C2 kernel
    (tmp_path / "profiles").mkdir()
    (tmp_path / "profiles" / "traffic.json").write_text(json.dumps({"search_kernel_dram_bytes_per_launch": 7.0}))
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))
    assert bench.ncu_traffic("c2_1Mx128_f32_l2") == 7.0 and bench.ncu_traffic("c4_10Mx128_i8_pq32") is None
