"""bench.py's output contract, checked on the CPU with the reference arm (the one arm that runs without a GPU):
exactly ONE line on stdout, JSON, with the keys the driver reads; and what --dump-outputs writes (on the GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--workload", "c3", "--ref-rows", "3000", "--ref-threads", "2"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "queries/s"
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data",
                "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 2 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0 and "workload" in d["config"]


def test_traffic_table_points_at_committed_captures():
    table = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    for e in table["captures"]:
        assert os.path.exists(os.path.join(ROOT, e["source"])), e["source"]
        assert e["dram_bytes_per_launch"] >= e["algorithmic_streamed_bytes_per_launch"] * 0.99


def test_clustered_corpus_generators_and_reference_arm():
    """--corpus clustered: rows and queries are centre + noise (host and device generators of one family), and the
    reference arm runs on it and says so in the workload name."""
    import importlib.util
    import numpy as np
    import torch
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    b.CORPUS = "clustered"
    dim = 48
    cen = b.centres_host(dim)
    assert cen.shape == (b.N_CENTRES, dim)

    def nearest(x):
        return np.sqrt(((x[:, None, :] - cen[None, :, :]) ** 2).sum(-1)).min(1).mean()

    host, dev, qs = b.gen_chunk_host(5, dim, 400), b.gen_chunk_device(torch, 5, dim, 400, device="cpu").numpy(), b.gen_queries(8, dim)
    want = b.CLUSTER_NOISE * np.sqrt(dim)
    for x in (host, dev, qs):
        assert x.dtype == np.float32 and abs(nearest(x) - want) < 0.15 * want
    assert np.array_equal(host, b.gen_chunk_host(5, dim, 400)) and not np.array_equal(host, b.gen_chunk_host(6, dim, 400))
    b.CORPUS = "gaussian"
    assert nearest(b.gen_chunk_host(5, dim, 400)) > 1.5 * want      # i.i.d. rows sit nowhere near a centre
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--workload", "c3", "--ref-rows", "2000", "--ref-threads", "2", "--corpus", "clustered"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.strip()][0])
    assert "[corpus: clustered]" in d["config"]["workload"] and d["value"] > 0


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    return b


def test_dump_outputs_stays_under_its_limit_with_a_fixed_sample(tmp_path):
    import numpy as np
    b = _bench_module()
    idx = np.arange(5000 * 10, dtype=np.int32).reshape(5000, 10)
    sc = -np.arange(5000 * 10, dtype=np.float32).reshape(5000, 10)
    b.dump_outputs(str(tmp_path / "all"), idx, sc)
    got = {n: np.load(tmp_path / "all" / f"{n}.npy") for n in ("query_rows", "topk_indices", "topk_scores")}
    assert got["topk_indices"].dtype == np.float64 and got["topk_scores"].dtype == np.float32
    assert np.array_equal(got["topk_indices"], idx) and np.array_equal(got["topk_scores"], sc)
    assert np.array_equal(got["query_rows"], np.arange(5000))
    b.DUMP_LIMIT = 1000 * (10 * 12 + 8)
    for d in ("s1", "s2"):
        b.dump_outputs(str(tmp_path / d), idx, sc)
    rows = np.load(tmp_path / "s1" / "query_rows.npy")
    assert rows.shape == (1000,) and np.all(np.diff(rows) > 0)
    assert sum(os.path.getsize(p) for p in (tmp_path / "s1").iterdir()) <= b.DUMP_LIMIT + 3 * 128
    for n in ("query_rows", "topk_indices", "topk_scores"):
        assert np.array_equal(np.load(tmp_path / "s1" / f"{n}.npy"), np.load(tmp_path / "s2" / f"{n}.npy"))
    assert np.array_equal(np.load(tmp_path / "s1" / "topk_indices.npy"), idx[rows.astype(int)])


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_lists_and_repeat(tmp_path):
    """Two runs with the same arguments dump the same lists, and those are the oracle's for the bench's own inputs."""
    import numpy as np
    from oracle import oracle as O
    b = _bench_module()
    n, nq, k, steps = 20000, 64, 10, 2
    lines = []
    for d in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c3", "--rows", str(n),
                              "--nq", str(nq), "--steps", str(steps), "--warmup", "1", "--no-cpu",
                              "--dump-outputs", str(tmp_path / d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        lines.append(json.loads([l for l in out.stdout.splitlines() if l.strip()][0]))
    assert [l["steps"] for l in lines] == [steps, steps]
    dumps = [{m: np.load(tmp_path / d / f"{m}.npy") for m in ("query_rows", "topk_indices", "topk_scores")}
             for d in ("a", "b")]
    for m in dumps[0]:
        assert np.array_equal(dumps[0][m], dumps[1][m]), m
    idx, sc = dumps[0]["topk_indices"], dumps[0]["topk_scores"]
    assert idx.shape == sc.shape == (nq, k) and np.array_equal(dumps[0]["query_rows"], np.arange(nq))
    w = b.WORKLOADS["c3"]
    rows = np.concatenate([b.gen_chunk_host(c, w["dim"], min(b.CHUNK, n - c * b.CHUNK)) for c in range(-(-n // b.CHUNK))])
    oidx = O.quantize_vectors(rows, sim=w["sim"], centroid=np.zeros(w["dim"], np.float32), want_unpacked=False)
    qs = b.gen_queries(nq, w["dim"])
    for i in (0, 31, 63):
        wi, ws = O.search_nearest_neighbors(qs[i], oidx, k, mode="canonical")
        assert idx[i].tolist() == wi.tolist() and sc[i].view(np.uint32).tolist() == ws.view(np.uint32).tolist()
