"""Search throughput of a device group (bbq_group_search: one process, one caller thread, one worker per GPU) at 1, 2,
4 and 8 GPUs on a C4-shaped search: 1024-d COSINE rows, 4096-query batches, k = 100.

The corpus is N seeded N(0,1) rows in host memory (--rows; one copy, sliced by the group), built with
bbq_group_index_build, or an image written by the sharded tools (--image PREFIX, loaded with bbq_group_index_load).
Per group size, one JSON line:

  build_s           wall time of the group build (or load)
  batch_ms, qps     wall time per 4096-query batch over --steps batches after --warmup, host pointers
  single_query_us   median wall time of one nq = 1, k = 100 search (groups of 1 and 2)
  plain_single_query_us, plain_batch_ms   the same on one GPU through bbq_search without a group (group size 1 only):
                    the difference is the cost of handing the call to the workers and back
  parity            the group's lists and score bits equal the 1-GPU group's for the first 64 queries

The card's name and power limit are read in the same run.

  python tools/group_scale.py --rows 4000000 --gpus 1 2 4 8 --out DIR
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card_info():
    import torch
    out = {"device": torch.cuda.get_device_name(0), "gpus_present": torch.cuda.device_count()}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=60)
        out["power_limit_w"] = float(q.stdout.strip().splitlines()[0])
    except Exception as e:
        out["power_limit_w"] = None
        out["power_limit_error"] = str(e)[:200]
    return out


def corpus(n, dim, seed=1234, chunk=1 << 18):
    rows = np.empty((n, dim), np.float32)
    for c0 in range(0, n, chunk):
        rows[c0:c0 + chunk] = np.random.default_rng(seed + c0 // chunk).standard_normal(
            (min(chunk, n - c0), dim), dtype=np.float32)
    return rows


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    t = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        t.append(time.perf_counter() - t0)
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=4_000_000)
    ap.add_argument("--dim", type=int, default=1024)
    ap.add_argument("--image", default=None, help="prefix of an index image to load instead of building")
    ap.add_argument("--gpus", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--nq", type=int, default=4096)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--single", type=int, default=200, help="nq = 1 calls timed")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    import bbq_b200
    bbq_b200.build_library()
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing to measure")
    info = card_info()
    cfg = {"queryBits": 4, "indexBits": 1, "quantizer": {"similarityFunction": "COSINE", "lambda": 0.1, "iters": 5}}
    rows = None if a.image else corpus(a.rows, a.dim)
    queries = corpus(a.nq, a.dim, seed=99)
    lines, ref = [], None
    for g in a.gpus:
        if g > info["gpus_present"]:
            lines.append({"gpus": g, "skipped": f"{info['gpus_present']} GPUs present"})
            continue
        fmt = bbq_b200.BinaryQuantizationFormat(cfg, devices=list(range(g)))
        t0 = time.perf_counter()
        gi = fmt.loadIndex(a.image) if a.image else fmt.quantizeVectors(rows)["quantizedVectors"]
        build_s = time.perf_counter() - t0
        t = timed(lambda: fmt.searchBatch(queries, gi, a.k), a.steps, a.warmup)
        line = {"gpus": g, "rows": gi.size(), "dim": a.dim, "nq": a.nq, "k": a.k, "source": "image" if a.image else "build",
                "build_s": round(build_s, 3), "batch_ms": round(1e3 * float(np.median(t)), 3),
                "batch_ms_min": round(1e3 * min(t), 3), "qps": round(a.nq / float(np.median(t)), 1)}
        got = fmt.searchBatch(queries[:64], gi, a.k)
        if ref is None:
            ref = got
        line["parity"] = bool(np.array_equal(got[0], ref[0]) and
                              np.array_equal(got[1].view(np.uint32), ref[1].view(np.uint32)))
        if g <= 2:
            t1 = timed(lambda: fmt.searchBatch(queries[:1], gi, a.k), a.single, 10)
            line["single_query_us"] = round(1e6 * float(np.median(t1)), 1)
        if g == 1:
            plain = bbq_b200.BinaryQuantizationFormat(cfg, device=0)
            del gi
            pi = plain.loadIndex(a.image) if a.image else plain.quantizeVectors(rows)["quantizedVectors"]
            t1 = timed(lambda: plain.searchBatch(queries[:1], pi, a.k), a.single, 10)
            tb = timed(lambda: plain.searchBatch(queries, pi, a.k), a.steps, a.warmup)
            line["plain_single_query_us"] = round(1e6 * float(np.median(t1)), 1)
            line["plain_batch_ms"] = round(1e3 * float(np.median(tb)), 3)
            del pi, plain
        else:
            del gi
        del fmt
        line.update(info)
        print(json.dumps(line), flush=True)
        lines.append(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "group_scale.jsonl"), "w") as f:
            for l in lines:
                f.write(json.dumps(l) + "\n")


if __name__ == "__main__":
    main()
