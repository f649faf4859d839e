"""One index image across row shards at scale: bbq_index_save_sharded / bbq_index_load_sharded on N GPUs, and the same
image reloaded on a different number of ranks through bbq_index_load_rows.  One process per GPU (the communicator id
travels over a queue, as in tests/test_gpu_sharded_nccl.py).  Every rank generates its contiguous slice of the bench
corpus (bench.gen_chunk_device; --corpus gaussian is BASELINE's C4 corpus) and builds its shard from it (reserve +
append), then:

  save    bbq_index_save_sharded of the N shards into ONE image (wall time, max over ranks; GB/s of the image)
  load    bbq_index_load_sharded of that image on the same N ranks (wall time, max over ranks; GB/s)
  parity  bbq_search_sharded lists of --nq queries before the save and after the load: bit-identical
  reshard the image loaded on --reload-ranks ranks (default N/2, at least 1; a different count from N where N > 1)
          through bbq_index_load_rows, one process per range, without a communicator; the partial checksums must sum
          to the header's and the per-range lists, merged by (score desc, id asc), must equal the lists before the save

The image goes to --dir (default: a new temporary directory, removed at the end).  The load right after the save reads
whatever the operating system still caches of the files: the line says so, and names the card and its power limit.

  python tools/image_shard_scale.py --gpus 8 --rows 100000000 --out DIR
"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)


def _fmt(bbq_b200, rank):
    return bbq_b200.createBinaryQuantizationFormat(
        {"queryBits": 4, "indexBits": 1, "quantizer": {"similarityFunction": "COSINE", "lambda": 0.1, "iters": 5}},
        device=rank)


def _search(torch, fmt, shard, queries, k):
    hq = torch.from_numpy(queries).pin_memory()
    hi = torch.empty((queries.shape[0], k), dtype=torch.int32).pin_memory()
    hs = torch.empty((queries.shape[0], k), dtype=torch.float32).pin_memory()
    cnt = fmt.searchShardedHost(hq.data_ptr(), queries.shape[0], shard, k, hi.data_ptr(), hs.data_ptr())
    return hi.numpy()[:, :cnt].copy(), hs.numpy()[:, :cnt].copy()


def worker(rank, world, a, prefix, ids, out):
    import torch
    torch.cuda.set_device(rank)
    import bench
    import bbq_b200
    from rerank_sharded_scale import card_info, gen_shard_rows
    bench.CORPUS = a.corpus
    n, dim = a.rows, a.dim
    r0, r1 = bbq_b200.shard_bounds(n, world, rank)
    fmt = _fmt(bbq_b200, rank)
    t0 = time.time()
    rows = gen_shard_rows(torch, bench, n, dim, r0, r1)
    shard = fmt.reserveIndex(max(r1 - r0, 1), dim, np.zeros(dim, np.float32))
    for p in range(0, r1 - r0, bench.CHUNK):
        q = min(r1 - r0, p + bench.CHUNK)
        fmt.appendRows(shard, d_rows_ptr=rows[p:q].data_ptr(), n=q - p)
    del rows
    fmt.setBase(shard, r0)
    torch.cuda.synchronize()
    build_s = time.time() - t0
    if world > 1:
        if rank == 0:
            cid = fmt.commUniqueId()
            for _ in range(world - 1):
                ids.put(cid)
        else:
            cid = ids.get(timeout=600)
        fmt.commInit(cid, rank, world)
    queries = bench.gen_queries(a.nq, dim)
    before = _search(torch, fmt, shard, queries, a.k)
    t = time.perf_counter()
    fmt.saveIndex(shard, prefix, sharded=True)        # collective and blocking: every rank returns after the last write
    save_s = time.perf_counter() - t
    del shard
    torch.cuda.synchronize()
    t = time.perf_counter()
    mine = fmt.loadIndex(prefix, sharded=True)
    load_s = time.perf_counter() - t
    after = _search(torch, fmt, mine, queries, a.k)
    if world > 1:
        fmt.commDestroy()
    out.put((rank, dict(save_s=save_s, load_s=load_s, build_s=build_s, card=card_info(rank), before=before,
                        after=after, rows=mine.size())))
    del mine, fmt
    torch.cuda.synchronize()


def range_worker(rank, ranges, a, prefix, out):
    """one process per range, no communicator: bbq_index_load_rows and a search of the range (global ids)"""
    import torch
    torch.cuda.set_device(rank % torch.cuda.device_count())
    import bench
    import bbq_b200
    bench.CORPUS = a.corpus
    r0, r1 = ranges[rank]
    fmt = _fmt(bbq_b200, rank % torch.cuda.device_count())
    t = time.perf_counter()
    part, parts = fmt.loadIndexRows(prefix, r0, r1 - r0)
    load_s = time.perf_counter() - t
    found = fmt.searchBatch(bench.gen_queries(a.nq, a.dim), part, a.k) if r1 > r0 else None
    out.put((rank, dict(load_s=load_s, parts=parts, found=found)))


def spawn(target, nproc, args, timeout):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = [ctx.Queue() for _ in range(2)]
    procs = [ctx.Process(target=target, args=(r,) + args(q)) for r in range(nproc)]
    for p in procs:
        p.start()
    out = q[-1]
    try:
        res = dict(out.get(timeout=timeout) for _ in range(nproc))
        for p in procs:
            p.join(300)
            if p.exitcode != 0:
                raise RuntimeError(f"a rank exited with {p.exitcode}")
    finally:
        for p in procs:     # no rank may be left in a collective
            if p.is_alive():
                p.kill()
    return [res[i] for i in range(nproc)]


def run(a, prefix):
    import bbq_b200
    from bbq_b200 import merge_host, shard_bounds
    import importlib
    image = importlib.import_module("better_binary_quantization_b200.host.image")
    r = spawn(worker, a.gpus, lambda q: (a.gpus, a, prefix, q[0], q[1]), a.timeout)
    image_bytes = os.path.getsize(prefix + ".veb") + os.path.getsize(prefix + ".vemb")
    before, after = r[0]["before"], r[0]["after"]
    same_ranks = all(np.array_equal(x["before"][0], before[0]) and np.array_equal(x["after"][0], after[0]) for x in r)
    parity = np.array_equal(before[0], after[0]) and np.array_equal(before[1].view(np.uint32), after[1].view(np.uint32))

    m = a.reload_ranks
    ranges = [shard_bounds(a.rows, m, i) for i in range(m)]
    rr = spawn(range_worker, m, lambda q: (ranges, a, prefix, q[1]), a.timeout)
    meta = image.read_metadata(prefix)
    sums = [0] * 5
    for x in rr:
        sums = [(s + p) & 0xFFFFFFFFFFFFFFFF for s, p in zip(sums, x["parts"])]
    checks_ok = sums == [meta["sectionChecksums"][s] for s in image.SECTIONS]
    found = [x["found"] for x in rr if x["found"] is not None]
    mi, ms = merge_host([f[0] for f in found], [f[1] for f in found], a.k)
    reshard = np.array_equal(mi, before[0]) and np.array_equal(ms.view(np.uint32), before[1].view(np.uint32))

    save = max(x["save_s"] for x in r)
    load = max(x["load_s"] for x in r)
    return {
        "tool": "tools/image_shard_scale.py", "corpus": a.corpus, "gpus": a.gpus, "rows": a.rows, "dim": a.dim,
        "image_bytes": image_bytes, "cards": sorted({x["card"]["device"] for x in r}),
        "power_limit_w": sorted({x["card"]["power_limit_w"] for x in r}, key=str),
        "save_sharded": {"s": save, "GB_per_s": image_bytes / save / 1e9},
        "load_sharded": {"s": load, "GB_per_s": image_bytes / load / 1e9},
        "reload_ranks": m, "load_rows_s_max": max(x["load_s"] for x in rr),
        "build_s_max": max(x["build_s"] for x in r),
        "search_lists_identical_after_load": bool(parity), "ranks_identical": bool(same_ranks),
        "reshard_lists_identical": bool(reshard), "reshard_checksums_sum_to_header": bool(checks_ok),
        "queries": a.nq, "k": a.k,
        "timing": "host wall clock around each blocking collective call, max over ranks; the load follows the save "
                  "directly, so it reads what the operating system still caches of the files; the reshard loads "
                  "run one process per range, concurrently, without a communicator",
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=0, help="ranks, one per GPU (default: every visible GPU)")
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=1024)
    ap.add_argument("--corpus", default="gaussian", choices=["gaussian", "clustered"])
    ap.add_argument("--nq", type=int, default=64)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--reload-ranks", type=int, default=0, help="ranks of the reshard (default: gpus // 2, at least 1)")
    ap.add_argument("--dir", default="", help="where the image is written (default: a new temporary directory)")
    ap.add_argument("--timeout", type=int, default=3000)
    ap.add_argument("--out", default="", help="directory for image_shard_scale.json (default: stdout only)")
    a = ap.parse_args()
    if a.gpus <= 0:
        import torch
        a.gpus = torch.cuda.device_count()
    if a.gpus <= 0:
        sys.exit("no GPU: this tool measures the device path and has nothing to fall back to")
    if a.reload_ranks <= 0:
        a.reload_ranks = max(1, a.gpus // 2)
    tmp = a.dir or tempfile.mkdtemp(prefix="bbq_image_")
    try:
        line = run(a, os.path.join(tmp, "index"))
    finally:
        if not a.dir:
            shutil.rmtree(tmp, ignore_errors=True)
    s = json.dumps(line)
    print(s, flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "image_shard_scale.json"), "a") as f:
            f.write(s + "\n")
    if not (line["search_lists_identical_after_load"] and line["ranks_identical"] and line["reshard_lists_identical"]
            and line["reshard_checksums_sum_to_header"]):
        sys.exit("parity failed")


if __name__ == "__main__":
    main()
