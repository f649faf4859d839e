"""The index build across row shards at scale, with the reference-order centroid chained across the GPUs.

The corpus is generated on the device from a seed (bench.gen_chunk_device: chunk c of bench.CHUNK rows is seeded by
SEED + c), so a row's values depend only on its global index and every world size builds the same corpus.  COSINE.
One process per GPU; rank r holds rows shard_bounds(N, world, r).

  collective (world >= 4, or --mode collective): every rank generates its rows into device memory and calls
      bbq_index_build_sharded_device, once with the NULL centroid (the chain) and once with that centroid passed in
      (no chain); chain = the difference of the two wall times, quantise = the second.
  streaming (world 1 and 2, or --mode streaming: the f32 rows of 100 M x 1024, 410 GB, do not fit): pass 1, rank by rank
      in rank order, bbq_centroid_accumulate_device over generated chunks (the running sum travels to the next rank over
      a queue), bbq_centroid_finish; pass 2, on every rank at once, bbq_index_reserve + bbq_index_append_device of the
      chunks generated again.  chain = pass 1, quantise = pass 2 (both include generating the rows).

Every run writes one JSON line to --out/build_sharded_<world>gpu_<rows>.json: wall times, rows/s, the SHA-256 of the
centroid's bytes, and the name and power limit of every card.  --compare checks that every such file in --out with the
same row count holds the same centroid.  --parity-rows R (R rows must fit one GPU) also builds R rows with the
collective entry and checks on every rank that its shard equals its slice of bbq_index_build of all R rows.

  python tools/build_sharded_scale.py --gpus 8 --rows 100000000 --parity-rows 10000000 --out profiles/
  python tools/build_sharded_scale.py --gpus 1 --rows 100000000 --out profiles/ --compare
"""
import argparse
import glob
import hashlib
import json
import os
import sys
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


def _chunks(bench, r0, r1):
    """(chunk, lo, hi): the generated chunks that hold rows [r0, r1), with the part of each inside the range"""
    c = r0 // bench.CHUNK
    while c * bench.CHUNK < r1:
        c0 = c * bench.CHUNK
        yield c, max(r0, c0), min(r1, c0 + bench.CHUNK)
        c += 1


def _gen(torch, bench, n, dim, c, lo, hi):
    c0 = c * bench.CHUNK
    return bench.gen_chunk_device(torch, c, dim, min(bench.CHUNK, n - c0))[lo - c0:hi - c0].contiguous()


def _join(fmt, ids, rank, world):
    if rank == 0:
        cid = fmt.commUniqueId()
        for _ in range(world - 1):
            ids.put(cid)
    else:
        cid = ids.get(timeout=600)
    fmt.commInit(cid, rank, world)


def worker(rank, world, a, mode, ids, chain_q, out):
    import torch
    torch.cuda.set_device(rank)
    import bench
    import bbq_b200
    from rerank_sharded_scale import card_info, gen_shard_rows
    n, dim = a.rows, a.dim
    r0, r1 = bbq_b200.shard_bounds(n, world, rank)
    fmt = _fmt(bbq_b200, rank)
    res = {"rank": rank, "rows": r1 - r0, "card": card_info(rank)}
    if mode == "collective":
        rows = gen_shard_rows(torch, bench, n, dim, r0, r1)
        _join(fmt, ids, rank, world)
        t = time.perf_counter()
        qv = fmt.quantizeVectorsDevice(rows.data_ptr(), r1 - r0, dim, sharded=True)["quantizedVectors"]
        total_s = time.perf_counter() - t
        cen = qv.getCentroid().copy()
        del qv
        t = time.perf_counter()
        qv = fmt.quantizeVectorsDevice(rows.data_ptr(), r1 - r0, dim, centroid=cen, sharded=True)["quantizedVectors"]
        res.update(quantise_s=time.perf_counter() - t, total_s=total_s)
        res["chain_s"] = total_s - res["quantise_s"]
        del qv, rows
    else:
        t = time.perf_counter()
        running = np.zeros(dim, np.float32) if rank == 0 else chain_q[rank].get(timeout=7200)
        t_turn = time.perf_counter()
        for c, lo, hi in _chunks(bench, r0, r1):
            x = _gen(torch, bench, n, dim, c, lo, hi)
            fmt.accumulateCentroid(running, lo, d_rows_ptr=x.data_ptr(), n=hi - lo)
            del x
        res["own_turn_s"] = time.perf_counter() - t_turn
        for r in range(world):              # the last rank's sum is the corpus's: it goes to every rank
            if r != rank and (r == rank + 1 or rank == world - 1):
                chain_q[r].put(running)
        if rank != world - 1:
            running = chain_q[rank].get(timeout=7200)
        cen = fmt.finishCentroid(running, n)
        res["chain_s"] = time.perf_counter() - t
        t = time.perf_counter()
        qv = fmt.reserveIndex(max(r1 - r0, 1), dim, cen)
        for c, lo, hi in _chunks(bench, r0, r1):
            x = _gen(torch, bench, n, dim, c, lo, hi)
            fmt.appendRows(qv, d_rows_ptr=x.data_ptr(), n=hi - lo)
            del x
        fmt.setBase(qv, r0)
        torch.cuda.synchronize()
        res["quantise_s"] = time.perf_counter() - t
        res["total_s"] = res["chain_s"] + res["quantise_s"]
        del qv
    res["centroid_sha256"] = hashlib.sha256(np.ascontiguousarray(cen, np.float32).tobytes()).hexdigest()
    if a.parity_rows:
        pn = a.parity_rows
        p0, p1 = bbq_b200.shard_bounds(pn, world, rank)
        if mode != "collective" and world > 1:
            _join(fmt, ids, rank, world)
        rows = gen_shard_rows(torch, bench, pn, dim, 0, pn)
        whole = fmt.quantizeVectorsDevice(rows.data_ptr(), pn, dim)["quantizedVectors"]
        mine = fmt.quantizeVectorsDevice(rows[p0:].data_ptr(), p1 - p0, dim, sharded=True)["quantizedVectors"]
        wp, wc = whole._export(p0, p1 - p0) if p1 > p0 else (None, None)
        sp, sc = mine.exportAll() if p1 > p0 else (None, None)
        res["parity_rows"] = pn
        res["parity"] = bool(whole.getCentroid().tobytes() == mine.getCentroid().tobytes() and
                             whole.getCentroidDP() == mine.getCentroidDP() and
                             (p1 == p0 or (np.array_equal(wp, sp) and np.array_equal(wc.view(np.uint64), sc.view(np.uint64)))))
        del whole, mine, rows
    if world > 1 and (mode == "collective" or a.parity_rows):
        fmt.commDestroy()
    out.put(res)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--dim", type=int, default=1024)
    ap.add_argument("--mode", choices=["auto", "collective", "streaming"], default="auto")
    ap.add_argument("--parity-rows", type=int, default=0)
    ap.add_argument("--out", required=True)
    ap.add_argument("--compare", action="store_true")
    a = ap.parse_args()
    import torch
    import torch.multiprocessing as mp
    world = a.gpus
    if torch.cuda.device_count() < world:
        sys.exit(f"needs {world} GPUs, this machine has {torch.cuda.device_count()}")
    mode = a.mode if a.mode != "auto" else ("collective" if world >= 4 else "streaming")
    ctx = mp.get_context("spawn")
    ids, out = ctx.Queue(), ctx.Queue()
    chain_q = [ctx.Queue() for _ in range(world)]
    t = time.perf_counter()
    procs = [ctx.Process(target=worker, args=(r, world, a, mode, ids, chain_q, out)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        ranks = sorted((out.get(timeout=7200) for _ in range(world)), key=lambda r: r["rank"])
        for p in procs:
            p.join(600)
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
    wall = time.perf_counter() - t
    line = {"tool": "build_sharded_scale", "mode": mode, "world": world, "rows": a.rows, "dim": a.dim,
            "similarity": "COSINE", "chain_s": max(r["chain_s"] for r in ranks),
            "quantise_s": max(r["quantise_s"] for r in ranks), "total_s": max(r["total_s"] for r in ranks),
            "process_wall_s": wall, "centroid_sha256": ranks[0]["centroid_sha256"],
            "same_centroid_on_every_rank": len({r["centroid_sha256"] for r in ranks}) == 1, "ranks": ranks}
    line["rows_per_s"] = a.rows / line["total_s"]
    line["chain_ns_per_row"] = 1e9 * line["chain_s"] / a.rows
    if a.parity_rows:
        line["parity_all_ranks"] = all(r["parity"] for r in ranks)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, f"build_sharded_{world}gpu_{a.rows}.json"), "w") as f:
        f.write(json.dumps(line) + "\n")
    print(json.dumps({k: v for k, v in line.items() if k != "ranks"}))
    ok = line["same_centroid_on_every_rank"] and line.get("parity_all_ranks", True)
    if a.compare:
        shas = {}
        for p in glob.glob(os.path.join(a.out, f"build_sharded_*gpu_{a.rows}.json")):
            with open(p) as f:
                shas[os.path.basename(p)] = json.loads(f.readline())["centroid_sha256"]
        print(json.dumps({"centroid_by_run": shas, "same": len(set(shas.values())) == 1}))
        ok &= len(set(shas.values())) == 1
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
