"""Oversampled search with exact re-rank across row shards at scale (bbq_search_rerank_sharded), beside the plain
sharded search on the same query batch.  One process per GPU (the communicator id travels over a queue, as in
tests/test_gpu_sharded_nccl.py).  Every rank generates its contiguous slice of the bench corpus (bench.gen_chunk_device,
so --corpus gaussian is BASELINE's C4 corpus) into one [rows, dim] tensor, builds its shard from it (reserve + append),
sets its base and attaches the same tensor as its original rows.  Per corpus, one JSON line:

  timing  wall time per --nq query batch of bbq_search_sharded (k) and bbq_search_rerank_sharded (k, factor), host
          pointers, the two calls alternated after a warm-up, max over ranks; card name and power limit read in the
          same run
  recall  recall@k of both against exact f32 cosine ground truth for the first --recall-queries queries (per-shard
          top-k over the rows tensor, as tools/recall_harness.py:exact_topk does, merged across ranks)
  parity  for --parity-queries sampled queries: the m = k*factor candidates of bbq_search_sharded(k = m), scored by
          oracle.cosine_similarity on the rows of their owners, stable-sorted by true score: the re-rank's output
          must equal that bit for bit

With --gpus 1 there is no communicator and the sharded entries are the single-index ones: the line then measures
what one rank's shard costs, without the exchange.

  python tools/rerank_sharded_scale.py --gpus 8 --rows 100000000 --corpus gaussian clustered --out DIR
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


def card_info(rank):
    import torch
    out = {"device": torch.cuda.get_device_name(rank)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(rank), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=60)
        out["power_limit_w"] = float(q.stdout.strip().splitlines()[0])
    except Exception as e:   # the number is still reported, marked as such
        out["power_limit_w"] = None
        out["power_limit_error"] = str(e)[:200]
    return out


def gen_shard_rows(torch, bench, n, dim, r0, r1):
    """Rows [r0, r1) of the bench corpus (chunk c seeded by SEED + c whatever the shard split) as one tensor."""
    rows = torch.empty((r1 - r0, dim), dtype=torch.float32, device="cuda")
    c = r0 // bench.CHUNK
    while c * bench.CHUNK < r1:
        c0 = c * bench.CHUNK
        lo, hi = max(r0, c0), min(r1, c0 + bench.CHUNK)
        chunk = bench.gen_chunk_device(torch, c, dim, min(bench.CHUNK, n - c0))
        rows[lo - r0:hi - r0] = chunk[lo - c0:hi - c0]
        del chunk
        c += 1
    torch.cuda.synchronize()
    return rows


def shard_exact_topk(torch, rows, queries_d, k, chunk=262144):
    """exact f32 cosine top-k of this shard (local ids, scores), normalisation in f64 as tools/recall_harness.py does"""
    qn = torch.nn.functional.normalize(queries_d.double(), dim=1).float()
    best_s = torch.full((queries_d.shape[0], k), -float("inf"), device=rows.device)
    best_i = torch.zeros((queries_d.shape[0], k), dtype=torch.int64, device=rows.device)
    for a in range(0, rows.shape[0], chunk):
        blk = torch.nn.functional.normalize(rows[a:a + chunk].double(), dim=1).float()
        s = qn @ blk.T
        cs, ci = torch.topk(s, min(k, s.shape[1]), dim=1)
        ms, mi = torch.cat([best_s, cs], 1), torch.cat([best_i, ci + a], 1)
        o = torch.argsort(ms, dim=1, descending=True, stable=True)[:, :k]
        best_s, best_i = torch.gather(ms, 1, o), torch.gather(mi, 1, o)
    return best_i.cpu().numpy(), best_s.cpu().numpy()


def worker(rank, world, a, corpus, ids, out):
    import ctypes as C
    import torch
    torch.cuda.set_device(rank)
    import bench
    import bbq_b200
    from oracle import oracle as O
    bench.CORPUS = corpus
    L = bbq_b200._native.load()
    n, dim, k, factor, nq = a.rows, a.dim, a.k, a.factor, a.nq
    m = k * factor
    r0, r1 = bbq_b200.shard_bounds(n, world, rank)
    t0 = time.time()
    fmt = bbq_b200.createBinaryQuantizationFormat(
        {"queryBits": 4, "indexBits": 1, "quantizer": {"similarityFunction": "COSINE", "lambda": 0.1, "iters": 5}},
        device=rank)
    rows = gen_shard_rows(torch, bench, n, dim, r0, r1)
    shard = fmt.reserveIndex(max(r1 - r0, 1), dim, np.zeros(dim, np.float32))
    for p in range(0, r1 - r0, bench.CHUNK):
        q = min(r1 - r0, p + bench.CHUNK)
        fmt.appendRows(shard, d_rows_ptr=rows[p:q].data_ptr(), n=q - p)
    assert L.bbq_index_set_base(shard._h, r0) == 0
    fmt.attachOriginalVectorsDevice(shard, rows.data_ptr())
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

    queries = bench.gen_queries(nq, dim)
    hq = torch.from_numpy(queries).pin_memory()
    si = torch.empty((nq, k), dtype=torch.int32).pin_memory()
    ss = torch.empty((nq, k), dtype=torch.float32).pin_memory()
    ri = torch.empty((nq, k), dtype=torch.int32).pin_memory()
    rq = torch.empty((nq, k), dtype=torch.float32).pin_memory()
    rt = torch.empty((nq, k), dtype=torch.float64).pin_memory()
    cnt = C.c_uint32(0)

    def search():
        return fmt.searchShardedHost(hq.data_ptr(), nq, shard, k, si.data_ptr(), ss.data_ptr())

    def rerank():
        st = L.bbq_search_rerank_sharded(shard._h, hq.data_ptr(), nq, k, factor, ri.data_ptr(), rq.data_ptr(),
                                         rt.data_ptr(), C.byref(cnt))
        if st != 0:
            raise RuntimeError(f"bbq_search_rerank_sharded: {st} {L.bbq_last_error().decode()}")
        return cnt.value

    for _ in range(a.warmup):
        search()
        rerank()
    t_search, t_rerank = [], []
    for _ in range(a.steps):          # alternated; both calls are collective and blocking, so ranks stay in step
        t = time.perf_counter()
        search()
        t_search.append((time.perf_counter() - t) * 1e3)
        t = time.perf_counter()
        rerank()
        t_rerank.append((time.perf_counter() - t) * 1e3)
    got_search, got_rerank = si.numpy().copy(), ri.numpy().copy()
    got_q, got_t = rq.numpy().copy(), rt.numpy().copy()

    # parity: the candidates of the sharded search at k = m for the sampled queries, scored by the oracle on the
    # rows this rank holds
    pq = np.sort(np.random.default_rng(7).choice(nq, a.parity_queries, replace=False))
    ci = torch.empty((nq, m), dtype=torch.int32).pin_memory()
    cs = torch.empty((nq, m), dtype=torch.float32).pin_memory()
    fmt.searchShardedHost(hq.data_ptr(), nq, shard, m, ci.data_ptr(), cs.data_ptr())
    cand, cand_s = ci.numpy()[pq].copy(), cs.numpy()[pq].copy()
    owned = {}
    for j, qi in enumerate(pq):
        for s, g in enumerate(cand[j]):
            if r0 <= g < r1:
                owned[(j, s)] = O.cosine_similarity(queries[qi], rows[g - r0].cpu().numpy())

    # exact ground truth of this shard for the recall queries
    nr = min(a.recall_queries, nq)
    ti, ts = shard_exact_topk(torch, rows, torch.from_numpy(queries[:nr]).cuda(), k)
    if world > 1:
        fmt.commDestroy()
    out.put((rank, dict(t_search=t_search, t_rerank=t_rerank, build_s=build_s, card=card_info(rank),
                        search=got_search[:nr], rerank=got_rerank, rerank_q=got_q, rerank_t=got_t, pq=pq, cand=cand,
                        cand_s=cand_s, owned=owned, truth_i=ti + r0, truth_s=ts, count=cnt.value)))
    del rows, shard, fmt
    torch.cuda.synchronize()


def run(a, corpus):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ids, out = ctx.Queue(), ctx.Queue()
    procs = [ctx.Process(target=worker, args=(r, a.gpus, a, corpus, ids, out)) for r in range(a.gpus)]
    for p in procs:
        p.start()
    try:
        res = dict(out.get(timeout=a.timeout) for _ in range(a.gpus))
        for p in procs:
            p.join(300)
            if p.exitcode != 0:
                raise RuntimeError(f"a rank exited with {p.exitcode}")
    finally:
        for p in procs:     # no rank may be left in a collective
            if p.is_alive():
                p.kill()
    k, m = a.k, a.k * a.factor
    r = [res[i] for i in range(a.gpus)]
    same = all(np.array_equal(x["rerank"], r[0]["rerank"]) and np.array_equal(x["rerank_t"].view(np.uint64),
                                                                                r[0]["rerank_t"].view(np.uint64))
               for x in r)
    # ground truth: per-shard exact top-k merged (score desc, then global id asc)
    ti = np.concatenate([x["truth_i"] for x in r], 1)
    ts = np.concatenate([x["truth_s"] for x in r], 1)
    truth = np.stack([ti[q][np.lexsort((ti[q], -ts[q]))[:k]] for q in range(ti.shape[0])])
    nr = truth.shape[0]

    def recall(found):
        return float(np.mean([len(set(f.tolist()) & set(t.tolist())) / k for f, t in zip(found[:nr], truth)]))

    # parity: every slot owned by exactly one rank, stable sort by the oracle's true score
    owned = {}
    for x in r:
        for key, v in x["owned"].items():
            assert key not in owned, "two ranks own one candidate"
            owned[key] = v
    cand, cand_s, pq = r[0]["cand"], r[0]["cand_s"], r[0]["pq"]
    parity_ok = True
    for j, qi in enumerate(pq):
        true = np.array([owned[(j, s)] for s in range(m)], np.float64)
        pos = np.argsort(-true, kind="stable")[:k]
        parity_ok &= r[0]["rerank"][qi].tolist() == cand[j][pos].tolist()
        parity_ok &= np.array_equal(r[0]["rerank_q"][qi].view(np.uint32), cand_s[j][pos].view(np.uint32))
        parity_ok &= np.array_equal(r[0]["rerank_t"][qi].view(np.uint64), true[pos].view(np.uint64))
    ts_ = np.max([x["t_search"] for x in r], 0)     # per step: the slowest rank
    tr_ = np.max([x["t_rerank"] for x in r], 0)
    line = {
        "tool": "tools/rerank_sharded_scale.py", "corpus": corpus, "gpus": a.gpus, "rows": a.rows,
        "rows_per_gpu": -(-a.rows // a.gpus), "dim": a.dim, "nq": a.nq, "k": k, "factor": a.factor, "m": m,
        "cards": sorted({x["card"]["device"] for x in r}),
        "power_limit_w": sorted({x["card"]["power_limit_w"] for x in r}, key=str),
        "search_sharded_ms": {"median": float(np.median(ts_)), "min": float(ts_.min()), "steps": [round(float(v), 3) for v in ts_]},
        "rerank_sharded_ms": {"median": float(np.median(tr_)), "min": float(tr_.min()), "steps": [round(float(v), 3) for v in tr_]},
        "added_ms_median": float(np.median(tr_ - ts_)),
        "qps": {"search_sharded": a.nq / (np.median(ts_) / 1e3), "rerank_sharded": a.nq / (np.median(tr_) / 1e3)},
        "recall_at_k": {"queries": nr, "search_sharded": recall(r[0]["search"]), "rerank_sharded": recall(r[0]["rerank"])},
        "parity": {"queries": len(pq), "ok": bool(parity_ok)}, "ranks_identical": bool(same),
        "count": r[0]["count"], "build_s_max": max(x["build_s"] for x in r),
        "timing": "host wall clock around each blocking call (host pointers, pinned), steps alternated after warm-up, "
                  "max over ranks per step" + ("" if a.gpus > 1 else "; one GPU: no communicator, so the entries are "
                                                 "the single-index bbq_search / bbq_search_rerank on this shard"),
    }
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=0, help="ranks, one per GPU (default: every visible GPU)")
    ap.add_argument("--rows", type=int, default=100_000_000)
    ap.add_argument("--dim", type=int, default=1024)
    ap.add_argument("--nq", type=int, default=4096)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--factor", type=int, default=3)
    ap.add_argument("--corpus", nargs="+", default=["gaussian", "clustered"], choices=["gaussian", "clustered"])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--recall-queries", type=int, default=256)
    ap.add_argument("--parity-queries", type=int, default=16)
    ap.add_argument("--timeout", type=int, default=3000)
    ap.add_argument("--out", default="", help="directory for r03_rerank_sharded_<corpus>.json (default: stdout only)")
    a = ap.parse_args()
    if a.gpus <= 0:
        import torch
        a.gpus = torch.cuda.device_count()
    if a.gpus <= 0:
        sys.exit("no GPU: this tool measures the device path and has nothing to fall back to")
    for corpus in a.corpus:
        line = run(a, corpus)
        s = json.dumps(line)
        print(s, flush=True)
        if a.out:
            os.makedirs(a.out, exist_ok=True)
            with open(os.path.join(a.out, f"r03_rerank_sharded_{corpus}.json"), "a") as f:
                f.write(s + "\n")
        if not line["parity"]["ok"] or not line["ranks_identical"]:
            sys.exit(f"{corpus}: parity failed")


if __name__ == "__main__":
    main()
