"""Oversampled search with exact re-rank across row shards (bbq_search_rerank_sharded, bbq_rerank_owned_device).

On one GPU: the shard-local step (bbq_rerank_owned_device) for 2, 3 and 8 ragged shards of one corpus, summed as
integers, gives the oracle's exact-score bits; the entry without a communicator is bbq_search_rerank; an index that
grew after its rows were attached is refused.  On two GPUs (skipped below that): every rank returns the oracle's
getOversampledTopKWithSort lists bit for bit, and a per-rank precondition that fails makes both ranks fail alike."""
import numpy as np
import pytest

from oracle import oracle as O
from tests.fixtures import gaussian, sincos_dataset, true_topk_cosine

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bbq():
    import bbq_b200
    bbq_b200.build_library()
    return bbq_b200


def _fmt(bbq, sim="COSINE", lam=0.1, iters=5, device=-1):
    return bbq.createBinaryQuantizationFormat(
        {"queryBits": 4, "indexBits": 1, "quantizer": {"similarityFunction": sim, "lambda": lam, "iters": iters}},
        device=device)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64 if np.asarray(a).dtype.itemsize == 8 else np.uint32)


# ---- one GPU: the shard-local step, shards emulated by slices of one index ------------------------------------
@pytest.mark.parametrize("n,dim,bounds", [
    (30000, 256, [0, 17000, 30000]),
    (30000, 256, [0, 10, 12000, 30000]),                                         # a shard smaller than m
    (30000, 256, [0, 5, 3000, 3001, 9000, 15000, 15020, 22000, 30000]),
    (7, 32, [0, 3, 7]),                                                          # k*factor > n: empty slots
])
def test_owned_scores_of_all_shards_sum_to_the_exact_bits(bbq, n, dim, bounds):
    import torch
    k, factor, nq = 10, 3, 9
    m = k * factor
    rows, qs = gaussian(n, dim, 3100 + len(bounds)), gaussian(nq, dim, 3200 + len(bounds))
    fmt = _fmt(bbq)
    whole = fmt.quantizeVectors(rows)["quantizedVectors"]
    packed, corr = whole.exportAll()
    cen = whole.getCentroid()
    dq = torch.from_numpy(qs).cuda()
    cand = torch.empty((nq, m), dtype=torch.int32, device="cuda")
    cand_score = torch.empty((nq, m), dtype=torch.float32, device="cuda")
    fmt.searchDevice(dq.data_ptr(), nq, whole, m, cand.data_ptr(), cand_score.data_ptr())
    torch.cuda.synchronize()
    ci = cand.cpu().numpy()
    assert (ci < 0).any() == (m > n)
    total = np.zeros((nq, m), np.uint64)
    for r0, r1 in zip(bounds[:-1], bounds[1:]):
        shard = fmt.adoptQuantized(packed[r0:r1], corr[r0:r1], cen)
        assert bbq._native.load().bbq_index_set_base(shard._h, r0) == 0
        fmt.attachOriginalVectors(shard, rows[r0:r1])
        out = torch.full((nq, m), -1, dtype=torch.int64, device="cuda")     # every word is written
        fmt.rerankOwnedDevice(shard, dq.data_ptr(), nq, cand.data_ptr(), m, out.data_ptr())
        torch.cuda.synchronize()
        words = out.cpu().numpy().view(np.uint64)
        owned = (ci >= r0) & (ci < r1)
        assert not words[~owned].any(), "a slot this shard does not hold is not 0"
        total += words
    for qi in range(nq):
        for j in range(m):
            if ci[qi, j] < 0:
                assert total[qi, j] == 0
            else:
                want = np.float64(O.cosine_similarity(qs[qi], rows[ci[qi, j]]))
                assert total[qi, j] == want.view(np.uint64), (qi, j)


def test_sharded_rerank_without_communicator_is_the_plain_rerank(bbq):
    rows, qs = gaussian(5000, 96, 3301), gaussian(6, 96, 3302)
    fmt = _fmt(bbq)
    qv = fmt.quantizeVectors(rows)["quantizedVectors"]
    fmt.attachOriginalVectors(qv, rows)
    a = fmt.searchOversampledBatch(qs, qv, 10, 3)
    b = fmt.searchOversampledBatch(qs, qv, 10, 3, sharded=True)
    assert fmt.commInfo()["world"] == 1
    assert a[0].shape == (6, 10) and np.array_equal(a[0], b[0])
    assert np.array_equal(_bits(a[1]), _bits(b[1])) and np.array_equal(_bits(a[2]), _bits(b[2]))


def test_rerank_limits_and_grown_index(bbq):
    dim = 64
    rows = gaussian(3000, dim, 3401)
    qs = rows[:2] + 0.01
    fmt = _fmt(bbq)
    qv = fmt.reserveIndex(3000, dim, np.zeros(dim, np.float32))
    fmt.appendRows(qv, rows[:2000])
    fmt.attachOriginalVectors(qv, rows[:2000])
    for sharded in (False, True):
        with pytest.raises(bbq.BbqError) as e:
            fmt.searchOversampledBatch(qs, qv, 100, 41, sharded=sharded)               # k * factor > 4096
        assert e.value.status == 9
        i, q, t = fmt.searchOversampledBatch(qs, qv, 0, 3, sharded=sharded)
        assert i.shape == (2, 0)
    fmt.appendRows(qv, rows[2000:])
    for sharded in (False, True):
        with pytest.raises(bbq.BbqError) as e:
            fmt.searchOversampledBatch(qs, qv, 10, 3, sharded=sharded)
        assert e.value.status == 10 and "rows attached for 2000 rows, index has 3000" in str(e.value)
    with pytest.raises(bbq.BbqError) as e:
        fmt.rerankOwnedDevice(qv, 1, 1, 1, 1, 1)                                       # refused before any launch
    assert e.value.status == 10
    fmt.attachOriginalVectors(qv, rows)
    a = fmt.searchOversampledBatch(qs, qv, 10, 3)
    b = fmt.searchOversampledBatch(qs, qv, 10, 3, sharded=True)
    assert a[0][:, 0].tolist() == [0, 1] and np.array_equal(a[0], b[0]) and np.array_equal(_bits(a[2]), _bits(b[2]))


# ---- two GPUs: the collective entry, one process per GPU --------------------------------------------------------
# (name, similarity, n, dim, nq, k, factor, lambda, iters)
CASES = [
    ("cosine_mma", "COSINE", 50_000, 256, 96, 10, 3, 0.1, 5),      # tensor-core scan
    ("cosine_popc", "COSINE", 50_000, 256, 3, 10, 3, 0.1, 5),      # popcount scan
    ("euclidean", "EUCLIDEAN", 3001, 128, 40, 10, 3, 0.1, 5),      # the re-rank is cosine whatever the index
    ("m_above_shard", "COSINE", 50, 64, 5, 12, 3, 0.1, 5),         # m = 36 > 25 rows per shard
    ("sincos", "COSINE", 100, 128, 10, 10, 3, 0.001, 20),          # tests/recall.test.ts:519,635
]


def _data(name, n, dim, nq):
    if name == "sincos":
        return sincos_dataset(dim, n, nq)
    return gaussian(n, dim, 3500 + n), gaussian(nq, dim, 3600 + n)


def _join(fmt, ids, rank, world):
    if rank == 0:
        cid = fmt.commUniqueId()
        for _ in range(world - 1):
            ids.put(cid)
    else:
        cid = ids.get(timeout=120)
    fmt.commInit(cid, rank, world)


def _worker_parity(rank, world, ids, out):
    import torch
    torch.cuda.set_device(rank)
    import bbq_b200
    results = {}
    for name, sim, n, dim, nq, k, factor, lam, iters in CASES:
        fmt = _fmt(bbq_b200, sim, lam, iters, device=rank)
        rows, qs = _data(name, n, dim, nq)
        cen = np.zeros(dim, np.float32)
        r0, r1 = bbq_b200.shard_bounds(n, world, rank)
        shard = fmt.quantizeVectors(rows[r0:r1], centroid=cen)["quantizedVectors"]
        assert bbq_b200._native.load().bbq_index_set_base(shard._h, r0) == 0
        fmt.attachOriginalVectors(shard, rows[r0:r1])
        _join(fmt, ids, rank, world)
        gi, gq, gt = fmt.searchOversampledBatch(qs, shard, k, factor, sharded=True)
        fmt.commDestroy()
        idx = O.quantize_vectors(rows, sim=sim, want_unpacked=False, lam=lam, iters=iters, centroid=cen)
        ok, rec = gi.shape == (nq, min(k, n)), 0.0
        for qi in range(nq):
            wi, wq, wt = O.oversampled_topk(qs[qi], rows, idx, k, factor, lam=lam, iters=iters)
            ok &= gi[qi].tolist() == wi.tolist()
            ok &= np.array_equal(_bits(gq[qi]), _bits(wq)) and np.array_equal(_bits(gt[qi]), _bits(wt))
            rec += len(set(gi[qi].tolist()) & set(true_topk_cosine(qs[qi], rows, k).tolist())) / k
        if name == "sincos":
            ok &= rec / nq >= 0.75
        results[name] = (bool(ok), gi.tobytes() + _bits(gq).tobytes() + _bits(gt).tobytes())
    out.put((rank, results))


def _worker_errors(rank, world, ids, out):
    import torch
    torch.cuda.set_device(rank)
    import bbq_b200
    n, dim = 4000, 64
    rows, qs = gaussian(n, dim, 3701), gaussian(4, dim, 3702)
    cen = np.zeros(dim, np.float32)
    r0, r1 = bbq_b200.shard_bounds(n, world, rank)
    got = []
    for case in ("rank1_without_rows", "overlapping_bases"):
        fmt = _fmt(bbq_b200, device=rank)
        shard = fmt.quantizeVectors(rows[r0:r1], centroid=cen)["quantizedVectors"]
        base = 0 if case == "overlapping_bases" else r0
        assert bbq_b200._native.load().bbq_index_set_base(shard._h, base) == 0
        if not (case == "rank1_without_rows" and rank == 1):
            fmt.attachOriginalVectors(shard, rows[r0:r1])
        _join(fmt, ids, rank, world)
        try:
            fmt.searchOversampledBatch(qs, shard, 10, 3, sharded=True)
            got.append((case, 0, ""))
        except bbq_b200.BbqError as e:
            got.append((case, e.status, str(e)))
        fmt.commDestroy()
    out.put((rank, got))


def _spawn(target, world):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    ctx = mp.get_context("spawn")
    ids, out = ctx.Queue(), ctx.Queue()
    procs = [ctx.Process(target=target, args=(r, world, ids, out)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        got = dict(out.get(timeout=600) for _ in range(world))
        for p in procs:
            p.join(240)
            assert p.exitcode == 0, "a rank failed or hung"
    finally:
        for p in procs:      # never leave a rank spinning in a collective on the GPU behind a failed test
            if p.is_alive():
                p.kill()
    return got


def test_sharded_rerank_equals_the_unsharded_oracle_on_every_rank():
    got = _spawn(_worker_parity, 2)
    for name, *_ in CASES:
        assert got[0][name][0] and got[1][name][0], name
        assert got[0][name][1] == got[1][name][1], f"{name}: the ranks returned different lists"


def test_failed_precondition_on_one_rank_fails_every_rank_alike():
    got = _spawn(_worker_errors, 2)
    for (case, s0, m0), (_, s1, m1) in zip(got[0], got[1]):
        assert s0 == s1 == 10, (case, s0, s1)
        assert m0 == m1 and m0, (case, m0, m1)
    assert "rank 1 has no original rows attached" in got[0][0][2]
    assert "overlap" in got[0][1][2]
