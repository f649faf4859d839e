"""GPU search across its own plan space: large k on the filtered path (both threshold rules, every scan engine), exact
ties at large k, large k on large shards without overflow, rows that score NaN, more than one query batch per call,
the oversampled re-rank at large m and the captured launch sequence at large k.  Every list is compared with the
oracle's canonical mode (f32 scores bit-equal, ids equal), and stats() proves which regime ran."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as O
from tests.fixtures import gaussian
from tests.test_gpu_parity import bits_equal, make_format, SIMS

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bbq():
    import bbq_b200
    bbq_b200.build_library()
    return bbq_b200


def device_rows(n, dim, seed):
    import torch
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return torch.randn((n, dim), generator=g, device="cuda", dtype=torch.float32)


def device_corpus(bbq, sim, n, dim, seed):
    """(packed, corr, centroid) of n seeded N(0,1) rows quantised on the device with a zero centroid."""
    import torch
    rows_d = device_rows(n, dim, seed)
    cen = np.zeros(dim, np.float32)
    qv = make_format(bbq, sim).quantizeVectorsDevice(rows_d.data_ptr(), n, dim, centroid=cen)["quantizedVectors"]
    packed, corr = qv.exportAll()
    del rows_d, qv
    torch.cuda.empty_cache()
    return packed, corr, cen


@pytest.fixture(scope="module")
def corpora(bbq):
    cache = {}

    def get(sim, n, dim):
        if (sim, n, dim) not in cache:
            cache[(sim, n, dim)] = device_corpus(bbq, sim, n, dim, 7000 + n + dim)
        return cache[(sim, n, dim)]
    return get


def oracle_index(packed, corr, cen, sim):
    return O.OracleIndex(cen, packed, None, corr, len(cen), sim, 1)


def check_oracle(gi, gs, qs, oidx, k, rows, qb=4):
    for qi in rows:
        wi, ws = O.search_nearest_neighbors(qs[qi], oidx, k, query_bits=qb, mode="canonical")
        assert gi[qi].tolist() == wi.tolist(), f"query {qi}: top-{k} list differs from the oracle"
        assert bits_equal(gs[qi], ws), f"query {qi}: scores differ from the oracle"


def spread(nq):
    return sorted({0, 1, nq // 2, nq - 2, nq - 1} & set(range(nq)))


# ---- 1. large k on the filtered path: both threshold rules, every scan engine -------------------------------------------
# k = 100 control; 128 / 129 = the running threshold of the tensor-core scan ends (RETIGHTEN_KMAX); 512 / 513 = the
# per-thread maxima give way to the maxima of 16384 bins; 4096 = K_MAX, the final select sorts up to 16384 candidates.
ENGINES = {
    "k1s": dict(nq=3, engine=1),                              # streaming popcount scan
    "tile": dict(nq=3, engine=1, popc_form="tile"),           # shared-memory tile popcount scan
    "narrow": dict(nq=5, engine=2, layout=1, passes=1),       # smallest tensor-core batch
    "wide": dict(nq=130, engine=2, layout=0, passes=1),
    "two_blocks": dict(nq=300, engine=2, layout=0, passes=2),
    "qb8": dict(nq=24, engine=2, qb=8),                       # two nibble columns per query
}
KS = [100, 128, 129, 512, 513, 1000, 4096]
CORPORA = [(40000, 128), (16385, 100), (40000, 100), (16385, 128)]   # 16385 = a 128-tile sample + a 1-row ragged tile
LARGE_K_CASES = [(eng, k, SIMS[(ei + ki) % 3]) + CORPORA[(ei + 2 * ki) % 4]
                 for ei, eng in enumerate(ENGINES) for ki, k in enumerate(KS)]


@pytest.mark.parametrize("eng,k,sim,n,dim", LARGE_K_CASES)
def test_filtered_path_large_k(bbq, corpora, eng, k, sim, n, dim):
    e = ENGINES[eng]
    qb, nq = e.get("qb", 4), e["nq"]
    packed, corr, cen = corpora(sim, n, dim)
    qs = gaussian(nq, dim, 9000 + k + nq)
    fmt = make_format(bbq, sim, qb=qb, popc_form=e.get("popc_form"))
    gi, gs = fmt.searchBatch(qs, fmt.adoptQuantized(packed, corr, cen), k)
    st = fmt.stats()
    assert st["last_path"] == 1 and st["last_overflow"] == 0 and st["last_engine"] == e["engine"], st
    for key in ("layout", "passes"):
        if key in e:
            assert st["mma_" + key] == e[key], st
    # the other engine on the same queries
    other = make_format(bbq, sim, qb=qb, scan="popc" if e["engine"] == 2 else "mma")
    oi, os_ = other.searchBatch(qs, other.adoptQuantized(packed, corr, cen), k)
    assert other.stats()["last_engine"] == 3 - e["engine"] and other.stats()["last_overflow"] == 0
    assert np.array_equal(gi, oi) and bits_equal(gs, os_)
    check_oracle(gi, gs, qs, oracle_index(packed, corr, cen, sim), k, spread(nq), qb)


# ---- 2. exact ties at large k ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sim", SIMS)
@pytest.mark.parametrize("k", [1000, 1500])       # the k-th place at the end of a tie group / inside the second one
@pytest.mark.parametrize("scan,nq", [("popc", 3), ("mma", 8)])
def test_large_k_ties_lower_index_first(bbq, sim, k, scan, nq):
    """40 distinct rows, each repeated 1000 times: every score is tied 1000 times across the sample's bins."""
    dim = 64
    idx = O.quantize_vectors(gaussian(40, dim, 61), sim=sim, want_unpacked=False, centroid=np.zeros(dim, np.float32))
    packed, corr = np.concatenate([idx.packed] * 1000), np.concatenate([idx.corr] * 1000)
    big = O.OracleIndex(idx.centroid, packed, None, corr, dim, sim, 1)
    fmt = make_format(bbq, sim, scan=scan)
    qs = gaussian(nq, dim, 62)
    gi, gs = fmt.searchBatch(qs, fmt.adoptQuantized(packed, corr, idx.centroid), k)
    st = fmt.stats()
    assert st["last_path"] == 1 and st["last_overflow"] == 0 and st["last_engine"] == (2 if scan == "mma" else 1)
    check_oracle(gi, gs, qs, big, k, range(nq))
    assert np.all(np.diff(gi[:, :1000], axis=1) == 40)       # the best row's 1000 copies, ascending ids


# ---- 3. large k on a large shard: the threshold sample grows with k*n for k > 512 too ---------------------------------------
@pytest.mark.parametrize("n,k", [(1_000_000, 1000), (250_000, 4096)])
@pytest.mark.parametrize("nq,engine", [(2, 1), (48, 2)])
def test_large_k_large_shard_does_not_overflow(bbq, corpora, n, k, nq, engine):
    sim, dim = "MAXIMUM_INNER_PRODUCT", 128
    packed, corr, cen = corpora(sim, n, dim)
    fmt = make_format(bbq, sim)
    qs = gaussian(nq, dim, 20261002)
    gi, gs = fmt.searchBatch(qs, fmt.adoptQuantized(packed, corr, cen), k)
    st = fmt.stats()
    assert st["last_engine"] == engine and st["last_path"] == 1
    assert st["last_overflow"] == 0, "ordinary data overflowed the candidate lists: the exact fallback ran"
    assert st["last_candidates"] <= nq * 8192
    check_oracle(gi, gs, qs, oracle_index(packed, corr, cen, sim), k, (0, nq - 1))


# ---- 4. fewer than k rows score finitely: NaN-scored rows fill the tail, by ascending id, on every path ----------------
def nan_heavy(packed, corr, finite, seed, pool=None):
    """upperInterval of every row but `finite` seeded ones (drawn from `pool`, default all rows) := NaN (a degenerate
    interval: the row scores NaN)."""
    pool = np.arange(len(corr)) if pool is None else pool
    keep = np.random.default_rng(seed).choice(pool, finite, replace=False)
    c = corr.copy()
    mask = np.ones(len(c), bool)
    mask[keep] = False
    c[mask, 1] = np.nan
    return packed, c


NAN_CASES = [(5, 10), (3000, 4096), (0, 10)]


@pytest.mark.parametrize("sim", SIMS)
@pytest.mark.parametrize("finite,k", NAN_CASES)
def test_fewer_than_k_finite_rows_every_path(bbq, corpora, sim, finite, k):
    dim = 128
    qs = gaussian(8, dim, 4242)
    for n in (40000, 9000):
        packed, corr = nan_heavy(*corpora(sim, 40000, dim)[:2], finite, 77 + finite)
        packed, corr, cen = packed[:n], corr[:n], np.zeros(dim, np.float32)
        oidx = oracle_index(packed, corr, cen, sim)
        wants = [O.search_nearest_neighbors(q, oidx, k, mode="canonical") for q in qs]
        nfin = int(np.isfinite(wants[0][1]).sum())
        assert nfin == min(k, int(np.isfinite(corr[:, 1]).sum())) and len(wants[0][0]) == min(k, n)
        assert np.all(np.diff(wants[0][0][nfin:]) > 0)            # the NaN tail by ascending id
        if finite == 0:
            assert wants[0][0].tolist() == list(range(k))
        runs = [("popc", None, 3), ("mma", None, 8), (None, 1, 8), (None, 2, 8)] if n > 16384 else [(None, None, 8)]
        for scan, force, nq in runs:
            fmt = make_format(bbq, sim, scan=scan, force_path=force)
            gi, gs = fmt.searchBatch(qs[:nq], fmt.adoptQuantized(packed, corr, cen), k)
            for qi in range(nq):
                assert gi[qi].tolist() == wants[qi][0].tolist(), (n, scan, force, qi)
                assert bits_equal(gs[qi], wants[qi][1]), (n, scan, force, qi)
            st = fmt.stats()
            if n <= 16384:
                assert st["last_path"] == 0
            elif force == 2:
                assert st["last_path"] == 2 and st["last_overflow"] == 0
            else:   # the filtered scan came up short and the exact chunked path redid the batch
                assert st["last_path"] == 2 and st["last_overflow"] == 1


@pytest.mark.parametrize("finite,k", NAN_CASES)
def test_fewer_than_k_finite_rows_sharded_merge(bbq, corpora, finite, k):
    """3 row shards (filtered path, direct path, filtered path), the middle one all NaN, merged by bbq_merge_topk_device."""
    import torch
    sim, dim, nq = "COSINE", 128, 6
    bounds = [0, 17000, 23000, 40000]
    pool = np.r_[0:bounds[1], bounds[2]:bounds[3]]
    packed, corr = nan_heavy(*corpora(sim, 40000, dim)[:2], finite, 91 + finite, pool)
    cen = np.zeros(dim, np.float32)
    qs = gaussian(nq, dim, 4343)
    fmt = make_format(bbq, sim)
    L = bbq._native.load()
    dq = torch.from_numpy(qs).cuda()
    all_idx = torch.empty((3, nq, k), dtype=torch.int32, device="cuda")
    all_sc = torch.empty((3, nq, k), dtype=torch.float32, device="cuda")
    keep = []
    for s in range(3):
        a, b = bounds[s], bounds[s + 1]
        qv = fmt.adoptQuantized(packed[a:b], corr[a:b], cen)
        assert L.bbq_index_set_base(qv._h, a) == 0
        assert L.bbq_search_device(qv._h, dq.data_ptr(), nq, k, all_idx[s].data_ptr(), all_sc[s].data_ptr(), None) == 0, \
            L.bbq_last_error()
        keep.append(qv)
    torch.cuda.synchronize()
    out_idx = torch.empty((nq, k), dtype=torch.int32, device="cuda")
    out_sc = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    assert L.bbq_merge_topk_device(fmt._ctx, all_idx.data_ptr(), all_sc.data_ptr(), 3, nq, k, out_idx.data_ptr(),
                                   out_sc.data_ptr(), None) == 0, L.bbq_last_error()
    torch.cuda.synchronize()
    check_oracle(out_idx.cpu().numpy(), out_sc.cpu().numpy(), qs, oracle_index(packed, corr, cen, sim), k, range(nq))


# ---- 5. more than one query batch (4096 queries) per call -----------------------------------------------------------------
@pytest.fixture(scope="module")
def batch_corpus(bbq):
    """60000 x 256 COSINE rows on the device, with the index and its f32 rows attached for the re-rank."""
    import torch
    n, dim = 60000, 256
    rows_d = device_rows(n, dim, 20261021)
    cen = np.zeros(dim, np.float32)
    fmt = make_format(bbq, "COSINE")
    qv = fmt.quantizeVectorsDevice(rows_d.data_ptr(), n, dim, centroid=cen)["quantizedVectors"]
    fmt.attachOriginalVectorsDevice(qv, rows_d.data_ptr())
    torch.cuda.synchronize()
    packed, corr = qv.exportAll()
    yield fmt, qv, oracle_index(packed, corr, cen, "COSINE")
    del qv, rows_d
    torch.cuda.empty_cache()


@pytest.mark.parametrize("k", [10, 100])
@pytest.mark.parametrize("nq,tail_engine", [(4099, 1), (8200, 2)])   # a tail of 3 on K1s, a tail of 8 on narrow K2
def test_more_than_one_query_batch(bbq, batch_corpus, k, nq, tail_engine):
    fmt, qv, oidx = batch_corpus
    qs = gaussian(nq, 256, 5000 + nq)
    gi, gs = fmt.searchBatch(qs, qv, k)
    st = fmt.stats()
    assert st["last_path"] == 1 and st["last_overflow"] == 0 and st["last_engine"] == tail_engine
    if tail_engine == 2:
        assert st["mma_layout"] == 1
    for q0 in range(0, nq, 4096):
        si, ss = fmt.searchBatch(qs[q0:q0 + 4096], qv, k)
        assert np.array_equal(si, gi[q0:q0 + 4096]) and bits_equal(ss, gs[q0:q0 + 4096]), q0
    check_oracle(gi, gs, qs, oidx, k, (0, 4095, 4096, 4097, nq - 1))


def test_bad_query_past_the_first_batch(bbq, batch_corpus):
    fmt, qv, _ = batch_corpus
    qs = gaussian(8200, 256, 5101)
    want_i, want_s = fmt.searchBatch(qs[:10], qv, 10)
    qs[5000, 17] = np.nan
    with pytest.raises(bbq.BbqError) as e:
        fmt.searchBatch(qs, qv, 10)
    assert e.value.status == 5
    v, p = C.c_int64(-1), C.c_int64(-1)
    bbq._native.load().bbq_last_error_pos(C.byref(v), C.byref(p))
    assert v.value == 5000
    gi, gs = fmt.searchBatch(qs[:10], qv, 10)                       # the context answers as before
    assert np.array_equal(gi, want_i) and bits_equal(gs, want_s)


def test_oversampled_more_than_one_query_batch(bbq, batch_corpus):
    fmt, qv, _ = batch_corpus
    qs = gaussian(4100, 256, 5202)
    gi, gq, gt = fmt.searchOversampledBatch(qs, qv, 10, 3)
    for q0 in (0, 4096):
        si, sq, stt = fmt.searchOversampledBatch(qs[q0:q0 + 4096], qv, 10, 3)
        assert np.array_equal(si, gi[q0:q0 + 4096]) and bits_equal(sq, gq[q0:q0 + 4096]) and bits_equal(stt, gt[q0:q0 + 4096])


# ---- 6. oversampled re-rank at large m = k * factor -------------------------------------------------------------------------
@pytest.mark.parametrize("k,factor", [(100, 40), (1000, 4), (4096, 1)])
@pytest.mark.parametrize("nq,engine", [(3, 1), (20, 2)])
@pytest.mark.parametrize("dups", [1, 10])       # 10: every row 10 times, equal true scores ordered by candidate position
def test_oversampled_rerank_large_m(bbq, k, factor, nq, engine, dups):
    import torch
    n, dim = 40000, 128
    rows_d = device_rows(n // dups, dim, 31337 + dups).repeat(dups, 1).contiguous()
    rows = rows_d.cpu().numpy()
    fmt = make_format(bbq, "COSINE")
    qv = fmt.quantizeVectorsDevice(rows_d.data_ptr(), n, dim)["quantizedVectors"]
    fmt.attachOriginalVectorsDevice(qv, rows_d.data_ptr())
    torch.cuda.synchronize()
    packed, corr = qv.exportAll()
    oidx = oracle_index(packed, corr, qv.getCentroid(), "COSINE")
    qs = gaussian(nq, dim, 31400 + nq)
    gi, gq, gt = fmt.searchOversampledBatch(qs, qv, k, factor)
    st = fmt.stats()
    assert st["last_path"] == 1 and st["last_overflow"] == 0 and st["last_engine"] == engine
    for qi in spread(nq):
        wi, wq, wt = O.oversampled_topk(qs[qi], rows, oidx, k, factor)
        assert gi[qi].tolist() == wi.tolist(), qi
        assert bits_equal(gq[qi], wq) and bits_equal(gt[qi], wt), qi
    del qv, rows_d
    torch.cuda.empty_cache()


# ---- 7. the captured launch sequence at large k -------------------------------------------------------------------------
def _direct_capture_replay(fmt, qv, qs, k):
    """Calls with one batch until the captured sequence has been replayed once.  The first call sizes the scratch
    buffers, which changes the key, so the sequence is captured on the third call and replayed on the fourth."""
    r0 = fmt.stats()["graph_replays"]
    out = []
    while fmt.stats()["graph_replays"] == r0:
        assert len(out) < 6, "the launch sequence was never replayed"
        out.append(fmt.searchBatch(qs, qv, k))
    assert len(out) >= 3 and fmt.stats()["graph_replays"] == r0 + 1   # direct calls, a capturing call, one replay
    for gi, gs in out[1:]:
        assert np.array_equal(gi, out[0][0]) and bits_equal(gs, out[0][1])
    return out[2]


def test_replayed_sequence_large_k(bbq, corpora):
    sim, n, dim, k = "EUCLIDEAN", 40000, 128, 1000
    packed, corr, cen = corpora(sim, n, dim)
    fmt = make_format(bbq, sim)
    qv = fmt.adoptQuantized(packed, corr, cen)
    qs = gaussian(8, dim, 6060)
    gi, gs = _direct_capture_replay(fmt, qv, qs, k)
    st = fmt.stats()
    assert st["last_path"] == 1 and st["last_engine"] == 2 and st["last_overflow"] == 0
    check_oracle(gi, gs, qs, oracle_index(packed, corr, cen, sim), k, (0, 3, 7))


def test_replayed_sequence_fewer_than_k_finite_rows(bbq, corpora):
    sim, dim, k = "EUCLIDEAN", 128, 1000
    packed, corr = nan_heavy(*corpora(sim, 40000, dim)[:2], 300, 606)
    cen = np.zeros(dim, np.float32)
    fmt = make_format(bbq, sim)
    qv = fmt.adoptQuantized(packed, corr, cen)
    qs = gaussian(8, dim, 6161)
    gi, gs = _direct_capture_replay(fmt, qv, qs, k)
    st = fmt.stats()
    assert st["last_path"] == 2 and st["last_overflow"] == 1       # the replayed filtered scan came up short
    check_oracle(gi, gs, qs, oracle_index(packed, corr, cen, sim), k, range(8))
