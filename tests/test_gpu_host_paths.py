"""GPU: host orchestration paths the other tests do not reach.  The hierarchical top-k merge over more than one level
(through bbq_merge_topk_device and through the exact chunked search), and the build loop shared by the one-shot and
the streaming builds.  Everything is compared bit for bit with the oracle or with another entry point."""
import numpy as np
import pytest

from oracle import oracle as O
from tests.fixtures import gaussian
from tests.test_gpu_parity import SIMS, bits_equal, make_format

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bbq():
    import bbq_b200
    bbq_b200.build_library()
    return bbq_b200


# ---- bbq_merge_topk_device: groups of max(2, 16384 / k) lists, so these take two levels ------------------------------
@pytest.mark.parametrize("k,sizes", [
    (4096, [700, 3000, 9000, 5000, 1200, 8000, 4100, 2000, 7000]),    # 9 lists, groups of 4
    (2000, [500, 1500] + [2400] * 15),                                # 17 lists, groups of 8
])
def test_merge_topk_device_multi_level(bbq, k, sizes):
    import torch
    n, dim, nq = sum(sizes), 64, 3
    rows, qs = gaussian(n, dim, 601 + k), gaussian(nq, dim, 602 + k)
    idx = O.quantize_vectors(rows, sim="COSINE", want_unpacked=False)
    fmt = make_format(bbq, "COSINE")
    L = bbq._native.load()
    lists = len(sizes)
    bounds = np.concatenate([[0], np.cumsum(sizes)])
    dq = torch.from_numpy(qs).cuda()
    all_idx = torch.empty((lists, nq, k), dtype=torch.int32, device="cuda")
    all_sc = torch.empty((lists, nq, k), dtype=torch.float32, device="cuda")
    keep = []
    for s in range(lists):
        a, b = int(bounds[s]), int(bounds[s + 1])
        qv = fmt.adoptQuantized(idx.packed[a:b], idx.corr[a:b], idx.centroid)
        assert L.bbq_index_set_base(qv._h, a) == 0
        st = L.bbq_search_device(qv._h, dq.data_ptr(), nq, k, all_idx[s].data_ptr(), all_sc[s].data_ptr(), None)
        assert st == 0, L.bbq_last_error()
        keep.append(qv)
    torch.cuda.synchronize()
    assert (all_idx < 0).any(), "a shard smaller than k leaves empty (-1) slots"
    out_idx = torch.empty((nq, k), dtype=torch.int32, device="cuda")
    out_sc = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    st = L.bbq_merge_topk_device(fmt._ctx, all_idx.data_ptr(), all_sc.data_ptr(), lists, nq, k, out_idx.data_ptr(),
                                 out_sc.data_ptr(), None)
    assert st == 0, L.bbq_last_error()
    torch.cuda.synchronize()
    gi, gs = out_idx.cpu().numpy(), out_sc.cpu().numpy()
    for qi, q in enumerate(qs):
        wi, ws = O.search_nearest_neighbors(q, idx, k, mode="canonical")
        assert gi[qi].tolist() == wi.tolist() and bits_equal(gs[qi], ws)


# ---- exact chunked path: 6 chunks of 16384 rows merged in groups of 4 at k = 4096 --------------------------------------
def test_exact_chunked_multi_level_merge(bbq):
    n, dim, nq, k = 90000, 64, 3, 4096
    rows, qs = gaussian(n, dim, 611), gaussian(nq, dim, 612)
    want = O.quantize_vectors(rows, sim="EUCLIDEAN", want_unpacked=False)
    fmt = make_format(bbq, "EUCLIDEAN", force_path=2)
    qv = fmt.adoptQuantized(want.packed, want.corr, want.centroid)
    gi, gs = fmt.searchBatch(qs, qv, k)
    assert fmt.stats()["last_path"] == 2
    for qi, q in enumerate(qs):
        wi, ws = O.search_nearest_neighbors(q, want, k, mode="canonical")
        assert gi[qi].tolist() == wi.tolist() and bits_equal(gs[qi], ws)


# ---- one-shot build == streaming build from host chunks == streaming build from device chunks ------------------------
@pytest.mark.parametrize("sim", SIMS)
@pytest.mark.parametrize("ib", [1, 2])
def test_streaming_build_equals_one_shot(bbq, sim, ib):
    import torch
    n, dim = 70000, 100                                     # crosses BUILD_CHUNK (32768) twice
    rows = gaussian(n, dim, 621 + ib)
    cen = gaussian(1, dim, 622)[0]
    fmt = bbq.createBinaryQuantizationFormat(
        {"queryBits": 4, "indexBits": ib, "quantizer": {"similarityFunction": sim, "lambda": 0.1, "iters": 5}})
    one = fmt.quantizeVectors(rows, centroid=cen)["quantizedVectors"]
    cuts = [0, 1, 40001, 40002, 65000, n]                   # ragged appends, one of them larger than a build chunk
    host = fmt.reserveIndex(n, dim, cen)
    for a, b in zip(cuts[:-1], cuts[1:]):
        fmt.appendRows(host, rows[a:b])
    d_rows = torch.from_numpy(rows).cuda()
    torch.cuda.synchronize()
    dev = fmt.reserveIndex(n, dim, cen)
    for a, b in zip(cuts[:-1], cuts[1:]):
        fmt.appendRows(dev, d_rows_ptr=d_rows[a:b].data_ptr(), n=b - a)
    want_packed, want_corr = one.exportAll()
    for qv in (host, dev):
        assert qv.size() == n
        packed, corr = qv.exportAll()
        assert np.array_equal(packed, want_packed) and bits_equal(corr, want_corr)
        assert bits_equal(qv.getCentroid(), one.getCentroid())
        assert np.float64(qv.getCentroidDP()).tobytes() == np.float64(one.getCentroidDP()).tobytes()
