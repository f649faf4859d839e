"""Device groups: one process and one caller thread over several GPUs (bbq_group_*).

Every group result is compared, bit for bit, with the single-GPU entry on one index of the whole corpus: the build's
exports and centroid (every similarity, indexBits 1 and 2, N not divisible by the group size, N below it), the search
lists, scores and counts (queryBits 1, 4 and 8; nq up to past one 4096-query step; k = 1, 100 and k > N), the re-rank's
ids, quantised scores and f64 true scores, and the saved image.  Errors read on the caller's thread equal the
single-index entry's.  Groups of 1 (no communicator), 2, 3 and all GPUs; sizes above the GPUs present are skipped."""
import ctypes as C
import os

import numpy as np
import pytest

from tests.fixtures import gaussian

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bbq():
    import bbq_b200
    bbq_b200.build_library()
    return bbq_b200


def _n_gpus():
    import torch
    return torch.cuda.device_count()


SIZES = ["1", "2", "3", "all"]


def _devices(size):
    n = _n_gpus()
    want = n if size == "all" else int(size)
    if want > n or (size == "all" and n in (1, 2, 3)):
        pytest.skip(f"needs {want} GPUs, {n} present" if want > n else "'all' equals a size covered already")
    return list(range(want))


def _cfg(sim="COSINE", index_bits=1, query_bits=4):
    return {"queryBits": query_bits, "indexBits": index_bits,
            "quantizer": {"similarityFunction": sim, "lambda": 0.1, "iters": 5}}


def _pair(bbq, devices, **kw):
    """(group format, single-GPU format on the group's first device)"""
    return (bbq.BinaryQuantizationFormat(_cfg(**kw), devices=devices),
            bbq.BinaryQuantizationFormat(_cfg(**kw), device=devices[0]))


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64 if a.dtype == np.float64 else np.uint32)


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("sim,index_bits", [("EUCLIDEAN", 1), ("COSINE", 1), ("MAXIMUM_INNER_PRODUCT", 1),
                                            ("COSINE", 2), ("EUCLIDEAN", 2)])
def test_build_exports_equal_the_whole_corpus_build(bbq, size, sim, index_bits):
    devices = _devices(size)
    gf, sf = _pair(bbq, devices, sim=sim, index_bits=index_bits)
    for n in (5003, 2):   # not divisible by 2 or 3; fewer rows than GPUs (empty shards)
        rows = gaussian(n, 100, 7100 + n)
        gi = gf.quantizeVectors(rows)["quantizedVectors"]
        si = sf.quantizeVectors(rows)["quantizedVectors"]
        assert isinstance(gi, bbq.GroupBinarizedByteVectorValues)
        assert gi.size() == n and gi.dimension() == 100
        assert np.array_equal(_bits(gi.getCentroid()), _bits(si.getCentroid()))
        assert _bits(np.float64(gi.getCentroidDP())) == _bits(np.float64(si.getCentroidDP()))
        gp, gc = gi.exportAll()
        sp, sc = si.exportAll()
        assert np.array_equal(gp, sp) and np.array_equal(_bits(gc), _bits(sc))
        # ranges that span shard boundaries, and single rows
        for first, count in ((0, n), (n // 3 - 2, 5), (n // 2 - 1, n), (n - 1, 1)):
            first = max(0, first)
            count = min(count, n - first)
            p, c = gi._export(first, count)
            assert np.array_equal(p, sp[first:first + count]) and np.array_equal(_bits(c), _bits(sc[first:first + count]))
        assert np.array_equal(gi.getUnpackedVector(n - 1), si.getUnpackedVector(n - 1))
        assert gi.getCorrectiveTerms(0) == si.getCorrectiveTerms(0)


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("query_bits", [1, 4, 8])
def test_search_equals_the_single_gpu_search(bbq, size, query_bits):
    devices = _devices(size)
    gf, sf = _pair(bbq, devices, sim="EUCLIDEAN", query_bits=query_bits)
    rows = gaussian(20011, 128, 7200)
    queries = gaussian(5000, 128, 7201)
    gi = gf.quantizeVectors(rows)["quantizedVectors"]
    si = sf.quantizeVectors(rows)["quantizedVectors"]
    for nq in (1, 8, 1024, 5000):
        for k in (1, 100):
            a = gf.searchBatch(queries[:nq], gi, k)
            b = sf.searchBatch(queries[:nq], si, k)
            assert np.array_equal(a[0], b[0]) and np.array_equal(_bits(a[1]), _bits(b[1])), (nq, k)
    # k > N, with empty tail slots the caller never sees (out_count = N)
    small = rows[:301]
    gs = gf.quantizeVectors(small)["quantizedVectors"]
    ss = sf.quantizeVectors(small)["quantizedVectors"]
    a, b = gf.searchBatch(queries[:8], gs, 310), sf.searchBatch(queries[:8], ss, 310)
    assert a[0].shape == (8, 301) and np.array_equal(a[0], b[0]) and np.array_equal(_bits(a[1]), _bits(b[1]))
    got = gf.searchNearestNeighbors(queries[0], gs, 5)
    want = sf.searchNearestNeighbors(queries[0], ss, 5)
    assert got == want


@pytest.mark.parametrize("size", SIZES)
def test_rerank_equals_the_single_gpu_rerank(bbq, size):
    devices = _devices(size)
    gf, sf = _pair(bbq, devices, sim="COSINE")
    rows = gaussian(9001, 96, 7300)
    queries = gaussian(300, 96, 7301)
    gi = gf.quantizeVectors(rows)["quantizedVectors"]
    si = sf.quantizeVectors(rows)["quantizedVectors"]
    with pytest.raises(bbq.BbqError) as eg:
        gf.searchOversampledBatch(queries[:2], gi, 10, 4)
    with pytest.raises(bbq.BbqError) as es:
        sf.searchOversampledBatch(queries[:2], si, 10, 4)
    assert (eg.value.status, str(eg.value)) == (es.value.status, str(es.value)) and es.value.status == 10
    gf.attachOriginalVectors(gi, rows)
    sf.attachOriginalVectors(si, rows)
    for k, factor in ((10, 4), (100, 5), (1, 1)):
        a = gf.searchOversampledBatch(queries, gi, k, factor)
        b = sf.searchOversampledBatch(queries, si, k, factor)
        assert np.array_equal(a[0], b[0]) and np.array_equal(_bits(a[1]), _bits(b[1])) and \
            np.array_equal(_bits(a[2]), _bits(b[2])), (k, factor)


@pytest.mark.parametrize("size", SIZES)
def test_images(bbq, size, tmp_path):
    devices = _devices(size)
    gf, sf = _pair(bbq, devices, sim="MAXIMUM_INNER_PRODUCT")
    rows = gaussian(7777, 128, 7400)
    gi = gf.quantizeVectors(rows)["quantizedVectors"]
    si = sf.quantizeVectors(rows)["quantizedVectors"]
    gf.saveIndex(gi, str(tmp_path / "g"))
    sf.saveIndex(si, str(tmp_path / "s"))
    for ext in (".veb", ".vemb"):
        assert (tmp_path / ("g" + ext)).read_bytes() == (tmp_path / ("s" + ext)).read_bytes(), ext
    # an image written by one GPU, loaded by this group (and the group's image by one GPU)
    lg = gf.loadIndex(str(tmp_path / "s"))
    ls = sf.loadIndex(str(tmp_path / "g"))
    assert lg.size() == 7777 and np.array_equal(_bits(lg.getCentroid()), _bits(si.getCentroid()))
    for x in (lg, ls):
        p, c = x.exportAll()
        sp, sc = si.exportAll()
        assert np.array_equal(p, sp) and np.array_equal(_bits(c), _bits(sc))
    q = gaussian(64, 128, 7401)
    a, b = gf.searchBatch(q, lg, 50), sf.searchBatch(q, si, 50)
    assert np.array_equal(a[0], b[0]) and np.array_equal(_bits(a[1]), _bits(b[1]))
    # a corrupted codes section
    veb = tmp_path / "s.veb"
    data = bytearray(veb.read_bytes())
    data[len(data) // 3] ^= 0x10
    veb.write_bytes(bytes(data))
    with pytest.raises(bbq.BbqError) as e:
        gf.loadIndex(str(tmp_path / "s"))
    assert e.value.status == 12


def test_a_group_of_another_size_loads_the_image(bbq, tmp_path):
    n = _n_gpus()
    if n < 2:
        pytest.skip("needs 2 GPUs")
    rows = gaussian(3001, 64, 7500)
    g2 = bbq.BinaryQuantizationFormat(_cfg(), devices=[0, 1])
    gi = g2.quantizeVectors(rows)["quantizedVectors"]
    g2.saveIndex(gi, str(tmp_path / "two"))
    want = gi.exportAll()
    for devs in ([1], list(range(min(n, 3)))):
        g = bbq.BinaryQuantizationFormat(_cfg(), devices=devs)
        got = g.loadIndex(str(tmp_path / "two")).exportAll()
        assert np.array_equal(got[0], want[0]) and np.array_equal(_bits(got[1]), _bits(want[1]))


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("sim", ["EUCLIDEAN", "COSINE"])
def test_errors_match_the_single_index_entries(bbq, size, sim):
    devices = _devices(size)
    gf, sf = _pair(bbq, devices, sim=sim)
    L = bbq._native.load()
    rows = gaussian(5003, 40, 7600)
    for bad in (np.nan, np.inf):
        r = rows.copy()
        r[5001, 7] = bad   # in the last rank's rows
        outcomes = []
        for f in (gf, sf):
            with pytest.raises(bbq.BbqError) as e:
                f.quantizeVectors(r)
            v, p = C.c_int64(), C.c_int64()
            L.bbq_last_error_pos(C.byref(v), C.byref(p))
            outcomes.append((e.value.status, str(e.value), L.bbq_last_error().decode(), v.value, p.value))
        assert outcomes[0] == outcomes[1] and outcomes[0][3] == 5001, outcomes
    gi = gf.quantizeVectors(rows)["quantizedVectors"]
    si = sf.quantizeVectors(rows)["quantizedVectors"]
    q = gaussian(3, 40, 7601)
    qn = q.copy()
    qn[1, 3] = np.nan
    cases = [lambda f, x: f.searchBatch(qn, x, 10), lambda f, x: f.searchBatch(q, x, -1),
             lambda f, x: f.searchBatch(q, x, 5000), lambda f, x: f.searchBatch(q[:, :39], x, 10),
             lambda f, x: f.searchNearestNeighbors(q[0, :30], x, 10)]
    for case in cases:
        got = []
        for f, x in ((gf, gi), (sf, si)):
            with pytest.raises(bbq.BbqError) as e:
                case(f, x)
            got.append((e.value.status, str(e.value)))
        assert got[0] == got[1], got
    # the group stays usable after every one of them
    a, b = gf.searchBatch(q, gi, 10), sf.searchBatch(q, si, 10)
    assert np.array_equal(a[0], b[0])


@pytest.mark.parametrize("size", ["1", "2"])
def test_destroy_with_a_live_index_and_collectives_on_group_contexts(bbq, size, tmp_path):
    devices = _devices(size)
    L = bbq._native.load()
    gf = bbq.BinaryQuantizationFormat(_cfg(), devices=devices)
    assert gf.devices() == devices
    rows = gaussian(1000, 64, 7700)
    gi = gf.quantizeVectors(rows)["quantizedVectors"]
    assert L.bbq_group_destroy(gf._group) == 10
    assert "still alive" in L.bbq_last_error().decode()
    gf.saveIndex(gi, str(tmp_path / "x"))
    ctx = gf.groupContext(len(devices) - 1)
    h = C.c_void_p()
    veb, vemb = os.fsencode(str(tmp_path / "x.veb")), os.fsencode(str(tmp_path / "x.vemb"))
    # collective entries on a group's context, from outside the group: refused, never a hang
    assert L.bbq_index_load_sharded(ctx, veb, vemb, C.byref(h)) == 10 and not h.value
    assert "device group" in L.bbq_last_error().decode()
    assert L.bbq_index_build_sharded(ctx, rows.ctypes.data, 1000, 64, None, C.byref(h)) == 10
    assert L.bbq_comm_destroy(ctx) == 10
    # non-collective members of a group context still work
    assert L.bbq_index_load(ctx, veb, vemb, C.byref(h)) == 0
    L.bbq_index_destroy(h)
    i, s = gf.searchBatch(rows[:4], gi, 3)
    assert i[:, 0].tolist() == [0, 1, 2, 3]


def test_lifetime_threads_and_per_rank_stats(bbq):
    devices = list(range(min(_n_gpus(), 4)))
    L = bbq._native.load()

    def tasks():
        return len(os.listdir("/proc/self/task"))

    def cycle():
        gf = bbq.BinaryQuantizationFormat(_cfg(), devices=devices)
        gi = gf.quantizeVectors(gaussian(20000, 128, 7800))["quantizedVectors"]
        before = []
        for r in range(len(devices)):
            st = bbq._native.BbqStats()
            assert L.bbq_get_stats(C.c_void_p(gf.groupContext(r)), C.byref(st)) == 0
            before.append(st.kernel_launches)
        gf.searchBatch(gaussian(64, 128, 7801), gi, 10)
        for r in range(len(devices)):
            st = bbq._native.BbqStats()
            assert L.bbq_get_stats(C.c_void_p(gf.groupContext(r)), C.byref(st)) == 0
            assert st.kernel_launches > before[r] and st.last_engine in (1, 2), r   # every rank ran its scan
        del gi
        assert L.bbq_group_destroy(gf._group) == 0
        gf._group = None

    cycle()   # the CUDA runtime's and NCCL's own threads of first use
    t0 = tasks()
    for _ in range(3):
        cycle()
    assert tasks() == t0


@pytest.mark.parametrize("size", SIZES)
def test_python_end_to_end_and_from_quantized(bbq, size):
    devices = _devices(size)
    gf, sf = _pair(bbq, devices, sim="COSINE")
    rows = gaussian(4099, 72, 7900)
    q = gaussian(40, 72, 7901)
    gi = gf.quantizeVectors(rows)["quantizedVectors"]
    si = sf.quantizeVectors(rows)["quantizedVectors"]
    assert gf.searchNearestNeighbors(q[0], gi, 20) == sf.searchNearestNeighbors(q[0], si, 20)
    a, b = gf.searchBatch(q, gi, 33), sf.searchBatch(q, si, 33)
    assert np.array_equal(a[0], b[0]) and np.array_equal(_bits(a[1]), _bits(b[1]))
    gf.attachOriginalVectors(gi, rows)
    sf.attachOriginalVectors(si, rows)
    a, b = gf.searchOversampledBatch(q, gi, 10, 3), sf.searchOversampledBatch(q, si, 10, 3)
    assert all(np.array_equal(_bits(x), _bits(y)) for x, y in zip(a, b))
    # serializeVectorData / deserializeVectorData through the group (from_quantized: one slice per GPU)
    ser = gf.serializeVectorData(rows)
    back = gf.deserializeVectorData(ser["vectorData"], ser["metadata"])
    assert isinstance(back, bbq.GroupBinarizedByteVectorValues)
    a, b = gf.searchBatch(q, back, 33), sf.searchBatch(q, si, 33)
    assert np.array_equal(a[0], b[0]) and np.array_equal(_bits(a[1]), _bits(b[1]))
    # members that run on the group's first GPU
    assert gf.quantizeQueryVector(q[0], gi.getCentroid())["quantizedQuery"].tolist() == \
        sf.quantizeQueryVector(q[0], si.getCentroid())["quantizedQuery"].tolist()
    with pytest.raises(bbq.BbqError) as e:
        gf.searchBatch(q, gi, 10, sharded=True)
    assert e.value.status == 10
    # a group index never reaches a bbq_index_* entry, and one-GPU members refuse a group format
    for call in (lambda: gf.quantizeQueryVector(q[0], gi), lambda: sf.quantizeQueryVector(q[0], gi),
                 lambda: sf.debugScores(q[0], gi), lambda: sf.setBase(gi, 0),
                 lambda: gf.quantizeVectorsDevice(0, 1, 72), lambda: gf.reserveIndex(10, 72, gi.getCentroid())):
        with pytest.raises(bbq.BbqError) as e:
            call()
        assert e.value.status == 10
    # the search-path quantisation of a one-GPU index still works on a group format's first GPU
    assert gf.quantizeQueryVector(q[0], si)["quantizedQuery"].tolist() == \
        sf.quantizeQueryVector(q[0], si)["quantizedQuery"].tolist()
