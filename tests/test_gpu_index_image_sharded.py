"""One index image across row shards: bbq_index_write_rows / _write_meta / _load_rows (shard-local) and
bbq_index_save_sharded / _load_sharded (collective).

On one GPU, shards are emulated as slices of one index (adoptQuantized of packed[r0:r1] plus bbq_index_set_base):
the image written shard by shard, in any order, equals bbq_index_save of the whole index byte for byte; row ranges load
back with partial checksums that sum to the header's, their rows equal the matching slices, and their merged searches
equal the whole-index search and the oracle bit for bit; an image written from 3 shards reloads as 2 ranges or whole;
a flipped bit inside one range changes that range's partial and fails a whole-range load; and the refusals.  On two
GPUs (skipped below that): the collective save equals a single-index save, the collective load searches like the
oracle on every rank, and a per-rank failure fails both ranks alike."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from tests.fixtures import gaussian

pytestmark = pytest.mark.gpu

M64 = (1 << 64) - 1


@pytest.fixture(scope="module")
def bbq():
    import bbq_b200
    bbq_b200.build_library()
    return bbq_b200


@pytest.fixture(scope="module")
def image():
    import importlib
    import bbq_b200  # noqa: F401  (registers the package under its importable name)
    return importlib.import_module("better_binary_quantization_b200.host.image")


def _fmt(bbq, sim="COSINE", index_bits=1, device=-1):
    return bbq.createBinaryQuantizationFormat(
        {"queryBits": 4, "indexBits": index_bits, "quantizer": {"similarityFunction": sim, "lambda": 0.1, "iters": 5}},
        device=device)


def _shard(fmt, packed, corr, cen, r0, r1):
    """rows [r0, r1) of an index as a shard of its own with base r0 (an empty one for r0 == r1)."""
    if r1 > r0:
        s = fmt.adoptQuantized(packed[r0:r1], corr[r0:r1], cen)
    else:
        s = fmt.reserveIndex(1, cen.size, cen)          # capacity 1, 0 rows
    fmt.setBase(s, r0)
    assert s.size() == r1 - r0
    return s


def _read(p):
    with open(p, "rb") as f:
        return f.read()


def _same_files(a, b):
    return _read(a + ".veb") == _read(b + ".veb") and _read(a + ".vemb") == _read(b + ".vemb")


def _sum(parts):
    out = [0] * 5
    for p in parts:
        out = [(x + y) & M64 for x, y in zip(out, p)]
    return out


def _header_sums(image, prefix):
    meta = image.read_metadata(prefix)
    return [meta["sectionChecksums"][s] for s in image.SECTIONS]


def _strides(image, dim):
    return (image.row_bytes_for(dim), 8, 8, 8, 4)


def _merged_search(bbq, fmt, shards, qs, k):
    """per-shard searchDevice (global ids through each base), merged by bbq_merge_topk_device -> (idx, score) [nq, k]"""
    import torch
    nq = qs.shape[0]
    shards = [s for s in shards if s.size() > 0]
    dq = torch.from_numpy(qs).cuda()
    li = torch.empty((len(shards), nq, k), dtype=torch.int32, device="cuda")
    ls = torch.empty((len(shards), nq, k), dtype=torch.float32, device="cuda")
    for j, s in enumerate(shards):
        fmt.searchDevice(dq.data_ptr(), nq, s, k, li[j].data_ptr(), ls[j].data_ptr())
    oi = torch.empty((nq, k), dtype=torch.int32, device="cuda")
    os_ = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    fmt.mergeTopKDevice(li.data_ptr(), ls.data_ptr(), len(shards), nq, k, oi.data_ptr(), os_.data_ptr())
    torch.cuda.synchronize()
    return oi.cpu().numpy(), os_.cpu().numpy()


SPLITS = {
    "two": lambda n: [0, n // 2 + 7, n],
    "three": lambda n: [0, 1000, 1001, n],                                       # a 1-row shard
    "eight": lambda n: [0, 5, 6, 900, 900, 1700, 2400, 2999, n],                 # a 1-row and an empty shard
}


# ---- 1. the image written shard by shard (in reverse order) is bbq_index_save of the whole index, byte for byte ----
@pytest.mark.parametrize("split", sorted(SPLITS))
@pytest.mark.parametrize("sim,dim", [("COSINE", 100), ("EUCLIDEAN", 128), ("MAXIMUM_INNER_PRODUCT", 768)])
def test_split_save_equals_whole_save(bbq, image, tmp_path, split, sim, dim):
    n = 3001
    rows = gaussian(n, dim, 4100 + dim)
    fmt = _fmt(bbq, sim)
    built = fmt.quantizeVectors(rows)["quantizedVectors"]
    packed, corr = built.exportAll()
    cen = built.getCentroid()
    whole = fmt.adoptQuantized(packed, corr, cen)
    a, b = str(tmp_path / "whole"), str(tmp_path / "split")
    fmt.saveIndex(whole, a)
    bounds = SPLITS[split](n)
    shards = [_shard(fmt, packed, corr, cen, r0, r1) for r0, r1 in zip(bounds[:-1], bounds[1:])]
    parts = {}
    for (r0, r1), s in reversed(list(zip(zip(bounds[:-1], bounds[1:]), shards))):
        parts[r0, r1] = fmt.writeIndexRows(s, b, n)
    fmt.writeIndexMeta(shards[-1], b, n, _sum(parts.values()))
    assert _same_files(a, b)
    assert _sum(parts.values()) == _header_sums(image, a)
    # each partial is the host reader's checksum of that slice of the section, counted from the image's row 0
    veb = _read(a + ".veb")
    meta = image.read_metadata(a)
    for (r0, r1), part in parts.items():
        for i, (name, stride) in enumerate(zip(image.SECTIONS, _strides(image, dim))):
            off = meta["sectionOffsets"][name]
            raw = veb[off + r0 * stride: off + r1 * stride]
            assert part[i] == image.section_checksum(raw, first_word=r0 * stride // 4), (r0, r1, name)


# ---- 2. row ranges of an image: partials, rows, and searches merged across ranges -----------------------------------
@pytest.mark.parametrize("sim,dim", [("COSINE", 128), ("EUCLIDEAN", 100), ("MAXIMUM_INNER_PRODUCT", 768)])
def test_range_load(bbq, image, tmp_path, sim, dim):
    n = 3001
    rows, qs = gaussian(n, dim, 4200 + dim), gaussian(9, dim, 4300 + dim)
    fmt = _fmt(bbq, sim)
    whole = fmt.quantizeVectors(rows)["quantizedVectors"]
    packed, corr = whole.exportAll()
    prefix = str(tmp_path / "index")
    fmt.saveIndex(whole, prefix)
    bounds = [0, 7, 8, 1500, 1500, 2222, n]                      # 7 rows, 1 row, an empty range
    shards, parts = [], []
    for r0, r1 in zip(bounds[:-1], bounds[1:]):
        s, part = fmt.loadIndexRows(prefix, r0, r1 - r0)
        assert s.size() == r1 - r0 and s.dimension() == dim
        assert s.getCentroidDP() == whole.getCentroidDP()
        p, c = s.exportAll()
        assert np.array_equal(p, packed[r0:r1]) and np.array_equal(c.view(np.uint64), corr[r0:r1].view(np.uint64))
        shards.append(s)
        parts.append(part)
    assert _sum(parts) == _header_sums(image, prefix)
    assert parts[3] == [0] * 5                                  # the empty range
    full = O.quantize_vectors(rows, sim=sim, want_unpacked=False)
    for k in (10, 20):                                          # 20 > the 7-row and the 1-row range
        gi, gs = _merged_search(bbq, fmt, shards, qs, k)
        wi, ws = fmt.searchBatch(qs, whole, k)
        assert np.array_equal(gi, wi) and np.array_equal(gs.view(np.uint32), ws.view(np.uint32)), k
        for qi in range(qs.shape[0]):
            oi, osc = O.search_nearest_neighbors(qs[qi], full, k, mode="canonical")
            assert gi[qi].tolist() == oi.tolist() and gs[qi].view(np.uint32).tolist() == osc.view(np.uint32).tolist()


# ---- 3. written from 3 shards, read as 2 ranges and as one index ----------------------------------------------------
def test_reshard(bbq, image, tmp_path):
    n, dim = 5000, 256
    rows, qs = gaussian(n, dim, 4401), gaussian(9, dim, 4402)
    fmt = _fmt(bbq, "COSINE")
    built = fmt.quantizeVectors(rows)["quantizedVectors"]
    packed, corr = built.exportAll()
    cen = built.getCentroid()
    prefix = str(tmp_path / "index")
    bounds3 = [0, 1234, 3333, n]
    shards3 = [_shard(fmt, packed, corr, cen, r0, r1) for r0, r1 in zip(bounds3[:-1], bounds3[1:])]
    fmt.writeIndexMeta(shards3[0], prefix, n, _sum([fmt.writeIndexRows(s, prefix, n) for s in shards3]))
    one = fmt.loadIndex(prefix)
    halves = [fmt.loadIndexRows(prefix, 0, 2500)[0], fmt.loadIndexRows(prefix, 2500, n - 2500)[0]]
    for k in (10, 100):
        wi, ws = fmt.searchBatch(qs, one, k)
        bi, bs = fmt.searchBatch(qs, built, k)
        gi, gs = _merged_search(bbq, fmt, halves, qs, k)
        assert np.array_equal(wi, bi) and np.array_equal(ws.view(np.uint32), bs.view(np.uint32))
        assert np.array_equal(gi, wi) and np.array_equal(gs.view(np.uint32), ws.view(np.uint32))


# ---- 4. a flipped bit inside one range ------------------------------------------------------------------------------
@pytest.mark.parametrize("section,row,byte", [("binaryValues", 1800, 3), ("upperInterval", 2100, 6)])
def test_corruption_inside_one_range(bbq, image, tmp_path, section, row, byte):
    n, dim = 3000, 128
    fmt = _fmt(bbq, "COSINE")
    whole = fmt.quantizeVectors(gaussian(n, dim, 4501))["quantizedVectors"]
    prefix = str(tmp_path / "index")
    fmt.saveIndex(whole, prefix)
    bounds = [0, 1000, 2500, n]
    clean = [fmt.loadIndexRows(prefix, r0, r1 - r0)[1] for r0, r1 in zip(bounds[:-1], bounds[1:])]
    meta = image.read_metadata(prefix)
    stride = meta["rowBytes"] if section == "binaryValues" else 8
    blob = bytearray(_read(prefix + ".veb"))
    blob[meta["sectionOffsets"][section] + row * stride + byte] ^= 0x04
    with open(prefix + ".veb", "wb") as f:
        f.write(blob)
    bad = [fmt.loadIndexRows(prefix, r0, r1 - r0)[1] for r0, r1 in zip(bounds[:-1], bounds[1:])]
    which = image.SECTIONS.index(section)
    assert bad[0] == clean[0] and bad[2] == clean[2]
    assert bad[1][which] != clean[1][which] and [x for i, x in enumerate(bad[1]) if i != which] == \
        [x for i, x in enumerate(clean[1]) if i != which]
    assert _sum(bad) != _header_sums(image, prefix)
    for load in (lambda: fmt.loadIndexRows(prefix, 0, n), lambda: fmt.loadIndex(prefix)):
        with pytest.raises(bbq.BbqError) as e:
            load()
        assert e.value.status == 12 and "checksum" in str(e.value)


# ---- 5. refusals, and the collective entries without a communicator ---------------------------------------------------
def test_refusals_and_entries_without_communicator(bbq, tmp_path):
    n, dim = 1000, 64
    rows = gaussian(n, dim, 4601)
    fmt = _fmt(bbq, "EUCLIDEAN")
    whole = fmt.quantizeVectors(rows)["quantizedVectors"]
    packed, corr = whole.exportAll()
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    fmt.saveIndex(whole, a)
    for first, count in ((0, n + 1), (990, 11), (n + 1, 0)):
        with pytest.raises(bbq.BbqError) as e:
            fmt.loadIndexRows(a, first, count)
        assert e.value.status == 10, (first, count)
    s, part = fmt.loadIndexRows(a, n, 0)
    assert s.size() == 0 and part == [0] * 5
    tail = _shard(fmt, packed, corr, whole.getCentroid(), 600, n)
    for total in (999, 600):
        with pytest.raises(bbq.BbqError) as e:
            fmt.writeIndexRows(tail, b, total)
        assert e.value.status == 10
        with pytest.raises(bbq.BbqError) as e:
            fmt.writeIndexMeta(tail, b, total, [0] * 5)
        assert e.value.status == 10
    # 2-bit indexes have no image, on any entry
    fmt2 = _fmt(bbq, "EUCLIDEAN", index_bits=2)
    two = fmt2.quantizeVectors(rows)["quantizedVectors"]
    for call in (lambda: fmt2.saveIndex(two, b), lambda: fmt2.saveIndex(two, b, sharded=True),
                 lambda: fmt2.writeIndexRows(two, b, n), lambda: fmt2.writeIndexMeta(two, b, n, [0] * 5),
                 lambda: fmt2.loadIndexRows(a, 0, 10), lambda: fmt2.loadIndex(a, sharded=True)):
        with pytest.raises(bbq.BbqError) as e:
            call()
        assert e.value.status == 9
    # without a communicator the collective entries are bbq_index_save / bbq_index_load
    assert fmt.commInfo()["world"] == 1
    fmt.saveIndex(whole, b, sharded=True)
    assert _same_files(a, b)
    l1, l2 = fmt.loadIndex(a), fmt.loadIndex(a, sharded=True)
    p1, c1 = l1.exportAll()
    p2, c2 = l2.exportAll()
    assert l2.size() == n and np.array_equal(p1, p2) and np.array_equal(c1.view(np.uint64), c2.view(np.uint64))
    qs = gaussian(5, dim, 4602)
    i1, s1 = fmt.searchBatch(qs, l1, 10)
    i2, s2 = fmt.searchBatch(qs, l2, 10, sharded=True)
    assert np.array_equal(i1, i2) and np.array_equal(s1.view(np.uint32), s2.view(np.uint32))


# ---- two GPUs: the collective entries, one process per GPU ----------------------------------------------------------
def _join(fmt, ids, rank, world):
    if rank == 0:
        cid = fmt.commUniqueId()
        for _ in range(world - 1):
            ids.put(cid)
    else:
        cid = ids.get(timeout=120)
    fmt.commInit(cid, rank, world)


def _worker_parity(rank, world, ids, out, tmp):
    import torch
    torch.cuda.set_device(rank)
    import bbq_b200
    n, dim, nq, k = 5001, 256, 9, 10
    rows, qs = gaussian(n, dim, 4701), gaussian(nq, dim, 4702)
    cen = np.zeros(dim, np.float32)
    fmt = _fmt(bbq_b200, "COSINE", device=rank)
    r0, r1 = bbq_b200.shard_bounds(n, world, rank)
    shard = fmt.quantizeVectors(rows[r0:r1], centroid=cen)["quantizedVectors"]
    fmt.setBase(shard, r0)
    _join(fmt, ids, rank, world)
    prefix = os.path.join(tmp, "sharded")
    fmt.saveIndex(shard, prefix, sharded=True)
    ok = True
    if rank == 0:                       # every rank has returned from the save: the files are complete
        whole = fmt.quantizeVectors(rows, centroid=cen)["quantizedVectors"]
        fmt.saveIndex(whole, os.path.join(tmp, "whole"))
        ok &= _same_files(prefix, os.path.join(tmp, "whole"))
    mine = fmt.loadIndex(prefix, sharded=True)
    ok &= mine.size() == r1 - r0
    gi, gs = fmt.searchBatch(qs, mine, k, sharded=True)
    fmt.commDestroy()
    full = O.quantize_vectors(rows, sim="COSINE", want_unpacked=False, centroid=cen)
    for qi in range(nq):
        wi, ws = O.search_nearest_neighbors(qs[qi], full, k, mode="canonical")
        ok &= gi[qi].tolist() == wi.tolist() and gs[qi].view(np.uint32).tolist() == ws.view(np.uint32).tolist()
    out.put((rank, (bool(ok), gi.tobytes() + gs.tobytes())))


def _worker_errors(rank, world, ids, out, tmp):
    import torch
    torch.cuda.set_device(rank)
    import bbq_b200
    n, dim = 4000, 64
    rows = gaussian(n, dim, 4801)
    cen = np.zeros(dim, np.float32)
    r0, r1 = bbq_b200.shard_bounds(n, world, rank)
    got = []
    for case in ("centroid", "gap", "corrupt"):
        fmt = _fmt(bbq_b200, device=rank)
        prefix = os.path.join(tmp, case)
        if case == "corrupt":
            if rank == 0:               # written and damaged (inside rank 1's rows) before any rank joins
                whole = fmt.quantizeVectors(rows, centroid=cen)["quantizedVectors"]
                fmt.saveIndex(whole, prefix)
                blob = bytearray(_read(prefix + ".veb"))
                blob[(n - 10) * 16 + 1] ^= 0x01
                with open(prefix + ".veb", "wb") as f:
                    f.write(blob)
            _join(fmt, ids, rank, world)
            call = lambda: fmt.loadIndex(prefix, sharded=True)
        else:
            c = cen + (1.0 if case == "centroid" and rank == 1 else 0.0)
            shard = fmt.quantizeVectors(rows[r0:r1], centroid=c)["quantizedVectors"]
            fmt.setBase(shard, r0 + (5 if case == "gap" and rank == 1 else 0))
            _join(fmt, ids, rank, world)
            call = lambda: fmt.saveIndex(shard, prefix, sharded=True)
        try:
            call()
            got.append((case, 0, ""))
        except bbq_b200.BbqError as e:
            got.append((case, e.status, str(e)))
        fmt.commDestroy()
    out.put((rank, got))


def _spawn(target, world, tmp):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    ctx = mp.get_context("spawn")
    ids, out = ctx.Queue(), ctx.Queue()
    procs = [ctx.Process(target=target, args=(r, world, ids, out, tmp)) for r in range(world)]
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


def test_sharded_save_and_load_on_two_gpus(tmp_path):
    got = _spawn(_worker_parity, 2, str(tmp_path))
    assert got[0][0] and got[1][0]
    assert got[0][1] == got[1][1], "the ranks returned different lists"


def test_a_failure_on_one_rank_fails_both_alike(tmp_path):
    got = _spawn(_worker_errors, 2, str(tmp_path))
    want = {"centroid": 10, "gap": 10, "corrupt": 12}
    for (case, s0, m0), (_, s1, m1) in zip(got[0], got[1]):
        assert s0 == s1 == want[case], (case, s0, s1)
        assert m0 == m1 and m0, (case, m0, m1)
    msgs = {case: m for case, _, m in got[0]}
    assert "centroid of rank 1" in msgs["centroid"]
    assert "held by no rank" in msgs["gap"]
    assert "checksum mismatch in section codes" in msgs["corrupt"]
