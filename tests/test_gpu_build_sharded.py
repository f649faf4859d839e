"""The reference centroid chained across row slices, and the index build across row shards.

On one GPU, shards are emulated as slices of one corpus: the running sum continued slice by slice
(bbq_centroid_accumulate / _device) and finished on the host (bbq_centroid_finish) equals, bit for bit, the centroid and
centroidDP of bbq_index_build over the whole corpus and the oracle's computeCentroid, for 2, 3 and 8 ragged slices (with
a 1-row and an empty one, edges off the 32768-row build chunk), host and device rows, every similarity and dims 100, 128
and 768; edge corpora (a first row of -0.0, cancelling rows, subnormals, unvalidated device rows holding Inf or NaN)
too.  reserve + append per slice with that centroid, plus setBase, gives the whole build's rows for indexBits 1 and 2,
and bbq_index_build_sharded without a communicator is bbq_index_build, errors included.  On two GPUs (skipped below
that): ragged shards and an empty rank, host and device rows, NULL and explicit centroid: every shard equals its slice of
the whole build, the sharded search equals the oracle, the sharded save equals a whole-index save, and every error gives
the same status, message and position on both ranks."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from tests.fixtures import gaussian

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bbq():
    import bbq_b200
    bbq_b200.build_library()
    return bbq_b200


def _fmt(bbq, sim="COSINE", index_bits=1, device=-1):
    return bbq.createBinaryQuantizationFormat(
        {"queryBits": 4, "indexBits": index_bits, "quantizer": {"similarityFunction": sim, "lambda": 0.1, "iters": 5}},
        device=device)


def _same(a, b):
    """bit-equal f32 arrays, any NaN equal to any NaN (the host finish keeps a payload the device may not)"""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    nan = np.isnan(a)
    return np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(np.uint32), b[~nan].view(np.uint32))


def _oracle_centroid(rows, sim):
    if sim == "COSINE":
        rows = np.stack([O.normalize_vector(r) for r in rows])
    return O.compute_centroid(rows)


def _chain(fmt, rows, bounds, device):
    """the running sum over the slices [bounds[i], bounds[i+1]) in order, then finished: the centroid of all rows"""
    import torch
    running = np.zeros(rows.shape[1], np.float32)
    d = torch.from_numpy(rows).cuda() if device else None
    for r0, r1 in zip(bounds[:-1], bounds[1:]):
        if device:
            fmt.accumulateCentroid(running, r0, d_rows_ptr=d[r0:].data_ptr() if r1 > r0 else 0, n=r1 - r0)
        else:
            fmt.accumulateCentroid(running, r0, rows=rows[r0:r1])
    return fmt.finishCentroid(running, rows.shape[0])


def _slice_shards(fmt, rows, bounds, cen):
    """each slice as a shard of its own: reserve + append with the given centroid, base set"""
    out = []
    for r0, r1 in zip(bounds[:-1], bounds[1:]):
        s = fmt.reserveIndex(max(r1 - r0, 1), rows.shape[1], cen)
        if r1 > r0:
            fmt.appendRows(s, rows=rows[r0:r1])
        fmt.setBase(s, r0)
        out.append(s)
    return out


def _same_rows(a, b):
    pa, ca = a
    pb, cb = b
    return np.array_equal(pa, pb) and np.array_equal(ca.view(np.uint64), cb.view(np.uint64))


SPLITS = {
    "two": lambda n: [0, 40001, n],
    "three": lambda n: [0, 32767, 32768, n],                                      # a 1-row slice across a chunk edge
    "eight": lambda n: [0, 5, 6, 30000, 30000, 50001, 65539, 69000, n],          # a 1-row and an empty slice
}
CORPORA = {("COSINE", 100): 100_003, ("EUCLIDEAN", 128): 85_001, ("MAXIMUM_INNER_PRODUCT", 768): 70_001}
_whole = {}


def _whole_build(bbq, sim, dim):
    if (sim, dim) not in _whole:
        n = CORPORA[sim, dim]
        rows = gaussian(n, dim, 5100 + dim)
        fmt = _fmt(bbq, sim)
        qv = fmt.quantizeVectors(rows)["quantizedVectors"]
        _whole[sim, dim] = (rows, fmt, qv, qv.exportAll(), _oracle_centroid(rows, sim))
    return _whole[sim, dim]


@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("split", sorted(SPLITS))
@pytest.mark.parametrize("sim,dim", sorted(CORPORA))
def test_chained_centroid_equals_whole_build(bbq, sim, dim, split, device):
    rows, fmt, whole, whole_rows, want = _whole_build(bbq, sim, dim)
    bounds = SPLITS[split](rows.shape[0])
    cen = _chain(fmt, rows, bounds, device)
    assert _same(cen, whole.getCentroid()) and _same(cen, want)
    shards = _slice_shards(fmt, rows, bounds, cen)
    for s, (r0, r1) in zip(shards, zip(bounds[:-1], bounds[1:])):
        assert s.getCentroidDP() == whole.getCentroidDP() and s.size() == r1 - r0
        if r1 > r0:
            assert _same_rows(s.exportAll(), (whole_rows[0][r0:r1], whole_rows[1][r0:r1]))


@pytest.mark.parametrize("sim", ["COSINE", "EUCLIDEAN", "MAXIMUM_INNER_PRODUCT"])
def test_slices_with_two_bit_codes(bbq, sim):
    n, dim = 40_003, 130
    rows = gaussian(n, dim, 5200)
    fmt = _fmt(bbq, sim, index_bits=2)
    whole = fmt.quantizeVectors(rows)["quantizedVectors"]
    p, c = whole.exportAll()
    bounds = [0, 1, 1, 32769, n]
    cen = _chain(fmt, rows, bounds, device=True)
    assert _same(cen, whole.getCentroid())
    for s, (r0, r1) in zip(_slice_shards(fmt, rows, bounds, cen), zip(bounds[:-1], bounds[1:])):
        if r1 > r0:
            assert _same_rows(s.exportAll(), (p[r0:r1], c[r0:r1]))


def _edge_rows(kind, n, dim):
    rows = gaussian(n, dim, 5300)
    if kind == "neg_zero":            # row 0 all -0.0, and one component -0.0 in every row: the sum stays -0.0
        rows[0] = -0.0
        rows[:, 3] = -0.0
    elif kind == "cancel":            # huge rows that cancel pairwise, around small ones
        rows[1::4] *= 1e30
        rows[2::4] = -rows[1::4][: rows[2::4].shape[0]]
    elif kind == "subnormal":
        rows *= np.float32(1e-41)
        rows[0, :5] = np.float32(1e-45)
    elif kind == "nonfinite":         # device rows are not validated
        rows[700, 4] = np.inf
        rows[900, 9] = -np.inf
        rows[1600, 2] = np.nan
    return rows


@pytest.mark.parametrize("sim", ["COSINE", "EUCLIDEAN", "MAXIMUM_INNER_PRODUCT"])
@pytest.mark.parametrize("kind", ["neg_zero", "cancel", "subnormal", "nonfinite"])
def test_edge_corpora(bbq, kind, sim):
    import torch
    n, dim = 3001, 64
    rows = _edge_rows(kind, n, dim)
    fmt = _fmt(bbq, sim)
    d = torch.from_numpy(rows).cuda()
    whole = fmt.quantizeVectorsDevice(d.data_ptr(), n, dim)["quantizedVectors"]
    want = _oracle_centroid(rows, sim)
    for bounds in ([0, 1, 1, 1500, n], [0, n]):      # a 1-row first slice: row 0 copied, the next slice added
        cen = _chain(fmt, rows, bounds, device=True)
        assert _same(cen, whole.getCentroid()) and _same(cen, want), bounds
        if kind != "nonfinite":
            assert _same(_chain(fmt, rows, bounds, device=False), cen)
    if kind == "neg_zero" and sim != "COSINE":      # (COSINE turns the zero row 0 into +0.0)
        assert np.float32(cen[3]).view(np.uint32) == 0x80000000
    if kind == "subnormal" and sim != "COSINE":
        assert np.any((cen != 0) & (np.abs(cen) < np.finfo(np.float32).tiny))


def test_build_sharded_without_communicator_is_build(bbq):
    import torch
    n, dim = 5003, 96
    rows = gaussian(n, dim, 5400)
    for sim in ("COSINE", "EUCLIDEAN"):
        fmt = _fmt(bbq, sim)
        assert fmt.commInfo()["world"] == 1
        plain = fmt.quantizeVectors(rows)["quantizedVectors"]
        d = torch.from_numpy(rows).cuda()
        for qv in (fmt.quantizeVectors(rows, sharded=True)["quantizedVectors"],
                   fmt.quantizeVectorsDevice(d.data_ptr(), n, dim, sharded=True)["quantizedVectors"],
                   fmt.quantizeVectors(rows, centroid=plain.getCentroid(), sharded=True)["quantizedVectors"]):
            assert _same(qv.getCentroid(), plain.getCentroid()) and qv.getCentroidDP() == plain.getCentroidDP()
            assert _same_rows(qv.exportAll(), plain.exportAll())
        bad = rows.copy()
        bad[17, 5] = np.inf
        for r in (bad, np.empty((0, dim), np.float32)):
            got = []
            for sharded in (False, True):
                with pytest.raises(bbq.BbqError) as e:
                    fmt.quantizeVectors(r, sharded=sharded)
                got.append((e.value.status, str(e.value)))
            assert got[0] == got[1], got
        assert got[0][0] == 3
    # host rows' validation errors name the vector in the whole corpus
    fmt = _fmt(bbq, "EUCLIDEAN")
    with pytest.raises(bbq.BbqError) as e:
        fmt.accumulateCentroid(np.zeros(dim, np.float32), 1000, rows=bad[10:20])
    assert e.value.status == 6 and str(e.value) == "向量 1007 位置 5 包含Infinity值"


# ---- two GPUs: the collective build, one process per GPU ----------------------------------------------------------
def _join(fmt, ids, rank, world):
    if rank == 0:
        cid = fmt.commUniqueId()
        for _ in range(world - 1):
            ids.put(cid)
    else:
        cid = ids.get(timeout=120)
    fmt.commInit(cid, rank, world)


def _read(p):
    with open(p, "rb") as f:
        return f.read()


def _worker_build(rank, world, ids, out, tmp):
    import torch
    torch.cuda.set_device(rank)
    import bbq_b200
    n, dim, nq, k = 50_003, 128, 6, 10
    rows, qs = gaussian(n, dim, 5500), gaussian(nq, dim, 5501)
    fmt = _fmt(bbq_b200, "COSINE", device=rank)
    whole = fmt.quantizeVectors(rows)["quantizedVectors"]
    wp, wc = whole.exportAll()
    full = O.quantize_vectors(rows, sim="COSINE", want_unpacked=False)
    explicit = gaussian(1, dim, 5502)[0]
    want_explicit = fmt.quantizeVectors(rows, centroid=explicit)["quantizedVectors"].exportAll()
    _join(fmt, ids, rank, world)
    d = torch.from_numpy(rows).cuda()
    ok, log = True, []
    for split in ([0, 30001, n], [0, 0, n], [0, n, n]):
        r0, r1 = split[rank], split[rank + 1]
        for device in (False, True):
            for given in (False, True):
                cen = explicit if given else None
                if device:
                    qv = fmt.quantizeVectorsDevice(d[r0:].data_ptr() if r1 > r0 else 0, r1 - r0, dim, centroid=cen,
                                                   sharded=True)["quantizedVectors"]
                else:
                    qv = fmt.quantizeVectors(rows[r0:r1], centroid=cen, sharded=True)["quantizedVectors"]
                wp_, wc_ = want_explicit if given else (wp, wc)
                c_ok = _same(qv.getCentroid(), explicit if given else whole.getCentroid())
                c_ok &= given or qv.getCentroidDP() == whole.getCentroidDP()
                r_ok = qv.size() == r1 - r0 and (r1 == r0 or _same_rows(qv.exportAll(), (wp_[r0:r1], wc_[r0:r1])))
                case_ok = bool(c_ok and r_ok)
                if not given and not device:
                    prefix = os.path.join(tmp, f"s{split[1]}")
                    fmt.saveIndex(qv, prefix, sharded=True)
                    if rank == 0:                # every rank has returned from the save: the files are complete
                        fmt.saveIndex(whole, os.path.join(tmp, "whole"))
                        case_ok &= _read(prefix + ".veb") == _read(os.path.join(tmp, "whole.veb"))
                        case_ok &= _read(prefix + ".vemb") == _read(os.path.join(tmp, "whole.vemb"))
                    if split[1] not in (0, n):
                        gi, gs = fmt.searchBatch(qs, qv, k, sharded=True)
                        for qi in range(nq):
                            oi, osc = O.search_nearest_neighbors(qs[qi], full, k, mode="canonical")
                            case_ok &= gi[qi].tolist() == oi.tolist() and \
                                gs[qi].view(np.uint32).tolist() == osc.view(np.uint32).tolist()
                log.append((split[1], device, given, case_ok))
                ok &= case_ok
    fmt.commDestroy()
    out.put((rank, (bool(ok), log)))


def _worker_errors(rank, world, ids, out, tmp):
    import torch
    torch.cuda.set_device(rank)
    import bbq_b200
    n, dim = 4000, 64
    rows = gaussian(n, dim, 5600)
    r0, r1 = bbq_b200.shard_bounds(n, world, rank)
    got = []
    for case in ("nan", "dims", "centroid", "empty"):
        fmt = _fmt(bbq_b200, "EUCLIDEAN", device=rank)
        _join(fmt, ids, rank, world)
        mine, cen = rows[r0:r1].copy(), None
        if case == "nan" and rank == 1:
            mine[33, 7] = np.nan
        if case == "dims" and rank == 1:
            mine = mine[:, :-1].copy()
        if case == "centroid":
            cen = np.full(dim, float(rank), np.float32)
        if case == "empty":
            mine = np.empty((0, dim), np.float32)
        try:
            fmt.quantizeVectors(mine, centroid=cen, sharded=True)
            got.append((case, 0, "", (-1, -1)))
        except bbq_b200.BbqError as e:
            import ctypes as C
            v, p = C.c_int64(), C.c_int64()
            bbq_b200._native.load().bbq_last_error_pos(C.byref(v), C.byref(p))
            got.append((case, e.status, str(e), (v.value, p.value)))
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
        got = dict(out.get(timeout=900) for _ in range(world))
        for p in procs:
            p.join(240)
            assert p.exitcode == 0, "a rank failed or hung"
    finally:
        for p in procs:      # never leave a rank spinning in a collective on the GPU behind a failed test
            if p.is_alive():
                p.kill()
    return got


def test_sharded_build_on_two_gpus(tmp_path):
    got = _spawn(_worker_build, 2, str(tmp_path))
    assert got[0][0] and got[1][0], (got[0][1], got[1][1])


def test_build_errors_agree_on_two_gpus(tmp_path):
    got = _spawn(_worker_errors, 2, str(tmp_path))
    want = {"nan": 5, "dims": 10, "centroid": 10, "empty": 3}
    for a, b in zip(got[0], got[1]):
        assert a == b, (a, b)
        assert a[1] == want[a[0]], a
    msgs = {case: (m, pos) for case, _, m, pos in got[0]}
    assert msgs["nan"] == ("向量 2033 位置 7 包含NaN值", (2033, 7))
    assert "rank 1 has dimension 63" in msgs["dims"][0]
    assert "centroid of rank 1" in msgs["centroid"][0]
    assert msgs["empty"][0] == "向量集合不能为空"
