"""Oracle vs fixtures generated FROM THE REFERENCE'S OWN SOURCE TEXT.

`tests/golden/from_ts/*.ts.json` were produced by executing the unmodified `src/index.ts` of the reference (and every
module it imports) with `tests/golden/from_ts/tsinterp.py` — a TypeScript-subset interpreter written for this purpose,
because no JavaScript runtime exists in the image or on the GPU box (profiles/r02_js_runtime_probe.txt) — through
`tests/golden/from_ts/make_golden_with_interp.py`.  Each fixture records the SHA-256 of the reference files that produced
it.  The oracle must reproduce them bit for bit: centroid (f32), every row's packed code and correctives (f64 bit
patterns), every row's f32 score, the heap-ordered top-k lists, `quantizeQueryVector` called directly, the statistics
of `computeQuantizationAccuracy`, and `getOversampledTopKWithHeap`.

`make_golden_from_ts.mjs` (the Node version of the generator) writes the same schema minus the extra members; a
fixture without them is accepted too."""
import glob
import json
import os
import struct

import numpy as np
import pytest

from oracle import oracle as O
from tests.fixtures import gaussian
from tests.golden.make_golden import CASES, case_inputs
from tests.golden.from_ts import live_cases as L
from tests.golden_util import HAVE_REFERENCE, REFERENCE_DIR

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "from_ts")
FIXTURES = sorted(glob.glob(os.path.join(HERE, "*.ts.json")))


def _f64_from_hex(rows):
    return np.array([[struct.unpack(">d", bytes.fromhex(h))[0] for h in row] for row in rows], np.float64)


def _u64(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def test_fixtures_from_the_reference_source_exist():
    assert len(FIXTURES) >= 11, "run tests/golden/from_ts/make_golden_with_interp.py (needs the reference)"
    sims = {json.load(open(p))["sim"] for p in FIXTURES}
    assert sims == {"EUCLIDEAN", "COSINE", "MAXIMUM_INNER_PRODUCT"}


@pytest.mark.parametrize("path", FIXTURES, ids=[os.path.basename(p)[:-len(".ts.json")] for p in FIXTURES])
def test_oracle_equals_the_typescript_reference(path):
    d = json.load(open(path))
    name = os.path.basename(path)[:-len(".ts.json")]
    n, dim, sim, qb, k, nq, lam, iters, data = CASES[name]
    assert (d["n"], d["dim"], d["sim"], d["queryBits"], d["k"]) == (n, dim, sim, qb, k)
    assert not d.get("console"), "the reference logged something (a fallback ran?)"
    base, queries = case_inputs(name)
    idx = O.quantize_vectors(base, sim=sim, index_bits=1, lam=lam, iters=iters)
    # quantizeVectors: centroid, correctives, codes
    assert idx.centroid.view(np.uint32).tolist() == d["centroid_bits"]
    assert np.array_equal(_u64(idx.corr), _u64(_f64_from_hex(d["corrections_bits"])))
    assert int(idx.packed.astype(np.uint64).sum()) == d["packed_sum"]
    if "packed_head" in d:
        assert idx.packed[:16].tolist() == d["packed_head"]
    for q, ref in zip(queries, d["queries"]):
        # searchNearestNeighbors: every row's f32 score and the heap-ordered list
        _, _, alls, _ = O.search_nearest_neighbors(q, idx, k, query_bits=qb, lam=lam, iters=iters, mode="heap", want_all=True)
        assert alls.view(np.uint32).tolist() == ref["all_score_bits"]
        hi, hs = O.search_nearest_neighbors(q, idx, k, query_bits=qb, lam=lam, iters=iters, mode="heap")
        assert hi.tolist() == ref["top_index"] and hs.view(np.uint32).tolist() == ref["top_score_bits"]
        # the canonical rule (score desc, id asc) returns the same SET whenever no exact tie straddles the k-th place
        ci, cs = O.search_nearest_neighbors(q, idx, k, query_bits=qb, lam=lam, iters=iters, mode="canonical")
        if len(alls) > k and np.sort(alls)[::-1][k - 1] != np.sort(alls)[::-1][k]:
            assert sorted(ci.tolist()) == sorted(ref["top_index"])
        if "k_beyond_n" in ref:               # k > vectorCount: min(k, n) results, the whole index in heap order
            bi, bs = O.search_nearest_neighbors(q, idx, ref["k_beyond_n"]["k"], query_bits=qb, lam=lam, iters=iters, mode="heap")
            assert bi.tolist() == ref["k_beyond_n"]["index"] and bs.view(np.uint32).tolist() == ref["k_beyond_n"]["score_bits"]
        if "quantize_query_once" in ref:      # quantizeQueryVector(query, centroid) as a direct member call
            codes, corr = O.quantize_query_vector_once(q, idx.centroid, sim, qb, lam, iters)
            assert codes.tolist() == ref["quantize_query_once"]["codes"]
            assert np.array_equal(_u64(corr), _u64(_f64_from_hex([ref["quantize_query_once"]["corrections_bits"]])[0]))
        if "oversampled_heap" in ref:         # getOversampledTopKWithHeap
            ov = ref["oversampled_heap"]
            oi, oq, ot = O.oversampled_topk(q, base, idx, k, ov["factor"], query_bits=qb, lam=lam, iters=iters, mode="heap")
            assert oi.tolist() == ov["index"] and oq.view(np.uint32).tolist() == ov["quantized_score_bits"]
            assert np.array_equal(_u64(ot), _u64(_f64_from_hex([ov["true_score_bits"]])[0]))
    if "accuracy" in d:                        # computeQuantizationAccuracy(rows[:nq], queries)
        m = d["accuracy"]["rows"]
        stats = O.compute_quantization_accuracy(base[:m], queries, sim, qb, lam, iters)
        for f in ("meanError", "maxError", "minError", "stdError", "correlation"):
            want = struct.unpack(">d", bytes.fromhex(d["accuracy"][f]))[0]
            assert np.float64(stats[f]).view(np.uint64) == np.float64(want).view(np.uint64), f


def _oracle_equals_stored(cases, stored):
    """The oracle against the reference's stored answers for `cases` (live_cases.py): correctives (f64 bit patterns), packed
    codes, the heap-ordered top-k list of every query and its f32 scores."""
    for name, sim, qb, lam, iters, k, base, queries in cases:
        idx = O.quantize_vectors(base, sim=sim, index_bits=1, lam=lam, iters=iters)
        res = [O.search_nearest_neighbors(q, idx, k, query_bits=qb, lam=lam, iters=iters, mode="heap") for q in queries]
        assert L.encode(idx.corr, idx.packed, [(i.tolist(), s) for i, s in res]) == stored[name], name


def _reference_equals_stored(cases, stored):
    """With a reference checkout: the reference source, interpreted now, gives the stored answers (guards them, and the
    interpreter, against going stale)."""
    if HAVE_REFERENCE:
        live = L.run_reference(REFERENCE_DIR, cases)
        for name, *_ in cases:
            assert live[name] == stored[name], name


@pytest.mark.parametrize("sim,qb,n,dim", [("COSINE", 4, 40, 24), ("EUCLIDEAN", 1, 30, 20), ("MAXIMUM_INNER_PRODUCT", 4, 36, 36)])
def test_reference_source_interpreted_live_equals_oracle(sim, qb, n, dim):
    """A tiny seeded case, two queries: the oracle gives the reference's answers (stored in live_cases.json; run through
    the reference source again when BBQ_REFERENCE_DIR names a checkout)."""
    cases = [c for c in L.fixed_cases() if c[0] == f"fixed_{sim}_{qb}_{n}x{dim}"]
    assert len(cases) == 1
    stored = L.load_stored()
    _oracle_equals_stored(cases, stored)
    _reference_equals_stored(cases, stored)


class _OracleBackedFormat:
    """The host interface's shape (quantizeVectors / searchBatch / debugScores / exportAll), answered by the oracle in
    CANONICAL order — a stand-in for the GPU format, so that the GPU-side checker of the reference fixtures
    (tests/test_zz_gpu_vs_reference_fixtures.py:check_against_fixture) is itself exercised on the CPU."""

    def __init__(self, sim, qb, lam, iters):
        self.sim, self.qb, self.lam, self.iters = sim, qb, lam, iters

    def quantizeVectors(self, base):
        idx = O.quantize_vectors(base, sim=self.sim, index_bits=1, lam=self.lam, iters=self.iters)

        class QV:
            def getCentroid(self_inner):
                return idx.centroid

            def exportAll(self_inner):
                return idx.packed, idx.corr
        qv = QV()
        qv.idx = idx
        return {"quantizedVectors": qv}

    def searchBatch(self, queries, qv, k):
        out = [O.search_nearest_neighbors(q, qv.idx, k, query_bits=self.qb, lam=self.lam, iters=self.iters, mode="canonical")
               for q in queries]
        return np.stack([o[0] for o in out]), np.stack([o[1] for o in out])

    def debugScores(self, q, qv):
        return O.search_nearest_neighbors(q, qv.idx, 1, query_bits=self.qb, lam=self.lam, iters=self.iters, mode="canonical",
                                          want_all=True)[2]


@pytest.mark.parametrize("path", FIXTURES, ids=[os.path.basename(p)[:-len(".ts.json")] for p in FIXTURES])
def test_gpu_side_checker_dry_run_with_the_oracle(path):
    from tests.test_zz_gpu_vs_reference_fixtures import check_against_fixture
    d = json.load(open(path))
    name = os.path.basename(path)[:-len(".ts.json")]
    n, dim, sim, qb, k, nq, lam, iters, data = CASES[name]
    check_against_fixture(_OracleBackedFormat(sim, qb, lam, iters), d, name)


def test_index_bits_2_build_equals_the_reference_and_its_search_behaviour_is_recorded():
    """indexBits = 2 (BASELINE configs[4] is queryBits = 8 / indexBits = 2).  Executed, the reference BUILDS such an index
    (2-bit codes, one per byte, + correctives) — the oracle reproduces that bit for bit — but cannot search it: the batch
    path fails, the per-vector fallback throws for queryBits = 8 (the recorded message) and, for queryBits = 4, scores
    with a formula that ignores the number of levels.  This repository's search over 2-bit indexes is therefore an
    EXTENSION (SURVEY §8c's generalisation, oracle/bbq_oracle.cpp:score_ext), and deliberately not that fallback."""
    d = json.load(open(os.path.join(HERE, "index_bits_2.behaviour.json")))
    base, queries = gaussian(d["n"], d["dim"], d["seed_base"]), gaussian(2, d["dim"], d["seed_queries"])
    for sim, ref in d["index_build"].items():
        idx = O.quantize_vectors(base, sim=sim, index_bits=2, lam=d["lambda"], iters=d["iters"])
        assert idx.centroid.view(np.uint32).tolist() == ref["centroid_bits"]
        assert np.array_equal(_u64(idx.corr), _u64(_f64_from_hex(ref["corrections_bits"])))
        assert idx.unpacked.tolist() == ref["codes"]
    for key, obs in d["search"].items():
        assert any("批量计算失败" in line for line in obs["console"])           # the batch path failed in every case
        if key.endswith("queryBits=8"):
            assert obs["threw"] == "Error: 不支持的查询位数: 8，只支持1位和4位"
        else:
            assert obs["threw"] is None
            sim = key.split()[0]
            idx = O.quantize_vectors(base, sim=sim, index_bits=2, lam=d["lambda"], iters=d["iters"])
            _, _, ext, _ = O.search_nearest_neighbors(queries[0], idx, 5, query_bits=4, mode="heap", want_all=True)
            assert ext.view(np.uint32).tolist() != obs["all_score_bits_of_the_fallback"]   # the extension is NOT the fallback


def test_host_messages_equal_the_executed_reference():
    """errors.behaviour.json holds the messages the reference throws (observed by executing it).  The parts of the host
    interface that need no GPU — the message templates the C-ABI status codes are mapped to, and the checks made in
    Python before any call — produce exactly those strings.  (The GPU-side half, which status and position the library
    reports for NaN / Infinity under each similarity function, is tests/test_zz_gpu_vs_reference_fixtures.py.)"""
    import importlib
    import bbq_b200  # noqa: F401  (registers the package under its importable name)
    fm = importlib.import_module("better_binary_quantization_b200.host.format")
    d = json.load(open(os.path.join(HERE, "errors.behaviour.json")))
    by = {(c["sim"], c["label"]): c["message"] for c in d["cases"]}
    assert fm._message(5, 3, 9, "build") == by[("EUCLIDEAN", "build NaN row 3 @9")]
    assert fm._message(6, 2, 4, "build") == by[("EUCLIDEAN", "build Infinity row 2 @4")]
    assert fm._message(5, 3, 0, "build") == by[("COSINE", "build NaN row 3 @9")]          # normalised first: NaN everywhere
    assert fm._message(5, 2, 4, "build") == by[("COSINE", "build Infinity row 2 @4")]     # Infinity / Infinity = NaN, in place
    assert fm._message(6, -1, 7, "search") == by[("EUCLIDEAN", "query NaN@30 + Infinity@7")]
    assert fm._message(6, -1, 12, "search") == by[("MAXIMUM_INNER_PRODUCT", "query -Infinity@12")]
    assert fm._message(5, -1, 5, "search") == by[("EUCLIDEAN", "query NaN@5")]
    assert fm._message(5, -1, 0, "search") == by[("COSINE", "query -Infinity@12")]
    assert fm._message(7, -1, -1, "search") == by[("COSINE", "k = -1")]
    assert fm._message(3, -1, -1, "build") == by[("COSINE", "empty vector set")]
    assert fm._message(4, -1, -1, "search") == by[("COSINE", "dimension mismatch")]
    assert fm._message(1, -1, -1, "") == by[("COSINE", "queryBits = 9")] and fm._message(2, -1, -1, "") == by[("COSINE", "indexBits = 0")]
    with pytest.raises(fm.BbqError) as e:
        fm._as_matrix([np.zeros(64, np.float32), np.zeros(10, np.float32)])
    assert str(e.value) == by[("COSINE", "ragged rows (row 1 has 10 of 64 dims)")]


def test_fuzz_reference_source_interpreted_live_equals_oracle():
    """150 random small configurations (live_cases.fuzz_cases: every similarity function, query bits 1..8, dims 1..70,
    1..40 rows, lambda 0..1, 0..20 iterations, scales 1e-3..1e3, duplicated and all-zero rows, signed zeros, integers,
    values near the f32 limit): correctives (f64 bit patterns), packed codes, the heap-ordered top-k list and its f32
    scores of the oracle are the reference's in every case (stored in live_cases.json; run through the reference source
    again when BBQ_REFERENCE_DIR names a checkout).  This is the comparison that found the signed-zero rule of
    Math.min / Math.max."""
    cases = L.fuzz_cases()
    assert len(cases) == 150
    stored = L.load_stored()
    _oracle_equals_stored(cases, stored)
    _reference_equals_stored(cases, stored)
