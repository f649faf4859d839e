"""The TypeScript drop-in class (better-binary-quantization_b200/bindings/ts/binaryQuantizationFormat.gpu.ts + errors.ts)
EXECUTED — installed into the reference package exactly as INTEGRATION.md says, run by the TypeScript-subset interpreter
(tests/golden/from_ts/tsinterp.py; there is no Node in the image), with a stand-in for the N-API addon whose compute engine
is the CPU oracle (tests/ts_dropin/oracle_addon.py: same function names, argument order, result shapes and error codes as
bindings/napi/bbq_napi.c).  What this checks is the TypeScript layer itself, which nothing had ever run: that it loads in
place of the reference's file with `src/index.ts` unchanged, marshals arguments and results correctly, keeps every public
member, and is indistinguishable from the reference's class to a caller — same values bit for bit, same Error messages —
including to the reference's own vitest file.  Needs a checkout of the reference in BBQ_REFERENCE_DIR (skipped
without one)."""
import json
import os
import struct
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden", "from_ts"))
from tests.fixtures import edge_dataset, gaussian  # noqa: E402
from tests.golden_util import HAVE_REFERENCE, REFERENCE_DIR as REF  # noqa: E402

pytestmark = pytest.mark.skipif(not HAVE_REFERENCE, reason="needs a checkout of the reference project in BBQ_REFERENCE_DIR")

SIMS = ["EUCLIDEAN", "COSINE", "MAXIMUM_INNER_PRODUCT"]


def _packages():
    import tsinterp as T
    from tests.ts_dropin.oracle_addon import load_dropin_package
    con_ref, con_gpu = [], []
    ref = T.Interp(log=lambda *a: con_ref.append(a), stub_modules=["/src/wasm/index.ts"])
    ref_ex = ref.load(os.path.join(REF, "src", "index.ts"))
    gpu, gpu_ex, addon = load_dropin_package(REF, ROOT, con_gpu)
    return T, (ref, ref_ex, con_ref), (gpu, gpu_ex, con_gpu), addon


def _bits64(x):
    return struct.pack(">d", float(x))


def _config(sim, qb):
    return {"queryBits": float(qb), "indexBits": 1.0, "quantizer": {"similarityFunction": sim, "lambda": 0.1, "iters": 5.0}}


@pytest.mark.parametrize("sim", SIMS)
@pytest.mark.parametrize("qb", [4, 1])
def test_dropin_class_is_indistinguishable_from_the_reference_class(sim, qb):
    T, (ref, ref_ex, con_ref), (gpu, gpu_ex, con_gpu), addon = _packages()
    n, dim, k = 48, 40, 6
    base, queries = edge_dataset(n, dim, 3, 9100 + qb)          # zero / duplicated / constant rows, zero query included
    out = {}
    for name, (I, ex) in (("ref", (ref, ref_ex)), ("gpu", (gpu, gpu_ex))):
        fmt = I.call(ex["createBinaryQuantizationFormat"], args=[_config(sim, qb)])      # the UNCHANGED src/index.ts factory
        rows = [I.float32(r.tolist()) for r in base]
        res = I.call(I.get(fmt, "quantizeVectors"), fmt, [rows])
        qv = res["quantizedVectors"]
        assert res["queryQuantizer"] is I.call(I.get(fmt, "getQuantizer"), fmt, [])     # :261 `this.quantizer`
        o = {"size": I.call(I.get(qv, "size"), qv, []), "dim": I.call(I.get(qv, "dimension"), qv, []),
             "centroid": list(I.call(I.get(qv, "getCentroid"), qv, []).a), "cdp": I.call(I.get(qv, "getCentroidDP"), qv, []),
             "corr": [], "packed": [], "unpacked": [], "search": [], "once": [], "config": I.call(I.get(fmt, "getConfig"), fmt, [])}
        for i in range(n):
            c = I.call(I.get(qv, "getCorrectiveTerms"), qv, [float(i)])
            o["corr"].append([_bits64(c[f]) for f in ("lowerInterval", "upperInterval", "additionalCorrection", "quantizedComponentSum")])
            o["packed"].append(list(I.call(I.get(qv, "vectorValue"), qv, [float(i)]).a))
            o["unpacked"].append(list(I.call(I.get(qv, "getUnpackedVector"), qv, [float(i)]).a))
        for q in queries:
            qa = I.float32(q.tolist())
            o["search"].append([(r["index"], r["score"]) for r in I.call(I.get(fmt, "searchNearestNeighbors"), fmt, [qa, qv, float(k)])])
            assert I.call(I.get(fmt, "searchNearestNeighbors"), fmt, [qa, qv, 0.0]) == []
            assert len(I.call(I.get(fmt, "searchNearestNeighbors"), fmt, [qa, qv, 2.5])) == 3                 # fractional k -> ceil(k)
            assert len(I.call(I.get(fmt, "searchNearestNeighbors"), fmt, [qa, qv, float(n + 9)])) == n        # k > n -> n results
            once = I.call(I.get(fmt, "quantizeQueryVector"), fmt, [qa, I.call(I.get(qv, "getCentroid"), qv, [])])
            qc = once["queryCorrections"]
            o["once"].append((list(once["quantizedQuery"].a), [_bits64(qc[f]) for f in ("lowerInterval", "upperInterval",
                                                                                        "additionalCorrection", "quantizedComponentSum")]))
        o["range"] = []
        for member, bad_ord in (("vectorValue", float(n)), ("vectorValue", -1.0), ("getCorrectiveTerms", float(n)), ("getUnpackedVector", float(n + 51))):
            with pytest.raises(T.JSThrow) as e:
                I.call(I.get(qv, member), qv, [bad_ord])
            o["range"].append(str(e.value))
        o["cdp_q"] = I.call(I.get(qv, "getCentroidDP"), qv, [I.float32(queries[0].tolist())])
        acc = I.call(I.get(fmt, "computeQuantizationAccuracy"), fmt, [rows[:3], [I.float32(q.tolist()) for q in queries]])
        o["acc"] = [_bits64(acc[f]) for f in ("meanError", "maxError", "minError", "stdError", "correlation")]
        # serializeVectorData -> deserializeVectorData.  Executed, the REFERENCE's serializeVectorData throws on any real
        # index: it runs packAsBinary over rows that are already packed (:499-500), and packAsBinary rejects bytes > 1.
        # The drop-in serialises the packed rows as they are, and the re-created index answers like the original.
        if name == "ref":
            with pytest.raises(T.JSThrow) as e:
                I.call(I.get(fmt, "serializeVectorData"), fmt, [rows])
            assert "1位量化值必须为0或1" in str(e.value)
            o["roundtrip"] = o["search"][0]
        else:
            ser = I.call(I.get(fmt, "serializeVectorData"), fmt, [rows])
            assert ser["metadata"]["vectorCount"] == float(n) and ser["metadata"]["dimensions"] == float(dim) and len(ser["vectorData"]) == n
            assert ser["metadata"]["centroidSquareMagnitude"] == o["cdp"]
            back = I.call(I.get(fmt, "deserializeVectorData"), fmt, [ser["vectorData"], ser["metadata"]])
            o["roundtrip"] = [(r["index"], r["score"]) for r in
                              I.call(I.get(fmt, "searchNearestNeighbors"), fmt, [I.float32(queries[0].tolist()), back, float(k)])]
        for member in ("getQuantizer", "getScorer"):                   # the helper objects src/index.ts hands out
            assert isinstance(I.call(I.get(fmt, member), fmt, []), T.JSObj)
        out[name] = o
    r, g = out["ref"], out["gpu"]
    for key in ("size", "dim", "centroid", "cdp", "cdp_q", "corr", "packed", "unpacked", "once", "acc", "range"):
        assert r[key] == g[key], key
    assert r["config"]["queryBits"] == g["config"]["queryBits"] and r["config"]["quantizer"] == g["config"]["quantizer"]
    for a, b in zip(r["search"] + [r["roundtrip"]], g["search"] + [g["roundtrip"]]):
        assert [s for _, s in a] == [s for _, s in b]              # the same scores, rank by rank
        scores = [s for _, s in a]
        if len(set(scores)) == len(scores):                        # no exact ties: the same list
            assert [i for i, _ in a] == [i for i, _ in b]
    assert not con_ref and not con_gpu
    assert {"create", "build", "info", "search", "rows", "quantizeQuery", "accuracy", "fromQuantized"} <= set(addon.calls)


def test_dropin_class_raises_the_reference_messages():
    """Every case of errors.behaviour.json (what the executed reference throws): the drop-in throws the same message —
    through its own argument checks, or the addon's status code mapped back by errors.ts."""
    T, _, (I, ex, _), addon = _packages()
    d = json.load(open(os.path.join(ROOT, "tests", "golden", "from_ts", "errors.behaviour.json")))
    rows, qs = gaussian(d["n"], d["dim"], d["rows_seed"]), gaussian(6, d["dim"], d["queries_seed"])
    made = {}

    def setup(sim):
        if sim not in made:
            fmt = I.call(ex["createBinaryQuantizationFormat"], args=[_config(sim, 4)])
            made[sim] = (fmt, I.call(I.get(fmt, "quantizeVectors"), fmt, [[I.float32(r.tolist()) for r in rows[:40]]])["quantizedVectors"])
        return made[sim]

    def run(c):
        fmt, qv = setup(c["sim"])
        search, quantize = I.get(fmt, "searchNearestNeighbors"), I.get(fmt, "quantizeVectors")
        label = c["label"]
        if c["what"] == "search" and "edits" in c:
            q = qs[2].copy()
            for pos, val in c["edits"].items():
                q[int(pos)] = float(val)
            return I.call(search, fmt, [I.float32(q.tolist()), qv, 5.0])
        if c["what"] == "build" and "row" in c:
            b = rows[:5].copy()
            b[c["row"], c["pos"]] = float(c["value"])
            return I.call(quantize, fmt, [[I.float32(x.tolist()) for x in b]])
        q0 = I.float32(qs[0].tolist())
        if label == "k = -1":
            return I.call(search, fmt, [q0, qv, -1.0])
        if label.startswith("k = 0"):
            return I.call(search, fmt, [q0, qv, 0.0])
        if label == "dimension mismatch":
            return I.call(search, fmt, [I.float32(qs[0][:10].tolist()), qv, 3.0])
        if label == "null query":
            return I.call(search, fmt, [None, qv, 3.0])
        if label == "null targets":
            return I.call(search, fmt, [q0, None, 3.0])
        if label == "empty vector set":
            return I.call(quantize, fmt, [[]])
        if label.startswith("ragged rows"):
            return I.call(quantize, fmt, [[I.float32(rows[0].tolist()), I.float32(rows[1][:10].tolist())]])
        if label == "queryBits = 9":
            return I.call(ex["createBinaryQuantizationFormat"], args=[{"queryBits": 9.0, "quantizer": {"similarityFunction": "COSINE"}}])
        if label == "indexBits = 0":
            return I.call(ex["createBinaryQuantizationFormat"], args=[{"indexBits": 0.0, "quantizer": {"similarityFunction": "COSINE"}}])
        raise AssertionError(label)

    for c in d["cases"]:
        if c["message"] is None:
            assert run(c) == []
            continue
        with pytest.raises(T.JSThrow) as e:
            run(c)
        v = e.value.value
        assert isinstance(v, T.JSObj) and T.to_str(I.get(v, "message")) == c["message"], (c["sim"], c["label"], str(e.value))


def test_reference_own_recall_tests_pass_on_the_dropin_class():
    """tests/recall.test.ts of the reference — which imports '../src/binaryQuantizationFormat' — run against the package
    with the drop-in installed: all eight tests pass, and the searches went through the addon."""
    import vitest_shim as V
    from tests.ts_dropin.oracle_addon import OracleAddon, dropin_interp_kwargs
    addon = OracleAddon()
    passed, failed, assertions, console = V.run_test_file(os.path.join(REF, "tests", "recall.test.ts"),
                                                          **dropin_interp_kwargs(REF, ROOT, addon))
    assert not failed, failed[:3]
    assert len(passed) == 8 and assertions > 100
    assert addon.calls.count("search") > 50 and "build" in addon.calls


def test_dropin_additive_members_execute():
    """searchBatch (one call for several queries) and attachOriginalVectors + searchOversampled (the device form of
    src/topKSelector.ts) — members the reference does not have: row i of searchBatch equals searchNearestNeighbors of
    query i, and the oversampled search returns what the reference's getOversampledTopKWithSort computes with the
    reference's own class (true cosine scores bit for bit)."""
    T, (ref, ref_ex, _), (gpu, gpu_ex, _), addon = _packages()
    n, dim, k, factor = 60, 32, 5, 3
    base, queries = gaussian(n, dim, 9300), gaussian(3, dim, 9301)
    fmt = gpu.call(gpu_ex["createBinaryQuantizationFormat"], args=[_config("COSINE", 4)])
    rows = [gpu.float32(r.tolist()) for r in base]
    qv = gpu.call(gpu.get(fmt, "quantizeVectors"), fmt, [rows])["quantizedVectors"]
    qs = [gpu.float32(q.tolist()) for q in queries]
    batch = gpu.call(gpu.get(fmt, "searchBatch"), fmt, [qs, qv, float(k)])
    assert len(batch) == 3
    for i, q in enumerate(qs):
        single = gpu.call(gpu.get(fmt, "searchNearestNeighbors"), fmt, [q, qv, float(k)])
        assert [(r["index"], r["score"]) for r in batch[i]] == [(r["index"], r["score"]) for r in single]
    gpu.call(gpu.get(fmt, "attachOriginalVectors"), fmt, [qv, rows])
    over = gpu.call(gpu.get(fmt, "searchOversampled"), fmt, [qs[0], qv, float(k), float(factor)])
    # the reference's selector over the reference's class
    sel = ref.load(os.path.join(REF, "src", "topKSelector.ts"))
    rfmt = ref.call(ref_ex["createBinaryQuantizationFormat"], args=[_config("COSINE", 4)])
    rrows = [ref.float32(r.tolist()) for r in base]
    rqv = ref.call(ref.get(rfmt, "quantizeVectors"), rfmt, [rrows])["quantizedVectors"]
    want = ref.call(sel["getOversampledTopKWithSort"], args=[ref.float32(queries[0].tolist()), rqv, rrows, float(k), float(factor), rfmt])
    assert [c["index"] for c in over] == [c["index"] for c in want]
    assert [_bits64(c["trueScore"]) for c in over] == [_bits64(c["trueScore"]) for c in want]
    assert [c["quantizedScore"] for c in over] == [c["quantizedScore"] for c in want]
    assert {"attachRows", "searchRerank"} <= set(addon.calls)
