"""Golden fixtures FROM THE REFERENCE'S OWN SOURCE TEXT.

No JavaScript / TypeScript runtime exists in this image or on the GPU box (profiles/r02_js_runtime_probe.txt), so
`make_golden_from_ts.mjs` (which needs Node) has never run.  This script does the same job with `tsinterp.py`, a
TypeScript-subset interpreter written for exactly this purpose: it loads the UNMODIFIED `<reference>/src/index.ts`
(every module it imports; only the async WASM bridge `src/wasm/index.ts` is loaded as an empty module — it is outside
the path), calls the reference's public API on the seeded inputs of `tests/golden/make_golden.py`, and writes
`<case>.ts.json` in the schema of the .mjs generator plus a few more members of the class:

  createBinaryQuantizationFormat(config)                       src/index.ts
  format.quantizeVectors(base)                                 src/binaryQuantizationFormat.ts:165-263
      -> centroid, every row's packed code + four corrective terms
  format.searchNearestNeighbors(q, qv, k) and (q, qv, n)       :308-412  -> top-k list, every row's f32 score
  format.quantizeQueryVector(q, centroid)                      :271-299  -> codes + correctives (ONE normalisation)
  format.computeQuantizationAccuracy(rows[:nq], queries)       :420-475  -> the five statistics
  getOversampledTopKWithHeap(q, qv, base, k, 3, format)        src/topKSelector.ts:29-78

Nothing of the reference is copied into the repository: the sources are read where they lie, the fixture records their
SHA-256 so that it is clear which text produced it.  `tests/test_golden_from_ts.py` compares the oracle with the
fixtures bit for bit; `tests/test_tsinterp.py` tests the interpreter itself.

    python tests/golden/from_ts/make_golden_with_interp.py [--reference <reference checkout>] [case ...]
"""
import argparse
import hashlib
import json
import os
import struct
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import tsinterp as T  # noqa: E402
from tests.golden.make_golden import CASES, case_inputs  # noqa: E402

OVERSAMPLE = 3


def f64bits(x):
    return struct.pack(">d", float(x)).hex()


def f32bits(x):
    return struct.unpack("<I", struct.pack("<f", float(x)))[0]


def load_reference(ref_root, console):
    interp = T.Interp(log=lambda *a: console.append(" ".join(map(str, a))), stub_modules=["/src/wasm/index.ts"])
    index = interp.load(os.path.join(ref_root, "src", "index.ts"))
    selector = interp.load(os.path.join(ref_root, "src", "topKSelector.ts"))
    files = {}
    for path in sorted(interp.modules):
        if path not in interp.stubbed:
            files[os.path.relpath(path, ref_root)] = hashlib.sha256(open(path, "rb").read()).hexdigest()
    return interp, index, selector, files


def run_case(name, ref_root):
    n, dim, sim, qb, k, nq, lam, iters, data = CASES[name]
    base, queries = case_inputs(name)
    console = []
    I, ex, sel, files = load_reference(ref_root, console)
    t0 = time.time()
    fmt = I.call(ex["createBinaryQuantizationFormat"], args=[
        {"queryBits": float(qb), "indexBits": 1.0, "quantizer": {"similarityFunction": sim, "lambda": lam, "iters": float(iters)}}])
    rows = [I.float32(r.tolist()) for r in base]
    qv = I.call(I.get(fmt, "quantizeVectors"), fmt, [rows])["quantizedVectors"]
    centroid = I.call(I.get(qv, "getCentroid"), qv, [])
    out = {"n": n, "dim": dim, "nq": nq, "k": k, "queryBits": qb, "sim": sim, "lambda": lam, "iters": iters,
           "engine": "tests/golden/from_ts/tsinterp.py (Python interpreter of the TypeScript subset) executing the unmodified "
                     "reference sources listed in reference_sha256; src/wasm/index.ts loaded as an empty module",
           "reference_sha256": files,
           "centroid_bits": [f32bits(x) for x in centroid.a], "corrections_bits": [], "packed_sum": 0, "packed_head": [],
           "queries": []}
    for i in range(n):
        c = I.call(I.get(qv, "getCorrectiveTerms"), qv, [float(i)])
        out["corrections_bits"].append([f64bits(c[f]) for f in ("lowerInterval", "upperInterval", "additionalCorrection",
                                                                "quantizedComponentSum")])
        packed = I.call(I.get(qv, "vectorValue"), qv, [float(i)]).a
        out["packed_sum"] += int(sum(packed))
        if i < 16:
            out["packed_head"].append(list(packed))
    t_build = time.time() - t0
    for q in queries:
        qa = I.float32(q.tolist())
        res = I.call(I.get(fmt, "searchNearestNeighbors"), fmt, [qa, qv, float(k)])
        every = I.call(I.get(fmt, "searchNearestNeighbors"), fmt, [qa, qv, float(n)])     # every row's f32 score, via k = n
        by_index = [None] * n
        for r in every:
            by_index[int(r["index"])] = f32bits(r["score"])
        beyond = I.call(I.get(fmt, "searchNearestNeighbors"), fmt, [qa, qv, float(n + 5)]) if n <= 200 else None   # k > n
        once = I.call(I.get(fmt, "quantizeQueryVector"), fmt, [qa, centroid])
        qc = once["queryCorrections"]
        over = I.call(sel["getOversampledTopKWithHeap"], args=[qa, qv, rows, float(k), float(OVERSAMPLE), fmt])
        out["queries"].append({
            "top_index": [int(r["index"]) for r in res], "top_score_bits": [f32bits(r["score"]) for r in res],
            "all_score_bits": by_index,
            **({"k_beyond_n": {"k": n + 5, "index": [int(r["index"]) for r in beyond],
                               "score_bits": [f32bits(r["score"]) for r in beyond]}} if beyond is not None else {}),
            "quantize_query_once": {"codes": [int(x) for x in once["quantizedQuery"].a],
                                    "corrections_bits": [f64bits(qc[f]) for f in ("lowerInterval", "upperInterval", "additionalCorrection",
                                                                                  "quantizedComponentSum")]},
            "oversampled_heap": {"factor": OVERSAMPLE, "index": [int(c["index"]) for c in over],
                                 "quantized_score_bits": [f32bits(c["quantizedScore"]) for c in over],
                                 "true_score_bits": [f64bits(c["trueScore"]) for c in over]}})
    if qb in (1, 4):     # (the single-vector scorer behind this member knows 1- and 4-bit queries only: it throws otherwise)
        m = min(nq, n)   # the member wants as many original vectors as queries (it re-quantises them): the first nq rows
        acc = I.call(I.get(fmt, "computeQuantizationAccuracy"), fmt, [rows[:m], [I.float32(q.tolist()) for q in queries]])
        out["accuracy"] = {"rows": m, **{f: f64bits(acc[f]) for f in ("meanError", "maxError", "minError", "stdError", "correlation")}}
    out["console"] = console          # the reference logs nothing on this path; a '批量计算失败' warning here would mean a fallback ran
    if any("失败" in line for line in console):
        raise RuntimeError(f"{name}: the reference fell back from its batch path: {console[:3]}")
    with open(os.path.join(HERE, name + ".ts.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print(f"wrote {name}.ts.json  (quantizeVectors {t_build:.1f}s, total {time.time() - t0:.1f}s, top of query 0: {out['queries'][0]['top_index'][:5]})",
          flush=True)


def run_index_bits_2(ref_root):
    """What the reference DOES for indexBits = 2 (BASELINE configs[4] names queryBits = 8 / indexBits = 2), observed by
    executing it: the index build works (2-bit codes, one per byte, + correctives) and is recorded here for the oracle
    to reproduce; searchNearestNeighbors fails inside the batch path (createDirectPackedBuffer: offset out of bounds),
    logs the fallback warning and goes through the per-vector scorer — which THROWS for queryBits = 8 and, for
    queryBits = 4, returns scores of its own formula (recorded as an observation; this repository's extension follows
    SURVEY §8c's generalisation instead and does not reproduce them)."""
    from tests.fixtures import gaussian
    n, dim = 40, 32
    base, queries = gaussian(n, dim, 5), gaussian(2, dim, 6)
    out = {"n": n, "dim": dim, "seed_base": 5, "seed_queries": 6, "lambda": 0.1, "iters": 5, "index_build": {}, "search": {}}
    for sim in ("EUCLIDEAN", "COSINE", "MAXIMUM_INNER_PRODUCT"):
        for qb in (8, 4):
            console = []
            I, ex, sel, files = load_reference(ref_root, console)
            out["reference_sha256"] = files
            fmt = I.call(ex["createBinaryQuantizationFormat"], args=[
                {"queryBits": float(qb), "indexBits": 2.0, "quantizer": {"similarityFunction": sim, "lambda": 0.1, "iters": 5.0}}])
            rows = [I.float32(r.tolist()) for r in base]
            qv = I.call(I.get(fmt, "quantizeVectors"), fmt, [rows])["quantizedVectors"]
            if qb == 8:
                corr, codes = [], []
                for i in range(n):
                    c = I.call(I.get(qv, "getCorrectiveTerms"), qv, [float(i)])
                    corr.append([f64bits(c[f]) for f in ("lowerInterval", "upperInterval", "additionalCorrection", "quantizedComponentSum")])
                    codes.append([int(x) for x in I.call(I.get(qv, "vectorValue"), qv, [float(i)]).a])
                out["index_build"][sim] = {"centroid_bits": [f32bits(x) for x in I.call(I.get(qv, "getCentroid"), qv, []).a],
                                           "corrections_bits": corr, "codes": codes}
            try:
                res = I.call(I.get(fmt, "searchNearestNeighbors"), fmt, [I.float32(queries[0].tolist()), qv, float(n)])
                by_index = [None] * n
                for r in res:
                    by_index[int(r["index"])] = f32bits(r["score"])
                observed = {"threw": None, "all_score_bits_of_the_fallback": by_index}
            except T.JSThrow as e:
                observed = {"threw": str(e)}
            observed["console"] = console
            out["search"][f"{sim} queryBits={qb}"] = observed
    with open(os.path.join(HERE, "index_bits_2.behaviour.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"), ensure_ascii=False)
    print("wrote index_bits_2.behaviour.json:", {k: (v["threw"] or "fallback scores") for k, v in out["search"].items()}, flush=True)


def run_errors(ref_root):
    """Which Error the reference throws for invalid inputs, observed by executing it (message text, and for NaN / Infinity
    the position it names: under COSINE the vector is normalised before the check, so a NaN anywhere is reported at
    position 0 and an Infinity turns into a NaN at its own position)."""
    import numpy as np
    from tests.fixtures import gaussian
    rows, qs = gaussian(300, 64, 11), gaussian(6, 64, 12)
    out = {"rows_seed": 11, "queries_seed": 12, "n": 300, "dim": 64, "cases": []}

    def attempt(label, spec, fn):
        try:
            fn()
            msg = None
        except T.JSThrow as e:
            v = e.value
            msg = T.to_str(I.get(v, "message")) if isinstance(v, T.JSObj) else T.to_str(v)
        out["cases"].append({"label": label, **spec, "message": msg})

    for sim in ("EUCLIDEAN", "COSINE", "MAXIMUM_INNER_PRODUCT"):
        I, ex, sel, files = load_reference(ref_root, [])
        out["reference_sha256"] = files
        fmt = I.call(ex["createBinaryQuantizationFormat"], args=[
            {"queryBits": 4.0, "indexBits": 1.0, "quantizer": {"similarityFunction": sim, "lambda": 0.1, "iters": 5.0}}])
        quantize, search = I.get(fmt, "quantizeVectors"), I.get(fmt, "searchNearestNeighbors")
        qv = I.call(quantize, fmt, [[I.float32(r.tolist()) for r in rows]])["quantizedVectors"]
        for label, edits in (("query NaN@30 + Infinity@7", {30: np.nan, 7: np.inf}), ("query -Infinity@12", {12: -np.inf}),
                             ("query NaN@5", {5: np.nan})):
            q = qs[2].copy()
            for pos, val in edits.items():
                q[pos] = val
            attempt(label, {"sim": sim, "what": "search", "edits": {str(k): str(v) for k, v in edits.items()}},
                    lambda q=q: I.call(search, fmt, [I.float32(q.tolist()), qv, 5.0]))
        for label, (r, pos, val) in (("build NaN row 3 @9", (3, 9, np.nan)), ("build Infinity row 2 @4", (2, 4, np.inf))):
            b = rows[:5].copy()
            b[r, pos] = val
            attempt(label, {"sim": sim, "what": "build", "row": r, "pos": pos, "value": str(val)},
                    lambda b=b: I.call(quantize, fmt, [[I.float32(x.tolist()) for x in b]]))
        if sim == "COSINE":
            q0 = I.float32(qs[0].tolist())
            attempt("k = -1", {"sim": sim, "what": "search"}, lambda: I.call(search, fmt, [q0, qv, -1.0]))
            attempt("k = 0 (returns [])", {"sim": sim, "what": "search"}, lambda: I.call(search, fmt, [q0, qv, 0.0]))
            attempt("dimension mismatch", {"sim": sim, "what": "search"}, lambda: I.call(search, fmt, [I.float32(qs[0][:10].tolist()), qv, 3.0]))
            attempt("null query", {"sim": sim, "what": "search"}, lambda: I.call(search, fmt, [None, qv, 3.0]))
            attempt("null targets", {"sim": sim, "what": "search"}, lambda: I.call(search, fmt, [q0, None, 3.0]))
            attempt("empty vector set", {"sim": sim, "what": "build"}, lambda: I.call(quantize, fmt, [[]]))
            attempt("ragged rows (row 1 has 10 of 64 dims)", {"sim": sim, "what": "build"},
                    lambda: I.call(quantize, fmt, [[I.float32(rows[0].tolist()), I.float32(rows[1][:10].tolist())]]))
            attempt("queryBits = 9", {"sim": sim, "what": "create"}, lambda: I.call(ex["createBinaryQuantizationFormat"], args=[
                {"queryBits": 9.0, "quantizer": {"similarityFunction": "COSINE"}}]))
            attempt("indexBits = 0", {"sim": sim, "what": "create"}, lambda: I.call(ex["createBinaryQuantizationFormat"], args=[
                {"indexBits": 0.0, "quantizer": {"similarityFunction": "COSINE"}}]))
    with open(os.path.join(HERE, "errors.behaviour.json"), "w") as f:
        json.dump(out, f, indent=1, ensure_ascii=False)
    print("wrote errors.behaviour.json:", len(out["cases"]), "cases", flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", default=os.environ.get("BBQ_REFERENCE_DIR"), required="BBQ_REFERENCE_DIR" not in os.environ)
    ap.add_argument("cases", nargs="*", default=list(CASES) + ["index_bits_2", "errors"])
    a = ap.parse_args()
    for nm in a.cases:
        if nm == "index_bits_2":
            run_index_bits_2(a.reference)
        elif nm == "errors":
            run_errors(a.reference)
        else:
            run_case(nm, a.reference)
