"""The cases tests/test_golden_from_ts.py once ran through the reference source live (three fixed tiny cases and a seeded
fuzz of 150 random configurations), with the answers stored in live_cases.json so that the oracle is compared with them
on every machine.  With a reference checkout the same cases are run through the reference again and must give the
stored answers.

    BBQ_REFERENCE_DIR=<reference checkout> python tests/golden/from_ts/live_cases.py     # rewrites live_cases.json
"""
import json
import os
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(HERE)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from tests.fixtures import gaussian  # noqa: E402

STORED = os.path.join(HERE, "live_cases.json")
FIELDS = ("lowerInterval", "upperInterval", "additionalCorrection", "quantizedComponentSum")


def fixed_cases():
    """-> [(name, sim, qb, lam, iters, k, base, queries)]: tiny seeded cases, two queries each, k = 5."""
    out = []
    for sim, qb, n, dim in (("COSINE", 4, 40, 24), ("EUCLIDEAN", 1, 30, 20), ("MAXIMUM_INNER_PRODUCT", 4, 36, 36)):
        out.append((f"fixed_{sim}_{qb}_{n}x{dim}", sim, qb, 0.1, 5, 5, gaussian(n, dim, 4242 + n), gaussian(2, dim, 4343 + n)))
    return out


def fuzz_cases():
    """-> the same list for 150 random small configurations (seed 7): every similarity function, query bits 1..8, dims
    1..70 (below and across the 8-dim packing boundary), 1..40 rows, lambda in {0, 0.001, 0.1, 0.5, 1}, 0 / 1 / 5 / 20
    iterations, component scales 1e-3..1e3, duplicated and all-zero rows; every sixth case each made of signed zeros
    only, of integers, or of values near the top of the f32 range.  One query each."""
    rng = np.random.default_rng(7)
    sims = ["EUCLIDEAN", "COSINE", "MAXIMUM_INNER_PRODUCT"]
    out = []
    for case in range(150):
        sim, qb = sims[rng.integers(3)], int(rng.integers(1, 9))
        dim, n = int(rng.choice([1, 2, 3, 5, 7, 8, 9, 15, 16, 17, 31, 33, 64, 70])), int(rng.integers(1, 40))
        lam, iters, k = float(rng.choice([0.1, 0.001, 0.5, 0.0, 1.0])), int(rng.choice([0, 1, 5, 20])), int(rng.integers(1, 12))
        scale = float(rng.choice([1.0, 1e-3, 1e3]))
        base = (rng.standard_normal((n, dim)) * scale).astype(np.float32)
        q = (rng.standard_normal(dim) * scale).astype(np.float32)
        if rng.random() < 0.3:
            base[rng.integers(n)] = base[0]
        if rng.random() < 0.2:
            base[rng.integers(n)] = 0
        kind = case % 6                                  # every sixth case each: an extreme shape
        if kind == 1:                                    # signed zeros only (Math.min(+0, -0) = -0 decides the interval's sign)
            base[:, ::2] = 0
            base[:, 1::2] = np.float32(-0.0) * base[:, 1::2]
        elif kind == 2:                                  # integers: exact ties and .5 roundings
            base, q = np.round(base).astype(np.float32), np.round(q).astype(np.float32)
        elif kind == 3:                                  # near the top of the f32 range
            base = (rng.standard_normal((n, dim)) * 1e30).astype(np.float32)
            q[0] = np.float32(3e38)
        out.append((f"fuzz_{case}_kind{kind}_{sim}_{qb}b_{n}x{dim}", sim, qb, lam, iters, k, base, q[None, :]))
    return out


def encode(corr, packed, results):
    """corr f64[n, 4], packed u8[n, bytes], results [(ids, f32 scores)] per query -> the stored (JSON) form."""
    return {"corr": [b"".join(struct.pack(">d", float(v)) for v in row).hex() for row in corr],
            "packed": [bytes(row.tolist()).hex() for row in packed],
            "top_index": [[int(i) for i in ids] for ids, _ in results],
            "top_score_bits": [np.asarray(sc, np.float32).view(np.uint32).tolist() for _, sc in results]}


def run_reference(reference_dir, cases):
    """Runs every case through the reference's own src/index.ts (tsinterp) -> {name: stored form}."""
    sys.path.insert(0, HERE)
    import tsinterp as T
    console = []
    interp = T.Interp(log=lambda *a: console.append(a), stub_modules=["/src/wasm/index.ts"])
    ex = interp.load(os.path.join(reference_dir, "src", "index.ts"))
    out = {}
    for name, sim, qb, lam, iters, k, base, queries in cases:
        fmt = interp.call(ex["createBinaryQuantizationFormat"], args=[
            {"queryBits": float(qb), "indexBits": 1.0, "quantizer": {"similarityFunction": sim, "lambda": lam, "iters": float(iters)}}])
        qv = interp.call(interp.get(fmt, "quantizeVectors"), fmt, [[interp.float32(r.tolist()) for r in base]])["quantizedVectors"]
        corr = [[interp.call(interp.get(qv, "getCorrectiveTerms"), qv, [float(i)])[f] for f in FIELDS] for i in range(len(base))]
        packed = np.array([list(interp.call(interp.get(qv, "vectorValue"), qv, [float(i)]).a) for i in range(len(base))], np.uint8)
        results = []
        for q in queries:
            res = interp.call(interp.get(fmt, "searchNearestNeighbors"), fmt, [interp.float32(q.tolist()), qv, float(k)])
            results.append(([int(r["index"]) for r in res], np.array([r["score"] for r in res], np.float32)))
        out[name] = encode(corr, packed, results)
    assert not console, console[:3]
    return out


def load_stored():
    with open(STORED) as f:
        return json.load(f)["cases"]


if __name__ == "__main__":
    ref = os.environ.get("BBQ_REFERENCE_DIR") or sys.exit("set BBQ_REFERENCE_DIR to a checkout of the reference project")
    cases = run_reference(ref, fixed_cases() + fuzz_cases())
    with open(STORED, "w") as f:
        json.dump({"source": "the reference's src/index.ts, executed by tsinterp.py (live_cases.py)", "cases": cases}, f,
                  separators=(",", ":"))
    print("wrote", STORED, len(cases), "cases")
