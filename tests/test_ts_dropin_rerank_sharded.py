"""The TypeScript drop-in's searchOversampled(..., sharded = true) executed under tsinterp with the oracle stand-in of
the addon: the flag routes the call to addon.searchRerankSharded, and the result object is read exactly as the one of
searchRerank.  The reference classes the drop-in imports are replaced by minimal stand-ins written here, so the test
needs no reference checkout."""
import os
import sys

import numpy as np

from tests.fixtures import gaussian
from tests.ts_dropin.oracle_addon import OracleAddon

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden", "from_ts"))
import tsinterp as T  # noqa: E402

TS = os.path.join(ROOT, "better-binary-quantization_b200", "bindings", "ts")

# just what binaryQuantizationFormat.gpu.ts imports from the reference's src/
STAND_INS = {
    "types.ts": "export enum VectorSimilarityFunction { EUCLIDEAN = 'EUCLIDEAN', COSINE = 'COSINE', "
                "MAXIMUM_INNER_PRODUCT = 'MAXIMUM_INNER_PRODUCT' }\n",
    "constants.ts": "export const QUERY_BITS = 4;\nexport const INDEX_BITS = 1;\n",
    "binaryQuantizationFormat.cpu.ts": "export class BinaryQuantizationFormat {\n"
                                       "  private config: any;\n"
                                       "  constructor(config: any) { this.config = config; }\n"
                                       "  getConfig(): any { return this.config; }\n"
                                       "  getQuantizer(): any { return null; }\n"
                                       "}\n",
}


class ShardedOracleAddon(OracleAddon):
    """One process holding the whole corpus is one shard of one: the sharded re-rank is the plain one."""

    f_searchRerankSharded = OracleAddon.f_searchRerank

    def exports(self):
        out = super().exports()

        def wrap(*a):
            self.calls.append("searchRerankSharded")
            return self.f_searchRerankSharded(*a)
        out["searchRerankSharded"] = wrap
        return out


def test_search_oversampled_sharded_flag_calls_the_sharded_addon_entry(tmp_path):
    src = tmp_path / "src"
    src.mkdir()
    for name, text in STAND_INS.items():
        (src / name).write_text(text)
    addon = ShardedOracleAddon()
    exports = addon.exports()
    interp = T.Interp(require=lambda spec: exports if spec.endswith("bbq_b200.node") else T.throw_type_error(spec),
                      path_overrides={str(src / "binaryQuantizationFormat.ts"): os.path.join(TS, "binaryQuantizationFormat.gpu.ts"),
                                      str(src / "errors.ts"): os.path.join(TS, "errors.ts")})
    mod = interp.load(str(src / "binaryQuantizationFormat.ts"))
    config = {"queryBits": 4.0, "indexBits": 1.0, "quantizer": {"similarityFunction": "COSINE", "lambda": 0.1, "iters": 5.0}}
    fmt = interp.construct(mod["BinaryQuantizationFormat"], [config])
    base, queries = gaussian(60, 32, 9400), gaussian(2, 32, 9401)
    rows = [interp.float32(r.tolist()) for r in base]
    qv = interp.call(interp.get(fmt, "quantizeVectors"), fmt, [rows])["quantizedVectors"]
    interp.call(interp.get(fmt, "attachOriginalVectors"), fmt, [qv, rows])
    search = interp.get(fmt, "searchOversampled")
    for q in queries:
        q = interp.float32(q.tolist())
        plain = interp.call(search, fmt, [q, qv, 5.0, 3.0])
        n_sharded = addon.calls.count("searchRerankSharded")
        sharded = interp.call(search, fmt, [q, qv, 5.0, 3.0, True])
        assert addon.calls.count("searchRerankSharded") == n_sharded + 1
        key = lambda rs: [(r["index"], r["quantizedScore"], np.float64(r["trueScore"]).view(np.uint64)) for r in rs]
        assert len(plain) == 5 and key(sharded) == key(plain)
    assert addon.calls.count("searchRerank") == len(queries)      # the default path still calls searchRerank
