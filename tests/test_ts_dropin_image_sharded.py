"""The TypeScript drop-in's saveIndex / loadIndex(..., sharded = true) and joinShardGroup without a shard, executed under
tsinterp with the oracle stand-in of the addon: the flags route to addon.saveIndexSharded / addon.loadIndexSharded, the
default path still calls saveIndex / loadIndex, and a rank that joins before it has a shard only runs commInit.  The
reference classes the drop-in imports are replaced by the minimal stand-ins of test_ts_dropin_rerank_sharded.py, so
the test needs no reference checkout."""
import os

import numpy as np

from tests.fixtures import gaussian
from tests.test_ts_dropin_rerank_sharded import STAND_INS, TS, T
from tests.ts_dropin.oracle_addon import OracleAddon, throw_status, typed


class ImageOracleAddon(OracleAddon):
    """Images kept in memory by path; one process holding the whole corpus is one shard of one, so the sharded entries
    store and return the same index as the plain ones."""

    def __init__(self):
        super().__init__()
        self.files = {}

    def exports(self):
        out = super().exports()
        for name in ("saveIndexSharded", "loadIndexSharded", "commInit", "setBase"):
            def wrap(*a, _n=name):
                self.calls.append(_n)
                return getattr(self, "f_" + _n)(*a)
            out[name] = wrap
        return out

    def f_saveIndex(self, h, veb, vemb):
        assert veb.endswith(".veb") and vemb.endswith(".vemb") and veb[:-4] == vemb[:-5]
        self.files[veb] = h
        return T.UNDEF

    def f_loadIndex(self, ctx, veb, vemb):
        if veb not in self.files:
            throw_status(11, message=f"cannot open '{vemb}'")
        return self.files[veb]

    f_saveIndexSharded = f_saveIndex
    f_loadIndexSharded = f_loadIndex

    def f_commInit(self, ctx, id_, rank, world):
        return T.UNDEF

    def f_setBase(self, h, base):
        return T.UNDEF


def test_image_sharded_flags_call_the_sharded_addon_entries(tmp_path):
    src = tmp_path / "src"
    src.mkdir()
    for name, text in STAND_INS.items():
        (src / name).write_text(text)
    addon = ImageOracleAddon()
    exports = addon.exports()
    interp = T.Interp(require=lambda spec: exports if spec.endswith("bbq_b200.node") else T.throw_type_error(spec),
                      path_overrides={str(src / "binaryQuantizationFormat.ts"): os.path.join(TS, "binaryQuantizationFormat.gpu.ts"),
                                      str(src / "errors.ts"): os.path.join(TS, "errors.ts")})
    mod = interp.load(str(src / "binaryQuantizationFormat.ts"))
    cls = mod["BinaryQuantizationFormat"]
    config = {"queryBits": 4.0, "indexBits": 1.0, "quantizer": {"similarityFunction": "COSINE", "lambda": 0.1, "iters": 5.0}}
    fmt = interp.construct(cls, [config])
    call = lambda name, *args: interp.call(interp.get(fmt, name), fmt, list(args))

    # a rank about to load its shard joins without one: commInit only
    gid = typed("Uint8Array", [0] * 128)
    call("joinShardGroup", gid, 0.0, 1.0)
    assert addon.calls[-1] == "commInit" and "setBase" not in addon.calls

    base, queries = gaussian(60, 32, 9500), gaussian(3, 32, 9501)
    rows = [interp.float32(r.tolist()) for r in base]
    qv = call("quantizeVectors", rows)["quantizedVectors"]
    call("joinShardGroup", gid, 0.0, 1.0, qv, 0.0)
    assert addon.calls[-2:] == ["commInit", "setBase"]

    prefix = str(tmp_path / "index")
    call("saveIndex", qv, prefix)
    assert addon.calls[-1] == "saveIndex"
    call("saveIndex", qv, prefix + "_s", True)
    assert addon.calls[-1] == "saveIndexSharded"
    plain = call("loadIndex", prefix)
    assert addon.calls[-2:] == ["loadIndex", "info"]            # (the handle's metadata is read once, on wrapping)
    sharded = call("loadIndex", prefix + "_s", True)
    assert addon.calls[-2:] == ["loadIndexSharded", "info"]
    qs = [interp.float32(q.tolist()) for q in queries]
    key = lambda res: [[(r["index"], np.float32(r["score"]).view(np.uint32)) for r in row] for row in res]
    want = key(call("searchBatch", qs, qv, 5.0))
    assert key(call("searchBatch", qs, plain, 5.0)) == want
    assert key(call("searchBatch", qs, sharded, 5.0, True)) == want
    assert addon.calls.count("saveIndex") == 1 and addon.calls.count("loadIndex") == 1
