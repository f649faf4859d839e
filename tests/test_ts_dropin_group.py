"""The TypeScript drop-in on a device group, executed under tsinterp with the oracle stand-in of the addon: with
config.devices or BBQ_DEVICES set, every member (the reference's own and the additive ones) reaches the group functions
of the addon and none of the single-GPU ones, and returns what the single-GPU class returns; sharded = true and
joinShardGroup throw; without either setting the class calls exactly what it calls without groups.  A group's stand-in
is one oracle index holding the whole corpus, which is what a group's results equal."""
import os
import sys

import pytest

from tests.fixtures import gaussian
from tests.test_ts_dropin_rerank_sharded import STAND_INS
from tests.ts_dropin.oracle_addon import OracleAddon

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden", "from_ts"))
import tsinterp as T  # noqa: E402

TS = os.path.join(ROOT, "better-binary-quantization_b200", "bindings", "ts")

GROUP_FUNCTIONS = {"groupCreate", "groupContext", "groupBuild", "groupFromQuantized", "groupLoadIndex", "groupSaveIndex",
                   "groupInfo", "groupRows", "groupAttachRows", "groupSearch", "groupSearchRerank"}


class GroupOracleAddon(OracleAddon):
    def __init__(self):
        super().__init__()
        self.images = {}
        self.devices = []

    def f_groupCreate(self, qb, ib, sim, lam, iters, devices):
        self.devices.append([int(d) for d in devices.a])
        return self.f_create(qb, ib, sim, lam, iters, -1)

    def f_groupContext(self, group):
        return group

    def f_groupSaveIndex(self, h, veb, vemb):
        self.images[(veb, vemb)] = h

    def f_groupLoadIndex(self, group, veb, vemb):
        return self.images[(veb, vemb)]

    f_groupBuild = OracleAddon.f_build
    f_groupFromQuantized = OracleAddon.f_fromQuantized
    f_groupInfo = OracleAddon.f_info
    f_groupRows = OracleAddon.f_rows
    f_groupAttachRows = OracleAddon.f_attachRows
    f_groupSearch = OracleAddon.f_search
    f_groupSearchRerank = OracleAddon.f_searchRerank

    def exports(self):
        out = super().exports()
        for n in GROUP_FUNCTIONS:
            def wrap(*a, _n=n):
                self.calls.append(_n)
                return getattr(self, "f_" + _n)(*a)
            out[n] = wrap
        return out


def _interp(tmp_path, addon, env=None):
    src = tmp_path / "src"
    src.mkdir(exist_ok=True)
    for name, text in STAND_INS.items():
        (src / name).write_text(text)
    exports = addon.exports()
    interp = T.Interp(require=lambda spec: exports if spec.endswith("bbq_b200.node") else T.throw_type_error(spec),
                      path_overrides={str(src / "binaryQuantizationFormat.ts"): os.path.join(TS, "binaryQuantizationFormat.gpu.ts"),
                                      str(src / "errors.ts"): os.path.join(TS, "errors.ts")})
    interp.globals.vars["process"]["env"].update(env or {})
    return interp, interp.load(str(src / "binaryQuantizationFormat.ts"))


def _config(**extra):
    return {"queryBits": 4.0, "indexBits": 1.0, "quantizer": {"similarityFunction": "COSINE", "lambda": 0.1, "iters": 5.0},
            **extra}


def _exercise(interp, fmt, base, queries, images=False):
    """every member on the path; -> comparable results"""
    call = lambda name, *a: interp.call(interp.get(fmt, name), fmt, list(a))
    rows = [interp.float32(r.tolist()) for r in base]
    qs = [interp.float32(q.tolist()) for q in queries]
    out = []
    qv = call("quantizeVectors", rows)["quantizedVectors"]
    g = lambda name, *a: interp.call(interp.get(qv, name), qv, list(a))
    out.append((g("size"), g("dimension"), list(g("getCentroid").a), g("getCentroidDP"), list(g("vectorValue", 3.0).a),
                list(g("getUnpackedVector", 5.0).a), dict(g("getCorrectiveTerms", 7.0))))
    key = lambda rs: [(r["index"], r["score"]) for r in rs]
    out.append(key(call("searchNearestNeighbors", qs[0], qv, 7.0)))
    out.append([key(r) for r in call("searchBatch", qs, qv, 9.0)])
    call("attachOriginalVectors", qv, rows)
    out.append([(r["index"], r["quantizedScore"], r["trueScore"]) for r in call("searchOversampled", qs[1], qv, 5.0, 3.0)])
    ser = call("serializeVectorData", rows)
    back = call("deserializeVectorData", ser["vectorData"], ser["metadata"])
    out.append(key(call("searchNearestNeighbors", qs[0], back, 7.0)))
    if images:   # (the stand-in keeps images of group indexes only)
        call("saveIndex", qv, "/img/x")
        out.append(key(call("searchNearestNeighbors", qs[0], call("loadIndex", "/img/x"), 7.0)))
    return out


@pytest.mark.parametrize("how", ["config", "env"])
def test_a_group_routes_every_member_to_the_group_functions(tmp_path, how):
    base, queries = gaussian(80, 24, 9600), gaussian(3, 24, 9601)
    addon = GroupOracleAddon()
    interp, mod = _interp(tmp_path, addon, env={"BBQ_DEVICES": "0, 1,2"} if how == "env" else None)
    cfg = _config(devices=[0.0, 1.0, 2.0]) if how == "config" else _config()
    fmt = interp.construct(mod["BinaryQuantizationFormat"], [cfg])
    got = _exercise(interp, fmt, base, queries, images=True)
    assert addon.devices == [[0, 1, 2]]
    assert set(addon.calls) <= GROUP_FUNCTIONS, set(addon.calls) - GROUP_FUNCTIONS
    assert GROUP_FUNCTIONS <= set(addon.calls), GROUP_FUNCTIONS - set(addon.calls)
    # the same results as the class without a group (whose image round trip the stand-in cannot run)
    (tmp_path / "plain").mkdir()
    p_interp, p_mod = _interp(tmp_path / "plain", OracleAddon())
    p_fmt = p_interp.construct(p_mod["BinaryQuantizationFormat"], [_config()])
    want = _exercise(p_interp, p_fmt, base, queries)
    assert got[:-1] == want and got[-1] == want[1]
    # quantizeQueryVector runs on the group's first GPU: the group's context
    q = interp.float32(queries[0].tolist())
    qv = interp.call(interp.get(fmt, "quantizeVectors"), fmt, [[interp.float32(r.tolist()) for r in base]])["quantizedVectors"]
    cen = interp.call(interp.get(qv, "getCentroid"), qv, [])
    interp.call(interp.get(fmt, "quantizeQueryVector"), fmt, [q, cen])
    assert addon.calls[-1] == "quantizeQuery"


def test_sharded_flags_and_join_throw_on_a_group(tmp_path):
    base, queries = gaussian(40, 16, 9700), gaussian(1, 16, 9701)
    addon = GroupOracleAddon()
    interp, mod = _interp(tmp_path, addon)
    fmt = interp.construct(mod["BinaryQuantizationFormat"], [_config(devices=[0.0, 1.0])])
    rows = [interp.float32(r.tolist()) for r in base]
    q = interp.float32(queries[0].tolist())
    qv = interp.call(interp.get(fmt, "quantizeVectors"), fmt, [rows])["quantizedVectors"]
    for name, args in (("quantizeVectors", [rows, True]), ("searchBatch", [[q], qv, 3.0, True]),
                       ("searchOversampled", [q, qv, 3.0, 2.0, True]), ("saveIndex", [qv, "/x", True]),
                       ("loadIndex", ["/x", True]), ("joinShardGroup", [interp.float32([0.0] * 128), 0.0, 2.0])):
        with pytest.raises(T.JSThrow) as e:
            interp.call(interp.get(fmt, name), fmt, args)
        assert "device group" in T.get_prop(e.value.value, "message"), name


def test_without_a_group_the_class_calls_what_it_calls_today(tmp_path):
    base, queries = gaussian(60, 20, 9800), gaussian(2, 20, 9801)
    addon = GroupOracleAddon()
    interp, mod = _interp(tmp_path, addon)
    fmt = interp.construct(mod["BinaryQuantizationFormat"], [_config()])
    _exercise(interp, fmt, base, queries)
    assert not set(addon.calls) & GROUP_FUNCTIONS
    assert addon.calls[:2] == ["create", "build"] and {"search", "rows", "attachRows", "searchRerank", "fromQuantized",
                                                       "info"} <= set(addon.calls)
