"""The reference centroid across slices of a corpus, without a GPU:

- bbq_centroid_finish equals numpy's f64 divide-then-round at N up to 2^31 - 17, for sums holding +-0, subnormals,
  +-Inf and NaN (a divide by float32(N) does not, once N > 2^24);
- the chain kernel's step, an f32 add, equals the reference's f64 add rounded to f32 (53 >= 2 * 24 + 2), checked by a
  host program on edge pairs and 10^7 random bit patterns;
- the TypeScript drop-in's quantizeVectors(vectors, sharded = true) under tsinterp with the oracle stand-in of the addon:
  the flag routes to addon.buildSharded and lets an empty rank through, the default path is unchanged."""
import os
import subprocess

import numpy as np
import pytest

from tests.fixtures import gaussian
from tests.test_ts_dropin_rerank_sharded import STAND_INS, TS, T
from tests.ts_dropin.oracle_addon import OracleAddon, throw_status


@pytest.fixture(scope="module")
def bbq():
    import bbq_b200
    bbq_b200.build_library()
    return bbq_b200


def _sums(seed):
    rng = np.random.default_rng(seed)
    edge = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1e-45, -1e-45, 1.1754942e-38, -3e-39, 3.4028235e38,
                     -3.4028235e38, 1.0, -1.0, 16777217.0], np.float32)
    rand = (rng.standard_normal(500) * 10.0 ** rng.integers(-40, 38, 500)).astype(np.float32)
    return np.concatenate([edge, rand, rng.integers(0, 1 << 32, 200, dtype=np.uint64).astype(np.uint32).view(np.float32)])


def _bits_equal(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    nan = np.isnan(a)
    return np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(np.uint32), b[~nan].view(np.uint32))


@pytest.mark.parametrize("n_total", [1, 3, 2 ** 24 + 1, 10 ** 8 + 7, 2 ** 31 - 17])
def test_centroid_finish_is_the_f64_divide(bbq, n_total):
    running = _sums(n_total % 1000)
    got = bbq.BinaryQuantizationFormat.finishCentroid(running, n_total)
    with np.errstate(all="ignore"):
        want = (running.astype(np.float64) / np.float64(n_total)).astype(np.float32)
        naive = running / np.float32(n_total)
    assert _bits_equal(got, want)
    if n_total > 2 ** 24:      # float32(N) is not N here: the obvious host code gives other centroids
        assert not _bits_equal(naive, want)


def test_centroid_finish_refusals(bbq):
    with pytest.raises(bbq.BbqError) as e:
        bbq.BinaryQuantizationFormat.finishCentroid(np.ones(4, np.float32), 0)
    assert e.value.status == 3


FADD_CHECK = r"""
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
static uint32_t bits(float x) { uint32_t u; memcpy(&u, &x, 4); return u; }
static float from(uint32_t u) { float x; memcpy(&x, &u, 4); return x; }
static int same(float a, float b) { return (std::isnan(a) && std::isnan(b)) || bits(a) == bits(b); }
static uint64_t s = 0x9E3779B97F4A7C15ull;
static uint64_t next() { uint64_t z = (s += 0x9E3779B97F4A7C15ull); z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
                         z = (z ^ (z >> 27)) * 0x94D049BB133111EBull; return z ^ (z >> 31); }
int main() {
  const uint32_t edge[] = {0x00000000u, 0x80000000u, 0x00000001u, 0x80000001u, 0x007FFFFFu, 0x807FFFFFu, 0x00800000u,
                           0x80800000u, 0x7F7FFFFFu, 0xFF7FFFFFu, 0x7F800000u, 0xFF800000u, 0x7FC00000u, 0x3F800000u,
                           0xBF800000u, 0x33800000u, 0x33800001u, 0x4B800000u, 0x4B800001u, 0x34000000u, 0x3F800001u};
  const int ne = sizeof edge / sizeof edge[0];
  long bad = 0, pairs = 0;
  for (int i = 0; i < ne; i++)
    for (int j = 0; j < ne; j++, pairs++) {
      const float a = from(edge[i]), b = from(edge[j]);
      bad += !same(a + b, (float)((double)a + (double)b));
    }
  for (long k = 0; k < 10000000; k++, pairs++) {
    const uint64_t r = next();
    float a = from((uint32_t)r), b = from((uint32_t)(r >> 32));
    if (k & 1) b = from((bits(a) & 0x80000000u) ^ (k & 2 ? 0x80000000u : 0) | ((bits(a) & 0x7FFFFFFFu) + (uint32_t)(r >> 40) % 64));
    bad += !same(a + b, (float)((double)a + (double)b));
  }
  printf("%ld %ld\n", pairs, bad);
  return 0;
}
"""


def test_f32_add_is_the_f64_add_rounded(tmp_path):
    """Every second random pair is a near-cancelling one (same magnitude up to 63 ulps, either sign), where a double
    rounding would show first."""
    src, exe = tmp_path / "fadd.cpp", tmp_path / "fadd"
    src.write_text(FADD_CHECK)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-o", str(exe), str(src)])
    pairs, bad = map(int, subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split())
    assert pairs == 21 * 21 + 10 ** 7 and bad == 0


class BuildShardedOracleAddon(OracleAddon):
    """One process holding the whole corpus is one shard of one: the sharded build is the plain one, and with no rows
    on the only rank the corpus is empty."""

    def exports(self):
        out = super().exports()

        def wrap(*a):
            self.calls.append("buildSharded")
            return self.f_buildSharded(*a)
        out["buildSharded"] = wrap
        return out

    def f_buildSharded(self, ctx, rows, n, dim, centroid):
        if int(n) == 0:
            throw_status(3, message="vector set must not be empty")
        return self.f_build(ctx, rows, n, dim, centroid)


def test_ts_quantize_vectors_sharded_flag_calls_build_sharded(tmp_path):
    src = tmp_path / "src"
    src.mkdir()
    for name, text in STAND_INS.items():
        (src / name).write_text(text)
    addon = BuildShardedOracleAddon()
    exports = addon.exports()
    interp = T.Interp(require=lambda spec: exports if spec.endswith("bbq_b200.node") else T.throw_type_error(spec),
                      path_overrides={str(src / "binaryQuantizationFormat.ts"): os.path.join(TS, "binaryQuantizationFormat.gpu.ts"),
                                      str(src / "errors.ts"): os.path.join(TS, "errors.ts")})
    mod = interp.load(str(src / "binaryQuantizationFormat.ts"))
    config = {"queryBits": 4.0, "indexBits": 1.0, "quantizer": {"similarityFunction": "COSINE", "lambda": 0.1, "iters": 5.0}}
    fmt = interp.construct(mod["BinaryQuantizationFormat"], [config])
    call = lambda name, *args: interp.call(interp.get(fmt, name), fmt, list(args))
    base, queries = gaussian(60, 32, 9600), gaussian(3, 32, 9601)
    rows = [interp.float32(r.tolist()) for r in base]

    plain = call("quantizeVectors", rows)["quantizedVectors"]
    assert "buildSharded" not in addon.calls and addon.calls.count("build") == 1
    sharded = call("quantizeVectors", rows, True)["quantizedVectors"]
    assert addon.calls.count("buildSharded") == 1 and addon.calls.count("build") == 1
    info = lambda qv: (call_get(qv, "size"), np.asarray(call_get(qv, "getCentroid").a, np.float32).tobytes())
    call_get = lambda obj, name: interp.call(interp.get(obj, name), obj, [])
    assert info(sharded) == info(plain)
    qs = [interp.float32(q.tolist()) for q in queries]
    key = lambda res: [[(r["index"], np.float32(r["score"]).view(np.uint32)) for r in row] for row in res]
    assert key(call("searchBatch", qs, sharded, 5.0)) == key(call("searchBatch", qs, plain, 5.0))

    # an empty rank reaches the addon with the flag (here the only rank, so the corpus is empty) ...
    with pytest.raises(T.JSThrow) as e:
        call("quantizeVectors", [], True)
    assert addon.calls[-1] == "buildSharded" and addon.calls.count("buildSharded") == 2
    assert T.get_prop(e.value.value, "message") == "向量集合不能为空"
    # ... and is refused before it without
    n_calls = len(addon.calls)
    with pytest.raises(T.JSThrow) as e:
        call("quantizeVectors", [])
    assert len(addon.calls) == n_calls and T.get_prop(e.value.value, "message") == "向量集合不能为空"
