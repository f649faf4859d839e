"""tests/golden/from_ts/tsinterp.py — the TypeScript-subset interpreter that produced the reference-source fixtures —
checked on its own: ECMAScript number semantics (the part the fixtures depend on), TypeScript syntax skipping, classes,
closures, modules.  Expected values are what any JavaScript engine prints for the same source (worked out by hand from
the ECMAScript rules: ToInt32 / ToUint32, Math.round half-up, Float32Array / Uint8Array stores, remainder sign, ...)."""
import math
import os
import struct
import sys

import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "from_ts"))
import tsinterp as T  # noqa: E402

from tests.golden_util import HAVE_REFERENCE, REFERENCE_DIR  # noqa: E402


def run(tmp_path, src, extra=None, fn="main", args=()):
    for name, text in (extra or {}).items():
        (tmp_path / name).write_text(text, encoding="utf-8")
    p = tmp_path / "main.ts"
    p.write_text(src, encoding="utf-8")
    log = []
    interp = T.Interp(log=lambda *a: log.append(" ".join(map(str, a))))
    ex = interp.load(str(p))
    return interp.call(ex[fn], args=list(args)), log


def f32(x):
    return struct.unpack("f", struct.pack("f", x))[0]


def test_number_semantics(tmp_path):
    out, _ = run(tmp_path, """
    export function main(): number[] {
      const u8 = new Uint8Array(4); u8[0] = 257; u8[1] = -1; u8[2] = 3.99; u8[3] = NaN;
      const i32 = new Int32Array(2); i32[0] = 2147483648; i32[1] = -2147483649;
      const f = new Float32Array(3); f[0] = 0.1; f[1] = 1e40; f[2] = 16777217;
      return [
        Math.round(2.5), Math.round(-2.5), Math.round(0.49999999999999994), Math.round(-0.4), Math.round(1e300),
        5 >>> 1, -5 >> 1, -5 >>> 28, 1 << 31, 0xFFFFFFFF | 0, 7 & 3, 6 ^ 3, ~5, 2 ** 10, (-8) % 3, 8 % -3, 5.5 % 2,
        1 / 0, -1 / 0, u8[0]!, u8[1]!, u8[2]!, u8[3]!, i32[0]!, i32[1]!, f[0]!, f[1]!, f[2]!,
        Math.max(1, 2, 3), Math.min(), Math.floor(-0.5), Math.ceil(-0.5), Math.trunc(-3.7), Math.sign(-2), Math.fround(0.1),
        Number.MAX_VALUE * 2, 0.1 + 0.2, parseInt('42px'), parseFloat('3.5e2x'), Number('0x10'), +true, 7 / 2 | 0,
      ];
    }""")
    want = [3.0, -2.0, 0.0, -0.0, 1e300,
            2.0, -3.0, 15.0, -2147483648.0, -1.0, 3.0, 5.0, -6.0, 1024.0, -2.0, 2.0, 1.5,
            math.inf, -math.inf, 1.0, 255.0, 3.0, 0.0, -2147483648.0, 2147483647.0, f32(0.1), math.inf, 16777216.0,
            3.0, math.inf, -1.0, -0.0, -3.0, -1.0, f32(0.1),
            math.inf, 0.30000000000000004, 42.0, 350.0, 16.0, 1.0, 3.0]
    assert len(out) == len(want)
    for i, (a, b) in enumerate(zip(out, want)):
        assert struct.pack("d", a) == struct.pack("d", b), (i, a, b)     # bit patterns: -0 and +0 differ


def test_nan_and_equality(tmp_path):
    out, _ = run(tmp_path, """
    export function main() {
      const n = 0 / 0;
      return [n === n, n !== n, Math.max(1, NaN), Math.min(NaN, 1), Number.isNaN(n), isNaN('x' as any), Number.isFinite(1 / 0),
              null == undefined, null === undefined, 1 == ('1' as any), 0 === -0, typeof n, typeof undefined, typeof null, typeof (() => 1),
              undefined ?? 'd', 0 ?? 'd', 0 || 'd', '' && 'x', [] ? 'truthy' : 'falsy', NaN ? 1 : 2];
    }""")
    assert out[0] is False and out[1] is True and math.isnan(out[2]) and math.isnan(out[3])
    assert out[4:] == [True, True, False, True, False, True, True, "number", "undefined", "object", "function",
                       "d", 0.0, "d", "", "truthy", 2.0]


def test_typescript_syntax_is_skipped(tmp_path):
    out, _ = run(tmp_path, """
    import type { Foo } from './types';
    import { twice, Kind, type Unused } from './lib';
    export interface Shape { area(): number; readonly name?: string }
    type Pair<T> = [T, T] | { first: T; second: T };
    type Fn = (a: number, b: number) => number;
    declare const notThere: number;
    export abstract class Nothing { }
    function id<T extends object = {}>(x: T): T { return x; }
    const add: Fn = (a: number, b: number): number => a + b;
    function over(a: number): number;
    function over(a: string): string;
    function over(a: any): any { return a; }
    export function main(n: number, opt?: { k: number }): Array<{ v: number }> {
      const m = new Map<string, Array<{ v: number }>>();
      const list: Array<{ v: number }> = [];
      let x = <number>(n as unknown as number);
      const y = opt!?.k ?? 7;
      const t = id<{ v: number }>({ v: x + y });
      list.push(t, { v: add(twice(2), 1) }, { v: Kind.B }, { v: over(5) satisfies number });
      m.set('a', list);
      return m.get('a')!;
    }""", {"lib.ts": "export const twice = (v: number) => v * 2;\nexport enum Kind { A, B, C = 10, D }\nexport type Unused = number;\n",
           "types.ts": "export interface Foo { a: number }\n"}, args=[3.0])
    assert [e["v"] for e in out] == [10.0, 5.0, 1.0, 5.0]


def test_classes_closures_and_control_flow(tmp_path):
    out, log = run(tmp_path, """
    class MinHeap<T> {
      private heap: T[] = [];
      private static created = 0;
      constructor(private readonly compareFn: (a: T, b: T) => number, public label: string = 'heap') { MinHeap.created++; }
      push(v: T): void { this.heap.push(v); this.heap.sort(this.compareFn); }
      pop(): T | undefined { return this.heap.shift(); }
      size(): number { return this.heap.length; }
      static count(): number { return MinHeap.created; }
    }
    export function main(n: number) {
      const h = new MinHeap<{ s: number; i: number }>((a, b) => a.s - b.s);
      for (let i = 0; i < n; i++) h.push({ s: (i * 7) % 5, i });
      const order: number[] = [];
      while (h.size() > 0) order.push(h.pop()!.i);
      const fns: Array<() => number> = [];
      for (let i = 0; i < 3; i++) fns.push(() => i * 10);           // per-iteration binding
      let sw = '';
      for (const v of [1, 2, 3, 4]) {
        switch (v) { case 1: sw += 'a'; case 2: sw += 'b'; break; case 3: continue; default: sw += 'd'; }
        sw += '.';
      }
      let tr = '';
      try { try { throw new RangeError('boom'); } finally { tr += 'f'; } } catch (e) { tr += (e as Error).name + ':' + (e as Error).message; }
      const { a, b = 5, ...rest } = { a: 1, c: 3, d: 4 } as any;
      const [p, , q = 9, ...tail] = [1, 2, undefined, 4, 5];
      const merged = { ...rest, a, b, [`k${p}`]: q };
      let count = 0;
      do { count++; } while (count < 3);
      console.log('done', count);
      return { order, fns: fns.map(f => f()), sw, tr, merged, tail, label: h.label, heaps: MinHeap.count(),
               stable: [{ k: 1, t: 'x' }, { k: 0, t: 'y' }, { k: 1, t: 'z' }, { k: 0, t: 'w' }].sort((u, v) => u.k - v.k).map(o => o.t).join('') };
    }""", args=[6.0])
    assert out["order"] == [0.0, 5.0, 3.0, 1.0, 4.0, 2.0]       # scores 0,2,4,1,3,0: stable sort keeps insertion order of ties
    assert out["fns"] == [0.0, 10.0, 20.0]
    assert out["sw"] == "ab.b.d."
    assert out["tr"] == "fRangeError:boom"
    assert out["merged"] == {"c": 3.0, "d": 4.0, "a": 1.0, "b": 5.0, "k1": 9.0}
    assert out["tail"] == [4.0, 5.0] and out["label"] == "heap" and out["heaps"] == 1.0 and out["stable"] == "ywxz"
    assert log == ["done 3"]


def test_arrays_strings_and_typed_arrays(tmp_path):
    out, _ = run(tmp_path, """
    export function main() {
      const a = Array.from({ length: 5 }, (_, j) => j * j);
      const t = new Float32Array([1.5, 2.5, 3.5]);
      const copy = new Float32Array(t); copy[0] = 9;
      const u = new Uint8Array(6); u.set([1, 2, 3], 2); u.fill(7, 0, 1);
      const sum = t.reduce((s, v) => s + v, 0);
      let viaOf = 0; for (const v of t) viaOf += v;
      return { a, sliced: a.slice(1, -1), idx: a.indexOf(9), inc: a.includes(16), t0: t[0], c0: copy[0], len: t.length, oob: t[10] === undefined,
               u: Array.from(u), sum, viaOf, str: `n=${1 / 4} ${[1, 2]} ${'ab'.padStart(4, '0')} ${(0.125).toFixed(2)} ${'x'.repeat(3)}`,
               spread: [...a.slice(0, 2), ...'hi'], max: Math.max(...a), filled: new Array(3).fill(0), joined: [1, null, 2].join('-'),
               keys: Object.keys({ z: 1, y: 2 }), entries: Object.entries({ q: 1 }), isArr: Array.isArray(t), every: a.every(v => v >= 0) };
    }""")
    assert out["a"] == [0.0, 1.0, 4.0, 9.0, 16.0] and out["sliced"] == [1.0, 4.0, 9.0] and out["idx"] == 3.0 and out["inc"] is True
    assert out["t0"] == 1.5 and out["c0"] == 9.0 and out["len"] == 3.0 and out["oob"] is True
    assert out["u"] == [7.0, 0.0, 1.0, 2.0, 3.0, 0.0] and out["sum"] == 7.5 and out["viaOf"] == 7.5
    assert out["str"] == "n=0.25 1,2 00ab 0.13 xxx"
    assert out["spread"] == [0.0, 1.0, "h", "i"] and out["max"] == 16.0 and out["filled"] == [0.0, 0.0, 0.0] and out["joined"] == "1--2"
    assert out["keys"] == ["z", "y"] and out["entries"] == [["q", 1.0]] and out["isArr"] is False and out["every"] is True


def test_modules_and_errors(tmp_path):
    out, _ = run(tmp_path, """
    export * from './consts';
    export { helper as renamed } from './lib';
    import * as lib from './lib';
    import { LIMIT } from './consts';
    export function main() { return lib.helper(LIMIT) + lib.DEFAULTS.step; }
    """, {"consts.ts": "export const LIMIT = 41;\n", "lib.ts": "export function helper(v: number) { return v + 1; }\nexport const DEFAULTS = { step: 0.5 } as const;\n"})
    assert out == 42.5
    with pytest.raises(T.JSThrow) as e:
        run(tmp_path, "export function main() { const o: any = undefined; return o.x; }")
    assert "Cannot read properties of undefined" in str(e.value)
    with pytest.raises(T.JSThrow) as e:
        run(tmp_path, "export function main() { throw new Error('向量集合不能为空'); }")
    assert str(e.value) == "Error: 向量集合不能为空"
    for bad in ("export async function main() { await 1; }", "export function* main() { yield 1; }",
                "export function main() { outer: for (;;) { break outer; } }"):
        with pytest.raises(SyntaxError):
            run(tmp_path, bad)


@pytest.mark.skipif(not HAVE_REFERENCE, reason="needs a checkout of the reference project in BBQ_REFERENCE_DIR")
@pytest.mark.parametrize("name,tests", [("utils.test.ts", 27), ("computeCentroid-correctness.test.ts", 2), ("recall.test.ts", 8)])
def test_reference_own_test_files_pass_under_the_interpreter(name, tests):
    """The reference's OWN vitest files, executed against the reference's own sources by the interpreter (a minimal
    describe / it / expect in vitest_shim.py; Math.random seeded): every test in them passes.  (The performance-sized
    files — batch-*.test.ts, simple-quantized-query.test.ts, recall-all-dimensions.test.ts: thousands of 1024-d vectors —
    are not run: an interpreter in Python is the wrong tool for those.)"""
    import vitest_shim as V
    passed, failed, assertions, console = V.run_test_file(os.path.join(REFERENCE_DIR, "tests", name))
    assert not failed, failed[:3]
    assert len(passed) == tests and assertions > 0
