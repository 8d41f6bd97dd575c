"""Conformance checks of oracle/jsmini.py — the interpreter that runs the reference's JavaScript for the parity pin.
Every expectation below is what ECMAScript specifies (and what V8 prints); the cases concentrate on the semantics the
reference's render path leans on: ToInt32 (`~~x`, shifts), typed-array stores, sparse / non-index array keys, number
formatting of property keys, automatic semicolon insertion, hoisting, closures, classes, modules' building blocks."""
import math

import numpy as np
import pytest

from oracle.jsmini import Interp, UNDEF, JSThrow


def run(src):
    I = Interp()
    env = I.run_source(src)
    I.drain()
    return I, env.vars


def val(expr, prelude=""):
    I, v = run(prelude + "\nvar __r = (" + expr + ")")
    return I.to_py(v["__r"])


@pytest.mark.parametrize("expr,expected", [
    ("~~3.7", 3), ("~~-3.7", -3), ("~~NaN", 0), ("~~Infinity", 0), ("~~-Infinity", 0), ("~~2147483648", -2147483648),
    ("~~-2147483649", 2147483647), ("~~4294967301", 5), ("~~(0.5 + 2.5)", 3), ("~~(0.5 + -0.6)", 0), ("~~undefined", 0),
    ("1 << 31", -2147483648), ("(1 << 31) >> 31", -1), ("(1 << 31) >>> 31", 1), ("-1 >>> 0", 4294967295), ("-1 >>> 28", 15),
    ("(0xf0 << 24) >> 28", -1), ("((0x8f & 0x0f) << 28) >> 28", -1), ("5 & 3", 1), ("5 | 3", 7), ("5 ^ 3", 6), ("~5", -6),
    ("1 << 32", 1), ("2 ** 31", 2147483648), ("7 / 2", 3.5), ("-7 % 3", -1), ("7 % -3", 1), ("5.5 % 2", 1.5),
    ("1 / 0", math.inf), ("-1 / 0", -math.inf), ("0.1 + 0.2", 0.30000000000000004), ("3 * '4'", 12), ("'3' + 4", "34"),
    ("1 + undefined !== 1 + undefined", True), ("null + 1", 1), ("true + 1", 2), ("[] + 1", "1"), ("+'0x10'", 16), ("+''", 0),
    ("typeof null", "object"), ("typeof undefined", "undefined"), ("typeof (() => 1)", "function"), ("typeof 1", "number"),
    ("null == undefined", True), ("null === undefined", False), ("'1' == 1", True), ("0 == ''", True), ("NaN == NaN", False),
    ("1 < 2 < 3", True), ("3 > 2 > 1", False), ("'b' > 'a'", True), ("undefined < 1", False), ("null >= 0", True),
    ("0 || 'x'", "x"), ("0 && 'x'", 0), ("null ?? 5", 5), ("0 ?? 5", 0), ("!''", True), ("!!NaN", False),
    ("Math.round(2.5)", 3), ("Math.round(-2.5)", -2), ("Math.round(0.49999999999999994)", 0), ("Math.max()", -math.inf),
    ("Math.min(1, NaN) !== Math.min(1, NaN)", True), ("Math.log10(0)", -math.inf), ("Math.log10(1000)", 3),
    ("Math.log10(-1) !== Math.log10(-1)", True), ("Math.abs(-0.5)", 0.5), ("Math.floor(-0.5)", -1), ("Math.sign(-3)", -1),
    ("parseInt('512px', 10)", 512), ("parseInt('abc', 10) || 30", 30), ("parseInt('0', 10) || 7", 7), ("parseFloat('433.92M')", 433.92),
    ("parseFloat('1e3k')", 1000), ("isNaN(parseFloat('x'))", True), ("(1234.5678).toFixed(2)", "1234.57"), ("(255).toString(16)", "ff"),
    ("'abc'.toUpperCase() + 'DEF'.toLowerCase()", "ABCdef"), ("'a.b.c'.lastIndexOf('.')", 3), ("'hello'.substr(1, 3)", "ell"),
    ("'hello'.substr(2)", "llo"), ("'hannWindow'.toLowerCase().startsWith('hann')", True), ("'x'[5] === undefined", True),
    ("`a${1 + 1}b${'c'}`", "a2bc"), ("[1, 2, 3].map(x => x * 2).join('-')", "2-4-6"), ("[3, 1, 2].sort().join()", "1,2,3"),
    ("[1, 2, 3].reduce((a, b) => a + b)", 6), ("[1, [2, 3]].length", 2), ("Array.isArray([])", True), ("[...[1, 2], 3].length", 3),
    ("Object.keys({b: 1, a: 2}).join()", "b,a"), ("'x' in {x: 1}", True), ("({a: 1}).hasOwnProperty('a')", True),
])
def test_expressions(expr, expected):
    got = val(expr)
    if isinstance(expected, float) and not math.isinf(expected):
        assert got == expected and isinstance(got, (int, float))
    else:
        assert got == expected and type(got) is type(expected) or (got == expected and isinstance(expected, (int, float)))


def test_arrays_sparse_and_non_index_keys():
    I, v = run("""
        var h = new Array(5).fill(0)
        h[-3] += 1            // a property named "-3", not an element: undefined + 1 = NaN
        h[NaN] = 7
        h[2.0] += 1
        h[7] = 1              // grows the array, holes read as undefined
        var hole = h[5], len = h.length, neg = h[-3], keys = []
        for (var k in h) keys.push(k)
        var a = new Array(3); var filled = a.fill(0).length
        var empty = new Array(2); var und = empty[0] === undefined
    """)
    assert v["hole"] is UNDEF and v["len"] == 8 and v["neg"] != v["neg"]
    assert I.to_py(v["keys"])[:8] == ["0", "1", "2", "3", "4", "5", "6", "7"] and set(I.to_py(v["keys"])[8:]) == {"-3", "NaN"}
    assert I.to_py(v["h"])[2] == 1 and v["filled"] == 3 and v["und"] is True


def test_typed_arrays_store_conversions():
    I, v = run("""
        var c = new Uint8ClampedArray(8)
        c[0] = 0.5; c[1] = 1.5; c[2] = 2.5; c[3] = -7; c[4] = 300; c[5] = NaN; c[6] = 254.5; c[7] = -Infinity
        var u = new Uint8Array(3); u[0] = 257; u[1] = -1; u[2] = 3.9
        var s = new Int16Array(new ArrayBuffer(4)); s[0] = 40000; s[1] = -1
        var f = new Float32Array(1); f[0] = 0.1
        var oob = c[8], sl = new ArrayBuffer(10).slice(2, 6).byteLength
        var view = new Uint8Array(new Uint16Array([0x1234]).buffer)
        var threw = false
        try { new Int16Array(new ArrayBuffer(3)) } catch (e) { threw = true }
    """)
    assert list(v["c"].arr) == [0, 2, 2, 0, 255, 0, 254, 0]            # round half to even, clamp, NaN -> 0
    assert list(v["u"].arr) == [1, 255, 3] and list(v["s"].arr) == [-25536, -1]
    assert float(v["f"].arr[0]) == float(np.float32(0.1)) and v["oob"] is UNDEF and v["sl"] == 4
    assert list(v["view"].arr) == [0x34, 0x12] and v["threw"] is True     # little endian; RangeError on odd byte length


def test_asi_hoisting_closures_classes():
    I, v = run("""
        const a = 1
        const b = a
            + 2                       // continuation line: no semicolon inserted
        let c = b
        ++c
        var early = hoisted()         // function declarations are hoisted
        function hoisted() { return typeof later }      // var is hoisted as undefined
        var later = 5
        function counter() { let n = 0; return () => ++n }
        const k = counter(); k(); k()
        var kv = k()
        class P {
            constructor(x) { this.x = x }
            get double() { return this.x * 2 }
            add(y = 10, ...rest) { return this.x + y + rest.length }
            static make() { return new P(7) }
        }
        var p = P.make()
        var r = [p.double, p.add(), p.add(1, 2, 3), p instanceof P, typeof P]
        function args() { return arguments.length + arguments[1] }
        var ar = args(5, 6, 7)
        var ret = (function () { return
            42 })()                    // `return` + newline returns undefined
        var sw = (function (x) { switch (x) { case 1: return 'one'; case 2: case 3: return 'few'; default: return 'many' } })
        var sws = [sw(1), sw(3), sw(9)]
        var fin = []
        try { try { throw 'boom' } finally { fin.push('f') } } catch (e) { fin.push(e) }
        var obj = { m() { return this.v }, v: 3, ['k' + 1]: 4 }
        const { v: vv, k1 } = obj
        var lab = 0
        for (let i = 0, j = 10; i < j; i++, j--) { if (i == 2) continue; if (i == 4) break; lab += i }
    """)
    assert v["b"] == 3 and v["c"] == 4 and v["early"] == "undefined" and v["kv"] == 3
    assert I.to_py(v["r"]) == [14, 17, 10, True, "function"] and v["ar"] == 9 and v["ret"] is UNDEF
    assert I.to_py(v["sws"]) == ["one", "few", "many"] and I.to_py(v["fin"]) == ["f", "boom"]
    assert v["vv"] == 3 and v["k1"] == 4 and v["lab"] == 0 + 1 + 3


def test_promises_run_after_the_current_job():
    I, v = run("""
        var log = []
        Promise.resolve(1).then(x => { log.push('then ' + x); return x + 1 }).then(x => log.push('then ' + x))
        new Promise((res, rej) => rej('no')).catch(e => log.push('caught ' + e))
        Promise.all([1, Promise.resolve(2)]).then(a => log.push('all ' + a.length))
        log.push('sync')
    """)
    assert I.to_py(v["log"])[0] == "sync" and set(I.to_py(v["log"])) == {"sync", "then 1", "then 2", "caught no", "all 2"}


def test_errors_are_js_errors():
    with pytest.raises(JSThrow):
        run("undefinedFunction()")
    with pytest.raises(JSThrow):
        run("var x = null; x.y")
    with pytest.raises(JSThrow, match="Length"):
        run("throw 'Length is not a power of 2'")
    with pytest.raises(SyntaxError):
        run("var = 3")
