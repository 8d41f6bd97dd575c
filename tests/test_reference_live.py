"""Randomised differential tests of the Python host mirror against the reference's own helper code, executed live by
oracle/jsmini.py.  Needs a checkout of the reference's sources, named by $SP_REFERENCE (its lib/ directory, as for
tools/make_ref_golden.py), and is skipped without one.  Nothing else in the suite replaces these comparisons: the stored
reference answers of tests/test_reference_js.py hold far fewer helper inputs (11 file names, 26 lookup keys, 6 slice
cases) and no worker message with n = 2 or 4, a single frame or a capture shorter than one frame.  Storing the
reference's answers to the seeded inputs below needs one run against that checkout."""
import os
import random

import numpy as np
import pytest

REFERENCE = os.environ.get("SP_REFERENCE", "")
pytestmark = pytest.mark.skipif(not os.path.isdir(REFERENCE), reason="needs the reference sources ($SP_REFERENCE)")


@pytest.fixture(scope="module")
def js():
    from oracle.jsmini import Interp
    return Interp(REFERENCE)


def test_parse_freq_rate_random_names(js):
    from oracle.jsmini import UNDEF
    from spectro_b200 import parse_freq_rate as P
    m = js.load_module("./parseFreqRate", REFERENCE)
    rnd = random.Random(20261017)
    parts = ["g", "001", "433.92M", "868M", "250k", "1024k", "2.4K", "10.7m", "x", "1e3k", "-", "_", ".", " ", "/", "cu8", "cs16", "CF32", "wav", "3.5", "0", "M", "k", "7.", ".5M"]
    for _ in range(400):
        name = "".join(rnd.choice(parts) + rnd.choice(["_", "-", ".", "", " ", "/"]) for _ in range(rnd.randint(0, 7)))
        assert P.parseFreqRate(name) == js.to_py(js.call(m["parseFreqRate"], UNDEF, [name])), name
        assert P.parseFormat(name) == js.to_py(js.call(m["parseFormat"], UNDEF, [name])), name


def test_lookup_random_keys(js):
    from oracle.jsmini import UNDEF, JSObject
    from spectro_b200 import utils
    lookup = js.load_module("./utils", REFERENCE)["lookup"]
    names = ["rectangularWindow", "bartlettWindow", "hammingWindow", "hannWindow", "blackmanWindow", "blackmanHarrisWindow",
             "cube1_cmap", "viridis_cmap", "hot_cmap", "afmhot_cmap", "gist_heat_cmap", "parabola_cmap", "sox_cmap", "naive_cmap"]
    tab = JSObject(js.object_proto)
    for k in names:
        tab.props[k] = k
    py_tab = {k: k for k in names}
    rnd = random.Random(7)
    for _ in range(500):
        base = rnd.choice(names)
        key = base[:rnd.randint(0, len(base))]
        key = "".join(c.upper() if rnd.random() < 0.3 else c for c in key) + rnd.choice(["", "", "x", "_"])
        got = js.to_py(js.call(lookup, UNDEF, [tab, key]))
        assert utils.lookup(py_tab, key) == got, key


def test_windows_random_sizes(js):
    from oracle.jsmini import UNDEF
    from spectro_b200 import windows
    m = js.load_module("./windows", REFERENCE)
    rnd = random.Random(3)
    for kind in ("rectangular", "bartlett", "hamming", "hann", "blackman", "blackmanHarris"):
        for n in (2, 3, 5, 16, 100, rnd.randint(6, 600), 1 << rnd.randint(3, 11)):
            r = js.call(m[kind + "Window"], UNDEF, [n])
            ref_w, ref_weight = js.to_py(js.get_prop(r, "window")), js.get_prop(r, "weight")
            mine = getattr(windows, kind + "Window")(n)
            assert mine["weight"] == ref_weight and list(mine["window"]) == ref_w, (kind, n)


def test_sampleview_decode_and_slice_random(js):
    from oracle.jsmini import UNDEF
    from oracle import oracle as O
    from spectro_b200.samples import SampleView
    SV = js.load_module("./samples", REFERENCE)["default"]
    rnd = random.Random(11)
    for fmt in ("CU4", "CS4", "CU8", "CS8", "CU12", "CS12", "CU16", "CS16", "CU32", "CS32", "CF32", "CU64", "CS64", "CF64"):
        sw = SampleView(fmt).sampleWidth
        count = rnd.randint(5, 40)
        raw = bytes(rnd.randrange(256) for _ in range(sw * count))
        if fmt in ("CF32", "CF64"):                      # keep the floats finite
            raw = np.random.default_rng(5).standard_normal(2 * count).astype("<f4" if fmt == "CF32" else "<f8").tobytes()
        sv = js.construct(SV, [fmt, js.from_py(raw)])
        ref = [[js.call(js.get_prop(sv, "sampleI"), sv, [i]), js.call(js.get_prop(sv, "sampleQ"), sv, [i])] for i in range(count)]
        assert np.array_equal(O.decode(fmt, raw), np.array(ref, np.float64)), fmt
        py = SampleView(fmt, raw)
        for _ in range(5):
            k = rnd.randint(1, 6)
            end = int(len(raw) / sw)
            for i in range(k):
                b = js.call(js.get_prop(sv, "slice"), sv, [i, k, 0, end])
                assert bytes(py.slice(i, k, 0, end)) == bytes(b.data), (fmt, i, k)


def test_worker_random_messages_equal_the_oracle():
    """Seeded random worker messages (format, N <= 256, width, hop, window, gain, range, colormap length, channel mode,
    waterfall, ragged tails, occasional NaN / silence) through the reference's unmodified lib/worker.js and through the C
    oracle: every reply field must be identical."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "tools"))
    from make_ref_golden import RefWorker, hist_to_np, injective_cmap
    from oracle import oracle as O
    from spectro_b200.samples import SampleView
    W = RefWorker()
    I = W.I
    rnd = random.Random(424242)
    fmts = list(O.FORMATS)
    wins = ["rectangular", "bartlett", "hamming", "hann", "blackman", "blackmanHarris"]
    checked = 0
    for case in range(70):
        fmt = rnd.choice(fmts)
        n = 1 << rnd.randint(3, 8)
        width = rnd.choice([2, 3, 5, 8, 13, 24, 33])
        hop = rnd.choice([0.0, 0.4, 1.0, 1.0, 2.3])
        S = n + int(hop * n * (width - 1)) + rnd.randint(0, 9)
        buf = bytearray(O.synth(fmt, 0, S, S, 1000 + case).tobytes())
        sv = SampleView(fmt)
        if rnd.random() < 0.2 and sv.sampleWidth > sv.elementSize:
            del buf[-sv.elementSize:]                                  # ragged tail (fractional sampleCount)
        if fmt == "CF32" and rnd.random() < 0.3:
            a = np.frombuffer(bytes(buf), "<f4").copy(); a[rnd.randrange(len(a))] = np.nan; buf = bytearray(a.tobytes())
        if rnd.random() < 0.1:
            buf = bytearray(len(buf))                                  # silence: log10(0)
        if len(buf) / sv.sampleWidth < n:
            continue
        window = rnd.choice(wins)
        gain, rng = rnd.choice([-10, 0, 6, 25]), rnd.choice([6, 30, 90, -30])
        cm = injective_cmap(rnd.choice([2, 64, 256, 300]))
        chm, wf = rnd.random() < 0.25, rnd.random() < 0.25
        windowc, weight = W.window(window, n)
        jcm = W.cmap(cm)
        r = W.post(dict(block_norm=1.0 / weight, gain=gain, range=rng, cmap=jcm, n=n, windowc=windowc, width=width, offset=case,
                        buffer=I.from_py(bytes(buf)), format=fmt, channelMode=chm, waterfall=wf))
        g = lambda k: I.get_prop(r, k)
        cmb = np.array(I.to_py(jcm), np.uint8)
        o = O.render(bytes(buf), fmt, n, width, np.array(I.to_py(windowc), np.float64), 1.0 / weight, gain, rng, cmb, chm, wf)
        label = (case, fmt, n, width, window, gain, rng, len(cm), chm, wf)
        assert np.array_equal(I.get_prop(g("imageData"), "data").arr, o.image.reshape(-1)), label
        assert np.array_equal(hist_to_np(I, g("cB_hist"))[0], o.cB_hist.astype(np.float64)), label
        assert np.array_equal(hist_to_np(I, g("c_hist"))[0], o.c_hist.astype(np.float64)), label
        for k in ("gauge_mins", "gauge_maxs", "gauge_amps"):
            assert np.array_equal(g(k).arr, getattr(o, k)), label + (k,)
        for k in ("dBfs_min", "dBfs_max"):
            a, b = float(g(k)), float(getattr(o, k))
            assert a == b or (a != a and b != b), label + (k, a, b)
        assert g("offset") == case
        checked += 1
    assert checked >= 60


def test_worker_degenerate_messages_equal_the_oracle():
    """Messages outside the worker's comfortable domain that the reference nevertheless answers (it never throws):
    one frame (stride = x/0), captures shorter than one frame (every frame reads `undefined`), n = 2 and 4."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "tools"))
    from make_ref_golden import RefWorker, hist_to_np, injective_cmap
    from oracle import oracle as O
    W = RefWorker()
    I = W.I
    cases = [("CU8", 8, 1, 8), ("CU8", 8, 1, 20), ("CS16", 16, 4, 10), ("CF32", 32, 3, 5), ("CS8", 64, 2, 63),
             ("CU8", 2, 7, 30), ("CS16", 4, 5, 21), ("CF32", 2, 2, 2), ("CU4", 4, 1, 3), ("CS12", 16, 3, 16)]
    for k, (fmt, n, width, S) in enumerate(cases):
        buf = O.synth(fmt, 0, S, S, 77 + k).tobytes()
        windowc, weight = W.window("hann" if n > 2 else "rectangular", n)
        cm = injective_cmap(256)
        jcm = W.cmap(cm)
        r = W.post(dict(block_norm=1.0 / weight, gain=6, range=30, cmap=jcm, n=n, windowc=windowc, width=width, offset=k,
                        buffer=I.from_py(buf), format=fmt, channelMode=False, waterfall=False))
        g = lambda key: I.get_prop(r, key)
        cmb = np.array(I.to_py(jcm), np.uint8)
        o = O.render(buf, fmt, n, width, np.array(I.to_py(windowc), np.float64), 1.0 / weight, 6, 30, cmb)
        label = (fmt, n, width, S)
        assert np.array_equal(I.get_prop(g("imageData"), "data").arr, o.image.reshape(-1)), label
        assert np.array_equal(hist_to_np(I, g("cB_hist"))[0], o.cB_hist.astype(np.float64)), label
        assert np.array_equal(hist_to_np(I, g("c_hist"))[0], o.c_hist.astype(np.float64)), label
        for key in ("gauge_mins", "gauge_maxs", "gauge_amps"):
            assert np.array_equal(g(key).arr, getattr(o, key)), label + (key,)
        for key in ("dBfs_min", "dBfs_max"):
            a, b = float(g(key)), float(getattr(o, key))
            assert a == b or (a != a and b != b), label + (key, a, b)
