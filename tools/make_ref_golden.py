"""Generate tests/golden/ref_js/*: outputs of the REFERENCE'S OWN SOURCE for the render path.

The reference is browser JavaScript and the image has no JS engine, so its unmodified files are executed by
oracle/jsmini.py (an ES-subset interpreter written for this purpose, test infrastructure only):

  lib/worker.js (+ lib/samples.js, lib/fft_nayuki.js, lib/polyfill.js)  -> one reply per request message
  lib/windows.js, lib/*cmap.js                                           -> `windowc`, `block_norm`, `cmap` of the message
  lib/utils.js (lookup), lib/parseFreqRate.js, SampleView.slice          -> host-helper known answers (ref_host.json)

The only caller-side lines restated here are the ones that build the message from those parts
(lib/spectroplot.js:1114-1116 block_norm = 1/weight, :1129-1130 cmap end points, :1213-1226 the message fields),
because lib/spectroplot.js itself needs a DOM.  The reference's lib/ directory ($SP_REFERENCE) is read at generation time
only; the fixtures and this script are committed, the tests never need it.  Re-run:  SP_REFERENCE=<reference>/lib python tools/make_ref_golden.py
"""
import hashlib
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
from oracle import oracle as O
from oracle.jsmini import Interp, JSObject, NativeFunction, UNDEF

REF = os.environ.get("SP_REFERENCE", "")
OUT = os.path.join(ROOT, "tests", "golden", "ref_js")


class RefWorker:
    """lib/worker.js loaded as a module into a worker-like global scope (onmessage / postMessage / self)."""

    def __init__(self):
        self.I = I = Interp(REF)
        G = I.globals.vars
        self.replies = []
        G["onmessage"] = None
        G["self"] = JSObject(I.object_proto)             # no self.performance -> the timing branch is skipped
        G["postMessage"] = NativeFunction(I, "postMessage", lambda t, a: (self.replies.append((a[0], a[1] if len(a) > 1 else None)), UNDEF)[1])
        I.load_module("./worker", REF)
        self.onmessage = G["onmessage"]
        self.windows = I.load_module("./windows", REF)
        self.cmaps = {}
        for m in ("cube1cmap", "matplotlibcmaps", "parabolacmap", "soxcmap", "naivecmap"):
            self.cmaps.update(I.load_module("./" + m, REF))

    def window(self, kind, n):
        r = self.I.call(self.windows[kind + "Window"], UNDEF, [n])
        return self.I.get_prop(r, "window"), self.I.get_prop(r, "weight")

    def cmap(self, name_or_table):
        """-> JS array of [r,g,b] with the end points overwritten (lib/spectroplot.js:1129-1130)."""
        I = self.I
        tab = self.I.to_py(self.cmaps[name_or_table + "_cmap"]) if isinstance(name_or_table, str) else [list(map(int, c)) for c in name_or_table]
        js = I.from_py(tab)
        js.list[0] = I.from_py([0, 0, 0])
        js.list[len(js.list) - 1] = I.from_py([255, 255, 255])
        return js

    def post(self, fields):
        I = self.I
        msg = JSObject(I.object_proto)
        for k, v in fields.items():
            msg.props[k] = v
        ev = JSObject(I.object_proto)
        ev.props["data"] = msg
        n0 = len(self.replies)
        I.call(self.onmessage, UNDEF, [ev])
        assert len(self.replies) == n0 + 1, "exactly one reply per request (lib/worker.js:140)"
        return self.replies[-1][0]


def hist_to_np(I, arr):
    """JS Array of counts -> (float64 values, {non-index property: value})."""
    vals = np.array([float("nan") if (x is UNDEF or x is None) else float(x) for x in arr.list], np.float64)
    extra = {k: (None if v != v else v) for k, v in arr.props.items()}
    return vals, extra


def injective_cmap(n):
    i = np.arange(n)
    return np.stack([i & 255, (i * 7 + 3) & 255, ((i >> 8) * 16 + (i * 37 & 15)) & 255], 1).astype(np.uint8)


def run_case(W, name, fmt, n, width, window, cmap, gain, rng, buf, channel_mode=False, waterfall=False, recipe=None):
    """recipe = (format, samples, seed) of a capture that is synth()'s output: the fixture stores it and the SHA-256 of the
    bytes instead of the bytes (tests/helpers.py load_fixture regenerates them), which keeps every file under 1 MB."""
    I = W.I
    t0 = time.time()
    windowc, weight = W.window(window, n)
    cm = W.cmap(cmap)
    fields = dict(block_norm=1.0 / weight, gain=gain, range=rng, cmap=cm, n=n, windowc=windowc, width=width, offset=7,
                  buffer=I.from_py(bytes(buf)), format=fmt, channelMode=channel_mode, waterfall=waterfall)   # lib/spectroplot.js:1213-1226
    r = W.post(fields)
    g = lambda k: I.get_prop(r, k)
    cB, cB_x = hist_to_np(I, g("cB_hist"))
    ch, ch_x = hist_to_np(I, g("c_hist"))
    img = I.get_prop(g("imageData"), "data").arr.copy()
    assert img.size == 4 * width * n
    os.makedirs(OUT, exist_ok=True)
    if recipe is not None:
        assert bytes(buf) == synth(*recipe), name
        cap = dict(synth_fmt=recipe[0], synth_samples=recipe[1], synth_seed=recipe[2], buf_sha256=hashlib.sha256(bytes(buf)).hexdigest())
    else:
        cap = dict(buf=np.frombuffer(bytes(buf), np.uint8))
    np.savez_compressed(
        os.path.join(OUT, name + ".npz"), **cap, fmt=fmt, n=n, width=width, window=window,
        windowc=np.array(I.to_py(windowc), np.float64), weight=float(weight), gain=gain, range=rng,
        cmap_name=cmap if isinstance(cmap, str) else "custom", cmap=np.array(I.to_py(cm), np.uint8),
        channel_mode=channel_mode, waterfall=waterfall, image=img, cB_hist=cB, cB_extra=json.dumps(cB_x), c_hist=ch,
        c_extra=json.dumps(ch_x), gauge_mins=g("gauge_mins").arr.copy(), gauge_maxs=g("gauge_maxs").arr.copy(),
        gauge_amps=g("gauge_amps").arr.copy(), dBfs_min=float(g("dBfs_min")), dBfs_max=float(g("dBfs_max")), offset=int(g("offset")))
    print("%-34s %5.1f s  dBfs %.4f .. %.4f  extra cB keys %s" % (name, time.time() - t0, g("dBfs_min"), g("dBfs_max"), list(cB_x)[:4]), flush=True)


def synth(fmt, S, seed):
    return O.synth(fmt, 0, S, S, seed).tobytes()


def render_cases(W):
    cm256, cm64, cm1000 = injective_cmap(256), injective_cmap(64), injective_cmap(1000)
    # ---- BASELINE shapes at fixture size
    run_case(W, "cu8_n1024_hann_cube1_w12", "CU8", 1024, 12, "hann", "cube1", 6, 30, synth("CU8", 1024 + 700 * 11 + 3, 0x5EC70101))
    run_case(W, "cs16_n4096_bh_viridis_w8", "CS16", 4096, 8, "blackmanHarris", "viridis", 6, 30, synth("CS16", 4096 * 8, 0x5EC70102))
    run_case(W, "cs16_n4096_hann_inj_w9", "CS16", 4096, 9, "hann", cm256, 6, 30, synth("CS16", 4096 * 6 + 1234, 0x5EC70103))
    run_case(W, "cf32_n8192_hann_inferno_w4", "CF32", 8192, 4, "hann", "inferno", 6, 30, synth("CF32", 8192 * 4, 0x5EC70104))
    run_case(W, "cf32_n32768_hann_inj_w3", "CF32", 32768, 3, "hann", cm256, 6, 30, synth("CF32", 32768 * 2 + 999, 0x5EC70105))
    run_case(W, "cf32_n65536_bh_viridis_w2", "CF32", 65536, 2, "blackmanHarris", "viridis", 6, 30, synth("CF32", 65536 * 2, 0x5EC70106),
             recipe=("CF32", 65536 * 2, 0x5EC70106))
    # ---- every format, every window, every colormap family
    run_case(W, "cu4_n64_rect_naive_w9", "CU4", 64, 9, "rectangular", "naive", 6, 30, synth("CU4", 700, 0x5EC70107))
    run_case(W, "cs4_n128_bartlett_sox_w20", "CS4", 128, 20, "bartlett", "sox", 6, 30, synth("CS4", 128 * 12 + 5, 0x5EC70108))
    run_case(W, "cs8_n128_rect_magma_w33_split", "CS8", 128, 33, "rectangular", "magma", 10, 40, synth("CS8", 5000, 0x5EC70109), channel_mode=True)
    run_case(W, "cu12_n512_blackman_parabola_w10", "CU12", 512, 10, "blackman", "parabola", 6, 30, synth("CU12", 512 * 7, 0x5EC7010A))
    run_case(W, "cs12_n256_hamming_hot_w7", "CS12", 256, 7, "hamming", "hot", 0, 60, synth("CS12", 3000, 0x5EC7010B))
    run_case(W, "cu16_n32_hann_afmhot_w11", "CU16", 32, 11, "hann", "afmhot", 6, 30, synth("CU16", 400, 0x5EC7010C))
    run_case(W, "cu32_n16_hann_gist_heat_w6", "CU32", 16, 6, "hann", "gist_heat", 6, 30, synth("CU32", 120, 0x5EC7010D))
    run_case(W, "cs32_n16_bh_plasma_w6", "CS32", 16, 6, "blackmanHarris", "plasma", 6, 30, synth("CS32", 120, 0x5EC7010E))
    run_case(W, "cu64_n8_hann_grayscale_w5", "CU64", 8, 5, "hann", "grayscale", 6, 30, synth("CU64", 60, 0x5EC7010F))
    run_case(W, "cs64_n8_hann_roentgen_w5", "CS64", 8, 5, "hann", "roentgen", 6, 30, synth("CS64", 60, 0x5EC70110))
    run_case(W, "cf64_n64_hann_phosphor_w8", "CF64", 64, 8, "hann", "phosphor", 6, 30, synth("CF64", 600, 0x5EC70111))
    run_case(W, "cf32_n256_hamming_inj_w10_wf", "CF32", 256, 10, "hamming", cm256, 0, 60, synth("CF32", 2600, 0x5EC70112), waterfall=True)
    run_case(W, "cs16_n2048_blackman_inj64_w5_wf_split", "CS16", 2048, 5, "blackman", cm64, 6, 30, synth("CS16", 2048 * 4, 0x5EC70113), channel_mode=True, waterfall=True)
    run_case(W, "cu8_n256_hann_inj1000_w6", "CU8", 256, 6, "hann", cm1000, 6, 30, synth("CU8", 2000, 0x5EC70114))
    # aliases and the unknown-format default (lib/samples.js:30-155)
    run_case(W, "alias_complex16s_n64_w5", "complex16s", 64, 5, "hann", "cube1", 6, 30, synth("CS8", 500, 0x5EC70115))
    run_case(W, "alias_cfile_n64_w5", "CFILE", 64, 5, "hann", "cube1", 6, 30, synth("CF32", 500, 0x5EC70116))
    run_case(W, "unknown_fmt_defaults_to_cu8_n64_w5", "XYZ", 64, 5, "hann", "cube1", 6, 30, synth("CU8", 500, 0x5EC70117))
    # ---- strides: overlapping, skipping, minimum width; gain / range corners
    run_case(W, "cu8_n256_overlap_w40", "CU8", 256, 40, "hann", cm256, 6, 30, synth("CU8", 1500, 0x5EC70118))
    run_case(W, "cu8_n256_skip_w5", "CU8", 256, 5, "hann", cm256, 6, 30, synth("CU8", 256 * 40 + 17, 0x5EC70119))
    run_case(W, "cs16_n128_w2", "CS16", 128, 2, "hann", cm256, 6, 30, synth("CS16", 1000, 0x5EC7011A))
    run_case(W, "cs16_n128_gain0_range90", "CS16", 128, 7, "hann", cm256, 0, 90, synth("CS16", 1000, 0x5EC7011B))
    run_case(W, "cs16_n128_gain30_range6", "CS16", 128, 7, "hann", cm256, 30, 6, synth("CS16", 1000, 0x5EC7011C))
    run_case(W, "cs16_n128_range_negative", "CS16", 128, 7, "hann", cm256, 6, -30, synth("CS16", 1000, 0x5EC7011D))
    # ---- ragged buffers (byteLength not a multiple of the sample width: fractional sampleCount, `undefined` reads)
    run_case(W, "cu8_n64_ragged_odd_bytes", "CU8", 64, 6, "hann", cm256, 6, 30, synth("CU8", 301, 0x5EC7011E)[:-1])
    run_case(W, "cu12_n32_ragged", "CU12", 32, 6, "hann", cm256, 6, 30, synth("CU12", 200, 0x5EC7011F)[:-2])
    run_case(W, "cs16_n64_ragged_half_sample", "CS16", 64, 6, "hann", cm256, 6, 30, synth("CS16", 301, 0x5EC70120)[:-2])
    # ---- special values: silence (log10(0) = -inf), NaN / inf input, levels above 0 dBFS (negative histogram index)
    run_case(W, "cs16_n64_zeros", "CS16", 64, 4, "hann", cm256, 6, 30, bytes(4 * 64 * 4))
    x = np.frombuffer(synth("CF32", 64 * 6, 0x5EC70121), "<f4").copy()
    x[2 * 70] = np.nan; x[2 * 200 + 1] = np.inf; x[2 * 330] = -np.inf
    run_case(W, "cf32_n64_nan_inf", "CF32", 64, 6, "hann", cm256, 6, 30, x.tobytes())
    y = (np.frombuffer(synth("CF32", 64 * 6, 0x5EC70122), "<f4") * 6.0).astype("<f4")
    run_case(W, "cf32_n64_above_0dbfs", "CF32", 64, 6, "rectangular", cm256, 6, 30, y.tobytes())
    z = np.zeros(2 * 64 * 3, "<f4"); z[0::2] = 1.0                       # full-scale DC, rectangular: bin 0 at exactly 0 dB
    run_case(W, "cf32_n64_fullscale_dc", "CF32", 64, 3, "rectangular", cm256, 0, 30, z.tobytes())


def host_fixtures(W):
    I = W.I
    out = {}
    out["windows"] = {}
    for kind in ("rectangular", "bartlett", "hamming", "hann", "blackman", "blackmanHarris"):
        for n in (8, 64, 1000, 4096):
            w, weight = W.window(kind, n)
            out["windows"]["%s/%d" % (kind, n)] = dict(weight=weight, window=I.to_py(w) if n <= 64 else None,
                                                       spot=[I.get_prop(w, i) for i in (0, 1, n // 3, n // 2, n - 1)])
    out["cmaps"] = {k: I.to_py(v) for k, v in W.cmaps.items()}
    utils = I.load_module("./utils", REF)
    tab = JSObject(I.object_proto)
    names = ["rectangularWindow", "bartlettWindow", "hammingWindow", "hannWindow", "blackmanWindow", "blackmanHarrisWindow"]
    for k in names:
        tab.props[k] = k
    ctab = JSObject(I.object_proto)
    for k in W.cmaps:                       # import order of lib/spectroplot.js is the table's key order
        ctab.props[k] = k
    keys = ["hann", "Hann", "HANN", "blackman", "blackmanHarris", "blackmanh", "ham", "rect", "bart", "nope", "", "b", "hannWindow"]
    out["lookup_windows"] = {k: I.to_py(I.call(utils["lookup"], UNDEF, [tab, k])) for k in keys}
    ckeys = ["cube1", "viridis", "hot", "parula", "sox", "naive", "gray", "mag", "Inferno", "afm", "gist", "p", "roentgen_cmap"]
    out["lookup_cmaps"] = {k: I.to_py(I.call(utils["lookup"], UNDEF, [ctab, k])) for k in ckeys}
    out["cmap_key_order"] = list(W.cmaps.keys())
    pfr = I.load_module("./parseFreqRate", REF)
    fnames = ["g001_433.92M_250k.cu8", "/a/b/test_868.3M_1000k.cs16", "x-10.7m-2.4K.cf32", "noext", "weird.name.CS8", "a_1e3k.cu8",
              "data_433M_250k_extra.cu8", "", "gfile001.data", "rtl_433_tests/tests/x/01/gfile_915M_1024k.complex16u", "a.b_3.5M.wav"]
    out["parseFreqRate"] = {f: I.to_py(I.call(pfr["parseFreqRate"], UNDEF, [f])) for f in fnames}
    out["parseFormat"] = {f: I.to_py(I.call(pfr["parseFormat"], UNDEF, [f])) for f in fnames}
    # SampleView: sampleCount and the fan-out slices (lib/samples.js:167, :253-258; lib/spectroplot.js:1206-1211)
    SV = I.load_module("./samples", REF)["default"]
    sl = {}
    for fmt, nbytes, count in (("CU8", 10000, 4), ("CS16", 10002, 3), ("CU12", 3001, 8), ("CF32", 4096, 5), ("CS4", 999, 16), ("CF64", 1600, 7)):
        sv = I.construct(SV, [fmt, I.from_py(bytes(nbytes))])
        sw = I.get_prop(sv, "sampleWidth")
        end = int(nbytes / sw)                                      # ~~(byteLength / sampleWidth)
        parts = []
        for i in range(count):
            b = I.call(I.get_prop(sv, "slice"), sv, [i, count, 0, end])
            parts.append(len(b.data))
        sl["%s/%d/%d" % (fmt, nbytes, count)] = dict(sampleWidth=sw, sampleCount=I.get_prop(sv, "sampleCount"), slice_bytes=parts)
    out["slices"] = sl
    # decode spot checks straight from SampleView.sampleI / sampleQ
    dec = {}
    for fmt in ("CU4", "CS4", "CU8", "CS8", "CU12", "CS12", "CU16", "CS16", "CU32", "CS32", "CF32", "CU64", "CS64", "CF64"):
        raw = O.synth(fmt, 0, 24, 24, 0x5EC70200).tobytes()
        sv = I.construct(SV, [fmt, I.from_py(raw)])
        vals = []
        for pos in range(24):
            vals.append([I.call(I.get_prop(sv, "sampleI"), sv, [pos]), I.call(I.get_prop(sv, "sampleQ"), sv, [pos])])
        dec[fmt] = dict(raw=list(raw), iq=vals)
    out["decode"] = dec
    # FFTNayuki: constructor error and a known transform
    FFT = I.load_module("./fft_nayuki", REF)["default"]
    try:
        I.construct(FFT, [12])
        out["fft_bad_length"] = None
    except Exception as ex:
        out["fft_bad_length"] = str(getattr(ex, "value", ex))
    f = I.construct(FFT, [16])
    re = I.from_py([math.cos(0.3 * i) + 0.01 * i for i in range(16)])
    im = I.from_py([math.sin(0.7 * i) for i in range(16)])
    out["fft16_in"] = [I.to_py(re), I.to_py(im)]
    I.call(I.get_prop(f, "transform"), f, [re, im])
    out["fft16_out"] = [I.to_py(re), I.to_py(im)]
    I.call(I.get_prop(f, "splitreal"), f, [re, im])
    out["fft16_split"] = [I.to_py(re), I.to_py(im)]
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, "ref_host.json"), "w") as fp:
        json.dump(out, fp)
    print("ref_host.json ok (%d windows, %d cmaps)" % (len(out["windows"]), len(out["cmaps"])))


def random_cases_large(W, count=16, seed=777):
    """The same at the sizes of the fused kernels (N = 1024 .. 4096: render_rc_kernel, render_r64_kernel and their waterfall /
    split-real variants), widths that leave partial tiles, ragged tails and NaN samples."""
    import random
    from spectro_b200.samples import SampleView
    rnd = random.Random(seed)
    wins = ["rectangular", "bartlett", "hamming", "hann", "blackman", "blackmanHarris"]
    for made in range(count):
        fmt = rnd.choice(["CS16", "CU8", "CF32", "CS8", "CU12", "CS4", "CU16", "CF32"])
        n = rnd.choice([1024, 2048, 4096, 4096])
        width = rnd.choice([8, 9, 12, 16, 17])
        hop = rnd.choice([0.5, 1.0, 1.0, 1.7])
        S = n + int(hop * n * (width - 1)) + rnd.randint(0, 9)
        buf = bytearray(synth(fmt, S, 0x5EC7F100 + made))
        sv = SampleView(fmt)
        ragged = rnd.random() < 0.3 and sv.sampleWidth > sv.elementSize
        if ragged:
            del buf[-sv.elementSize:]
        nan = fmt == "CF32" and rnd.random() < 0.4
        if nan:
            a = np.frombuffer(bytes(buf), "<f4").copy(); a[rnd.randrange(len(a))] = np.nan; buf = bytearray(a.tobytes())
        window, gain, rng = rnd.choice(wins), rnd.choice([0, 6, 25]), rnd.choice([30, 90, -30])
        cm = injective_cmap(rnd.choice([64, 256, 256]))
        chm, wf = rnd.random() < 0.4, rnd.random() < 0.4
        name = "big%02d_%s_n%d_w%d%s%s%s%s" % (made, fmt.lower(), n, width, "_split" if chm else "", "_wf" if wf else "",
                                             "_ragged" if ragged else "", "_nan" if nan else "")
        run_case(W, name, fmt, n, width, window, cm, gain, rng, bytes(buf), chm, wf)


def random_cases(W, count=40, seed=20261017):
    """Seeded random points of the option space at small sizes (the GPU suite has no access to the reference: these widen the
    set of reference replies it is compared with)."""
    import random
    from spectro_b200.samples import SampleView
    rnd = random.Random(seed)
    fmts = list(O.FORMATS)
    wins = ["rectangular", "bartlett", "hamming", "hann", "blackman", "blackmanHarris"]
    made = 0
    while made < count:
        fmt = rnd.choice(fmts)
        n = 1 << rnd.randint(3, 9)
        width = rnd.choice([2, 3, 5, 8, 13, 24, 33, 40])
        hop = rnd.choice([0.0, 0.4, 1.0, 1.0, 2.3])
        S = n + int(hop * n * (width - 1)) + rnd.randint(0, 9)
        buf = bytearray(synth(fmt, S, 0x5EC7F000 + made))
        sv = SampleView(fmt)
        ragged = rnd.random() < 0.2 and sv.sampleWidth > sv.elementSize
        if ragged:
            del buf[-sv.elementSize:]
        nan = fmt == "CF32" and rnd.random() < 0.3
        if nan:
            a = np.frombuffer(bytes(buf), "<f4").copy(); a[rnd.randrange(len(a))] = np.nan; buf = bytearray(a.tobytes())
        if len(buf) / sv.sampleWidth < n:
            continue
        window, gain, rng = rnd.choice(wins), rnd.choice([-10, 0, 6, 25]), rnd.choice([6, 30, 90, -30])
        cm = injective_cmap(rnd.choice([2, 64, 256, 300]))
        chm, wf = rnd.random() < 0.25, rnd.random() < 0.25
        name = "rnd%02d_%s_n%d_w%d%s%s%s%s" % (made, fmt.lower(), n, width, "_split" if chm else "", "_wf" if wf else "",
                                             "_ragged" if ragged else "", "_nan" if nan else "")
        run_case(W, name, fmt, n, width, window, cm, gain, rng, bytes(buf), chm, wf)
        made += 1


def round2_option_cases(W):
    """channelMode / turnFlip at the reference's menu sizes (lib/example.html:23-84), at widths that put whole groups of 8 frames on
    render_w_kernel (added when it took over both options from the generic kernel)."""
    cm256 = injective_cmap(256)
    run_case(W, "r2_cs16_n1024_hann_w17_split", "CS16", 1024, 17, "hann", cm256, 6, 30, synth("CS16", 1024 * 9 + 77, 0x5EC70201), channel_mode=True)
    run_case(W, "r2_cu8_n512_bh_viridis_w24_split_wf", "CU8", 512, 24, "blackmanHarris", "viridis", 6, 30, synth("CU8", 512 * 13 + 5, 0x5EC70202), channel_mode=True, waterfall=True)
    run_case(W, "r2_cf32_n256_hann_w40_split", "CF32", 256, 40, "hann", cm256, 0, 60, synth("CF32", 256 * 21 + 9, 0x5EC70203), channel_mode=True)
    run_case(W, "r2_cs16_n1024_blackman_w16_wf", "CS16", 1024, 16, "blackman", cm256, 6, 30, synth("CS16", 1024 * 16, 0x5EC70204), waterfall=True)
    run_case(W, "r2_cs8_n64_hamming_w72_wf_split", "CS8", 64, 72, "hamming", cm256, 6, 30, synth("CS8", 64 * 40 + 3, 0x5EC70205), channel_mode=True, waterfall=True)


if __name__ == "__main__":
    sys.path.insert(0, os.path.join(ROOT, "spectroplot-js_b200"))
    W = RefWorker()
    if "--round2-options" in sys.argv:
        round2_option_cases(W)
        sys.exit(0)
    if "--large-only" not in sys.argv:
        host_fixtures(W)
        render_cases(W)
        random_cases(W)
    random_cases_large(W)
