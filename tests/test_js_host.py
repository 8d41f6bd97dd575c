"""The JavaScript host layer (js/gpu_worker.js, js/spectroplot_headless.js) executed by oracle/jsmini.py.

CPU suite: the addon the JS files `require` is backed by the float64 oracle, so the protocol / controller LOGIC is
tested without a GPU (worker message protocol, FIFO replies, ignored probe, error -> onerror, format aliases, option
parsers, single flight, fan-out + merge == the reference's fan-out).  GPU suite: the same JS, the addon backed by the
C-ABI engine (sp_render), against the reference-worker fixtures."""
import glob
import os

import numpy as np
import pytest

from helpers import load_fixture
from js_host import JsHost, typed
from oracle import oracle as O
from oracle.jsmini import JSObject, JSArray, NativeFunction, UNDEF, JSThrow

REFJS = os.path.join(os.path.dirname(__file__), "golden", "ref_js")


def oracle_render(buf, fmt, n, width, windowc, block_norm, gain, rng, cmap, channel_mode, waterfall):
    r = O.render(buf, fmt, n, width, windowc, block_norm, gain, rng, cmap, channel_mode, waterfall)
    return dict(image=r.image, gauge_mins=r.gauge_mins, gauge_maxs=r.gauge_maxs, gauge_amps=r.gauge_amps,
                cB_hist=r.cB_hist, c_hist=r.c_hist, dBfs_min=r.dBfs_min, dBfs_max=r.dBfs_max)


def message(I, f, **over):
    m = dict(block_norm=1.0 / float(f["weight"]), gain=float(f["gain"]), range=float(f["range"]), n=int(f["n"]), width=int(f["width"]),
             offset=7, format=str(f["fmt"]), channelMode=bool(f["channel_mode"]), waterfall=bool(f["waterfall"]))
    m.update(over)
    msg = I.from_py(m)
    msg.props["cmap"] = I.from_py([list(map(int, c)) for c in f["cmap"]])
    msg.props["windowc"] = I.from_py(f["windowc"].tolist())
    msg.props["buffer"] = I.from_py(f["buf"].tobytes())
    return msg


def load(name):
    return load_fixture(os.path.join(REFJS, name + ".npz"))


def post(host, worker, msg):
    I = host.I
    replies, errors = [], []
    worker.props["onmessage"] = NativeFunction(I, "onmessage", lambda t, a: (replies.append(a[0]), UNDEF)[1])
    worker.props["onerror"] = NativeFunction(I, "onerror", lambda t, a: (errors.append(a[0]), UNDEF)[1])
    I.call(I.get_prop(worker, "postMessage"), worker, [msg])
    assert replies == [], "the reply must be asynchronous (after postMessage returns), like a real worker's"
    I.drain()
    return replies, errors


def check_reply(I, reply, f, exact):
    d = I.get_prop(reply, "data")
    g = lambda k: I.get_prop(d, k)
    assert g("offset") == 7
    img = I.get_prop(g("imageData"), "data")
    assert img.kind == "Uint8ClampedArray" and len(img.arr) == 4 * int(f["n"]) * int(f["width"])
    assert isinstance(g("cB_hist"), JSArray) and len(g("cB_hist").list) == 1000 and len(g("c_hist").list) == len(f["cmap"])
    assert all(isinstance(x, (int, float)) for x in g("c_hist").list)          # plain Numbers, as the reference posts them
    bad = (img.arr.reshape(-1, 4) != f["image"].reshape(-1, 4)).any(axis=1).sum()
    if exact:
        assert bad == 0 and np.array_equal(np.array(g("c_hist").list, float), f["c_hist"])
        assert np.array_equal(np.array(g("cB_hist").list, float), f["cB_hist"])
        assert g("dBfs_min") == float(f["dBfs_min"]) and g("dBfs_max") == float(f["dBfs_max"])
        for k in ("gauge_mins", "gauge_maxs", "gauge_amps"):
            assert np.array_equal(g(k).arr, f[k])
    else:
        assert bad <= max(1, int(1e-3 * int(f["n"]) * int(f["width"])))
        assert abs(g("dBfs_max") - float(f["dBfs_max"])) <= 0.01
        for k in ("gauge_mins", "gauge_maxs", "gauge_amps"):
            assert np.abs(g(k).arr.astype(int) - f[k].astype(int)).max() <= 1


# ------------------------------------------------------------------ CPU: protocol logic of js/gpu_worker.js
def test_gpu_worker_js_protocol_against_reference_replies():
    host = JsHost(oracle_render)
    I = host.I
    w = I.construct(host.GpuWorker, [3])
    assert host.log == [("create", 3)]
    # the {transferable} probe and anything without .buffer is ignored (lib/worker.js:159, lib/spectroplot.js:118-119)
    probe = I.from_py({"transferable": b"x"})
    replies, errors = post(host, w, probe)
    assert replies == [] and errors == [] and len(host.log) == 1
    for name in ("cu8_n256_overlap_w40", "cs8_n128_rect_magma_w33_split", "cf32_n256_hamming_inj_w10_wf",
                 "alias_complex16s_n64_w5", "alias_cfile_n64_w5", "unknown_fmt_defaults_to_cu8_n64_w5", "cu12_n512_blackman_parabola_w10"):
        f = load(name)
        replies, errors = post(host, w, message(I, f))
        assert len(replies) == 1 and errors == []
        check_reply(I, replies[0], f, exact=True)
    # two messages posted back to back are answered in order (FIFO per worker, lib/spectroplot.js:111-115)
    fa, fb = load("cs16_n128_w2"), load("cs16_n128_gain0_range90")
    replies = []
    w.props["onmessage"] = NativeFunction(I, "onmessage", lambda t, a: (replies.append(a[0]), UNDEF)[1])
    I.call(I.get_prop(w, "postMessage"), w, [message(I, fa, offset=1)])
    I.call(I.get_prop(w, "postMessage"), w, [message(I, fb, offset=2)])
    I.drain()
    assert [I.get_prop(I.get_prop(r, "data"), "offset") for r in replies] == [1, 2]
    I.call(I.get_prop(w, "terminate"), w, [])
    assert host.log[-1] == ("destroy", 3) and I.get_prop(w, "engine") is None


def test_gpu_worker_js_errors_go_to_onerror():
    def failing(*a):
        raise RuntimeError("SP_E_BAD_N: n must be a power of two")
    host = JsHost(failing)
    I = host.I
    w = I.construct(host.GpuWorker, [])
    replies, errors = post(host, w, message(I, load("cs16_n128_w2")))
    assert replies == [] and len(errors) == 1 and "SP_E_BAD_N" in I.get_prop(errors[0], "message")
    w.props["onerror"] = None                       # without a handler the error propagates instead of hanging the promise
    with pytest.raises(JSThrow):
        I.call(I.get_prop(w, "postMessage"), w, [message(I, load("cs16_n128_w2"))])


def test_format_ids_follow_sampleview_aliases():
    host = JsHost(oracle_render)
    fid = lambda s: host.I.call(host.formatId, UNDEF, [s])
    assert [fid(f) for f in ("cu4", "CS4", "cu8", "CS8", "CU12", "CS12", "CU16", "cs16", "CU32", "CS32", "CU64", "CS64", "cf32", "CF64")] == list(range(14))
    assert fid("data") == 2 and fid("COMPLEX16U") == 2 and fid("complex16s") == 3 and fid("cfile") == 12 and fid("COMPLEX") == 12
    assert fid("whatever") == 2 and fid("") == 2               # unknown -> CU8 (lib/samples.js:149-155)


# ------------------------------------------------------------------ CPU: js/spectroplot_headless.js over the mirrors of the reference's modules
def test_headless_spectroplot_js_matches_reference_fanout():
    host = JsHost(oracle_render)
    I = host.I
    Spectroplot = host.spectroplot_class(host.mirror_deps())
    opts = I.from_py({"fftN": "256", "windowF": "hann", "cmap": "hot", "gain": "6", "range": 30, "clientWidth": 500, "workerCount": 3})
    sp = I.construct(Spectroplot, [opts])
    g = lambda k: I.get_prop(sp, k)
    call = lambda name, *a: I.call(g(name), sp, list(a))
    assert [t for t in host.log] == [("create", 0)] * 3
    # no data yet: nothing to render, but a drop-in caller's `.then` must still work (lib/spectroplot.js:1097: Promise.resolve())
    assert host.await_(call("setOption", "fftN", 512)) is UNDEF
    assert g("fftN") == 512
    S = 30000
    buf = O.synth("CS16", 0, S, S, 9).tobytes()
    filedata = I.from_py({"name": "g001_433.92M_250k.cs16", "size": len(buf), "type": ""})
    filedata.props["fileBuffer"] = I.from_py(buf)
    res = host.await_(call("setData", filedata))
    assert g("center_freq") == 433920000.0 and g("sample_rate") == 250000.0 and g("sampleFormat") == "CS16"
    width = 500 - (40 + 60 + 100)
    assert I.get_prop(res, "width") == width == g("width") and I.get_prop(res, "height") == 512
    hot = I.to_py(host.mirror_deps().props["cmaps"].props["hot_cmap"])
    assert hot[0] == [0, 0, 0] and hot[-1] == [255, 255, 255]          # the shared table was overwritten in place (:1129-1130)
    w, wt = O.window("hann", 512)
    ora = O.render(buf, "CS16", 512, width, w, 1 / wt, 6, 30, np.array(hot, np.uint8), workers=3)
    img = I.get_prop(res, "image").arr.reshape(512, width, 4)
    assert np.array_equal(img, ora.image)
    assert np.array_equal(np.array(I.get_prop(res, "c_hist").list, np.int64), ora.c_hist.astype(np.int64))
    assert np.array_equal(np.array(I.get_prop(res, "cB_hist").list, np.int64), ora.cB_hist.astype(np.int64))
    assert I.get_prop(res, "dBfs_min") == ora.dBfs_min and I.get_prop(res, "dBfs_max") == ora.dBfs_max
    for k in ("gauge_mins", "gauge_maxs", "gauge_amps"):
        assert np.array_equal(I.get_prop(res, k).arr, getattr(ora, k))
    # single flight: a request made while one is pending returns the pending promise and is dropped (:1099)
    p1 = call("setOptions", I.from_py({"gain": "12", "cmap": "viridis", "windowF": "blackman"}))
    p2 = call("setOption", "gain", 20)
    assert p1 is p2 and g("gain") == 20
    renders_before = sum(1 for t in host.log if t[0] == "render")       # the three messages of p1 are already posted
    r1 = host.await_(p1)
    assert sum(1 for t in host.log if t[0] == "render") == renders_before == 6   # setData's 3 + p1's 3; the second request rendered nothing
    assert I.get_prop(r1, "width") == width
    assert g("inProcess") is False
    # zoom: half steps inside [1, 8] (:513-527); waterfall via turnFlip
    assert host.await_(call("zoomOut")) is UNDEF               # already at zoom 1: Promise.resolve() (:514)
    r2 = host.await_(call("zoomIn"))
    assert g("zoom") == 1.5 and I.get_prop(r2, "width") == int(500 * 1.5 - 200)
    r3 = host.await_(call("setOptions", I.from_py({"turnFlip": "flip", "zoom": "1", "fftN": "128"})))
    assert I.get_prop(r3, "waterfall") is True
    wf_width = int(3200 - 200)                                            # innerHeight stand-in
    w, wt = O.window("blackman", 128)
    vir = I.to_py(host.mirror_deps().props["cmaps"].props["viridis_cmap"])
    ora = O.render(buf, "CS16", 128, wf_width, w, 1 / wt, 20, 30, np.array(vir, np.uint8), waterfall=True, workers=3)
    assert np.array_equal(I.get_prop(r3, "image").arr, ora.image.reshape(-1))
    call("destroy")
    assert [t[0] for t in host.log[-3:]] == ["destroy"] * 3


def test_headless_spectroplot_js_rejects_instead_of_hanging():
    state = {"fail": False}

    def sometimes(*a):
        if state["fail"]:
            raise RuntimeError("SP_E_RANGE: sampleCount < n")
        return oracle_render(*a)
    host = JsHost(sometimes)
    I = host.I
    Spectroplot = host.spectroplot_class(host.mirror_deps())
    sp = I.construct(Spectroplot, [I.from_py({"fftN": 64, "clientWidth": 300, "workerCount": 2})])
    buf = O.synth("CU8", 0, 4000, 4000, 5).tobytes()
    fd = I.from_py({"name": "x_100M_1000k.cu8"})
    fd.props["fileBuffer"] = I.from_py(buf)
    state["fail"] = True
    with pytest.raises(JSThrow):
        host.await_(I.call(I.get_prop(sp, "setData"), sp, [fd]))
    assert I.get_prop(sp, "inProcess") is False                      # not stuck (the reference would be, lib/spectroplot.js:1277-1284)
    state["fail"] = False
    res = host.await_(I.call(I.get_prop(sp, "setOption"), sp, ["gain", 3]))
    assert I.get_prop(res, "width") == 100


# ------------------------------------------------------------------ GPU: the same JS over the C-ABI engine
@pytest.mark.gpu
def test_gpu_worker_js_over_the_c_abi(engine):
    def gpu_render(buf, fmt, n, width, windowc, block_norm, gain, rng, cmap, channel_mode, waterfall):
        return engine.render(buf, fmt, n, width, windowc, block_norm, gain, rng, cmap, channel_mode, waterfall)
    host = JsHost(gpu_render)
    I = host.I
    w = I.construct(host.GpuWorker, [0])
    for name in ("cu8_n1024_hann_cube1_w12", "cs16_n4096_bh_viridis_w8", "cf32_n8192_hann_inferno_w4", "cs4_n128_bartlett_sox_w20",
                 "cs16_n2048_blackman_inj64_w5_wf_split", "alias_cfile_n64_w5"):
        f = load(name)
        replies, errors = post(host, w, message(I, f))
        assert len(replies) == 1 and errors == []
        check_reply(I, replies[0], f, exact=False)
    # an engine error (n not a power of two) reaches onerror with the C ABI's message
    f = load("cs16_n128_w2")
    replies, errors = post(host, w, message(I, f, n=100))
    assert replies == [] and len(errors) == 1 and "SP_E" in I.get_prop(errors[0], "message")
    I.call(I.get_prop(w, "terminate"), w, [])
