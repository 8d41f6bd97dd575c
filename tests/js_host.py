"""Runs the repository's JavaScript host layer (spectroplot-js_b200/js/*.js) under oracle/jsmini.py (no Node.js in the
image).  The N-API addon those files `require` is replaced by an object with the same three functions
(create / render / destroy, see js/spectro_napi.c) that calls a Python render function: the C-ABI engine on a GPU
box, the float64 oracle in the CPU suite."""
import os

import numpy as np

from oracle.jsmini import Interp, JSObject, JSArray, JSTypedArray, JSArrayBuffer, NativeFunction, UNDEF, JSThrow, js_to_string

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
JS = os.path.join(ROOT, "spectroplot-js_b200", "js")
REF_HOST = os.path.join(ROOT, "tests", "golden", "ref_js", "ref_host.json")
FORMATS = ["CU4", "CS4", "CU8", "CS8", "CU12", "CS12", "CU16", "CS16", "CU32", "CS32", "CU64", "CS64", "CF32", "CF64"]


def typed(I, kind, arr):
    buf = JSArrayBuffer(I, bytearray(np.ascontiguousarray(arr).tobytes()))
    return I.construct(I.globals.vars[kind], [buf])


def make_addon(I, render_fn, log):
    """render_fn(buf, fmt, n, width, windowc, block_norm, gain, range, cmap[len,3], channel_mode, waterfall) -> dict."""
    addon = JSObject(I.object_proto)
    engines = {}

    def create(this, a):
        h = JSObject(I.object_proto)
        engines[id(h)] = int(a[0]) if a and a[0] is not UNDEF else 0
        log.append(("create", engines[id(h)]))
        return h

    def destroy(this, a):
        log.append(("destroy", engines.pop(id(a[0]), None)))
        return UNDEF

    def render(this, a):
        ctx = a[1]
        g = lambda k: I.get_prop(ctx, k)
        assert id(a[0]) in engines, "render on a destroyed engine"
        buf = g("buffer")
        assert isinstance(buf, JSArrayBuffer), "ctx.buffer must be an ArrayBuffer (napi_get_arraybuffer_info)"
        wc, cm = g("windowc"), g("cmap")
        assert isinstance(wc, JSTypedArray) and wc.kind == "Float64Array", "ctx.windowc must be a Float64Array"
        assert isinstance(cm, JSTypedArray) and cm.kind in ("Uint8Array", "Uint8ClampedArray"), "ctx.cmap must be a Uint8Array or Uint8ClampedArray(len*3)"
        n, width = int(g("n")), int(g("width"))
        log.append(("render", FORMATS[int(g("format"))], n, width))
        try:
            r = render_fn(bytes(buf.data), FORMATS[int(g("format"))], n, width, wc.arr.copy(), float(g("block_norm")), float(g("gain")),
                          float(g("range")), cm.arr.reshape(-1, 3).copy(), bool(g("channelMode")), bool(g("waterfall")))
        except Exception as ex:                      # the addon throws a JS Error with sp_last_error()
            err = JSObject(I.object_proto)
            err.props["message"] = str(ex)
            raise JSThrow(err)
        out = JSObject(I.object_proto)
        out.props["image"] = typed(I, "Uint8ClampedArray", np.asarray(r["image"], np.uint8).reshape(-1))
        for k in ("gauge_mins", "gauge_maxs", "gauge_amps"):
            out.props[k] = typed(I, "Uint8ClampedArray", np.asarray(r[k], np.uint8))
        out.props["cB_hist"] = typed(I, "BigUint64Array", np.asarray(r["cB_hist"], np.uint64))
        out.props["c_hist"] = typed(I, "BigUint64Array", np.asarray(r["c_hist"], np.uint64))
        out.props["dBfs_min"], out.props["dBfs_max"] = float(r["dBfs_min"]), float(r["dBfs_max"])
        out.props["device_ms"] = float(r.get("device_ms", 0.0))
        return out
    for name, fn in (("create", create), ("destroy", destroy), ("render", render)):
        addon.props[name] = NativeFunction(I, name, fn)
    return addon


class JsHost:
    def __init__(self, render_fn):
        self.I = I = Interp(JS)
        self.log = []
        self._deps = None
        addon = make_addon(I, render_fn, self.log)
        self.worker_mod = I.require_file(os.path.join(JS, "gpu_worker.js"), lambda spec: addon if spec.endswith("spectro_napi.node") else None)
        self.GpuWorker = I.get_prop(self.worker_mod, "GpuWorker")
        self.formatId = I.get_prop(self.worker_mod, "formatId")

    def mirror_deps(self):
        """The reference's pure modules that js/spectroplot_headless.js takes injected (windows, cmaps, lookup,
        parseFreqRate / parseFormat, SampleView), served by the package's Python mirrors of them, which
        tests/test_reference_js.py pins to the reference's own answers.  Built once per host: the cmap tables are
        shared objects that the controller overwrites in place, as the reference's are."""
        if self._deps is not None:
            return self._deps
        import json
        from spectro_b200 import cmaps, parse_freq_rate, utils, windows
        from spectro_b200.samples import SampleView
        I = self.I
        native = lambda name, fn: NativeFunction(I, name, fn)
        win = JSObject(I.object_proto)
        for kind in ("rectangular", "bartlett", "hamming", "hann", "blackman", "blackmanHarris"):   # lib/windows.js order
            fn = getattr(windows, kind + "Window")
            win.props[kind + "Window"] = native(kind + "Window", lambda t, a, fn=fn: I.from_py(fn(int(a[0]))))
        cm = JSObject(I.object_proto)
        with open(REF_HOST) as f:                     # key order of the reference's merged tables (lookup prefix matches)
            for name in json.load(f)["cmap_key_order"]:
                cm.props[name] = I.from_py([list(map(int, c)) for c in cmaps.cmaps[name]])

        def lookup(this, a):
            return utils.lookup(a[0].props, a[1] if len(a) > 1 else UNDEF)

        def sample_view(a):
            sv = SampleView(js_to_string(a[0]), None, *[None if x is UNDEF else x for x in a[2:4]])
            obj = JSObject(I.object_proto)

            def sync():
                obj.props.update(format=sv.format, sampleWidth=sv.sampleWidth, sampleRate=sv.sampleRate, sampleCount=sv.sampleCount)

            def load_buffer(this, b):
                sv.loadBuffer(bytes(b[0].data))
                obj.props["buffer"] = b[0]
                sync()
                return I.call(I.get_prop(I.globals.vars["Promise"], "resolve"), UNDEF, [obj])
            obj.props.update(buffer=None, loadBuffer=native("loadBuffer", load_buffer),
                             slice=native("slice", lambda t, b: JSArrayBuffer(I, bytearray(sv.slice(*[int(x) for x in b[:4]])))))
            sync()
            return obj
        deps = JSObject(I.object_proto)
        deps.props.update(windows=win, cmaps=cm, lookup=native("lookup", lookup),
                          parseFreqRate=native("parseFreqRate", lambda t, a: I.from_py(parse_freq_rate.parseFreqRate(js_to_string(a[0])))),
                          parseFormat=native("parseFormat", lambda t, a: parse_freq_rate.parseFormat(js_to_string(a[0]))),
                          SampleView=NativeFunction(I, "SampleView", None, sample_view), Worker=self.GpuWorker)
        self._deps = deps
        return deps

    def spectroplot_class(self, deps):
        create = self.I.require_file(os.path.join(JS, "spectroplot_headless.js"))
        return self.I.call(create, UNDEF, [deps])

    def await_(self, promise):
        self.I.drain()
        state, value = self.I.promise_state(promise)
        assert state != "pending", "promise still pending after the job queue drained"
        if state == "rejected":
            raise JSThrow(value)
        return value
