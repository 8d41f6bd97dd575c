"""js/spectro_napi.c — the N-API addon — compiled against tests/napi_stub (a fake Node-API runtime, since the image has
no Node.js) and driven through its exported create / render / destroy exactly as js/gpu_worker.js calls them.
CPU suite: it builds warning-free, registers its three functions and `create` throws the C ABI's message when there is
no GPU (no CPU fallback).  GPU suite: `render` marshals a worker message into sp_request / sp_reply and its outputs
match the reference-worker fixtures."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
STUB = os.path.join(ROOT, "tests", "napi_stub")
LIBDIR = os.path.join(ROOT, "spectroplot-js_b200", "lib")
REFJS = os.path.join(ROOT, "tests", "golden", "ref_js")
K_UNDEF, K_NUM, K_BOOL, K_OBJ, K_AB, K_TA, K_EXT, K_FN = range(8)
U8, U8C, F64, BU64 = 1, 2, 8, 10                     # napi_typedarray_type


@pytest.fixture(scope="module")
def fk():
    out = os.path.join(STUB, "_build")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "fake_addon.so")
    cmd = ["gcc", "-shared", "-fPIC", "-O1", "-Wall", "-Wextra", "-Werror", "-I" + STUB, "-I" + os.path.join(ROOT, "include"),
           os.path.join(STUB, "fake_napi.c"), os.path.join(ROOT, "spectroplot-js_b200", "js", "spectro_napi.c"),
           "-L" + LIBDIR, "-lspectro_b200", "-Wl,-rpath," + LIBDIR, "-o", so]
    subprocess.check_call(cmd)                         # -Werror: the addon must compile cleanly against the N-API signatures
    lib = C.CDLL(so)
    P = C.c_void_p
    for name, res, args in (("fk_env_new", P, []), ("fk_load", P, [P]), ("fk_number", P, [C.c_double]), ("fk_bool", P, [C.c_int]),
                            ("fk_object", P, []), ("fk_array", P, [C.c_uint32, C.POINTER(P)]), ("fk_arraybuffer", P, [P, C.c_size_t]), ("fk_typedarray", P, [C.c_int, P, C.c_size_t, C.c_size_t]),
                            ("fk_set", None, [P, C.c_char_p, P]), ("fk_get", P, [P, P, C.c_char_p]), ("fk_kind", C.c_int, [P]),
                            ("fk_num", C.c_double, [P]), ("fk_data", P, [P]), ("fk_len", C.c_size_t, [P]), ("fk_ta_type", C.c_int, [P]),
                            ("fk_call", P, [P, P, C.c_size_t, C.POINTER(P)]), ("fk_error", C.c_char_p, [P])):
        f = getattr(lib, name)
        f.restype, f.argtypes = res, args
    return lib


class Addon:
    def __init__(self, lib):
        self.lib = lib
        self.env = lib.fk_env_new()
        self.exports = lib.fk_load(self.env)

    def fn(self, name):
        return self.lib.fk_get(self.env, self.exports, name.encode())

    def call(self, name, *args):
        argv = (C.c_void_p * max(1, len(args)))(*args)
        r = self.lib.fk_call(self.env, self.fn(name), len(args), argv)
        if r is None:
            raise RuntimeError((self.lib.fk_error(self.env) or b"").decode())
        return r

    def ab(self, data: bytes):
        return self.lib.fk_arraybuffer(data, len(data))

    def ta(self, kind, arr):
        arr = np.ascontiguousarray(arr)
        return self.lib.fk_typedarray(kind, self.ab(arr.tobytes()), 0, arr.size)

    def ctx(self, f, **over):
        lib = self.lib
        o = lib.fk_object()
        vals = dict(format=f["format_id"], n=int(f["n"]), width=int(f["width"]), block_norm=1.0 / float(f["weight"]), gain=float(f["gain"]),
                    range=float(f["range"]))
        vals.update({k: v for k, v in over.items() if k in vals})
        for k, v in vals.items():
            lib.fk_set(o, k.encode(), lib.fk_number(float(v)))
        lib.fk_set(o, b"buffer", self.ab(f["buf"].tobytes()))
        lib.fk_set(o, b"windowc", over.get("windowc") or self.ta(F64, f["windowc"].astype(np.float64)))
        lib.fk_set(o, b"cmap", self.ta(U8, f["cmap"].astype(np.uint8).reshape(-1)))
        lib.fk_set(o, b"channelMode", lib.fk_bool(int(bool(f["channel_mode"]))))
        lib.fk_set(o, b"waterfall", lib.fk_bool(int(bool(f["waterfall"]))))
        return o

    def typed_out(self, obj, key, kind, dtype):
        v = self.lib.fk_get(self.env, obj, key.encode())
        assert self.lib.fk_kind(v) == K_TA and self.lib.fk_ta_type(v) == kind, key
        n = self.lib.fk_len(v)
        return np.frombuffer(C.string_at(self.lib.fk_data(v), n * np.dtype(dtype).itemsize), dtype=dtype).copy()


def load(name):
    from spectro_b200 import _lib
    from spectro_b200.samples import SampleView
    from helpers import load_fixture
    f = load_fixture(os.path.join(REFJS, name + ".npz"))
    f["format_id"] = _lib.FORMATS.index(SampleView(str(f["fmt"])).canonical)
    return f


def test_addon_registers_and_has_no_cpu_fallback(fk):
    a = Addon(fk)
    assert fk.fk_kind(a.exports) == K_OBJ
    for name in ("create", "render", "destroy"):
        assert fk.fk_kind(a.fn(name)) == K_FN, name
    import torch
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CUDA device|SP_E_NO_DEVICE|no CPU fallback"):
            a.call("create", fk.fk_number(0))


@pytest.mark.gpu
def test_addon_render_matches_reference_replies(fk):
    a = Addon(fk)
    eng = a.call("create", fk.fk_number(0))
    assert fk.fk_kind(eng) == K_EXT
    for name in ("cu8_n1024_hann_cube1_w12", "cs16_n4096_bh_viridis_w8", "cf32_n8192_hann_inferno_w4", "cu12_n512_blackman_parabola_w10",
                 "cs16_n2048_blackman_inj64_w5_wf_split", "cs16_n64_zeros"):
        f = load(name)
        n, width = int(f["n"]), int(f["width"])
        r = a.call("render", eng, a.ctx(f))
        img = a.typed_out(r, "image", U8C, np.uint8)
        assert img.size == 4 * n * width
        bad = (img.reshape(-1, 4) != f["image"].reshape(-1, 4)).any(axis=1).sum()
        assert bad <= max(1, int(1e-3 * n * width)), name
        c_hist = a.typed_out(r, "c_hist", BU64, np.uint64)
        cB_hist = a.typed_out(r, "cB_hist", BU64, np.uint64)
        assert c_hist.size == len(f["cmap"]) and cB_hist.size == 1000 and int(c_hist.sum()) == n * width
        assert np.abs(c_hist.astype(np.float64) - f["c_hist"]).sum() <= 2 * bad
        for k in ("gauge_mins", "gauge_maxs", "gauge_amps"):
            assert np.abs(a.typed_out(r, k, U8C, np.uint8).astype(int) - f[k].astype(int)).max() <= 1, (name, k)
        dmax = fk.fk_num(fk.fk_get(a.env, r, b"dBfs_max"))
        assert dmax == float(f["dBfs_max"]) or abs(dmax - float(f["dBfs_max"])) <= 0.01
        assert fk.fk_num(fk.fk_get(a.env, r, b"device_ms")) > 0
    # engine errors become JS exceptions carrying sp_last_error(): the reference's own string (lib/fft_nayuki.js:39)
    f = load("cs16_n128_w2")
    with pytest.raises(RuntimeError, match="not a power of 2"):
        a.call("render", eng, a.ctx(f, n=100))
    # a windowc that is not a typed array is refused by napi_get_typedarray_info, not read as garbage
    with pytest.raises(RuntimeError, match="napi_get_typedarray_info"):
        a.call("render", eng, a.ctx(f, windowc=a.ab(f["windowc"].tobytes())))
    # windowc of the wrong element type or shorter than n would be read out of bounds on the JS heap: refused
    F32 = 7
    with pytest.raises(RuntimeError, match="Float64Array"):
        a.call("render", eng, a.ctx(f, windowc=fk.fk_typedarray(F32, a.ab(f["windowc"].astype(np.float32).tobytes()), 0, int(f["n"]))))
    with pytest.raises(RuntimeError, match="shorter than n"):
        a.call("render", eng, a.ctx(f, windowc=a.ta(F64, f["windowc"].astype(np.float64)[: int(f["n"]) // 2])))
    with pytest.raises(RuntimeError, match="width out of range"):
        a.call("render", eng, a.ctx(f, width=0))
    a.call("destroy", eng)
    # create([devices]): one engine over several GPUs (sp_create with ndev > 1); with one GPU in the box a one-element list
    import torch
    ids = list(range(min(torch.cuda.device_count(), 8)))
    items = (C.c_void_p * len(ids))(*[fk.fk_number(float(i)) for i in ids])
    multi = a.call("create", fk.fk_array(len(ids), items))
    f = load("cu8_n256_overlap_w40")
    r = a.call("render", multi, a.ctx(f))
    img = a.typed_out(r, "image", U8C, np.uint8)
    assert (img.reshape(-1, 4) != f["image"].reshape(-1, 4)).any(axis=1).sum() <= 10
    a.call("destroy", multi)
