"""Pins against the REFERENCE'S OWN CODE.

tests/golden/ref_js/ holds replies of the unmodified reference worker (lib/worker.js + lib/samples.js +
lib/fft_nayuki.js, message parts from lib/windows.js and the lib/*cmap.js tables) and known answers of its host
helpers (lib/utils.js lookup, lib/parseFreqRate.js, SampleView.slice), produced by tools/make_ref_golden.py, which
executes those files with oracle/jsmini.py (no JS engine exists in the image).  Here:

  * CPU (-m "not gpu"): the C oracle and the Python host mirror must reproduce the reference's outputs EXACTLY
    (image bytes, both histograms, gauges, dBfs_min / dBfs_max, window tables and weights, colormap tables, name
    lookup, file-name parsing, fan-out slices, decoded samples);
  * GPU (-m gpu): the CUDA path, called through the worker protocol (GpuWorker.postMessage -> sp_render), must match
    the reference's replies within BASELINE.json's bars (<= 0.1 % of pixels one colour step off, histograms equal up to
    those ties, gauges +-1, dBfs_min / dBfs_max within 0.01 dB).
"""
import glob
import json
import math
import os

import numpy as np
import pytest

from helpers import PIXEL_FRAC, DB_TOL, DB_FLOOR_STRICT, DB_FLOOR_REF, DB_TOL_FLOOR_MAX, cmap_index_image, load_fixture as load
from oracle import oracle as O

REF = os.path.join(os.path.dirname(__file__), "golden", "ref_js")
CASES = sorted(glob.glob(os.path.join(REF, "*.npz")))
IDS = [os.path.basename(p)[:-4] for p in CASES]


def canonical(fmt):
    from spectro_b200.samples import SampleView
    return SampleView(fmt).canonical


def same_float(a, b):
    return a == b or (a != a and b != b)


def test_fixture_inventory():
    assert len(CASES) >= 92 and os.path.exists(os.path.join(REF, "ref_host.json"))
    fmts = {canonical(load(p)["fmt"]) for p in CASES}
    assert fmts == {"CU4", "CS4", "CU8", "CS8", "CU12", "CS12", "CU16", "CS16", "CU32", "CS32", "CU64", "CS64", "CF32", "CF64"}
    assert {load(p)["window"] for p in CASES} == {"rectangular", "bartlett", "hamming", "hann", "blackman", "blackmanHarris"}


# ------------------------------------------------------------------ CPU: oracle == reference worker, exactly
@pytest.mark.parametrize("path", CASES, ids=IDS)
def test_oracle_equals_reference_worker(path):
    f = load(path)
    n, width = int(f["n"]), int(f["width"])
    r = O.render(f["buf"].tobytes(), canonical(f["fmt"]), n, width, f["windowc"], 1.0 / float(f["weight"]), float(f["gain"]),
                 float(f["range"]), f["cmap"], bool(f["channel_mode"]), bool(f["waterfall"]))
    assert np.array_equal(r.image.reshape(-1), f["image"]), "image bytes"
    assert np.array_equal(r.cB_hist.astype(np.float64), f["cB_hist"]), "cB_hist"
    assert np.array_equal(r.c_hist.astype(np.float64), f["c_hist"]), "c_hist"
    for k in ("gauge_mins", "gauge_maxs", "gauge_amps"):
        assert np.array_equal(getattr(r, k), f[k]), k
    assert same_float(r.dBfs_min, float(f["dBfs_min"])) and same_float(r.dBfs_max, float(f["dBfs_max"]))
    # pixels whose level is above +0.05 dB land on a negative, non-index key in the reference (lib/worker.js:105-106)
    # and are in no bin: totals account for them
    dropped = len(json.loads(f["cB_extra"]))
    assert (int(f["cB_hist"].sum()) == n * width) == (dropped == 0)
    assert int(f["c_hist"].sum()) == n * width and json.loads(f["c_extra"]) == {}


def test_reference_reply_echoes_offset_and_shapes():
    f = load(CASES[0])
    assert int(f["offset"]) == 7 and f["cB_hist"].shape == (1000,) and f["c_hist"].shape == (len(f["cmap"]),)
    assert f["image"].shape == (4 * int(f["width"]) * int(f["n"]),)


# ------------------------------------------------------------------ CPU: host mirror == reference helpers, exactly
@pytest.fixture(scope="module")
def host():
    with open(os.path.join(REF, "ref_host.json")) as fp:
        return json.load(fp)


def test_windows_equal_reference(host):
    from spectro_b200 import windows
    for key, ref in host["windows"].items():
        kind, n = key.split("/")
        n = int(n)
        mine = getattr(windows, kind + "Window")(n)
        assert mine["weight"] == ref["weight"], key
        w = np.asarray(mine["window"], np.float64)
        if ref["window"] is not None:
            assert np.array_equal(w, np.array(ref["window"])), key
        assert [w[i] for i in (0, 1, n // 3, n // 2, n - 1)] == ref["spot"], key
        ow, owt = O.window(kind, n)                       # the oracle's table is the same one
        assert owt == ref["weight"] and np.array_equal(ow, w), key


def test_cmap_tables_equal_reference(host):
    from spectro_b200 import cmaps
    assert set(cmaps.cmaps) == set(host["cmaps"])
    for name, ref in host["cmaps"].items():
        assert [list(map(int, c)) for c in cmaps.cmaps[name]] == ref, name
    assert len(host["cmaps"]["parabola_cmap"]) == 64 and all(len(v) == 256 for k, v in host["cmaps"].items() if k != "parabola_cmap")


def test_lookup_equals_reference(host):
    from spectro_b200 import utils, cmaps
    names = ["rectangularWindow", "bartlettWindow", "hammingWindow", "hannWindow", "blackmanWindow", "blackmanHarrisWindow"]
    table = {k: k for k in names}
    for key, ref in host["lookup_windows"].items():
        assert utils.lookup(table, key) == ref, key
    ctab = {k: k for k in host["cmap_key_order"]}
    for key, ref in host["lookup_cmaps"].items():
        assert utils.lookup(ctab, key) == ref, key
    assert host["lookup_cmaps"]["parula"] is None         # the demo's 'parula' resolves to nothing (-> cube1 default)


def test_parse_freq_rate_equals_reference(host):
    from spectro_b200 import parse_freq_rate as P
    for name, ref in host["parseFreqRate"].items():
        assert P.parseFreqRate(name) == ref, name
    for name, ref in host["parseFormat"].items():
        assert P.parseFormat(name) == ref, name


def test_sampleview_slices_equal_reference(host):
    from spectro_b200.samples import SampleView
    for key, ref in host["slices"].items():
        fmt, nbytes, count = key.split("/")
        nbytes, count = int(nbytes), int(count)
        sv = SampleView(fmt, bytes(nbytes))
        assert sv.sampleWidth == ref["sampleWidth"] and sv.sampleCount == ref["sampleCount"], key
        end = int(nbytes / sv.sampleWidth)
        assert [len(sv.slice(i, count, 0, end)) for i in range(count)] == ref["slice_bytes"], key


def test_decode_equals_reference(host):
    for fmt, ref in host["decode"].items():
        got = O.decode(fmt, bytes(ref["raw"]))
        assert np.array_equal(got, np.array(ref["iq"], np.float64)), fmt


def test_fft_known_answer(host):
    assert host["fft_bad_length"] == "Length is not a power of 2"      # lib/fft_nayuki.js:38-39
    re, im = (np.array(a) for a in host["fft16_in"])
    out = np.array(host["fft16_out"][0]) + 1j * np.array(host["fft16_out"][1])
    assert np.abs(out - np.fft.fft(re + 1j * im)).max() < 1e-13       # forward sign, unscaled
    sr, si = host["fft16_split"]
    assert si[0] == 0 and sr[8] == 0 and si[8] == 0                   # lib/fft_nayuki.js:105-107


# ------------------------------------------------------------------ GPU: CUDA path == reference worker within the bars
def is_injective(cmap):
    key = (cmap[:, 0].astype(np.int64) << 16) | (cmap[:, 1].astype(np.int64) << 8) | cmap[:, 2]
    return len(set(key.tolist())) == len(cmap)


@pytest.mark.gpu
@pytest.mark.parametrize("path", CASES, ids=IDS)
def test_gpu_worker_equals_reference_worker(path):
    import spectro_b200
    f = load(path)
    n, width = int(f["n"]), int(f["width"])
    w = spectro_b200.GpuWorker(0)
    replies = []
    w.onmessage = replies.append
    w.postMessage(dict(block_norm=1.0 / float(f["weight"]), gain=float(f["gain"]), range=float(f["range"]),
                       cmap=[list(map(int, c)) for c in f["cmap"]], n=n, windowc=f["windowc"].tolist(), width=width, offset=7,
                       buffer=f["buf"].tobytes(), format=str(f["fmt"]), channelMode=bool(f["channel_mode"]),
                       waterfall=bool(f["waterfall"])))
    w.terminate()
    assert len(replies) == 1
    d = replies[0]["data"]
    assert d["offset"] == 7
    img, ref = d["imageData"]["data"].reshape(-1, 4), f["image"].reshape(-1, 4)
    npx = n * width
    if "nan_inf" in path:
        # A frame that holds a +-inf SAMPLE has bins that are +-inf (white) or inf - inf = NaN (black); which bin gets
        # which depends on the order of the butterflies (the reference's radix-2 vs the kernel's radix-64), so those two
        # frames (columns 3 and 5) are only required to be black / white.  The NaN frame (column 1: every bin NaN) and
        # the ordinary frames are held to the usual bars.
        cols = np.arange(npx) % width
        special = (cols == 3) | (cols == 5)
        black, white = np.array([0, 0, 0, 255]), np.array([255, 255, 255, 255])
        assert ((img[special] == black).all(axis=1) | (img[special] == white).all(axis=1)).all()
        assert ((ref[special] == black).all(axis=1) | (ref[special] == white).all(axis=1)).all()
        assert (img[cols == 1] == black).all() and (ref[cols == 1] == black).all()
        assert (img[~special] != ref[~special]).any(axis=1).sum() <= 1
        assert int(d["c_hist"].sum()) == npx and float(d["dBfs_max"]) == float(f["dBfs_max"]) == math.inf
        return
    tol = max(1, int(PIXEL_FRAC * npx))
    bad = (img != ref).any(axis=1)
    nbad = int(bad.sum())
    assert nbad <= tol, f"{nbad}/{npx} pixels differ from the reference"
    assert (img[:, 3] == 255).all()
    if nbad and is_injective(f["cmap"]):
        gi, ri = cmap_index_image(img[bad][None], f["cmap"]), cmap_index_image(ref[bad][None], f["cmap"])
        assert (gi >= 0).all() and np.abs(gi - ri).max() <= 1, "a differing pixel is more than one colour step off"
    assert int(np.abs(d["c_hist"].astype(np.float64) - f["c_hist"]).sum()) <= 2 * nbad, "c_hist"
    assert int(d["c_hist"].sum()) == npx
    assert np.abs(d["cB_hist"].astype(np.float64) - f["cB_hist"]).sum() <= 2 * max(2, tol), "cB_hist"
    for k in ("gauge_mins", "gauge_maxs", "gauge_amps"):
        assert np.abs(d[k].astype(int) - f[k].astype(int)).max() <= 1, k
    for k in ("dBfs_min", "dBfs_max"):
        a, b = float(d[k]), float(f[k])
        if math.isfinite(b) and b > DB_FLOOR_STRICT:
            assert abs(a - b) <= DB_TOL, (k, a, b)
        elif math.isfinite(b) and b > DB_FLOOR_REF:
            assert abs(a - b) <= DB_TOL_FLOOR_MAX, (k, a, b)
        elif math.isfinite(b):       # below -120 dBFS both values are round-off (float64 there, fp32 here): only "below the floor"
            assert a <= DB_FLOOR_REF + DB_TOL_FLOOR_MAX, (k, a, b)
        else:
            assert same_float(a, b), (k, a, b)
