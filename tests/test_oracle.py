"""CPU tests of the oracle (test infrastructure) — runs without a GPU.

The reference has no tests.  The primary pin is tests/test_reference_js.py (replies of the reference's own source,
run by oracle/jsmini.py); this file holds the secondary ones: SURVEY.md Appendix B (derived known-answers), the
agreement of two independent restatements (C radix-2 vs numpy pocketfft), mathematical identities, and the
restatement-generated golden fixtures."""
import glob
import os
import struct

import numpy as np
import pytest

from oracle import oracle as O, np_restatement as R
from helpers import injective_cmap, load_fixture

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("n,kind,weight,bn_db", [
    (8, "hann", 3.5, -5.440680443502757), (8, "blackmanHarris", 2.51131, -3.999003260062321),
    (1024, "hann", 511.5000000000002, -27.088456380481794), (1024, "hamming", 552.5000000000002, -27.423322823571485),
    (1024, "bartlett", 511.49951124144707, -27.08845223062365), (4096, "hann", 2047.5000000000048, -33.11223910432457),
    (4096, "blackman", 1719.899999999995, -32.355031964943365),
    (4096, "blackmanHarris", 1469.0813100000016, -31.670458335758774)])
def test_window_weights_appendix_b1(n, kind, weight, bn_db):
    w, wt = O.window(kind, n)
    assert wt == weight
    assert 10 * np.log10(1 / wt) == bn_db
    w2, wt2 = R.window(kind, n)
    assert wt2 == wt and np.array_equal(w, w2)


def test_window_spot_values():
    assert O.window("hann", 8)[0][1] == 0.1882550990706332
    assert O.window("blackman", 64)[0][0] == -1.3877787807814457e-17
    assert O.window("blackmanHarris", 64)[0][0] == 6.0000000000001025e-05
    assert (O.window("rectangular", 16)[0] == 1.0).all()


def test_decode_appendix_b2():
    assert np.array_equal(O.decode("CU8", bytes([0, 127, 128, 255])).ravel(), [-1.0, -0.00392156862745098, 0.00392156862745098, 1.0])
    assert np.array_equal(O.decode("CU4", bytes([0xA3]))[0], [0.3333333333333333, -0.6])
    assert np.array_equal(O.decode("CS4", bytes([0xA3]))[0], [-0.75, 0.375])
    assert np.array_equal(O.decode("CU12", bytes([0x21, 0x43, 0x65]))[0], [-0.6087912087912087, -0.2087912087912088])
    assert np.array_equal(O.decode("CS12", bytes([0xFF, 0x8F, 0x80]))[0], [-0.00048828125, -0.99609375])
    b = struct.pack("<IIII", 0x89ABCDEF, 0xC0000000, 0x89ABCDEF, 0xC0000000)
    assert O.decode("CU64", b)[0, 0] == 0.5000000001252112
    assert O.decode("CS64", b)[0, 0] == -0.4999999998747889


@pytest.mark.parametrize("fmt", O.FORMATS)
def test_decode_two_restatements_agree(fmt):
    rng = np.random.default_rng(7)
    raw = rng.integers(0, 256, 48 * 64, dtype=np.uint8)
    if fmt in ("CF32", "CF64"):
        raw = rng.standard_normal(48 * 64 // (4 if fmt == "CF32" else 8)).astype("<f4" if fmt == "CF32" else "<f8").view(np.uint8)
    a = O.decode(fmt, raw.tobytes())
    b = R.decode_all(fmt, raw.tobytes())
    assert a.shape == b.shape and np.array_equal(a, b)


def test_format_aliases_and_default():
    L = O.lib()
    f = lambda s: L.spo_format_from_name(s.encode())
    assert f("data") == f("CU8") == f("complex16u") == f("nonsense") == 2       # lib/samples.js:48,149
    assert f("complex16s") == 3 and f("cfile") == f("COMPLEX") == 12
    assert [L.spo_sample_width(i) for i in range(14)] == [1, 1, 2, 2, 3, 3, 4, 4, 8, 8, 16, 16, 8, 16]


def test_out_of_range_reads_follow_js_undefined():
    # CU8 with an odd byte count: the last Q is `undefined` -> NaN; CU4 past the end reads 0 bits -> -1
    a = O.decode("CU8", bytes([10, 20, 30]), 0, 2)
    assert a[0, 0] == (10 - 127.5) * (1 / 127.5) and np.isnan(a[1, 1]) and not np.isnan(a[1, 0])
    assert np.array_equal(O.decode("CU4", bytes([0xFF]), 0, 2)[1], [-1.0, -1.0])
    assert np.array_equal(O.decode("CS12", bytes([0xFF]), 0, 1)[0], [255 / 2048.0, 0.0])


@pytest.mark.parametrize("n", [2, 8, 64, 1024])
def test_fft_matches_naive_dft(n):
    rng = np.random.default_rng(n)
    x = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    re, im = O.fft(x.real, x.imag)
    k = np.arange(n)
    ref = (x[None, :] * np.exp(-2j * np.pi * k[:, None] * k[None, :] / n)).sum(1)
    assert np.allclose(re + 1j * im, ref, rtol=0, atol=1e-9 * n)


def test_fft_rejects_non_power_of_two():
    with pytest.raises(ValueError):
        O.fft(np.zeros(12), np.zeros(12))


def test_splitreal_separates_two_real_channels():
    n = 64
    rng = np.random.default_rng(3)
    l, r = rng.standard_normal(n), rng.standard_normal(n)
    re, im = O.fft(l, r)
    re, im = O.splitreal(re, im)
    L, Rr = np.fft.fft(l), np.fft.fft(r)
    i = np.arange(1, n // 2)
    assert np.allclose(re[i] + 1j * im[i], L[i])
    # the right channel's bin i lands at index n-i (lib/fft_nayuki.js:112-117)
    assert np.allclose(re[n - i], Rr[i].real) and np.allclose(im[n - i], Rr[i].imag)
    assert im[0] == 0 and re[n // 2] == 0 and im[n // 2] == 0
    z = np.fft.fft(l + 1j * r)
    assert np.allclose(R.splitreal(z[None, :])[0], re + 1j * im)


def test_full_scale_tone_is_0_db():
    n, width = 256, 4
    t = np.arange(n * width)
    z = np.exp(2j * np.pi * 32 * t / n)
    buf = np.stack([z.real, z.imag], 1).astype("<f8").tobytes()
    w, wt = O.window("rectangular", n)
    r = O.render(buf, "CF64", n, width, w, 1 / wt, 0, 30, injective_cmap(256), taps=True)
    assert np.abs(r.db[:, 32]).max() < 1e-9 and abs(r.dBfs_max) < 1e-9
    assert int(r.c_hist.sum()) == n * width


def test_appendix_b3_end_to_end():
    g = np.load(os.path.join(GOLD, "appendix_b3.npz"))
    w, wt = O.window("hann", 8)
    cmap = np.stack([np.arange(256)] * 3, 1).astype(np.uint8)
    r = O.render(g["buf"].tobytes(), "CU8", 8, 4, w, 1 / 3.5, 6, 30, cmap, taps=True)
    assert wt == 3.5
    assert np.array_equal(r.image[..., 0], g["gray_image"])
    assert np.array_equal(r.gauge_mins, g["gauge_mins"]) and np.array_equal(r.gauge_maxs, g["gauge_maxs"])
    assert np.array_equal(r.gauge_amps, g["gauge_amps"])
    assert r.dBfs_min == float(g["dBfs_min"]) and r.dBfs_max == float(g["dBfs_max"])
    assert np.allclose(r.db[0] + 6, g["frame0_dbfs"], atol=5e-7)
    assert int(r.cB_hist.sum()) == 32 and np.nonzero(r.cB_hist)[0][0] == 15 and np.nonzero(r.cB_hist)[0][-1] == 129


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLD, "c*.npz"))))
def test_oracle_reproduces_golden(path):
    g = load_fixture(path)
    r = O.render(g["buf"].tobytes(), str(g["fmt"]), int(g["n"]), int(g["width"]), g["windowc"], 1.0 / float(g["weight"]),
                 float(g["gain"]), float(g["range"]), g["cmap"], bool(g["channel_mode"]), bool(g["waterfall"]), taps=True)
    assert np.array_equal(r.image, g["image"]) and np.array_equal(r.gray, g["gray"])
    assert np.array_equal(r.cB_hist, g["cB_hist"]) and np.array_equal(r.c_hist, g["c_hist"])
    for k in ("gauge_mins", "gauge_maxs", "gauge_amps"):
        assert np.array_equal(getattr(r, k), g[k])
    assert r.dBfs_min == float(g["dBfs_min"]) and r.dBfs_max == float(g["dBfs_max"])


def test_special_values():
    # all-zero input: log10(0) = -inf -> cB bin 0 (T(+inf) = 0), colour 0, min = -inf (SURVEY A.4)
    n, width = 16, 3
    w, wt = O.window("hann", n)
    r = O.render(bytes(4 * n * width), "CS16", n, width, w, 1 / wt, 6, 30, injective_cmap(256), taps=True)
    assert r.cB_hist[0] == n * width and r.c_hist[0] == n * width and r.dBfs_min == -np.inf and r.dBfs_max == -200.0
    assert (r.gauge_mins == 0).all() and (r.gauge_amps == 0).all()
    # NaN input poisons the frame: every bin -> cB bin 0, colour 0, min/max untouched
    x = np.zeros((n * width, 2), "<f4"); x[5, 1] = np.nan; x[:, 0] = 0.25
    r = O.render(x.tobytes(), "CF32", n, width, w, 1 / wt, 6, 30, injective_cmap(256), taps=True)
    assert (r.gray[0] == 0).all() and (r.cbk[0] == 0).all() and np.isnan(r.db[0]).all()


def test_fanout_matches_reference_slicing():
    # lib/spectroplot.js:1206-1228: disjoint slices, per-slice stride, merged histograms
    n, width, workers = 64, 40, 4
    buf = O.synth("CU8", 0, 5000, 5000, 11).tobytes()
    w, wt = O.window("hann", n)
    cm = injective_cmap(256)
    whole = O.render(buf, "CU8", n, width, w, 1 / wt, 6, 30, cm, workers=workers)
    sl = 2 * (5000 // workers)
    acc = np.zeros(1000, np.uint64)
    for i in range(workers):
        part = O.render(buf[i * sl:(i + 1) * sl], "CU8", n, width // workers, w, 1 / wt, 6, 30, cm)
        acc += part.cB_hist
        assert np.array_equal(whole.image[:, i * 10:(i + 1) * 10], part.image)
    assert np.array_equal(acc, whole.cB_hist)


def test_synth_is_counter_based():
    a = O.synth("CS16", 0, 1000, 5000, 42)
    b = O.synth("CS16", 300, 200, 5000, 42)
    assert np.array_equal(a[4 * 300:4 * 500], b)
    v = a.view("<i2").astype(float)
    assert 0.3 < np.abs(v).max() / 32768 < 0.8
