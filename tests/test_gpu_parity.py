"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle on the
same seeded inputs, against the committed golden fixtures, and through size-independent
properties at larger sizes.  Tolerances are BASELINE.json's (see helpers.py)."""
import glob
import os

import ctypes as C

import numpy as np
import pytest

from helpers import check_parity, injective_cmap, gray_from_image, cmap_index_image, load_fixture, DB_TOL, DB_FLOOR_REF
from oracle import oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
CM256 = injective_cmap(256)


def run_both(engine, buf, fmt, n, width, window="hann", gain=6, rng=30, cmap=CM256, channel_mode=False,
             waterfall=False, want_db=True, label=""):
    w, wt = O.window(window, n)
    ora = O.render(buf, fmt, n, width, w, 1 / wt, gain, rng, cmap, channel_mode, waterfall, taps=True)
    gpu = engine.render(buf, fmt, n, width, w, 1 / wt, gain, rng, cmap, channel_mode, waterfall)
    db = engine.render_db(buf, fmt, n, width, w, 1 / wt, gain, rng, cmap, channel_mode) if want_db else None
    nbad = check_parity(gpu, ora, cmap, n, width, waterfall, db, label or f"{fmt} n={n} w={width} {window}")
    return gpu, ora, nbad


# ------------------------------------------------------------------ decode: bit-exact
@pytest.mark.parametrize("fmt", O.FORMATS)
def test_decode_bit_exact(engine, fmt):
    """gpu_fp32 == fround(reference_f64) for every sample (exhaustive code tables for <= 16 bit)."""
    rng = np.random.default_rng(1234)
    if fmt in ("CU4", "CS4"):
        raw = np.arange(256, dtype=np.uint8)
    elif fmt in ("CU8", "CS8"):
        raw = np.stack([np.arange(256), np.arange(256)[::-1]], 1).astype(np.uint8).ravel()
    elif fmt in ("CU12", "CS12"):
        c = np.arange(4096); q = c[::-1]
        raw = np.stack([c & 255, (c >> 8) | ((q & 15) << 4), q >> 4], 1).astype(np.uint8).ravel()
    elif fmt in ("CU16", "CS16"):
        raw = np.stack([np.arange(65536), np.arange(65536)[::-1]], 1).astype("<u2").view(np.uint8).ravel()
    elif fmt == "CF32":
        raw = np.concatenate([rng.standard_normal(1 << 16), [0.0, -0.0, np.inf, -np.inf, np.nan, 1e-40, 3e38, 1.0]]).astype("<f4").view(np.uint8)
    elif fmt == "CF64":
        raw = np.concatenate([rng.standard_normal(1 << 16) * 10.0 ** rng.integers(-30, 30, 1 << 16), [0.0, 1e-300, 1e300, np.nan]]).astype("<f8").view(np.uint8)
    else:
        raw = rng.integers(0, 256, (1 << 16) * 16, dtype=np.uint8)
        edge = np.array([0, 0xFFFFFFFF, 0x80000000, 0x7FFFFFFF, 1, 0xFFFFFF7F, 0x00000080, 0x01000000], "<u4").view(np.uint8)
        raw = np.concatenate([edge, edge[::-1].copy(), raw])
    with np.errstate(over="ignore"):
        ref = O.decode(fmt, raw).astype(np.float32)       # fround
    got = engine.decode(fmt, raw)
    assert got.shape == ref.shape
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)) or np.array_equal(
        got[~np.isnan(ref)].view(np.uint32), ref[~np.isnan(ref)].view(np.uint32)) and np.array_equal(np.isnan(got), np.isnan(ref))


def test_decode_out_of_range_follows_js(engine):
    for fmt, raw in (("CU8", bytes([10, 20, 30])), ("CU4", bytes([0xFF])), ("CS12", bytes([0xFF])),
                     ("CS16", bytes([1, 2, 3, 4, 5, 6])), ("CS64", bytes(range(20))), ("CU64", bytes(range(28)))):
        cnt = len(raw) // O.SAMPLE_WIDTH[O.FORMATS.index(fmt)] + 2
        ref = O.decode(fmt, raw, 0, cnt).astype(np.float32)
        got = engine.decode(fmt, raw, 0, cnt)
        assert np.array_equal(np.isnan(got), np.isnan(ref)), fmt
        assert np.array_equal(got[~np.isnan(ref)], ref[~np.isnan(ref)]), fmt


def test_synth_generator_bit_identical(engine):
    total = 100000
    for fmt in O.FORMATS:
        sw = O.SAMPLE_WIDTH[O.FORMATS.index(fmt)]
        d = engine.alloc(5000 * sw)
        engine.synth_fill(d, fmt, 777, 5000, total, 0xABCDEF)
        got = np.empty(5000 * sw, np.uint8)
        engine.d2h(got, d)
        engine.free(d)
        assert np.array_equal(got, O.synth(fmt, 777, 5000, total, 0xABCDEF)), fmt


# ------------------------------------------------------------------ golden fixtures
def test_appendix_b3(engine):
    g = np.load(os.path.join(GOLD, "appendix_b3.npz"))
    w, wt = O.window("hann", 8)
    cmap = injective_cmap(256)
    r = engine.render(g["buf"].tobytes(), "CU8", 8, 4, w, 1 / 3.5, 6, 30, cmap)
    gray = gray_from_image(r["image"], cmap, 8, 4)
    y = np.where(np.arange(8) <= 4, 4 - np.arange(8), 12 - np.arange(8))
    img = np.zeros((8, 4), int); img[y[None, :], np.arange(4)[:, None]] = gray
    assert np.abs(img - g["gray_image"].astype(int)).max() <= 1 and (img != g["gray_image"]).sum() <= 1
    assert np.abs(r["gauge_mins"].astype(int) - g["gauge_mins"]).max() <= 1
    assert np.abs(r["gauge_maxs"].astype(int) - g["gauge_maxs"]).max() <= 1
    assert np.array_equal(r["gauge_amps"], g["gauge_amps"])
    assert abs(r["dBfs_min"] - float(g["dBfs_min"])) < DB_TOL and abs(r["dBfs_max"] - float(g["dBfs_max"])) < DB_TOL
    assert int(r["cB_hist"].sum()) == 32 and int(r["c_hist"].sum()) == 32


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLD, "c*.npz"))))
def test_golden_fixture(engine, path):
    g = load_fixture(path)
    fmt, n, width = str(g["fmt"]), int(g["n"]), int(g["width"])
    cm, wf, lr = g["cmap"], bool(g["waterfall"]), bool(g["channel_mode"])
    r = engine.render(g["buf"].tobytes(), fmt, n, width, g["windowc"], 1.0 / float(g["weight"]), float(g["gain"]),
                      float(g["range"]), cm, lr, wf)
    db = engine.render_db(g["buf"].tobytes(), fmt, n, width, g["windowc"], 1.0 / float(g["weight"]), float(g["gain"]),
                          float(g["range"]), cm, lr)

    class Ora:
        pass
    o = Ora()
    for k in ("image", "gray", "db", "cB_hist", "c_hist", "gauge_mins", "gauge_maxs", "gauge_amps"):
        setattr(o, k, g[k])
    o.dBfs_min, o.dBfs_max = float(g["dBfs_min"]), float(g["dBfs_max"])
    check_parity(r, o, cm, n, width, wf, db, os.path.basename(path))


# ------------------------------------------------------------------ oracle parity sweeps
@pytest.mark.parametrize("n", [8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096])
def test_all_single_kernel_sizes(engine, n):
    width = 37                                   # awkward width: fractional stride, partial tiles
    S = n * 20 + 13
    buf = O.synth("CS16", 0, S, S, 0x5EC70000 + n).tobytes()
    run_both(engine, buf, "CS16", n, width, "hann")


@pytest.mark.parametrize("n", [8192, 16384, 32768, 65536])
def test_four_step_sizes(engine, n):
    width = 12
    S = n * 5 + 77
    buf = O.synth("CF32", 0, S, S, 0x5EC71000 + n).tobytes()
    run_both(engine, buf, "CF32", n, width, "blackmanHarris")


@pytest.mark.parametrize("fmt", O.FORMATS)
def test_all_formats_render(engine, fmt):
    n, width = 1024, 24
    S = 30000
    buf = O.synth(fmt, 0, S, S, 0x5EC72000).tobytes()
    run_both(engine, buf, fmt, n, width, "blackman")


@pytest.mark.parametrize("window", O.WINDOWS)
def test_all_windows(engine, window):
    n, width = 512, 32
    S = 512 * 32
    buf = O.synth("CU8", 0, S, S, 0x5EC73000).tobytes()
    run_both(engine, buf, "CU8", n, width, window)           # hop == n exactly (stride = n - n/(w-1)... fractional)


def test_wide_rows_fast_path_and_hop_n(engine):
    """width % 4 == 0 and S = width*n: stride is exactly... (S-n)/(w-1) = n: the headline geometry."""
    n, width = 4096, 64
    S = n * width
    buf = O.synth("CS16", 0, S, S, 0x5EC74000).tobytes()
    run_both(engine, buf, "CS16", n, width, "blackmanHarris")
    n, width = 256, 1000                                      # several slots per CTA, partial last tile
    S = n * width
    buf = O.synth("CS16", 0, S, S, 0x5EC74001).tobytes()
    run_both(engine, buf, "CS16", n, width, "hann", want_db=False)


def test_overlapping_and_skipping_strides(engine):
    n = 1024
    S = 50000
    buf = O.synth("CU8", 0, S, S, 0x5EC75000).tobytes()
    run_both(engine, buf, "CU8", n, 400, "hann", want_db=False)      # stride ~ 123: heavy overlap
    run_both(engine, buf, "CU8", n, 12, "hann", want_db=False)       # stride ~ 4452: skips data
    run_both(engine, buf, "CU8", n, 3000 // 8, "hann", want_db=False)


@pytest.mark.parametrize("cmap_len", [2, 64, 256, 1000])
def test_cmap_lengths_and_ranges(engine, cmap_len):
    n, width = 256, 20
    S = 8000
    buf = O.synth("CS8", 0, S, S, 0x5EC76000).tobytes()
    cm = injective_cmap(cmap_len)
    for gain, rng in ((0, 6), (6, 30), (40, 120), (90, 10)):
        run_both(engine, buf, "CS8", n, width, "hamming", gain, rng, cm, want_db=False,
                 label=f"cmap{cmap_len} gain{gain} range{rng}")


@pytest.mark.parametrize("n", [64, 1024, 4096, 8192, 65536])
def test_channel_mode_and_waterfall(engine, n):
    """split-real (lib/fft_nayuki.js:103-119) and the waterfall layout at every kernel class, including the
    four-step sizes where bin k and bin n-k come from different sub-sequences."""
    width = 16 if n <= 8192 else 8
    S = n * (4 if n > 8192 else 16) + 5
    buf = O.synth("CS16", 0, S, S, 0x5EC77000 + n).tobytes()
    run_both(engine, buf, "CS16", n, width, "hann", channel_mode=True)
    run_both(engine, buf, "CS16", n, width, "hann", waterfall=True)
    run_both(engine, buf, "CS16", n, width, "hann", channel_mode=True, waterfall=True)


def test_special_values(engine):
    n, width = 64, 8
    w, wt = O.window("hann", n)
    # all zero: -inf dB -> cB bin 0, colour 0, min == -inf
    r = engine.render(bytes(4 * n * width), "CS16", n, width, w, 1 / wt, 6, 30, CM256)
    assert r["cB_hist"][0] == n * width and r["c_hist"][0] == n * width
    assert r["dBfs_min"] == -np.inf and r["dBfs_max"] == -200.0
    assert (r["gauge_mins"] == 0).all() and (r["gauge_amps"] == 0).all()
    # NaN poisons exactly the frames that contain it
    x = np.full((n * width, 2), 0.25, "<f4"); x[5, 1] = np.nan
    buf = x.tobytes()
    ora = O.render(buf, "CF32", n, width, w, 1 / wt, 6, 30, CM256, taps=True)
    gpu = engine.render(buf, "CF32", n, width, w, 1 / wt, 6, 30, CM256)
    g = gray_from_image(gpu["image"], CM256, n, width)
    assert np.array_equal(g == 0, ora.gray == 0) and (g[0] == 0).all()
    assert gpu["cB_hist"][0] >= n
    # full-scale tone in a rectangular window sits at 0 dB
    t = np.arange(n * width)
    z = np.exp(2j * np.pi * 5 * t / n)
    buf = np.stack([z.real, z.imag], 1).astype("<f4").tobytes()
    w, wt = O.window("rectangular", n)
    db = engine.render_db(buf, "CF32", n, width, w, 1 / wt, 0, 30, CM256)
    assert np.abs(db[:, 5]).max() < 1e-3


def test_ragged_buffer_tail(engine):
    """CU8 with an odd byte count: sampleCount is fractional and the last frame reads one
    `undefined` (NaN) component (SURVEY A.2) — the reference renders that frame as colour 0."""
    n, width = 32, 5
    raw = O.synth("CU8", 0, 200, 200, 5).tobytes() + b"\x80"
    run_both(engine, raw, "CU8", n, width, "hann", want_db=False)
    raw12 = O.synth("CU12", 0, 100, 100, 6).tobytes() + b"\x12"        # CU12: missing bytes read as 0 bits
    run_both(engine, raw12, "CU12", n, width, "hann", want_db=False)


def test_error_codes(engine):
    import spectro_b200
    w, wt = O.window("hann", 64)
    buf = bytes(4 * 64 * 4)
    def code(**kw):
        a = dict(buf=buf, fmt="CS16", n=64, width=4, windowc=w, block_norm=1 / wt, gain=6, range_=30, cmap=CM256)
        a.update(kw)
        with pytest.raises(spectro_b200.SpError) as ei:
            engine.render(**a)
        return ei.value.name
    assert code(n=48, windowc=np.ones(48)) == "SP_E_BAD_N"           # 'Length is not a power of 2'
    assert code(width=0) == "SP_E_BAD_WIDTH"
    assert code(buf=bytes(7)) == "SP_E_RAGGED"
    assert code(n=1, windowc=np.ones(1)) == "SP_E_BAD_N"
    assert code(n=1 << 19, windowc=np.ones(1 << 19)) == "SP_E_BAD_N"
    assert code(cmap=CM256[:1]) == "SP_E_BAD_CMAP"
    assert code(fmt=99) == "SP_E_BAD_FORMAT"
    # and the engine still works afterwards
    engine.render(buf, "CS16", 64, 4, w, 1 / wt, 6, 30, CM256)


@pytest.mark.parametrize("fmt,n,width,S", [("CU8", 8, 1, 8), ("CU8", 8, 1, 20), ("CS16", 16, 4, 10), ("CF32", 32, 3, 5), ("CS8", 64, 2, 63),
                                           ("CU8", 2, 7, 30), ("CS16", 4, 5, 21), ("CF32", 2, 2, 2), ("CU4", 4, 1, 3), ("CS12", 16, 3, 16),
                                           ("CS16", 4096, 3, 1000), ("CF32", 8192, 2, 5000), ("CS16", 2, 64, 640), ("CU8", 4, 100, 1000)])
def test_degenerate_messages_are_answered_like_the_reference(engine, fmt, n, width, S):
    """One frame (stride = x/0 -> frame at sample 0), captures shorter than a frame (every read past the array is
    `undefined`), n = 2 and 4: the reference worker answers all of them (lib/worker.js:50,72), and so does the engine
    (oracle pinned to the reference on these cases by tests/test_reference_live.py)."""
    raw = O.synth(fmt, 0, S, S, 31 + n + width).tobytes()
    run_both(engine, raw, fmt, n, width, "hann" if n > 2 else "rectangular", want_db=False)


@pytest.mark.parametrize("n,width,slots,lead", [(8192, 200, 4, 2), (8192, 136, 4, 4), (16384, 96, 5, 1), (65536, 40, 4, 2), (32768, 67, 0, 0)])
def test_big_kernel_ring_wraps(engine, monkeypatch, n, width, slots, lead):
    """render_big_kernel with a ring of only 4-5 blocks: every slot is reused several times (P waits for the F items of the
    slot's previous block, F for the 32 P items of its own), overlapping hops, the < 8-frame remainder on the generic path."""
    monkeypatch.setenv("SP_FOURSTEP", "ring")              # (short captures take the HBM-scratch form by default)
    if slots:
        monkeypatch.setenv("SP_BIG_SLOTS", str(slots))
        monkeypatch.setenv("SP_BIG_LEAD", str(lead))
    S = int(n * (width - 1) * 0.37) + n + 11
    raw = O.synth("CS16", 0, S, S, 99 + n).tobytes()
    gpu, ora, nbad = run_both(engine, raw, "CS16", n, width, "hann", want_db=False)
    g2 = engine.render(raw, "CS16", n, width, *O.window("hann", n)[:1], 1 / O.window("hann", n)[1], 6, 30, CM256)
    assert np.array_equal(g2["image"], gpu["image"]) and np.array_equal(g2["cB_hist"], gpu["cB_hist"])     # repeatable


@pytest.mark.parametrize("form", ["ring", "hbm"])
@pytest.mark.parametrize("n,width", [(131072, 8), (262144, 4)])
def test_sizes_above_65536(engine, monkeypatch, n, width, form):
    """lib/fft_nayuki.js:38-39 accepts any power of two; the four-step path covers n up to 262144 (pre-pass radix 32 / 64),
    in both of its forms."""
    monkeypatch.setenv("SP_FOURSTEP", form)
    S = n * 2 + 77
    raw = O.synth("CS16", 0, S, S, 5).tobytes()
    run_both(engine, raw, "CS16", n, width, "blackmanHarris", want_db=True)


# ------------------------------------------------------------------ sharding: N shards == 1 shard, exactly
@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("n,width,S", [(1024, 208, 150001), (4096, 72, 200003), (128, 203, 20011)])
def test_frame_range_shards_reproduce_the_whole_message(engine, world, n, width, S):
    """plan_shards cuts on multiples of 8 frames, so every frame keeps the kernel it has in the unsharded message (the fused
    kernels take whole groups of 8 frames, the generic kernel the rest): images, gauges and statistics are bit-identical."""
    from spectro_b200 import sharding
    fmt, sw = "CS16", 4
    buf = O.synth(fmt, 0, S, S, 0x5EC78000).tobytes()
    w, wt = O.window("hann", n)
    whole = engine.render(buf, fmt, n, width, w, 1 / wt, 6, 30, CM256)
    parts = []
    for sh in sharding.plan_shards(S, n, width, world):
        if sh["width"] == 0:
            continue
        sub = buf[sh["sample_first"] * sw:(sh["sample_first"] + sh["sample_count"]) * sw]
        r = engine.render(sub, fmt, n, sh["width"], w, 1 / wt, 6, 30, CM256,
                          shard=sharding.shard_fields(sh, S, sw, width))
        assert np.array_equal(r["image"], whole["image"][:, sh["frame_first"]:sh["frame_first"] + sh["width"]])
        for k in ("gauge_mins", "gauge_maxs", "gauge_amps"):
            assert np.array_equal(r[k], whole[k][sh["frame_first"]:sh["frame_first"] + sh["width"]])
        parts.append(r)
    m = sharding.merge_stats(parts)
    assert np.array_equal(m["cB_hist"], whole["cB_hist"]) and np.array_equal(m["c_hist"], whole["c_hist"])
    assert m["dBfs_min"] == whole["dBfs_min"] and m["dBfs_max"] == whole["dBfs_max"]


def test_frame_range_shards_of_an_odd_width(engine):
    """A total width that is not a multiple of 8 keeps the whole message on the generic kernel while its shards (cut on
    multiples of 8) use the fused one: the two fp32 FFTs may then differ at quantisation ties, never by more."""
    from spectro_b200 import sharding
    fmt, sw, n, width, S = "CS16", 4, 1024, 203, 150001
    buf = O.synth(fmt, 0, S, S, 0x5EC78000).tobytes()
    w, wt = O.window("hann", n)
    whole = engine.render(buf, fmt, n, width, w, 1 / wt, 6, 30, CM256)
    gw = gray_from_image(whole["image"], CM256, n, width)
    nbad = 0
    for sh in sharding.plan_shards(S, n, width, 3):
        sub = buf[sh["sample_first"] * sw:(sh["sample_first"] + sh["sample_count"]) * sw]
        r = engine.render(sub, fmt, n, sh["width"], w, 1 / wt, 6, 30, CM256, shard=sharding.shard_fields(sh, S, sw, width))
        d = gray_from_image(r["image"], CM256, n, sh["width"]) - gw[sh["frame_first"]:sh["frame_first"] + sh["width"]]
        assert np.abs(d).max() <= 1
        nbad += int((d != 0).sum())
    assert nbad <= 1e-3 * n * width


# ------------------------------------------------------------------ properties at larger sizes
def test_properties_at_scale(engine):
    """C2-like geometry (cs16, N=4096, hop N) at 16 Mi samples, device resident, checked through
    size-independent properties: histogram totals, determinism, sampled frames vs the oracle."""
    n, width = 4096, 4096
    S = n * width
    d = engine.alloc(S * 4)
    engine.synth_fill(d, "CS16", 0, S, S, 0x5EC70002)
    w, wt = O.window("blackmanHarris", n)
    r1 = engine.render(d, "CS16", n, width, w, 1 / wt, 6, 30, CM256, byte_length=S * 4)
    r2 = engine.render(d, "CS16", n, width, w, 1 / wt, 6, 30, CM256, byte_length=S * 4)
    engine.free(d)
    assert int(r1["c_hist"].sum()) == n * width
    assert int(r1["cB_hist"].sum()) <= n * width and int(r1["cB_hist"].sum()) >= n * width - 1000
    for k in ("image", "cB_hist", "c_hist", "gauge_mins", "gauge_maxs", "gauge_amps"):
        assert np.array_equal(r1[k], r2[k]), k                # deterministic (integer atomics only)
    # colour histogram == histogram of the image itself
    g = gray_from_image(r1["image"][:, :256], CM256, n, 256)
    # sampled frames against the oracle (frames are independent: stride == n exactly)
    for x in (0, 1, 255):
        fb = O.synth("CS16", x * n, n, S, 0x5EC70002).tobytes() + O.synth("CS16", 0, n, S, 0x5EC70002).tobytes()
        o = O.render(fb, "CS16", n, 2, w, 1 / wt, 6, 30, CM256, taps=True)
        d_ = g[x].astype(int) - o.gray[0].astype(int)
        assert np.abs(d_).max() <= 1 and (d_ != 0).sum() <= 8


@pytest.mark.parametrize("tag,fmt,n,window,S", [
    ("C1", "CU8", 1024, "hann", 9765 * 1024),                 # BASELINE configs[0]: 10 s @ 1 MS/s, hop N (9 765 frames)
    ("C2", "CS16", 4096, "blackmanHarris", 100 << 20),        # configs[1], the headline: 100 Mi samples, 25 600 frames
    ("C3", "CF32", 32768, "hann", 1 << 30),                   # configs[2] at zoom x1: 2^30 samples (8 GiB + a 4 GiB image)
    ("C4", "CU12", 512, "bartlett", 1 << 26),                 # configs[3]: one packed format on the small-N kernel
    ("C5", "CF32", 65536, "hann", 1 << 31)])                  # configs[4]: two of the eight shards of the 2^33-sample capture
def test_baseline_configs_at_full_size(engine, tag, fmt, n, window, S):
    """BASELINE.json's configurations at their stated sizes, device resident, generated on the device: histogram totals
    (64-bit counters), and groups of 8 frames - first, last, spread - against the float64 oracle (at hop N a group of 8
    frames is itself a message of 8 N samples with the same frame positions), pixels and gauges."""
    from spectro_b200 import _lib
    sw = _lib.load().sp_sample_width(_lib.format_id(fmt))
    width = S // n
    seed = 0x5EC70000 + n
    w, wt = O.window(window, n)
    d_in = engine.alloc(S * sw + 256)
    engine.synth_fill(d_in, fmt, 0, S, S, seed)
    d_img, d_g = engine.alloc(4 * width * n), engine.alloc(3 * width)
    d_hist, d_mm = engine.alloc(8 * (1000 + len(CM256))), engine.alloc(16)
    try:
        rq, keep = engine.make_request(d_in, fmt, n, width, w, 1 / wt, 6, 30, CM256, byte_length=S * sw)
        rp = engine.render_enqueue(rq, d_img, (d_g, d_g + width, d_g + 2 * width), d_hist, d_hist + 8000, d_mm)
        engine.render_finish(rp)
        hist = np.empty(1000 + len(CM256), np.uint64)
        engine.d2h(hist, d_hist)
        assert int(hist[1000:].sum()) == width * n
        assert width * n - 1000 <= int(hist[:1000].sum()) <= width * n
        gauges = np.empty(3 * width, np.uint8)
        engine.d2h(gauges, d_g)
        rows = (n // 2 - np.arange(n)) % n                                           # bin -> row, lib/worker.js:90
        groups = sorted({int(round(i * (width - 8) / 4)) // 8 * 8 for i in range(5)})
        off1 = px = 0
        for x in groups:
            raw = O.synth(fmt, x * n, 8 * n, S, seed)
            ora = O.render(raw, fmt, n, 8, w, 1 / wt, 6, 30, CM256, taps=True)
            # the group's pixels: 8 consecutive columns of every image row (32 bytes at pitch 4 * width)
            tile = np.empty((n, 8, 4), np.uint8)
            row = np.empty(32, np.uint8)
            for y in range(0, n, max(1, n // 512)):                                   # up to 512 rows per group keep the test quick
                engine.d2h(row, d_img + 4 * (y * width + x))
                tile[y] = row.reshape(8, 4)
            ys = np.arange(0, n, max(1, n // 512))
            gi = cmap_index_image(tile[ys], CM256)
            oi = np.empty((n, 8), np.int64)
            oi[rows, :] = ora.gray.T.astype(np.int64)
            d = np.abs(gi - oi[ys])
            assert d.max() <= 1, (tag, x, int(d.max()))
            off1 += int((d == 1).sum()); px += d.size
            for k, name in enumerate(("gauge_mins", "gauge_maxs", "gauge_amps")):
                assert np.abs(gauges[k * width + x:k * width + x + 8].astype(int) - getattr(ora, name).astype(int)).max() <= 1, (tag, name, x)
        assert off1 <= max(2, int(1e-3 * px)), (tag, off1, px)
    finally:
        for d in (d_in, d_img, d_g, d_hist, d_mm):
            engine.free(d)


# ------------------------------------------------------------------ pipelined host path == single shot
@pytest.mark.parametrize("case", [("CS16", 1024, 1000, 700, False), ("CU8", 256, 4001, 300, False),
                                  ("CS16", 4096, 800, 4096, False), ("CF32", 512, 1500, 512, True),
                                  ("CF32", 8192, 200, 5000, False)])
def test_pipelined_host_path_is_bit_identical(engine, case, monkeypatch):
    """Long host-buffer messages are streamed in frame-range chunks over three CUDA streams
    (H2D / render / D2H overlap); the chunks are shards of the same message, so nothing may change."""
    fmt, n, width, hop, wf = case
    S = hop * (width - 1) + n + 3
    buf = O.synth(fmt, 0, S, S, 0x5EC79000 + n).tobytes()
    w, wt = O.window("hann", n)
    monkeypatch.setenv("SP_PIPE_MB", "0")
    one = engine.render(buf, fmt, n, width, w, 1 / wt, 6, 30, CM256, waterfall=wf)
    monkeypatch.setenv("SP_PIPE_MB", "1")
    pin = __import__("spectro_b200").PinnedBuffer(len(buf))
    pin.array[:] = np.frombuffer(buf, np.uint8)
    pipe = engine.render(pin.array, fmt, n, width, w, 1 / wt, 6, 30, CM256, waterfall=wf)
    for k in ("image", "cB_hist", "c_hist", "gauge_mins", "gauge_maxs", "gauge_amps"):
        assert np.array_equal(one[k], pipe[k]), k
    assert one["dBfs_min"] == pipe["dBfs_min"] and one["dBfs_max"] == pipe["dBfs_max"]
    assert pipe["kernel_launches"] > one["kernel_launches"]          # it really was chunked
    pin.free()


def test_zoom_levels_in_one_pass(engine):
    """C3 shape at test size: zoom x1/x2/x4/x8 images of one capture from ONE upload (sp_render_zooms); every level
    has its own stride (SURVEY A.6) and must equal the separately rendered message exactly, and the x1 level must
    hold parity with the oracle."""
    fmt, n, base = "CF32", 2048, 24
    S = n * base + 777
    buf = O.synth(fmt, 0, S, S, 0x5EC70003).tobytes()
    w, wt = O.window("blackmanHarris", n)
    widths = [base * z for z in (1, 2, 4, 8)]
    outs = engine.render_zooms(buf, fmt, n, widths, w, 1 / wt, 6, 30, CM256)
    for width, o in zip(widths, outs):
        one = engine.render(buf, fmt, n, width, w, 1 / wt, 6, 30, CM256)
        for k in ("image", "cB_hist", "c_hist", "gauge_mins", "gauge_maxs", "gauge_amps"):
            assert np.array_equal(one[k], o[k]), (width, k)
        assert one["dBfs_min"] == o["dBfs_min"] and one["dBfs_max"] == o["dBfs_max"]
    ora = O.render(buf, fmt, n, widths[0], w, 1 / wt, 6, 30, CM256, taps=True)
    check_parity(outs[0], ora, CM256, n, widths[0], False, None, "zoom x1")


# ------------------------------------------------------------------ the N = 4096 "64 x 64" kernel (render_r64_kernel)
# Reached with spectrogram layout, cmap_len <= 256, width % 8 == 0 and at least 16 frames inside the buffer.
@pytest.mark.parametrize("fmt", O.FORMATS)
def test_r64_all_formats(engine, fmt):
    n, width, hop = 4096, 48, 1501                       # overlapping frames at a fractional stride
    S = hop * (width - 1) + n + 5
    buf = O.synth(fmt, 0, S, S, 0x5EC7A000).tobytes()
    gpu, ora, _ = run_both(engine, buf, fmt, n, width, "blackmanHarris", want_db=False)
    if fmt in ("CU4", "CS4", "CU8", "CS8", "CU12", "CS12", "CU16", "CS16", "CF32"):      # formats with a specialised build
        assert "render_r64_kernel" in engine.kernel_plan(fmt, n)


@pytest.mark.parametrize("gain,rng,cmap_len", [(0, 60, 256), (-20, 5, 256), (6, 30, 64), (40, 100, 2), (6, -30, 256)])
def test_r64_colour_scales(engine, gain, rng, cmap_len):
    """The joint histogram index must decode for any gain / range / colormap length (lib/worker.js:37-39,111-113)."""
    n, width = 4096, 32
    S = n * width
    buf = O.synth("CS16", 0, S, S, 0x5EC7A001).tobytes()
    run_both(engine, buf, "CS16", n, width, "hann", gain=gain, rng=rng, cmap=injective_cmap(cmap_len), want_db=False)


def test_r64_non_finite_pixels(engine):
    """|X|^2 == 0, +inf and NaN take the per-frame fix-up path of the joint histogram (~~(+-Infinity) == ~~NaN == 0)."""
    n, width = 4096, 32
    w, wt = O.window("hann", n)
    # every other group of frames silent: d0 = -inf -> bin 0, colour 0, min -inf
    x = np.frombuffer(O.synth("CS16", 0, n * width, n * width, 0x5EC7A002).tobytes(), "<i2").reshape(width, n, 2).copy()
    x[3:9] = 0
    x[20] = 0
    buf = x.tobytes()
    ora = O.render(buf, "CS16", n, width, w, 1 / wt, 6, 30, CM256, taps=True)
    gpu = engine.render(buf, "CS16", n, width, w, 1 / wt, 6, 30, CM256)
    check_parity(gpu, ora, CM256, n, width, False, None, "r64 silent frames")
    assert gpu["cB_hist"][0] >= 7 * n and gpu["dBfs_min"] == -np.inf
    # float input: a NaN poisons its frame (every bin NaN: colour 0, dB bin 0); a silent frame next to it
    f = np.frombuffer(O.synth("CF32", 0, n * width, n * width, 0x5EC7A003).tobytes(), "<f4").reshape(width, n, 2).copy()
    f[2, 100, 0] = np.nan
    f[11] = 0
    buf = f.tobytes()
    with np.errstate(all="ignore"):
        ora = O.render(buf, "CF32", n, width, w, 1 / wt, 6, 30, CM256, taps=True)
    gpu = engine.render(buf, "CF32", n, width, w, 1 / wt, 6, 30, CM256)
    g = gray_from_image(gpu["image"], CM256, n, width)
    for fr in (2, 11):
        assert np.array_equal(g[fr], ora.gray[fr]), fr
    ties = 2 * int(1e-3 * n * width)                          # quantisation ties of the ordinary pixels (helpers.PIXEL_FRAC)
    assert int(np.abs(gpu["cB_hist"].astype(np.int64) - ora.cB_hist.astype(np.int64)).sum()) <= ties
    assert int(np.abs(gpu["c_hist"].astype(np.int64) - ora.c_hist.astype(np.int64)).sum()) <= ties
    assert gpu["cB_hist"][0] == ora.cB_hist[0] and gpu["c_hist"][0] >= 2 * n
    assert gpu["dBfs_min"] == ora.dBfs_min == -np.inf and abs(gpu["dBfs_max"] - ora.dBfs_max) <= DB_TOL
    # +inf samples and |X|^2 beyond fp32 range are outside the reference's domain (samples lie in [-1, 1]); which bins
    # become NaN and which +inf then depends on the butterfly order, so only the bookkeeping is checked: every pixel is
    # counted once in c_hist, and the other frames are untouched
    f[5, 7, 1] = np.inf
    f[9, :, :] *= np.float32(3e19)
    gpu2 = engine.render(f.tobytes(), "CF32", n, width, w, 1 / wt, 6, 30, CM256)
    assert int(gpu2["c_hist"].sum()) == n * width
    g2 = gray_from_image(gpu2["image"], CM256, n, width)
    keep = [i for i in range(width) if i not in (5, 9)]
    assert np.array_equal(g2[keep], g[keep])


@pytest.mark.parametrize("form", ["ring", "hbm"])
@pytest.mark.parametrize("n,width", [(8192, 32), (16384, 48), (32768, 16), (65536, 16)])
def test_r64_four_step(engine, monkeypatch, n, width, form):
    monkeypatch.setenv("SP_FOURSTEP", form)
    S = n * width // 2 + n + 9                                 # ~50 % overlap
    buf = O.synth("CS16", 0, S, S, 0x5EC7A100 + n).tobytes()
    run_both(engine, buf, "CS16", n, width, "hann", want_db=False)


def test_r64_matches_generic_kernel(engine):
    """The same message through render_r64_kernel (spectrogram) and render_kernel (waterfall layout is not
    eligible for the fast path): the two fp32 FFTs may only differ at quantisation ties."""
    n, width = 4096, 64
    S = n * width
    buf = O.synth("CS16", 0, S, S, 0x5EC7A004).tobytes()
    w, wt = O.window("blackmanHarris", n)
    a = engine.render(buf, "CS16", n, width, w, 1 / wt, 0, 90, CM256)
    b = engine.render(buf, "CS16", n, width, w, 1 / wt, 0, 90, CM256, waterfall=True)
    ga = gray_from_image(a["image"], CM256, n, width)
    gb = gray_from_image(b["image"], CM256, n, width, waterfall=True)
    d = ga - gb
    assert np.abs(d).max() <= 1 and (d != 0).sum() <= 2e-3 * d.size
    assert np.abs(a["c_hist"].astype(np.int64) - b["c_hist"].astype(np.int64)).sum() <= 2 * (d != 0).sum()
    assert np.abs(a["cB_hist"].astype(np.int64) - b["cB_hist"].astype(np.int64)).sum() <= 4e-3 * d.size
    assert np.array_equal(a["gauge_amps"], b["gauge_amps"])


# ------------------------------------------------------------------ N = 512 / 1024 / 2048 as 64 x C (render_rc_kernel)
@pytest.mark.parametrize("n", [256, 512, 1024, 2048])
@pytest.mark.parametrize("fmt", ["CS16", "CU8", "CF32", "CU12", "CS4"])
def test_rc_sizes_and_formats(engine, n, fmt):
    tile = 65536 // n
    width, hop = 3 * tile + 8, int(n * 0.37) + 1              # three full tiles + a remainder for the generic kernel
    S = hop * (width - 1) + n + 3
    buf = O.synth(fmt, 0, S, S, 0x5EC7B000 + n).tobytes()
    run_both(engine, buf, fmt, n, width, "hann", want_db=False)
    assert ("render_rc_kernel" if n == 2048 else "render_w_kernel") in engine.kernel_plan(fmt, n)


@pytest.mark.parametrize("n", [256, 512, 1024, 2048])
def test_rc_hop_n_and_non_finite(engine, n):
    tile = 65536 // n
    width = 2 * tile
    S = n * width
    w, wt = O.window("blackmanHarris", n)
    x = np.frombuffer(O.synth("CS16", 0, S, S, 0x5EC7B100 + n).tobytes(), "<i2").reshape(width, n, 2).copy()
    x[5:9] = 0
    x[tile + 3] = 0
    buf = x.tobytes()
    ora = O.render(buf, "CS16", n, width, w, 1 / wt, 6, 30, CM256, taps=True)
    gpu = engine.render(buf, "CS16", n, width, w, 1 / wt, 6, 30, CM256)
    check_parity(gpu, ora, CM256, n, width, False, None, f"rc n={n} silent frames")
    assert gpu["cB_hist"][0] >= 5 * n and gpu["dBfs_min"] == -np.inf
    f = np.frombuffer(O.synth("CF32", 0, S, S, 0x5EC7B200 + n).tobytes(), "<f4").reshape(width, n, 2).copy()
    f[2, 100, 0] = np.nan
    buf = f.tobytes()
    with np.errstate(all="ignore"):
        ora = O.render(buf, "CF32", n, width, w, 1 / wt, 0, 60, CM256, taps=True)
    gpu = engine.render(buf, "CF32", n, width, w, 1 / wt, 0, 60, CM256)
    check_parity(gpu, ora, CM256, n, width, False, None, f"rc n={n} NaN frame")


def test_repeated_renders_are_bit_identical(engine):
    """Race detector of last resort: the fused kernels hand tiles between warpgroups through mbarriers (which
    compute-sanitizer racecheck does not model); twelve renders of the same message must agree to the last byte and count."""
    for fmt, n, width in (("CS16", 4096, 64), ("CU8", 1024, 200), ("CS4", 128, 300), ("CF32", 8192, 24)):
        S = n * (width // 2) + 999
        buf = O.synth(fmt, 0, S, S, 0x5EC7A000 + n).tobytes()
        w, wt = O.window("hann", n)
        first = engine.render(buf, fmt, n, width, w, 1 / wt, 6, 30, CM256)
        for _ in range(11):
            again = engine.render(buf, fmt, n, width, w, 1 / wt, 6, 30, CM256)
            for k in ("image", "cB_hist", "c_hist", "gauge_mins", "gauge_maxs", "gauge_amps"):
                assert np.array_equal(first[k], again[k]), (fmt, n, k)
            assert first["dBfs_min"] == again["dBfs_min"] and first["dBfs_max"] == again["dBfs_max"]


# ------------------------------------------------------------------ randomized sweep over the whole option space
def _random_cases(count, seed):
    rng = np.random.default_rng(seed)
    fmts = list(O.FORMATS)
    cases = []
    for i in range(count):
        n = int(2 ** rng.integers(3, 15))                       # 8 .. 16384
        fmt = fmts[int(rng.integers(0, len(fmts)))]
        width = int(rng.choice([2, 3, 7, 8, 9, 15, 16, 17, 24, 31, 33, 40, 64, 65, 100]))
        if n >= 4096:
            width = min(width, 24)
        hop = float(rng.choice([0.0, 0.37, 1.0, 1.0, 2.5]))     # x n: all frames on one position ... skipping data
        S = n + int(hop * n * (width - 1)) + int(rng.integers(0, 50))
        window = O.WINDOWS[int(rng.integers(0, len(O.WINDOWS)))]
        gain = int(rng.choice([-10, 0, 6, 20, 45]))
        rng_db = int(rng.choice([6, 30, 60, 120, -30]))
        cmap_len = int(rng.choice([2, 64, 256, 256, 300]))
        chm = bool(rng.integers(0, 4) == 0)
        wf = bool(rng.integers(0, 4) == 0)
        ragged = int(rng.integers(0, 5) == 0)
        cases.append((i, fmt, n, width, S, window, gain, rng_db, cmap_len, chm, wf, ragged))
    return cases


@pytest.mark.parametrize("case", _random_cases(72, 20261017), ids=lambda c: "r%02d-%s-n%d-w%d" % (c[0], c[1], c[2], c[3]))
def test_randomized_option_sweep(engine, case):
    """Seeded random points of (format, N, width, hop, window, gain, range, cmap length, channel mode, waterfall, ragged tail):
    every one must meet the parity bars against the oracle (which equals the reference, tests/test_reference_js.py)."""
    i, fmt, n, width, S, window, gain, rng_db, cmap_len, chm, wf, ragged = case
    buf = O.synth(fmt, 0, S, S, 0x5EC7B000 + i).tobytes()
    sw = O.SAMPLE_WIDTH[O.fmt_id(fmt)]
    if ragged:                                               # drop a partial sample: keep the typed-array element size
        elem = 1 if sw <= 3 else (2 if sw == 4 else (8 if fmt == "CF64" else 4))
        if sw > elem:
            buf = buf[:len(buf) - elem]
    if len(buf) // sw < n:
        pytest.skip("shorter than one frame")
    run_both(engine, buf, fmt, n, width, window, gain, rng_db, injective_cmap(cmap_len), chm, wf, want_db=not chm,
             label="random case %d" % i)


def test_async_messages_equal_synchronous_renders(engine):
    """sp_render_async / sp_render_wait: messages in flight two at a time through the pipelined host path (the device chunk
    buffers, the accumulators and the gauges are shared by consecutive messages) must reproduce sp_render byte for byte, whatever
    the order of waits; different windows / colormaps / sizes in a row exercise the table re-uploads between overlapping messages."""
    import spectro_b200
    msgs = [("CS16", 4096, 1000, "hann", CM256, False), ("CS16", 4096, 1000, "hann", CM256, False), ("CU8", 1024, 2400, "blackmanHarris", injective_cmap(64), False),
            ("CS16", 4096, 520, "bartlett", CM256, True), ("CF32", 512, 3000, "hann", CM256, False), ("CS16", 4096, 1000, "hann", CM256, False)]
    bufs, sync = [], []
    for i, (fmt, n, width, win, cm, wf) in enumerate(msgs):
        S = n * (width // 2 + 3) + 29
        pb = spectro_b200.PinnedBuffer(S * O.SAMPLE_WIDTH[O.fmt_id(fmt)])
        pb.array[:] = np.frombuffer(O.synth(fmt, 0, S, S, 0xA5A50000 + i).tobytes(), np.uint8)
        bufs.append(pb)
        w, wt = O.window(win, n)
        sync.append(engine.render(pb.array, fmt, n, width, w, 1 / wt, 6, 30, cm, waterfall=wf))
        assert sync[-1]["kernel_launches"] > 0
    outs = [spectro_b200.PinnedBuffer(4 * m[1] * m[2]) for m in msgs]
    handles = []
    for i, (fmt, n, width, win, cm, wf) in enumerate(msgs):
        w, wt = O.window(win, n)
        handles.append(engine.render_async(bufs[i].array, fmt, n, width, w, 1 / wt, 6, 30, cm, waterfall=wf, out_image=outs[i].array))
    for i in (1, 0, 2, 5, 4, 3):                               # any order, also after the slot was recycled
        r = engine.wait(handles[i])
        for k in ("image", "cB_hist", "c_hist", "gauge_mins", "gauge_maxs", "gauge_amps"):
            assert np.array_equal(r[k], sync[i][k]), (i, k)
        assert r["dBfs_min"] == sync[i]["dBfs_min"] and r["dBfs_max"] == sync[i]["dBfs_max"], i
    # a synchronous render between asynchronous ones
    h = engine.render_async(bufs[0].array, *msgs[0][:3], *(lambda w: (w[0], 1 / w[1]))(O.window("hann", 4096)), 6, 30, CM256, out_image=outs[0].array)
    w, wt = O.window("hann", 4096)
    mid = engine.render(bufs[1].array, "CS16", 4096, 1000, w, 1 / wt, 6, 30, CM256)
    r = engine.wait(h)
    assert np.array_equal(mid["image"], sync[1]["image"]) and np.array_equal(r["image"], sync[0]["image"])


# ------------------------------------------------------------------ multi-device engine (sp_create with ndev > 1)
def _gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs")
def test_multi_device_engine_equals_single_device(engine):
    """One C-ABI engine over several GPUs: sp_render shards a whole host-buffer message by frame range (cuts on multiples of
    8 frames, global positions, halo) and the devices write their bands straight into the caller's image; histograms and
    min / max are merged like lib/spectroplot.js:1229-1238.  The result must be the single-device result, byte for byte."""
    import spectro_b200
    ndev = min(_gpu_count(), 8)
    multi = spectro_b200.Engine(list(range(ndev)))
    assert multi.lib.sp_device_count(multi.h) == ndev
    try:
        cases = [("CS16", 4096, 1024, 4096, False, False), ("CU8", 1024, 4000, 700, False, False), ("CF32", 512, 960, 512, True, False),
                 ("CS16", 4096, 200, 3000, False, True), ("CF32", 8192, 64, 8192, False, False), ("CS8", 128, 4003, 100, False, False),
                 ("CU12", 256, 24, 256, False, False)]
        for fmt, n, width, hop, wf, chm in cases:
            S = hop * (width - 1) + n + 5
            buf = O.synth(fmt, 0, S, S, 0x5EC7C000 + n).tobytes()
            w, wt = O.window("hann", n)
            one = engine.render(buf, fmt, n, width, w, 1 / wt, 6, 30, CM256, channel_mode=chm, waterfall=wf)
            many = multi.render(buf, fmt, n, width, w, 1 / wt, 6, 30, CM256, channel_mode=chm, waterfall=wf)
            exact = width % 8 == 0
            for k in ("image", "cB_hist", "c_hist", "gauge_mins", "gauge_maxs", "gauge_amps"):
                if exact:
                    assert np.array_equal(one[k], many[k]), (fmt, n, width, k)
                elif k == "image":                             # odd widths: a frame may change kernels at a cut (ties only)
                    assert (one[k] != many[k]).any(axis=2).mean() <= 1e-3
            for k, tol in (("dBfs_min", 0.05), ("dBfs_max", 0.01)):
                assert one[k] == many[k] or (not exact and abs(one[k] - many[k]) <= tol), (fmt, n, width, k, one[k], many[k])
            assert int(many["c_hist"].sum()) == n * width
            if width >= 16 * ndev:
                assert many["kernel_launches"] > one["kernel_launches"]      # it really ran on several devices
        # a ragged tail travels with the last shard; errors carry the device's message
        buf = O.synth("CU8", 0, 40001, 40001, 5).tobytes()[:-1]
        w, wt = O.window("hann", 256)
        one = engine.render(buf, "CU8", 256, 800, w, 1 / wt, 6, 30, CM256)
        many = multi.render(buf, "CU8", 256, 800, w, 1 / wt, 6, 30, CM256)
        assert np.array_equal(one["image"], many["image"]) and np.array_equal(one["cB_hist"], many["cB_hist"])
        with pytest.raises(spectro_b200.SpError, match="power of 2"):
            multi.render(buf, "CU8", 100, 800, w[:100], 1 / wt, 6, 30, CM256)
        # pinned input: every device streams its own byte range through the pipelined path
        S = 4096 * 2048
        pin = spectro_b200.PinnedBuffer(S * 4)
        pin.array[:] = O.synth("CS16", 0, S, S, 77)
        w, wt = O.window("blackmanHarris", 4096)
        one = engine.render(pin.array, "CS16", 4096, 2048, w, 1 / wt, 6, 30, CM256)
        many = multi.render(pin.array, "CS16", 4096, 2048, w, 1 / wt, 6, 30, CM256)
        for k in ("image", "cB_hist", "c_hist", "gauge_mins", "gauge_maxs", "gauge_amps"):
            assert np.array_equal(one[k], many[k]), k
        pin.free()
    finally:
        multi.close()


@pytest.mark.parametrize("fmt,n,W", [("CS16", 4096, 256), ("CF32", 8192, 64), ("CU8", 512, 1000)])
def test_render_shards_nccl_merge_equals_single_device(engine, fmt, n, W):
    """sp_render_shards (C ABI, no torch): device-GENERATED shards on a multi-device engine, the histograms and min / max merged
    by ONE grouped NCCL all-reduce on the engines' streams (lib/spectroplot.js:1229-1238 over NVLink) == the single-device
    result.  Needs two GPUs."""
    import torch
    import spectro_b200
    from spectro_b200 import sharding, _lib
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    G = 2
    S = n * W // 2 + 5
    sw = _lib.load().sp_sample_width(_lib.format_id(fmt))
    w, wt = O.window("hann", n)
    seed = 0xC5C5 + n
    # single device: the whole message from a device-generated capture
    d_all = engine.alloc(S * sw + 256)
    engine.synth_fill(d_all, fmt, 0, S, S, seed)
    host = np.empty(S * sw, np.uint8)
    engine.d2h(host, d_all)
    engine.free(d_all)
    one = engine.render(host, fmt, n, W, w, 1 / wt, 6, 30, CM256)
    multi = spectro_b200.Engine(list(range(G)))
    try:
        plan = sharding.plan_shards(S, n, W, G)
        rqs, rps, bufs, keep = [], [], [], []
        for g, sh in enumerate(plan):
            multi.select_device(g)
            nb = sh["sample_count"] * sw
            d_in = multi.alloc(nb + 256)
            multi.synth_fill(d_in, fmt, sh["sample_first"], sh["sample_count"], S, seed)      # generated on ITS device
            d_img, d_g = multi.alloc(4 * sh["width"] * n), multi.alloc(3 * sh["width"])
            d_hist, d_mm = multi.alloc(8 * (1000 + len(CM256))), multi.alloc(16)
            rq, k = multi.make_request(d_in, fmt, n, sh["width"], w, 1 / wt, 6, 30, CM256, byte_length=nb,
                                       shard=sharding.shard_fields(sh, S, sw, W))
            keep.append(k)
            p = lambda v: C.c_void_p(int(v))
            rps.append(_lib.Reply(p(d_img), p(d_g), p(d_g + sh["width"]), p(d_g + 2 * sh["width"]), p(d_hist), p(d_hist + 8000),
                                  0.0, 0.0, 0.0, 0, p(d_mm)))
            rqs.append(rq)
            bufs.append((d_in, d_img, d_g, d_hist, d_mm))
        out = multi.render_shards(rqs, rps)
        for g, sh in enumerate(plan):
            multi.select_device(g)
            d_in, d_img, d_g, d_hist, d_mm = bufs[g]
            img = np.empty((n, sh["width"], 4), np.uint8)
            multi.d2h(img, d_img)
            assert np.array_equal(img, one["image"][:, sh["frame_first"]:sh["frame_first"] + sh["width"]]), g
            hist = np.empty(1000 + len(CM256), np.uint64)
            multi.d2h(hist, d_hist)
            # EVERY device holds the histograms of the whole message after the all-reduce
            assert np.array_equal(hist[:1000], one["cB_hist"]) and np.array_equal(hist[1000:], one["c_hist"]), g
            assert out[g].dBfs_min == one["dBfs_min"] and out[g].dBfs_max == one["dBfs_max"], g
            gg = np.empty(3 * sh["width"], np.uint8)
            multi.d2h(gg, d_g)
            assert np.array_equal(gg[:sh["width"]], one["gauge_mins"][sh["frame_first"]:sh["frame_first"] + sh["width"]])
            for d in bufs[g]:
                multi.free(d)
    finally:
        multi.close()


def test_render_shards_needs_a_multi_device_engine(engine):
    import spectro_b200
    from spectro_b200 import _lib
    rq = _lib.Request()
    rp = _lib.Reply()
    rc = engine.lib.sp_render_shards(engine.h, C.byref(rq), C.byref(rp))
    assert _lib.ERRORS[rc] == "SP_E_INVAL" and b"multi-device" in engine.lib.sp_last_error(engine.h)


def test_pipelined_shard_with_an_oversized_buffer(engine, monkeypatch):
    """A frame-range shard whose host buffer is the WHOLE capture (buffer_first_sample = 0) on the pipelined path: each chunk
    must take only the samples its frames read - the last chunk used to span to the end of the buffer and trip the
    staging-buffer check with SP_E_RANGE."""
    import spectro_b200
    monkeypatch.setenv("SP_PIPE_MB", "1")
    fmt, n, W = "CS16", 1024, 4096
    S = n * W // 2 + 7
    buf = O.synth(fmt, 0, S, S, 4242).tobytes()
    w, wt = O.window("hann", n)
    whole = engine.render(buf, fmt, n, W, w, 1 / wt, 6, 30, CM256)
    x0, x1 = 512, 2048                                   # a sub-range well inside: its frames end far before the buffer does
    shard = dict(total_byte_length=len(buf), total_width=W, frame_first=x0, buffer_first_sample=0)
    part = engine.render(buf, fmt, n, x1 - x0, w, 1 / wt, 6, 30, CM256, shard=shard)
    assert np.array_equal(part["image"], whole["image"][:, x0:x1])
    for k in ("gauge_mins", "gauge_maxs", "gauge_amps"):
        assert np.array_equal(part[k], whole[k][x0:x1]), k


@pytest.mark.parametrize("fmt,n,width", [("CS16", 4096, 40), ("CS16", 4096, 21), ("CF32", 4096, 64), ("CU8", 1024, 200), ("CS16", 2048, 37),
                                         ("CF32", 512, 136), ("CS4", 256, 300), ("CS16", 128, 1100), ("CU8", 64, 2100)])
def test_waterfall_on_the_fused_kernels(engine, fmt, n, width):
    """turnFlip / waterfall (lib/worker.js:116) through render_w_kernel / render_rc_kernel / render_r64_kernel: frame x is image row W - 1 - x,
    bin b is column (b + n/2 - 1) mod n; full and partial tiles, plus the same message through the pipelined host path."""
    S = n * (width // 2 + 3) + 11
    buf = O.synth(fmt, 0, S, S, 0x5EC7D000 + n + width).tobytes()
    gpu, ora, nbad = run_both(engine, buf, fmt, n, width, "hann", waterfall=True, want_db=False)
    assert gpu["image"].shape == (width, n, 4)
    plain = engine.render(buf, fmt, n, width, *O.window("hann", n)[:1], 1 / O.window("hann", n)[1], 6, 30, CM256)
    # the waterfall picture is the spectrogram transposed and flipped both ways, exactly: both layouts come from the same
    # kernel (render_w_kernel, render_rc_kernel or render_r64_kernel) at every fused size
    flipped = plain["image"].transpose(1, 0, 2)[::-1, ::-1]
    assert np.array_equal(gpu["image"], flipped)
    for k in ("cB_hist", "c_hist", "gauge_mins", "gauge_maxs", "gauge_amps"):
        assert np.array_equal(gpu[k], plain[k]), k


@pytest.mark.parametrize("fmt,n,width,wf", [("CS16", 64, 2100, False), ("CU8", 128, 1100, False), ("CS16", 256, 520, True), ("CF32", 512, 270, False),
                                            ("CS16", 512, 136, False), ("CU8", 1024, 140, False), ("CS8", 1024, 72, True)])
def test_split_real_on_the_warp_kernel(engine, fmt, n, width, wf):
    """channelMode inside render_w_kernel (N = 64 .. 1024, the reference's everyday sizes): bin i pairs with bin n - i in lane
    (T - t) mod T of the same frame, exchanged through the frame's area of the warp's buffer; full and partial tiles, both layouts."""
    S = n * (width // 2 + 3) + 17
    buf = O.synth(fmt, 0, S, S, 0x5EC7F000 + n + width).tobytes()
    gpu, ora, nbad = run_both(engine, buf, fmt, n, width, "hann", channel_mode=True, waterfall=wf, want_db=False)
    plan = engine.kernel_plan(fmt, n, True)
    assert "render_w_kernel" in plan and "split-real" in plan
    g = gray_from_image(gpu["image"], CM256, n, width, wf)
    assert (g[:, n // 2] == 0).all() and gpu["dBfs_min"] == -np.inf


@pytest.mark.parametrize("fmt,width,wf", [("CS16", 40, False), ("CF32", 21, False), ("CS16", 24, True), ("CU8", 64, False)])
def test_split_real_on_the_fused_kernel(engine, fmt, width, wf):
    """channelMode (two real channels, lib/fft_nayuki.js:103-119) inside render_r64_kernel: bin i pairs with bin n - i held by
    thread 64 - t, exchanged through the stream's buffer; bins 0 and n/2 follow the reference (imag[0] = 0, both parts of n/2 = 0)."""
    n = 4096
    S = n * (width // 2 + 3) + 17
    buf = O.synth(fmt, 0, S, S, 0x5EC7E000 + width).tobytes()
    gpu, ora, nbad = run_both(engine, buf, fmt, n, width, "hann", channel_mode=True, waterfall=wf, want_db=False)
    assert "render_r64_kernel" in engine.kernel_plan(fmt, n)
    # the n/2 row is -inf (|X|^2 == 0): colour 0 and dB bin 0 (~~(+Infinity) == 0), like the reference
    g = gray_from_image(gpu["image"], CM256, n, width, wf)
    assert (g[:, n // 2] == 0).all() and gpu["dBfs_min"] == -np.inf
