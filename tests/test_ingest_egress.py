"""The steps either side of the render path (SURVEY §8f rows 2-4): capture ingestion incl. the WAV front end, image egress."""
import io
import json
import os
import struct
import wave

import numpy as np
import pytest

from helpers import restored_cmap_tables
from oracle import oracle as O


@pytest.fixture(autouse=True)
def _shipped_cmap_tables():
    with restored_cmap_tables():
        yield


def wav_bytes(frames, rate=48000, width=2):
    """frames: int array [n][channels] -> PCM WAV bytes (python's wave module)."""
    b = io.BytesIO()
    with wave.open(b, "wb") as w:
        w.setnchannels(frames.shape[1]); w.setsampwidth(width); w.setframerate(rate)
        if width == 2:
            w.writeframes(frames.astype("<i2").tobytes())
        elif width == 1:
            w.writeframes(frames.astype(np.uint8).tobytes())
        elif width == 3:
            raw = frames.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :3]
            w.writeframes(raw.tobytes())
    return b.getvalue()


def test_wav_front_end_matches_webaudio_scaling():
    from spectro_b200.ingest import decode_wav
    x = np.array([[0, 32767], [-32768, 1], [16384, -16384]], np.int64)
    d, rate, ch = decode_wav(wav_bytes(x, 44100, 2))
    assert rate == 44100 and ch == 2 and d.dtype == np.float32
    assert np.array_equal(d, (x / 32768.0).astype(np.float32).reshape(-1))
    # mono is duplicated into both channels, extra channels are dropped (lib/samples.js:268-275, 286-293)
    d, _, ch = decode_wav(wav_bytes(x[:, :1], 8000, 2))
    assert ch == 1 and np.array_equal(d.reshape(-1, 2)[:, 0], d.reshape(-1, 2)[:, 1])
    x3 = np.array([[1, 2, 3], [4, 5, 6]], np.int64)
    d, _, ch = decode_wav(wav_bytes(x3, 8000, 2))
    assert ch == 3 and np.array_equal(d, (x3[:, :2] / 32768.0).astype(np.float32).reshape(-1))
    d, _, _ = decode_wav(wav_bytes(np.array([[0, 255], [128, 64]]), 8000, 1))            # 8-bit is unsigned
    assert np.array_equal(d, np.array([-1.0, 127 / 128, 0.0, -0.5], np.float32))
    d, _, _ = decode_wav(wav_bytes(np.array([[-8388608, 8388607]]), 8000, 3))
    assert np.array_equal(d, np.array([-1.0, 8388607 / 8388608], np.float32))
    # IEEE float WAV
    f = np.array([0.25, -0.5, 1.5, 0.0], "<f4")
    body = b"WAVE" + b"fmt " + struct.pack("<IHHIIHH", 16, 3, 2, 1000, 8000, 8, 32) + b"data" + struct.pack("<I", f.nbytes) + f.tobytes()
    d, rate, _ = decode_wav(b"RIFF" + struct.pack("<I", len(body)) + body)
    assert rate == 1000 and np.array_equal(d, f)
    with pytest.raises(ValueError):
        decode_wav(b"not a wav file at all")
    with pytest.raises(NotImplementedError):
        decode_wav(b"RIFF" + struct.pack("<I", 36) + b"WAVE" + b"fmt " + struct.pack("<IHHIIHH", 16, 85, 2, 1000, 8000, 8, 0) + b"data" + struct.pack("<I", 0))


def test_sampleview_wav_becomes_cf32():
    from spectro_b200.samples import SampleView
    x = (np.arange(40).reshape(20, 2) * 1000 - 9000).astype(np.int64)
    sv = SampleView("wav")
    assert sv.format == "CF32" and sv.sampleWidth == 8                       # lib/samples.js:141-148
    sv.loadBuffer(wav_bytes(x, 22050))
    assert sv.sampleCount == 20 and sv.sampleRate == 22050
    assert np.array_equal(np.frombuffer(sv.buffer, "<f4"), (x / 32768.0).astype(np.float32).reshape(-1))
    got = O.decode("CF32", sv.buffer)
    assert np.array_equal(got, (x / 32768.0).astype(np.float32).astype(np.float64))
    with pytest.raises(NotImplementedError):
        SampleView("mp3").loadBuffer(b"\x00" * 64)


def test_load_capture_and_name_parsing(tmp_path):
    from spectro_b200.ingest import load_capture
    from spectro_b200.parse_freq_rate import parseFormat, parseFreqRate
    raw = O.synth("CU8", 0, 5000, 5000, 3).tobytes()
    p = tmp_path / "g017_868.3M_1024k.cu8"
    p.write_bytes(raw)
    fd = load_capture(str(p), pinned=False)
    assert fd["name"] == "g017_868.3M_1024k.cu8" and fd["size"] == len(raw) and bytes(fd["fileBuffer"]) == raw
    assert parseFormat(fd["name"]) == "CU8" and parseFreqRate(fd["name"]) == {"freq": 868300000.0, "rate": 1024000.0}


def test_png_round_trip_and_tiles(tmp_path):
    from spectro_b200 import egress
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (64, 300, 4), dtype=np.uint8)
    img[..., 3] = 255
    data = egress.png_bytes(img)
    assert np.array_equal(egress.read_png_rgba(data), img)
    try:                                                         # an independent decoder, when the image has one
        from PIL import Image
        assert np.array_equal(np.array(Image.open(io.BytesIO(data)).convert("RGBA")), img)
    except ImportError:
        pass
    tiles = egress.write_tiles(str(tmp_path / "t"), img, tile_width=128)
    assert [os.path.basename(t) for t in tiles] == ["tile_00000000.png", "tile_00000128.png", "tile_00000256.png"]
    back = np.concatenate([egress.read_png_rgba(open(t, "rb").read()) for t in tiles], axis=1)
    assert np.array_equal(back, img)
    with pytest.raises(ValueError):
        egress.png_bytes(img[..., :3])


def test_write_reply_from_a_reference_fixture(tmp_path):
    from spectro_b200 import egress
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_js", "cu8_n256_overlap_w40.npz"))
    n, width = int(g["n"]), int(g["width"])
    reply = dict(image=g["image"].reshape(n, width, 4), cB_hist=g["cB_hist"], c_hist=g["c_hist"], gauge_mins=g["gauge_mins"],
                 gauge_maxs=g["gauge_maxs"], gauge_amps=g["gauge_amps"], dBfs_min=float(g["dBfs_min"]), dBfs_max=float(g["dBfs_max"]))
    meta = egress.write_reply(str(tmp_path / "r"), reply)
    assert meta["width"] == width and meta["height"] == n and sum(meta["c_hist"]) == n * width
    assert json.load(open(tmp_path / "r.json")) == meta
    assert np.array_equal(egress.read_png_rgba(open(tmp_path / "r.png", "rb").read()), reply["image"])


@pytest.mark.gpu
def test_file_to_pyramid_on_the_gpu(engine, tmp_path):
    """file -> pinned host -> pipelined render -> PNG tiles; a WAV capture through setData(path); a zoom pyramid on disk."""
    import spectro_b200
    from spectro_b200 import egress, ingest, windows, cmaps
    n, width = 1024, 2000
    S = 700 * (width - 1) + n
    raw = O.synth("CS16", 0, S, S, 77).tobytes()
    path = tmp_path / "cap_433.92M_250k.cs16"
    path.write_bytes(raw)
    fd = ingest.load_capture(str(path))
    assert fd["pinned"] is not None                                           # page-locked: the pipelined path overlaps the copies
    w = windows.hannWindow(n)
    cm = cmaps.cmap_bytes([list(c) for c in cmaps.cmaps["viridis_cmap"]])
    r = engine.render(fd["fileBuffer"], "CS16", n, width, np.array(w["window"]), 1 / w["weight"], 6, 30, cm)
    ora = O.render(raw, "CS16", n, width, np.array(w["window"]), 1 / w["weight"], 6, 30, cm)
    assert (r["image"] != ora.image).any(axis=2).mean() <= 1e-3
    tiles = egress.write_tiles(str(tmp_path / "tiles"), r["image"], 512)
    assert len(tiles) == 4 and np.array_equal(egress.read_png_rgba(open(tiles[1], "rb").read()), r["image"][:, 512:1024])
    fd["pinned"].free()
    # WAV through the headless API: decoded to CF32, left / right channel mode
    t = np.arange(40000)
    pcm = np.stack([12000 * np.sin(2 * np.pi * 0.05 * t), 8000 * np.sin(2 * np.pi * 0.11 * t)], 1).astype(np.int64)
    import io, wave
    b = io.BytesIO()
    with wave.open(b, "wb") as wf:
        wf.setnchannels(2); wf.setsampwidth(2); wf.setframerate(48000); wf.writeframes(pcm.astype("<i2").tobytes())
    wpath = tmp_path / "stereo.wav"
    wpath.write_bytes(b.getvalue())
    sp = spectro_b200.Spectroplot({"fftN": 512, "windowF": "hann", "cmap": "cube1", "channelMode": "L/R", "clientWidth": 600})
    res = sp.setData(str(wpath))
    assert sp.sampleView.format == "CF32" and sp.sample_rate == 48000 and res["image"].shape == (512, 400, 4)
    cf32 = (pcm / 32768.0).astype("<f4").tobytes()
    end = int(len(b.getvalue()) / 8)                                          # the reference sizes the slice from the FILE bytes (:1207)
    cube = [list(c) for c in cmaps.cmaps["cube1_cmap"]]
    wh = windows.hannWindow(512)
    ora = O.render(cf32[:8 * end], "CF32", 512, 400, np.array(wh["window"]), 1 / wh["weight"], 6, 30, cmaps.cmap_bytes(cube), True)
    assert (res["image"] != ora.image).any(axis=2).mean() <= 1e-3
    sp.destroy()
    # zoom pyramid of one capture on disk
    buf = O.synth("CF32", 0, 2048 * 24 + 5, 2048 * 24 + 5, 9).tobytes()
    wb = windows.blackmanHarrisWindow(2048)
    levels = egress.write_pyramid(str(tmp_path / "pyr"), engine, buf, "CF32", 2048, 24, (1, 2, 4), np.array(wb["window"]), 1 / wb["weight"], 6, 30, cm, 64)
    assert [l["meta"]["width"] for l in levels] == [24, 48, 96] and all(sum(l["meta"]["c_hist"]) == 2048 * l["meta"]["width"] for l in levels)
    assert len(levels[2]["tiles"]) == 2


@pytest.mark.gpu
def test_command_line_file_to_png(engine, tmp_path):
    """python -m spectro_b200 capture -> PNG + JSON: name parsing, option parsers, render, egress in one go."""
    import subprocess, sys
    from spectro_b200 import egress, windows, cmaps
    S = 200000
    raw = O.synth("CU8", 0, S, S, 21).tobytes()
    cap = tmp_path / "g005_433.92M_250k.cu8"
    cap.write_bytes(raw)
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), "..", "spectroplot-js_b200"))
    out = subprocess.run([sys.executable, "-m", "spectro_b200", str(cap), "--fftN", "1024", "--windowF", "hann", "--cmap", "viridis",
                          "--width", "800", "--out", str(tmp_path / "pic")], cwd=root, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    info = json.loads(out.stdout.strip().splitlines()[-1])
    assert info["format"] == "CU8" and info["center_freq"] == 433920000.0 and info["sample_rate"] == 250000.0
    assert info["width"] == 800 and info["height"] == 1024
    img = egress.read_png_rgba(open(tmp_path / "pic.png", "rb").read())
    w = windows.hannWindow(1024)
    cm = [list(c) for c in cmaps.cmaps["viridis_cmap"]]
    cm[0] = [0, 0, 0]; cm[-1] = [255, 255, 255]
    ora = O.render(raw, "CU8", 1024, 800, np.array(w["window"]), 1 / w["weight"], 6, 30, cmaps.cmap_bytes(cm))
    assert img.shape == ora.image.shape and (img != ora.image).any(axis=2).mean() <= 1e-3
    meta = json.load(open(tmp_path / "pic.json"))
    assert sum(meta["c_hist"]) == 800 * 1024
