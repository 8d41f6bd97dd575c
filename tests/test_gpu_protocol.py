"""The drop-in surface on a real GPU: worker message protocol and the headless Spectroplot API,
checked against the oracle's restatement of the reference's caller-side fan-out."""
import numpy as np
import pytest

from helpers import gray_from_image, restored_cmap_tables
from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _shipped_cmap_tables():
    with restored_cmap_tables():
        yield


def test_worker_message_protocol(engine):
    import spectro_b200
    from spectro_b200 import cmaps, windows
    w = spectro_b200.GpuWorker(0)
    replies = []
    w.onmessage = replies.append
    w.postMessage({"transferable": b"x"})                      # probe without .buffer: ignored (lib/worker.js:159)
    assert replies == []
    n, width = 512, 40
    S = 512 * 40
    buf = O.synth("CU8", 0, S, S, 3).tobytes()
    win = windows.hannWindow(n)
    cmap = [list(c) for c in cmaps.cmaps["viridis_cmap"]]
    cmap[0] = [0, 0, 0]; cmap[-1] = [255, 255, 255]
    msg = dict(block_norm=1.0 / win["weight"], gain=6, range=30, cmap=cmap, n=n, windowc=win["window"], width=width,
               offset=120, buffer=buf, format="cu8", channelMode=False, waterfall=False)
    w.postMessage(msg, [buf])
    assert len(replies) == 1
    d = replies[0]["data"]
    assert set(d) >= {"cB_hist", "c_hist", "dBfs_min", "dBfs_max", "offset", "gauge_mins", "gauge_maxs", "gauge_amps", "imageData"}
    assert d["offset"] == 120 and len(d["cB_hist"]) == 1000 and len(d["c_hist"]) == 256
    assert d["imageData"]["data"].shape == (4 * width * n,) and len(d["gauge_mins"]) == width
    ora = O.render(buf, "CU8", n, width, np.array(win["window"]), 1.0 / win["weight"], 6, 30, cmaps.cmap_bytes(cmap))
    img = d["imageData"]["data"].reshape(n, width, 4)
    assert (img != ora.image).any(axis=2).mean() <= 1e-3
    assert int(np.abs(d["c_hist"].astype(np.int64) - ora.c_hist.astype(np.int64)).sum()) <= 2 * int(1e-3 * n * width) + 2
    # unknown format strings fall back to CU8 like SampleView (lib/samples.js:149-155)
    msg2 = dict(msg, format="whatever")
    w.postMessage(msg2)
    assert np.array_equal(replies[1]["data"]["imageData"]["data"], d["imageData"]["data"])
    w.terminate()


def test_headless_spectroplot_matches_reference_fanout(engine):
    import spectro_b200
    from spectro_b200 import cmaps
    S = 60000
    buf = O.synth("CS16", 0, S, S, 9).tobytes()
    sp = spectro_b200.Spectroplot({"fftN": "1024", "windowF": "hann", "cmap": "hot", "gain": "6", "range": 30,
                                   "clientWidth": 1000, "workerCount": 2})
    assert sp.setOption("fftN", 512) is None                     # no data yet: processData returns nothing (:1097)
    res = sp.setData({"fileBuffer": buf, "name": "g001_433.92M_250k.cs16", "size": len(buf), "type": ""})
    assert sp.center_freq == 433920000.0 and sp.sample_rate == 250000.0 and sp.sampleFormat == "CS16"
    width = 1000 - (40 + 60 + 100)                               # clientWidth*zoom - (freqWidth + dbfsWidth + histWidth)
    assert res["width"] == width == sp.width and res["image"].shape == (512, width, 4)
    cm = [list(c) for c in cmaps.cmaps["hot_cmap"]]              # processData overwrote the endpoints in place (:1129-1130)
    assert cm[0] == [0, 0, 0] and cm[-1] == [255, 255, 255]
    w, wt = O.window("hann", 512)
    ora = O.render(buf, "CS16", 512, width, w, 1 / wt, 6, 30, cmaps.cmap_bytes(cm), workers=2)
    assert (res["image"] != ora.image).any(axis=2).mean() <= 1e-3
    assert abs(res["dBfs_max"] - ora.dBfs_max) < 0.01
    assert int(res["c_hist"].sum()) == int(ora.c_hist.sum())
    # setOptions re-renders; zoom steps by 0.5 within [1, 8] (:513-527)
    r2 = sp.setOptions({"gain": "12", "cmap": "viridis"})
    assert sp.gain == 12 and r2["width"] == width
    assert sp.zoomOut() is None
    sp.zoomIn()
    assert sp.zoom == 1.5 and sp.result["width"] == int(1000 * 1.5 - 200)
    sp.destroy()
