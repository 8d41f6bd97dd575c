"""Generate tests/golden/*.npz: small input/output vectors for the render path.

These vectors come from the
independent numpy restatement (oracle/np_restatement.py) and are cross-checked against the C
restatement before being written; SURVEY.md Appendix B's derived known-answers are stored too.
These are restatement-vs-restatement vectors; the pins against the reference's own code are
tests/golden/ref_js/ (tools/make_ref_golden.py).  Re-run:  python tools/make_golden.py
"""
import hashlib, os, sys
import numpy as np
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
from oracle import oracle as O, np_restatement as R

OUT = os.path.join(ROOT, "tests", "golden")
BUF_INLINE_MAX = 1 << 18                # larger seeded captures are stored as their recipe: every fixture stays under 1 MB
os.makedirs(OUT, exist_ok=True)


def injective_cmap(n):
    i = np.arange(n)
    return np.stack([i & 255, (i * 7 + 3) & 255, ((i >> 8) * 16 + (i * 37 & 15)) & 255], 1).astype(np.uint8)


def case(name, fmt, n, width, window, gain, rng, cmap, nsamples, seed, channel_mode=False, waterfall=False):
    buf = O.synth(fmt, 0, nsamples, nsamples, seed).tobytes()
    w, weight = R.window(window, n)
    r = R.render(buf, fmt, n, width, w, 1.0 / weight, gain, rng, cmap, channel_mode, waterfall)
    c = O.render(buf, fmt, n, width, w, 1.0 / weight, gain, rng, cmap, channel_mode, waterfall, taps=True)
    # cross-check the two restatements before trusting either
    bad = int((r["gray"] != c.gray).sum())
    assert bad <= max(1, r["gray"].size // 100000), (name, bad)
    fin = np.isfinite(c.db) & np.isfinite(r["db"])
    assert np.abs(r["db"][fin] - c.db[fin]).max() < 1e-9, name
    if len(buf) > BUF_INLINE_MAX:       # the recipe instead of the bytes (tests/helpers.py load_fixture regenerates them)
        cap = dict(synth_fmt=fmt, synth_samples=nsamples, synth_seed=seed, buf_sha256=hashlib.sha256(buf).hexdigest())
    else:
        cap = dict(buf=np.frombuffer(buf, np.uint8))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **cap, fmt=fmt, n=n, width=width,
                        window=window, windowc=w, weight=weight, gain=gain, range=rng, cmap=cmap,
                        channel_mode=channel_mode, waterfall=waterfall, image=c.image, gray=c.gray,
                        db=c.db.astype(np.float64), cB_hist=c.cB_hist, c_hist=c.c_hist, gauge_mins=c.gauge_mins,
                        gauge_maxs=c.gauge_maxs, gauge_amps=c.gauge_amps, dBfs_min=c.dBfs_min, dBfs_max=c.dBfs_max)
    print(name, "ok; restatement gray mismatches:", bad)


if __name__ == "__main__":
    cm256 = injective_cmap(256)
    case("cu8_n1024_hann_w48", "CU8", 1024, 48, "hann", 6, 30, cm256, 20000, 0x5EC70001)
    case("cs16_n4096_bh_w24", "CS16", 4096, 24, "blackmanHarris", 6, 30, cm256, 4096 * 24, 0x5EC70002)
    case("cf32_n256_hamming_w40_wf", "CF32", 256, 40, "hamming", 0, 60, cm256, 9000, 0x5EC70003, waterfall=True)
    case("cs8_n128_rect_w33_lr", "CS8", 128, 33, "rectangular", 10, 40, injective_cmap(64), 5000, 0x5EC70004, channel_mode=True)
    case("cu12_n512_blackman_w16", "CU12", 512, 16, "blackman", 6, 30, cm256, 512 * 16, 0x5EC70005)
    # Appendix B.3 (SURVEY.md): derived known-answer
    buf = bytes([(37 * j + 11) % 256 for j in range(40)])
    np.savez_compressed(os.path.join(OUT, "appendix_b3.npz"), buf=np.frombuffer(buf, np.uint8),
                        gray_image=np.array([[255, 255, 255, 255], [247, 255, 255, 255], [199, 255, 238, 238],
                                             [241, 255, 255, 250], [243, 232, 218, 197], [255, 249, 255, 255],
                                             [255, 255, 255, 255], [255, 255, 255, 255]], np.uint16),
                        gauge_mins=np.array([149, 182, 168, 147], np.uint8), gauge_maxs=np.array([243, 233, 240, 240], np.uint8),
                        gauge_amps=np.array([255, 255, 255, 255], np.uint8), dBfs_min=-12.852073819239978,
                        dBfs_max=-1.5306197856730837,
                        frame0_dbfs=np.array([-1.413285, -1.588836, -6.584125, -0.925007, 1.872985, 3.72409, 4.46938, 2.135198]))
    print("appendix_b3 ok")
