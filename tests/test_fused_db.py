"""dB accuracy of the fused render kernels, read back from their own pictures.

The dB tap (sp_render_db) always runs render_kernel, so the dB bars of BASELINE.json (helpers.py) reach the kernels that draw
the pictures - render_w_kernel, render_rc_kernel, render_r64_kernel, render_big_kernel and the sub-frame render_r64_kernel of the
four-step transform - only through their colours.  At a colour range of R = 0.64 dB one step of a 256-entry colormap is
R / 256 = 0.0025 dB, and a pixel that is not clamped (0 < g < cmax) places the kernel's own d0 in an interval of that width
(lib/worker.js:111-112):
    g = floor(0.5 + cmax + (d0 + gain) * cmap_len / R)   =>   d0 in [(g - 0.5 - cmax) R / cmap_len - gain, (g + 0.5 - cmax) R / cmap_len - gain)
A sweep of the gain whose unclamped windows tile the levels from the strongest bin down to below -60 (-120 dBFS conventional)
brackets every pixel the bars speak of.  The distance from the float64 oracle's d0 to a pixel's bracket is a lower bound on the
kernel's error, within R / 256 of it.  The self-check runs the sweep on render_kernel, whose d0 the dB tap returns, so the colour
to dB mapping and the gain handling are proved on the device before the fused kernels are measured with them.
"""
import time

import numpy as np
import pytest

from helpers import DB_FLOOR_REF, DB_FLOOR_STRICT, DB_TOL, DB_TOL_FLOOR_MAX, PIXEL_FRAC, bin_to_row, injective_cmap
from oracle import oracle as O

pytestmark = pytest.mark.gpu

R = 0.64                          # colour range of the sweep: 0.0025 dB per step of a 256-entry colormap
CM256 = injective_cmap(256)
# render_kernel's band rms (bracketed the same way) times K_PEER, plus one colour step, bounds a fused kernel's band rms.
# Ratios measured on a B200 (1000 W): 0.57 ... 1.08 for every case but w-cs16-n64 (1.55, a band of 16 pixels); K_PEER is
# 1.5 x the largest.  A relative error of 1e-6 on the entries of render_r64_kernel's / render_rc_kernel's twiddle table
# gives ratios of 2.9 ... 5.9 (profiles/r07_fused_db.txt).
K_PEER = 2.3


def colour_indices(image, cmap, n, width, waterfall=False):
    """RGBA picture -> [width][n] colour indices in FFT bin order, -1 where a pixel is not in the (injective) cmap: the layout
    of helpers.gray_from_image, with one sorted lookup of the 24-bit RGB keys so that a sweep of ~90 pictures stays quick."""
    key = lambda a: (a[..., 0].astype(np.int64) << 16) | (a[..., 1].astype(np.int64) << 8) | a[..., 2].astype(np.int64)
    ck = key(np.asarray(cmap))
    order = np.argsort(ck, kind="stable")
    sk = ck[order]
    assert (np.diff(sk) != 0).all(), "cmap not injective"
    k = key(image)
    pos = np.minimum(np.searchsorted(sk, k), len(sk) - 1)
    idx = np.where(sk[pos] == k, order[pos], -1)
    y = bin_to_row(n)
    if waterfall:
        return idx[(width - 1 - np.arange(width))[:, None], (n - 1 - y)[None, :]]
    return idx[y[None, :], np.arange(width)[:, None]]


def cb_edge_ties(ora_db):
    """check_parity's allowance for cB_hist: pixels whose reference level lies within 2e-4 dB of a 0.1 dB bin edge
    (lib/worker.js:105: ~~(2.5 - 10 * d0)) may sit in the neighbouring bin."""
    x = 2.5 - 10.0 * np.asarray(ora_db, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        fr = np.abs(x - np.round(x))
    return int((fr[np.isfinite(fr)] < 2e-3).sum())


def sweep_tops(top, bottom, cmap_len, range_=R):
    """Upper ends of the unclamped windows [t - (cmax - 0.5) q, t - 0.5 q) from top down past bottom (q = range / cmap_len),
    one colour step of overlap between neighbours so that no level falls between two windows."""
    q = range_ / cmap_len
    step = (cmap_len - 3) * q
    k = max(0, int(np.ceil((top - bottom - (cmap_len - 2) * q) / step))) + 1
    return top + 0.5 * q - step * np.arange(k)


def brackets_of(gray, gain, cmap_len, range_, lo, hi):
    """Narrow lo / hi to the bracket of d0 that each unclamped colour index of one render gives."""
    cmax, q = cmap_len - 1, range_ / cmap_len
    ok = (gray > 0) & (gray < cmax)
    lo[ok] = (gray[ok] - 0.5 - cmax) * q - gain
    hi[ok] = (gray[ok] + 0.5 - cmax) * q - gain


def quantised_brackets(d0, tops, cmap_len, range_=R):
    """The brackets the sweep would give for the levels d0, computed with the reference's colour rule in float64."""
    cmax, q = cmap_len - 1, range_ / cmap_len
    lo, hi = np.full(d0.shape, -np.inf), np.full(d0.shape, np.inf)
    d = d0.astype(np.float64)
    with np.errstate(invalid="ignore"):
        for top in tops:
            gu = cmax + (d - top) / q
            g = np.where(np.isfinite(gu), np.floor(0.5 + np.clip(gu, 0, cmax)), 0).astype(np.int64)
            brackets_of(g, -top, cmap_len, range_, lo, hi)
    return lo, hi


def sweep(engine, buf, fmt, n, width, windowc, block_norm, cmap, tops, channel_mode=False, waterfall=False, range_=R):
    """Render the message once per window top (gain = -top) -> (lo, hi, replies): the per-pixel bracket [lo, hi) of the
    kernel's d0 as [width][n] in FFT bin order (-inf / +inf where no render left the pixel unclamped), and the replies of the
    renders with the picture replaced by the bincount of its colour indices ("picture_hist") and the gain added."""
    cml = len(cmap)
    lo, hi = np.full((width, n), -np.inf), np.full((width, n), np.inf)
    replies = []
    for top in tops:
        gain = -float(top)
        r = engine.render(buf, fmt, n, width, windowc, block_norm, gain, range_, cmap, channel_mode, waterfall)
        assert (r["image"][..., 3] == 255).all(), "alpha"
        g = colour_indices(r["image"], cmap, n, width, waterfall)
        assert (g >= 0).all(), f"gain {gain}: pixel colour not in the colormap"
        brackets_of(g, gain, cml, range_, lo, hi)
        r["image"] = None
        r["picture_hist"] = np.bincount(g.ravel(), minlength=cml)
        r["gain"] = gain
        replies.append(r)
    return lo, hi, replies


def bracket_stats(lo, hi, ref):
    """Distance from the oracle's d0 to the bracket: max above DB_FLOOR_STRICT and in the band down to DB_FLOOR_REF; rms of
    (bracket midpoint - oracle) over the band; pixels of the bars without a bracket."""
    fin = np.isfinite(ref)
    has = np.isfinite(lo) & np.isfinite(hi)
    with np.errstate(invalid="ignore"):
        err = np.where(ref < lo, lo - ref, np.where(ref > hi, ref - hi, 0.0))
        mid = (lo + hi) / 2 - ref
    strict = fin & (ref > DB_FLOOR_STRICT) & has
    band = fin & (ref > DB_FLOOR_REF) & ~(ref > DB_FLOOR_STRICT) & has
    return dict(max_strict=float(err[strict].max()) if strict.any() else 0.0,
                max_floor=float(err[band].max()) if band.any() else 0.0,
                rms_floor=float(np.sqrt(np.mean(mid[band] ** 2))) if band.any() else 0.0,
                n_strict=int(strict.sum()), n_floor=int(band.sum()),
                missing=int((fin & (ref > DB_FLOOR_REF) & ~has).sum()))


def _fmt_stats(s):
    return f"max {s['max_strict']:.4f} / band max {s['max_floor']:.4f} / band rms {s['rms_floor']:.4f} dB"


def _message(fmt, n, width, hop, extra, seed):
    """A synth capture of hop * (width - 1) + n + extra samples: with extra < hop the stride is fractional and the last frame
    still lies inside the buffer, so every frame of a width that is a multiple of 8 stays on the fused kernel."""
    S = hop * (width - 1) + n + extra
    stride = (S - n) / (width - 1)
    assert int(0.5 + stride * (width - 1)) + n <= S
    return O.synth(fmt, 0, S, S, seed).tobytes()


def _sweep_range(ref):
    """Window tops from just above the strongest bin to below DB_FLOOR_REF, with room for a kernel error that misses the bars."""
    top = float(np.nanmax(np.where(np.isfinite(ref), ref, np.nan)))
    return top + 0.1, DB_FLOOR_REF - 0.1


def _check_statistics(replies, ora, label):
    """c_hist is the bincount of the render's own picture; cB_hist, dBfs_min and dBfs_max depend on neither gain nor range."""
    first = replies[0]
    for r in replies:
        assert np.array_equal(r["c_hist"].astype(np.int64), r["picture_hist"]), f"{label} gain {r['gain']}: c_hist"
        assert np.array_equal(r["cB_hist"], first["cB_hist"]), f"{label} gain {r['gain']}: cB_hist changed with the gain"
        assert r["dBfs_min"] == first["dBfs_min"] and r["dBfs_max"] == first["dBfs_max"], f"{label} gain {r['gain']}: min / max"
    npix = ora.db.size
    cb_d = int(np.abs(first["cB_hist"].astype(np.int64) - ora.cB_hist.astype(np.int64)).sum())
    edge = cb_edge_ties(ora.db)
    assert cb_d <= 2 * max(2, int(PIXEL_FRAC * npix), edge), f"{label}: cB_hist differs by {cb_d} (ties allowed: {edge})"


# ------------------------------------------------------------------ the instrument on render_kernel
@pytest.mark.parametrize("fmt,n,width,hop,window,cmap_len,channel_mode", [
    ("CS16", 32, 1024, 32, "hann", 256, False),                  # only render_kernel exists at N = 32
    ("CS16", 4096, 16, 4096, "blackmanHarris", 257, False),      # more than 256 colours: no fused kernel takes the message
    ("CF32", 8192, 16, 8192, "hann", 256, True),                 # split-real: prepass_kernel, render_kernel, spectrum_epilogue_kernel
], ids=["n32", "n4096-257colours", "n8192-splitreal"])
def test_instrument_reads_render_kernels_db(engine, fmt, n, width, hop, window, cmap_len, channel_mode):
    """The picture sweep of a message that render_kernel draws must bracket the d0 that sp_render_db returns for it, pixel by
    pixel (widened by 0.01 colour steps for the kernel's fp32 colour arithmetic)."""
    cm = injective_cmap(cmap_len)
    buf = _message(fmt, n, width, hop, 0, 0x5EC7D800 + n)
    w, wt = O.window(window, n)
    ora = O.render(buf, fmt, n, width, w, 1 / wt, 0, R, cm, channel_mode, taps=True)
    tops = sweep_tops(*_sweep_range(ora.db), cmap_len)
    lo, hi, replies = sweep(engine, buf, fmt, n, width, w, 1 / wt, cm, tops, channel_mode)
    db = engine.render_db(buf, fmt, n, width, w, 1 / wt, 0, R, cm, channel_mode).astype(np.float64)
    has = np.isfinite(lo) & np.isfinite(hi)
    slack = 0.01 * R / cmap_len
    out = has & ~((db >= lo - slack) & (db < hi + slack))
    assert not out.any(), (f"{int(out.sum())} of {int(has.sum())} d0 values outside their bracket, e.g. {db[out][:4]} in "
                           f"[{lo[out][:4]}, {hi[out][:4]})")
    st = bracket_stats(lo, hi, ora.db)
    assert st["missing"] == 0 and st["n_strict"] > 0 and st["n_floor"] > 0, st
    _check_statistics(replies, ora, f"render_kernel {fmt} n={n}")


# ------------------------------------------------------------------ the fused kernels against the bars
# (id, kernel named by kernel_plan, format, n, width, hop, extra samples, window, waterfall, channel mode, SP_FOURSTEP)
CASES = [
    ("w-cs16-n64", "render_w_kernel", "CS16", 64, 2048, 64, 0, "hann", False, False, None),                # P = 8
    ("w-cs16-n128", "render_w_kernel", "CS16", 128, 1024, 97, 7, "blackmanHarris", False, False, None),   # P = 16
    ("w-cs16-n256", "render_w_kernel", "CS16", 256, 512, 256, 0, "hann", False, False, None),
    ("w-cs16-n512", "render_w_kernel", "CS16", 512, 256, 389, 11, "blackman", False, False, None),         # P = 32
    ("w-cs16-n1024", "render_w_kernel", "CS16", 1024, 128, 1024, 0, "hann", False, False, None),
    ("w-cu8-n1024-C1", "render_w_kernel", "CU8", 1024, 128, 1024, 0, "hann", False, False, None),
    ("w-cf32-n512-waterfall", "render_w_kernel", "CF32", 512, 256, 512, 0, "hann", True, False, None),
    ("w-cs16-n128-splitreal", "render_w_kernel", "CS16", 128, 1024, 128, 0, "hann", False, True, None),
    ("w-cs16-n1024-splitreal", "render_w_kernel", "CS16", 1024, 128, 1024, 0, "hann", False, True, None),
    ("rc-cs16-n2048", "render_rc_kernel", "CS16", 2048, 128, 2048, 0, "blackmanHarris", False, False, None),
    ("rc-cf32-n2048-waterfall", "render_rc_kernel", "CF32", 2048, 64, 1501, 5, "hann", True, False, None),
    ("r64-cs16-C2", "render_r64_kernel", "CS16", 4096, 48, 4096, 0, "blackmanHarris", False, False, None),
    ("r64-cf32-hop1501", "render_r64_kernel", "CF32", 4096, 48, 1501, 5, "blackmanHarris", False, False, None),
    ("r64-cu8-hop1501", "render_r64_kernel", "CU8", 4096, 48, 1501, 5, "blackmanHarris", False, False, None),
    ("r64-cs4-hop1501", "render_r64_kernel", "CS4", 4096, 48, 1501, 5, "blackmanHarris", False, False, None),
    ("r64-cs16-waterfall", "render_r64_kernel", "CS16", 4096, 32, 4096, 0, "hann", True, False, None),
    ("r64-cs16-splitreal", "render_r64_kernel", "CS16", 4096, 32, 4096, 0, "hann", False, True, None),
    ("big-cf32-n8192", "render_big_kernel", "CF32", 8192, 64, 8192, 0, "hann", False, False, "ring"),       # R = 2
    ("big-cf32-n32768-C3", "render_big_kernel", "CF32", 32768, 32, 32768, 0, "hann", False, False, "ring"),  # R = 8
    ("big-cf32-n65536-C5", "render_big_kernel", "CF32", 65536, 16, 65536, 0, "hann", False, False, "ring"),  # R = 16
    ("sub-cf32-n16384", "render_r64_kernel", "CF32", 16384, 32, 16384, 0, "hann", False, False, "hbm"),
    ("sub-cf32-n65536", "render_r64_kernel", "CF32", 65536, 16, 65536, 0, "hann", False, False, "hbm"),
    # R = 64; the sub-frame kernel takes whole groups of 8 frames, so this one picture has 2 M pixels
    ("sub-cf32-n262144", "render_r64_kernel", "CF32", 262144, 8, 262144, 0, "blackmanHarris", False, False, "hbm"),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_fused_kernel_meets_the_db_bars(engine, monkeypatch, case):
    """Every bracket of a fused kernel's picture sweep lies within DB_TOL of the oracle above DB_FLOOR_STRICT and within
    DB_TOL_FLOOR_MAX in the band down to DB_FLOOR_REF, whose midpoints have an rms error of at most DB_TOL; the kernel stays
    within K_PEER of render_kernel's band rms, and its picture is not render_kernel's."""
    label, kernel, fmt, n, width, hop, extra, window, wf, chm, form = case
    if form:
        monkeypatch.setenv("SP_FOURSTEP", form)
    assert width % 8 == 0
    plan = engine.kernel_plan(fmt, n, chm)
    assert kernel in plan, plan
    if chm:
        assert "split-real" in plan, plan
    t0 = time.perf_counter()
    buf = _message(fmt, n, width, hop, extra, 0x5EC7D000 + n + width)
    w, wt = O.window(window, n)
    ora = O.render(buf, fmt, n, width, w, 1 / wt, 0, R, CM256, chm, wf, taps=True)
    tops = sweep_tops(*_sweep_range(ora.db), 256)
    lo, hi, replies = sweep(engine, buf, fmt, n, width, w, 1 / wt, CM256, tops, chm, wf)
    st = bracket_stats(lo, hi, ora.db)
    # render_kernel on the same message, bracketed the same way
    db = engine.render_db(buf, fmt, n, width, w, 1 / wt, 0, R, CM256, chm)
    plo, phi = quantised_brackets(db, tops, 256)
    peer = bracket_stats(plo, phi, ora.db)
    has = np.isfinite(lo) & np.isfinite(hi)
    differ = int((has & ~((db >= lo) & (db < hi))).sum())
    secs = time.perf_counter() - t0
    print(f"\n{label}: {kernel} {_fmt_stats(st)} | render_kernel {_fmt_stats(peer)} | band rms ratio "
          f"{st['rms_floor'] / max(peer['rms_floor'], 1e-12):.3f} | {st['n_strict']} + {st['n_floor']} pixels, {differ} brackets "
          f"exclude render_kernel's d0 | {len(tops)} renders, {secs:.1f} s")
    assert st["max_strict"] <= DB_TOL, f"{label}: dB error >= {st['max_strict']} above -100 dBFS"
    assert st["max_floor"] <= DB_TOL_FLOOR_MAX, f"{label}: dB error >= {st['max_floor']} in the -120..-100 dBFS band"
    assert st["rms_floor"] <= DB_TOL, f"{label}: rms dB error {st['rms_floor']} in the -120..-100 dBFS band"
    assert st["rms_floor"] <= K_PEER * peer["rms_floor"] + R / 256, (label, st, peer)
    assert st["missing"] == 0, f"{label}: {st['missing']} pixels above {DB_FLOOR_REF} without a bracket"
    assert st["n_strict"] > 0 and st["n_floor"] > 0, st
    assert differ > 0, f"{label}: every bracket holds render_kernel's d0: the picture did not come from {kernel}"
    _check_statistics(replies, ora, label)
