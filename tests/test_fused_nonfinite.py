"""Silent frames (|X|^2 == 0 everywhere: dB = -inf) and a frame with a NaN sample through every fused render kernel.
All four kernels share one fix-up for zero / +inf / NaN magnitudes (csrc/sp_fused.cuh: fixup_nonfinite, the reference's
~~(+-Infinity) == ~~NaN == 0 rule); each case here reaches it through a different kernel and compares with the oracle."""
import numpy as np
import pytest

from helpers import check_parity, injective_cmap
from oracle import oracle as O

pytestmark = pytest.mark.gpu
CM256 = injective_cmap(256)
SILENT = [5, 6, 7, 8, 11]                               # frames zeroed in the integer capture


# (n, width, kernel, channel_mode, waterfall, four-step form)
CASES = [
    (64, 600, "render_w_kernel", False, False, None),
    (512, 128, "render_w_kernel", False, False, None),
    (2048, 64, "render_rc_kernel", False, False, None),
    (4096, 48, "render_r64_kernel", False, False, None),
    (4096, 48, "render_r64_kernel", False, True, None),      # waterfall layout: the OPT instantiation
    (4096, 48, "render_r64_kernel", True, False, None),      # split-real: the OPT instantiation
    (8192, 24, "render_big_kernel", False, False, "ring"),
    (65536, 16, "render_big_kernel", False, False, "ring"),
]


@pytest.mark.parametrize("n,width,kernel,channel_mode,waterfall,form", CASES)
def test_fused_kernel_silent_and_nan_frames(engine, monkeypatch, n, width, kernel, channel_mode, waterfall, form):
    if form:
        monkeypatch.setenv("SP_FOURSTEP", form)
    label = f"{kernel} n={n} channel_mode={channel_mode} waterfall={waterfall}"
    for fmt in ("CS16", "CF32"):
        assert kernel in engine.kernel_plan(fmt, n, channel_mode), (fmt, engine.kernel_plan(fmt, n, channel_mode))
    S = n * width
    w, wt = O.window("blackmanHarris", n)
    x = np.frombuffer(O.synth("CS16", 0, S, S, 0x5EC7B300 + n).tobytes(), "<i2").reshape(width, n, 2).copy()
    x[SILENT] = 0
    buf = x.tobytes()
    ora = O.render(buf, "CS16", n, width, w, 1 / wt, 6, 30, CM256, channel_mode, waterfall, taps=True)
    gpu = engine.render(buf, "CS16", n, width, w, 1 / wt, 6, 30, CM256, channel_mode, waterfall)
    check_parity(gpu, ora, CM256, n, width, waterfall, None, f"{label} silent frames")
    assert gpu["cB_hist"][0] >= len(SILENT) * n and gpu["dBfs_min"] == -np.inf
    f = np.frombuffer(O.synth("CF32", 0, S, S, 0x5EC7B400 + n).tobytes(), "<f4").reshape(width, n, 2).copy()
    f[2, n // 3, 0] = np.nan                          # a NaN sample inside every frame size
    buf = f.tobytes()
    with np.errstate(all="ignore"):
        ora = O.render(buf, "CF32", n, width, w, 1 / wt, 0, 60, CM256, channel_mode, waterfall, taps=True)
    gpu = engine.render(buf, "CF32", n, width, w, 1 / wt, 0, 60, CM256, channel_mode, waterfall)
    check_parity(gpu, ora, CM256, n, width, waterfall, None, f"{label} NaN frame")
