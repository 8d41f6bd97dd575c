"""Back-to-back N = 4096 messages on one stream.  render_r64_kernel starts behind the previous message's finalize_kernel before
that has completed (programmatic dependent launch) and takes its tiles from a counter shared by its CTAs: every reply must
still equal, byte for byte, the same message rendered alone.  Each check also runs with SP_NO_PDL=1 (plain stream order),
in a child process because the switch is read once per process."""
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import injective_cmap

pytestmark = pytest.mark.gpu

N = 4096
FMT, SW = "CS16", 4
CM = injective_cmap(256)
# (capture seed, window, gain, range, width): A and B share their dB / colour settings and so do C and D, so that A -> B,
# B -> A, C -> D and D -> C overlap, while B -> C and D -> A (new window, LUT constants) fall back to plain stream order.
# Widths: 150 tiles of 16 frames (more than the SMs), a partial last tile (1000 = 62 * 16 + 8), 13 tiles (fewer than the
# SMs) and 100 tiles + a partial one.
MESSAGES = {"A": (1, "hann", 6, 30, 2400), "B": (2, "hann", 6, 30, 1000),
            "C": (1, "blackmanHarris", 20, 60, 200), "D": (2, "blackmanHarris", 20, 60, 1608)}
ORDER = "ABABCDCDA"
MAX_W = max(m[4] for m in MESSAGES.values())


class Outputs:
    """Device buffers of one reply: image, three gauge rows, cB | c histograms, dBfs min / max."""

    def __init__(self, eng, width):
        self.eng, self.width = eng, width
        self.img, self.g = eng.alloc(4 * width * N), eng.alloc(3 * width)
        self.hist, self.mm = eng.alloc(8 * (1000 + len(CM))), eng.alloc(16)

    def enqueue(self, rq):
        w = self.width
        return self.eng.render_enqueue(rq, self.img, (self.g, self.g + w, self.g + 2 * w), self.hist, self.hist + 8000, self.mm)

    def read(self):
        out = {"image": np.empty(4 * self.width * N, np.uint8), "gauges": np.empty(3 * self.width, np.uint8),
               "hist": np.empty(1000 + len(CM), np.uint64), "minmax": np.empty(2, np.float64)}
        for k, d in zip(out, (self.img, self.g, self.hist, self.mm)):
            self.eng.d2h(out[k], d)
        return out

    def free(self):
        for d in (self.img, self.g, self.hist, self.mm):
            self.eng.free(d)


def _request(eng, cap, name):
    from oracle import oracle as O
    _, window, gain, rng, width = MESSAGES[name]
    w, wt = O.window(window, N)
    return eng.make_request(cap, FMT, N, width, w, 1 / wt, gain, rng, CM, byte_length=width * N * SW)


def _same(a, b, label):
    for k in a:
        assert np.array_equal(a[k], b[k]), (label, k)


def back_to_back(eng):
    caps = {}
    for seed in (1, 2):
        caps[seed] = eng.alloc(MAX_W * N * SW + 256)
        eng.synth_fill(caps[seed], FMT, 0, MAX_W * N, MAX_W * N, 0x5EC7C000 + seed)
    alone = {}
    outs = []
    try:
        for name, m in MESSAGES.items():                     # each message alone, the stream drained before and after
            o = Outputs(eng, m[4])
            outs.append(o)
            rq, keep = _request(eng, caps[m[0]], name)
            rp = o.enqueue(rq)
            eng.render_finish(rp)
            alone[name] = o.read()
            assert rp.device_ms > 0, name
        run = [Outputs(eng, MESSAGES[name][4]) for name in ORDER]
        outs += run
        for name, o in zip(ORDER, run):                      # one stream, no host sync in between
            rq, keep = _request(eng, caps[MESSAGES[name][0]], name)
            rp = o.enqueue(rq)
        eng.render_finish(rp)
        assert rp.device_ms > 0
        for i, (name, o) in enumerate(zip(ORDER, run)):
            _same(o.read(), alone[name], f"message {i} ({name}) of {ORDER}")
    finally:
        for o in outs:
            o.free()
        for d in caps.values():
            eng.free(d)


def capture_rewritten_on_the_stream(eng):
    """A torch kernel on the engine's stream overwrites the capture right before the next message is enqueued."""
    import torch
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    width = MESSAGES["A"][4]
    nbytes = width * N * SW
    x = torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)
    y = torch.empty_like(x)
    cap = torch.empty_like(x)
    eng.synth_fill(x.data_ptr(), FMT, 0, width * N, width * N, 0x5EC7C101)
    eng.synth_fill(y.data_ptr(), FMT, 0, width * N, width * N, 0x5EC7C102)
    torch.cuda.synchronize()
    outs = [Outputs(eng, width) for _ in range(4)]
    try:
        eng.set_stream(stream.cuda_stream)
        for o, src in ((outs[0], x), (outs[1], y)):          # references: each capture alone
            rq, keep = _request(eng, src.data_ptr(), "A")
            eng.render_finish(o.enqueue(rq))
        ref = [outs[0].read(), outs[1].read()]
        with torch.cuda.stream(stream):
            torch.bitwise_or(x, 0, out=cap)                  # an elementwise kernel, not a copy
            rq, keep = _request(eng, cap.data_ptr(), "A")
            outs[2].enqueue(rq)
            torch.bitwise_or(y, 0, out=cap)                  # rewrites the capture between the two renders
            rq, keep = _request(eng, cap.data_ptr(), "A")
            rp = outs[3].enqueue(rq)
        eng.render_finish(rp)
        _same(outs[2].read(), ref[0], "render before the rewrite")
        _same(outs[3].read(), ref[1], "render after the rewrite")
    finally:
        eng.set_stream(None)
        for o in outs:
            o.free()


def _in_child_without_pdl(check):
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    code = ("import sys; sys.path[:0] = %r; import spectro_b200, test_render_overlap as t; e = spectro_b200.Engine(0); "
            "t.%s(e); e.close()" % ([root, os.path.join(root, "spectroplot-js_b200"), os.path.join(root, "tests")], check))
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, "-c", code], env=dict(os.environ, SP_NO_PDL="1"), capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


@pytest.mark.parametrize("pdl", [True, False], ids=["pdl", "no_pdl"])
def test_back_to_back_messages_equal_isolated_renders(engine, pdl):
    if pdl:
        back_to_back(engine)
    else:
        _in_child_without_pdl("back_to_back")


@pytest.mark.parametrize("pdl", [True, False], ids=["pdl", "no_pdl"])
def test_capture_rewritten_by_a_kernel_before_enqueue(engine, pdl):
    if pdl:
        capture_rewritten_on_the_stream(engine)
    else:
        _in_child_without_pdl("capture_rewritten_on_the_stream")
