"""Render a fixed set of messages that covers every kernel route and print, per message, kernel_launches and a SHA-256 of
the reply (image, gauges, both histograms, dBfs min / max), one line each.  Two libraries compute the same thing when their
outputs are identical:

    SP_LIB=/path/a/libspectro_b200.so python tools/route_digests.py > a.txt
    SP_LIB=/path/b/libspectro_b200.so python tools/route_digests.py > b.txt
    diff a.txt b.txt

The set: five specialised formats (CS16, CU8, CF32, CU4, CS12) and two runtime-switch formats (CU32, CF64) at N = 16 .. 4096,
widths 104 and 37, channel mode and waterfall on and off; a 300-colour map; the dB tap; a capture shorter than one frame;
frame-range shards; the host pipeline (SP_PIPE_MB=1); the four-step sizes n = 8192 / 32768 in both forms (SP_FOURSTEP),
n = 16384 / 65536 in the HBM-scratch form, and n = 131072 / 262144, so that prepass_kernel runs at every R = 2 .. 64; and the
sp_decode tap of all 14 formats over a span that runs past the end of the buffer: 579 lines.  Needs a GPU."""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "spectroplot-js_b200"), os.path.join(ROOT, "tests")]

import spectro_b200  # noqa: E402
from spectro_b200 import _lib, sharding  # noqa: E402
from oracle import oracle as O  # noqa: E402
from helpers import injective_cmap  # noqa: E402

CM256, CM300 = injective_cmap(256), injective_cmap(300)


def digest(r):
    h = hashlib.sha256()
    for k in ("image", "gauge_mins", "gauge_maxs", "gauge_amps", "cB_hist", "c_hist"):
        if r.get(k) is not None:
            h.update(np.ascontiguousarray(r[k]).tobytes())
    h.update(np.array([r["dBfs_min"], r["dBfs_max"]], np.float64).tobytes())
    return h.hexdigest()


def main():
    eng = spectro_b200.Engine(0)
    caps = {}

    def capture(fmt, S, seed=0x5EC7):
        if (fmt, S, seed) not in caps:
            caps[(fmt, S, seed)] = O.synth(fmt, 0, S, S, seed).tobytes()
        return caps[(fmt, S, seed)]

    def render(tag, fmt, n, width, S, cm=CM256, env=None, **kw):
        old = {k: os.environ.get(k) for k in (env or {})}
        os.environ.update(env or {})
        try:
            w, wt = O.window("hann", n)
            r = eng.render(capture(fmt, S), fmt, n, width, w, 1 / wt, 6, 30, cm, **kw)
        finally:
            for k, v in old.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
        print(f"{tag} launches={r['kernel_launches']} {digest(r)}", flush=True)
        return r

    for fmt in ("CS16", "CU8", "CF32", "CU4", "CS12", "CU32", "CF64"):
        for lg in range(4, 13):
            n = 1 << lg
            for width in (104, 37):
                for cm in (False, True):
                    for wf in (False, True):
                        render(f"{fmt} n={n} w={width} cm={int(cm)} wf={int(wf)}", fmt, n, width, 24 * n + 1001,
                               channel_mode=cm, waterfall=wf)
    for n in (256, 1024, 4096):
        render(f"CS16 n={n} cmap=300", "CS16", n, 104, 24 * n + 1001, cm=CM300)
        w, wt = O.window("hann", n)
        db = eng.render_db(capture("CS16", 24 * n + 1001), "CS16", n, 40, w, 1 / wt, 6, 30, CM256)
        print(f"CS16 n={n} db-tap {hashlib.sha256(db.tobytes()).hexdigest()}", flush=True)
    render("CS16 n=1024 short capture", "CS16", 1024, 16, 600)
    for n, width, S in ((1024, 208, 150001), (2048, 96, 170003), (4096, 72, 200003)):
        for sh in sharding.plan_shards(S, n, width, 3):
            if sh["width"]:
                buf = capture("CS16", S)[sh["sample_first"] * 4:(sh["sample_first"] + sh["sample_count"]) * 4]
                w, wt = O.window("hann", n)
                r = eng.render(buf, "CS16", n, sh["width"], w, 1 / wt, 6, 30, CM256,
                               shard=sharding.shard_fields(sh, S, 4, width))
                print(f"CS16 n={n} shard {sh['frame_first']}+{sh['width']} launches={r['kernel_launches']} {digest(r)}", flush=True)
    for n in (256, 1024, 2048, 4096):
        for wf in (False, True):
            render(f"CS16 n={n} pipelined wf={int(wf)}", "CS16", n, 900, 300 * n + 77, env={"SP_PIPE_MB": "1"}, waterfall=wf)
    for n in (8192, 32768):
        for form in ("ring", "hbm", ""):
            for cm in (False, True):
                for fmt in ("CF32", "CS16"):
                    render(f"{fmt} n={n} fourstep={form or 'auto'} cm={int(cm)}", fmt, n, 48, 40 * n + 3001,
                           env={"SP_FOURSTEP": form} if form else None, channel_mode=cm)
    render("CF32 n=32768 waterfall", "CF32", 32768, 48, 40 * 32768 + 3001, waterfall=True)
    for n in (16384, 65536):                                 # prepass_kernel at R = 4 and 16
        for cm in (False, True):
            for fmt in ("CF32", "CS16"):
                render(f"{fmt} n={n} fourstep=hbm cm={int(cm)}", fmt, n, 24, 26 * n + 3001, env={"SP_FOURSTEP": "hbm"}, channel_mode=cm)
    for n in (131072, 262144):
        for cm in (False, True):
            render(f"CF32 n={n} cm={int(cm)}", "CF32", n, 12, 14 * n + 5, channel_mode=cm)
    for fmt in _lib.FORMATS:
        sw = eng.lib.sp_sample_width(_lib.format_id(fmt))
        buf = capture(fmt, 4000)[: 4000 * sw - (1 if sw > 1 else 0)]      # a ragged end where the format allows one
        d = eng.decode(fmt, buf, 3900, 160)                                 # runs 60 samples past the end
        print(f"{fmt} decode {hashlib.sha256(d.tobytes()).hexdigest()}", flush=True)
    eng.close()


if __name__ == "__main__":
    main()
