#!/usr/bin/env python
"""End-to-end (pinned host -> pinned host) time of the C2 message as a function of the pipeline chunk size
(SP_PIPE_MB), plus raw PCIe copy rates for reference.  usage (under gpurun): python tools/e2e_sweep.py"""
import os, sys, time, subprocess, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if len(sys.argv) > 1 and sys.argv[1] == "child":
    for p in (ROOT, os.path.join(ROOT, "spectroplot-js_b200")):
        sys.path.insert(0, p)
    import numpy as np, torch, spectro_b200
    from spectro_b200 import windows, cmaps
    n, width = 4096, 25600
    S = n * width
    eng = spectro_b200.Engine(0)
    d = eng.alloc(S * 4)
    eng.synth_fill(d, "CS16", 0, S, S, 0x5EC70001)
    pin_in = spectro_b200.PinnedBuffer(S * 4); eng.d2h(pin_in.array, d)
    pin_img = spectro_b200.PinnedBuffer(4 * width * n)
    w = windows.blackmanHarrisWindow(n); ww = np.array(w["window"]); wt = float(w["weight"])
    cm = cmaps.cmap_bytes([list(c) for c in cmaps.cmaps["viridis_cmap"]])
    ts = []
    for i in range(6):
        t0 = time.perf_counter()
        out = eng.render(pin_in.array, "CS16", n, width, ww, 1 / wt, 6, 30, cm, out_image=pin_img.array)
        ts.append(time.perf_counter() - t0)
    ms = 1e3 * min(ts[1:])
    print(json.dumps(dict(pipe_mb=os.environ.get("SP_PIPE_MB"), ms=ms, gsamples_s=S / ms / 1e6, launches=out["kernel_launches"],
                          gbs_each_way=S * 4 / ms / 1e6)), flush=True)
    if os.environ.get("SP_PIPE_MB") == "32":
        # raw copies: H2D alone, D2H alone, both at once
        a = torch.empty(S * 4, dtype=torch.uint8, device="cuda"); b = torch.empty(S * 4, dtype=torch.uint8, device="cuda")
        ha = torch.empty(S * 4, dtype=torch.uint8).pin_memory(); hb = torch.empty(S * 4, dtype=torch.uint8).pin_memory()
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        def t(f):
            torch.cuda.synchronize(); t0 = time.perf_counter(); f(); torch.cuda.synchronize(); return time.perf_counter() - t0
        def h2d():
            with torch.cuda.stream(s1): a.copy_(ha, non_blocking=True)
        def d2h():
            with torch.cuda.stream(s2): hb.copy_(b, non_blocking=True)
        for name, f in (("h2d", h2d), ("d2h", d2h), ("both", lambda: (h2d(), d2h()))):
            f(); dt = min(t(f) for _ in range(3))
            print(json.dumps(dict(raw=name, ms=dt * 1e3, gbs=S * 4 / dt / 1e9)), flush=True)
    sys.exit(0)
for mb in ("8", "16", "32", "64", "128", "0"):
    env = dict(os.environ, SP_PIPE_MB=mb)
    subprocess.run([sys.executable, __file__, "child"], env=env)
