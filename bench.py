#!/usr/bin/env python
"""bench.py — headline benchmark of the render path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path
    python bench.py ... --dump-outputs DIR      # also write what the last timed step computed (dump_outputs)

Workload (BASELINE.json configs[1], "C2"): cs16 capture of 100 Mi complex samples PER GPU, FFT
N=4096, Blackman-Harris window, Viridis colormap, dB histogram + colour histogram + min/max/amp
gauges, spectrogram layout, hop == N (width = samples/N, so stride is exactly N and every sample is
read once).  One "step" = one full render of the capture.  N>1: the capture is N times longer and
is sharded by contiguous frame range (weak scaling); each rank renders its frames with the GLOBAL
stride and the histograms / min / max are merged with NCCL all-reduces (no data-path collective).

Prints ONE JSON line (rank 0).  `value` = device-resident input -> device-resident outputs;
`e2e` = the same through the public host-buffer API (pinned host input -> pinned host outputs,
H2D and D2H inside the timed region).  Beside the C2 headline the line carries
  * `configs`: device-resident throughput and roofline fraction of the other BASELINE.json configs (C1, C3 x1..x8,
    one C4 point per kernel family, C5 shard-sized) - N=1 only, `--no-configs` skips it;
  * `c5_strong` (N>1): ONE cf32 capture (2^33 samples at N=8), FFT N=65536, frame-range sharded with halo, strong scaling;
  * `parity_check`: sampled frame groups of the TIMED C2 output against the float64 oracle (pixels off by one colour
    step, dB error per band), so every bench record carries parity at full size.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "spectroplot-js_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "Msamples/s rendered to RGBA spectrogram (N=4096) and % of B200 HBM roofline"
UNIT = "Msamples/s"
FMT, N_FFT, WINDOW, CMAP, GAIN, RANGE = "CS16", 4096, "blackmanHarris", "viridis", 6, 30
SAMPLES_PER_GPU = 100 * (1 << 20)           # 104 857 600 complex samples (419 MB of cs16)
SEED = 0x5EC70002
SW = 4                                      # bytes per cs16 sample
ALG_BYTES_PER_SAMPLE = SW + 4.0             # input + RGBA at hop N (SURVEY.md §8(d)); gauges/hist negligible


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def viridis_cmap():
    from spectro_b200 import cmaps
    cm = [list(c) for c in cmaps.cmaps["viridis_cmap"]]
    cm[0] = [0, 0, 0]; cm[-1] = [255, 255, 255]          # caller-side overwrite, lib/spectroplot.js:1129-1130
    return cmaps.cmap_bytes(cm)


def window_f64():
    from spectro_b200 import windows
    w = windows.blackmanHarrisWindow(N_FFT)
    return np.array(w["window"], np.float64), float(w["weight"])


# ----------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation of the path (the float64 restatement in
# oracle/, since no JavaScript engine exists in this image), all host threads, fan-out exactly as
# lib/spectroplot.js:1206-1228 does it (one slice per worker thread).
# ----------------------------------------------------------------------------------------------
WORKLOAD = ("C2: cs16 100Mi samples/GPU, FFT N=4096, Blackman-Harris, Viridis, hop N "
            "(width {width}), dB+colour histograms, min/max/amp gauges")


def run_reference(args):
    """The reference's CPU implementation of the path on the SAME workload as our arm's N=1 run: the whole C2 capture
    (100 Mi samples, width 25 600) per step, fan-out over all host threads as lib/spectroplot.js:1206-1228."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle as O
    cores = os.cpu_count() or 1
    S = SAMPLES_PER_GPU
    frames = S // N_FFT
    buf = O.synth(FMT, 0, S, S, SEED)
    w, wt = window_f64()
    cm = viridis_cmap()
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        O.render(buf, FMT, N_FFT, frames, w, 1.0 / wt, GAIN, RANGE, cm, workers=cores)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
    ms = 1e3 * float(np.mean(times))
    val = S / (ms * 1e-3) / 1e6
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD.format(width=frames), "samples_total": S, "frames_total": frames,
                       "note": f"the whole C2 capture per step on {cores} worker threads (fan-out as lib/spectroplot.js:1206-1228); "
                               "at N>1 the reference renders one GPU's share (it has no multi-device path)"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{S} samples per step (the whole C2 capture); C float64 restatement of lib/worker.js (oracle/), "
                                       "an upper bound on the JS worker's speed"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)
    return 0


def cpu_baseline_sample():
    """Bounded CPU run of the same workload on the box's host cores (rank 0, N=1 only)."""
    from oracle import oracle as O
    cores = os.cpu_count() or 1
    frames = 1024 * cores
    S = frames * N_FFT
    buf = O.synth(FMT, 0, S, S, SEED)
    w, wt = window_f64()
    cm = viridis_cmap()
    O.render(buf[: 4 * N_FFT * 64 * cores], FMT, N_FFT, 64 * cores, w, 1.0 / wt, GAIN, RANGE, cm, workers=cores)  # warm
    t0 = time.perf_counter()
    O.render(buf, FMT, N_FFT, frames, w, 1.0 / wt, GAIN, RANGE, cm, workers=cores)
    dt = time.perf_counter() - t0
    return {"value": S / dt / 1e6, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"first {S} samples ({frames} frames) of the C2 capture, one pass, {cores} threads; "
                      "C float64 restatement of lib/worker.js (no JS engine in the image)"}


def bind_to_gpu_numa_node(index: int):
    """One process per GPU: run (and therefore allocate the page-locked staging buffers) on the CPUs of the GPU's own
    NUMA node, so that the e2e leg's H2D / D2H copies do not cross the socket interconnect.  Best effort."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:                      # nvml: 00000000:1B:00.0, sysfs: 0000:1b:00.0
            bus = bus[4:]
        base = "/sys/bus/pci/devices/" + bus
        node = int(open(base + "/numa_node").read())
        cpus = set()
        for part in open(base + "/local_cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"node": node, "cpus": len(cpus)}
    except Exception:
        return None



# ----------------------------------------------------------------------------------------------
# parity at full size: frame groups of the TIMED output against the float64 oracle (the checker, never the thing measured)
# ----------------------------------------------------------------------------------------------
def oracle_parity_sample(eng, torch, d_img, width, total_samples, w, wt, cm, groups=6):
    """Groups of 8 consecutive frames of the C2 render (first, last, evenly spread): at hop N a group is itself a message
    of 8N samples with stride N, so the oracle renders exactly the frames the GPU rendered.  Pixels come from the image
    the timed steps wrote; dB values from the engine's dB tap on the same samples."""
    from oracle import oracle as O
    xs = sorted({int(round(i * (width - 8) / max(1, groups - 1))) // 8 * 8 for i in range(groups)})
    lut = {(int(c[0]) << 16) | (int(c[1]) << 8) | int(c[2]): i for i, c in enumerate(cm)}
    img = d_img.view(N_FFT, width, 4)
    off1 = worse = px = 0
    err_hi = err_lo = 0.0
    sq_lo, n_lo = 0.0, 0
    for x in xs:
        raw = O.synth(FMT, x * N_FFT, 8 * N_FFT, total_samples, SEED)
        ora = O.render(raw, FMT, N_FFT, 8, w, 1.0 / wt, GAIN, RANGE, cm, taps=True)
        g = img[:, x:x + 8, :].cpu().numpy().astype(np.int64)
        key = (g[..., 0] << 16) | (g[..., 1] << 8) | g[..., 2]
        gi = np.vectorize(lambda k: lut.get(int(k), -1000))(key)                 # colour index per pixel [row][frame]
        rows = (N_FFT // 2 - np.arange(N_FFT)) % N_FFT                           # bin -> row (lib/worker.js:90)
        oi = np.empty_like(gi)
        oi[rows, :] = ora.gray.T.astype(np.int64)                                # oracle taps are [frame][bin]
        d = np.abs(gi - oi)
        off1 += int((d == 1).sum()); worse += int((d > 1).sum()); px += d.size
        db = eng.render_db(raw, FMT, N_FFT, 8, w, 1.0 / wt, GAIN, RANGE, cm)     # [frame][bin], dBfs - gain
        ref = ora.db
        # bands on the conventional 20 log10 scale: the reference's dB is 10 log10|X| = half of it
        e = np.abs(db.astype(np.float64) - ref)
        hi, lo = ref > -50.0, (ref <= -50.0) & (ref > -60.0)
        if hi.any(): err_hi = max(err_hi, float(e[hi].max()))
        if lo.any():
            err_lo = max(err_lo, float(e[lo].max())); sq_lo += float((e[lo] ** 2).sum()); n_lo += int(lo.sum())
    return {"frames_checked": 8 * len(xs), "frame_groups_at": xs, "pixels_checked": px, "pixels_off_by_one_step": off1,
            "pixels_off_by_more": worse, "off_by_one_fraction": off1 / max(1, px),
            "max_db_err_above_-100dBFS": err_hi, "max_db_err_-120..-100dBFS": err_lo,
            "rms_db_err_-120..-100dBFS": (sq_lo / n_lo) ** 0.5 if n_lo else 0.0,
            "checker": "oracle/ (float64 restatement of lib/worker.js pinned to the reference's own replies)"}


DUMP_FRAMES = 512                           # picture columns kept by --dump-outputs: 4096 x 512 x 4 float32 = 32 MiB


def dump_outputs(out_dir, torch, d_img, d_g, stats, width, world, ncm):
    """--dump-outputs: what the last timed C2 step handed its caller, one DIR/<name>.npy per array, so that two builds
    can be compared output for output.  The RGBA picture (419 MB) is kept at DUMP_FRAMES frames chosen by a fixed seed
    (all N_FFT rows each, their indices in image_frames.npy); gauges, both histograms and dBfs_min / dBfs_max are whole.
    At N > 1 rank 0 writes: the picture sample, its frame indices and the gauges are rank 0's own shard (frames counted
    from its first frame), while the histograms and dBfs_min / dBfs_max are merged over all ranks.  Integers are stored
    as float32 / float64, exactly."""
    from spectro_b200 import sharding
    _, d_hist, d_mm, d_gath = stats
    if world > 1:
        hist, mn, mx = sharding.fold_gathered(torch, d_gath, 1000 + ncm)
    else:
        hist, (mn, mx) = d_hist, d_mm.tolist()
    frames = np.sort(np.random.default_rng(SEED).choice(width, min(width, DUMP_FRAMES), replace=False))
    img = d_img.view(N_FFT, width, 4).index_select(1, torch.from_numpy(frames).to(d_img.device))
    g = d_g.view(3, width).cpu().numpy().astype(np.float32)
    hist = hist.cpu().numpy().astype(np.float64)
    arrays = {"image": img.cpu().numpy().astype(np.float32), "image_frames": frames.astype(np.float64),
              "gauge_mins": g[0], "gauge_maxs": g[1], "gauge_amps": g[2], "cB_hist": hist[:1000], "c_hist": hist[1000:],
              "dBfs_min_max": np.array([mn, mx], np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------------------------
# the other BASELINE.json configs, device resident (N=1): what only builder-run sweeps showed in round 1
# ----------------------------------------------------------------------------------------------
def run_config(eng, torch, stream, dev, tag, fmt, n, zoom, window, cmname, S, steps=3):
    from spectro_b200 import windows, cmaps, _lib
    sw = _lib.load().sp_sample_width(_lib.format_id(fmt))
    width = zoom * S // n
    if zoom > 1:
        width = width // 8 * 8
    w = getattr(windows, window + "Window")(n)
    cm = [list(c) for c in cmaps.cmaps[cmname + "_cmap"]]
    cm[0] = [0, 0, 0]; cm[-1] = [255, 255, 255]
    cmb = cmaps.cmap_bytes(cm)
    nbytes = S * sw
    d_in = torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)
    eng.synth_fill(d_in.data_ptr(), fmt, 0, S, S, 0x5EC70010)
    d_img = torch.empty(4 * width * n, dtype=torch.uint8, device=dev)
    d_g = torch.empty(3 * width, dtype=torch.uint8, device=dev)
    d_hist = torch.zeros(1000 + len(cmb), dtype=torch.int64, device=dev)
    d_mm = torch.zeros(2, dtype=torch.float64, device=dev)
    ww = np.array(w["window"], np.float64)

    def step():
        rq, keep = eng.make_request(d_in.data_ptr(), fmt, n, width, ww, 1.0 / float(w["weight"]), 6, 30, cmb, byte_length=nbytes)
        return eng.render_enqueue(rq, d_img.data_ptr(), (d_g.data_ptr(), d_g.data_ptr() + width, d_g.data_ptr() + 2 * width),
                                  d_hist.data_ptr(), d_hist.data_ptr() + 8000, d_mm.data_ptr())
    for _ in range(3):
        rp = step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        rp = step()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    eng.render_finish(rp)
    total = int(d_hist[1000:].sum().item())
    alg = S * sw + 4.0 * width * n                                  # SURVEY 8(d): sampleWidth + 4 n / H bytes per sample
    peak, _ = measured_peaks()
    out = {"case": tag, "format": fmt, "n": n, "zoom": zoom, "window": window, "cmap": cmname, "samples": S, "width": width,
           "hop": (S - n) / (width - 1), "ms_per_render": ms, "msamples_s": S / ms / 1e3, "algorithmic_gb": alg / 1e9,
           "frac_of_measured_hbm": alg / ms / 1e6 / peak, "launches": rp.kernel_launches, "hist_total_ok": total == width * n,
           "plan": eng.kernel_plan(fmt, n)}
    del d_in, d_img, d_g
    torch.cuda.empty_cache()
    return out


def configs_block(eng, torch, stream, dev):
    """(tag, format, N, zoom, window, colormap, samples).  C3 / C5 are sized to fit one GPU beside each other's buffers:
    C3 at 2^30 samples (the stated size: images of 4 + 8 + 16 + 32 GiB, one level resident at a time), C5 shard-sized
    (2^30 of the 2^33 samples: what one of 8 GPUs renders)."""
    cases = [("C1 cu8 N=1024 Hann Cube1 hop N", "CU8", 1024, 1, "hann", "cube1", 9765 * 1024)]
    cases += [(f"C3 cf32 N=32768 Inferno zoom x{z}", "CF32", 32768, z, "hann", "inferno", 1 << 30) for z in (1, 2, 4, 8)]
    cases += [("C4 cs4 N=128 (render_w_kernel)", "CS4", 128, 1, "blackmanHarris", "viridis", 1 << 26),
              ("C4 cu12 N=512 (render_w_kernel)", "CU12", 512, 1, "blackmanHarris", "viridis", 1 << 26),
              ("C4 cs16 N=128 (render_w_kernel)", "CS16", 128, 1, "hann", "viridis", 1 << 26),
              ("C4 cs16 N=256 (render_w_kernel)", "CS16", 256, 1, "hann", "viridis", 1 << 26),
              ("C4 cs16 N=512 (render_w_kernel)", "CS16", 512, 1, "hann", "viridis", 1 << 26),
              ("C4 cs4 N=2048 (render_rc_kernel)", "CS4", 2048, 1, "blackmanHarris", "viridis", 1 << 26),
              ("C4 cu12 N=4096 (render_r64_kernel)", "CU12", 4096, 1, "blackmanHarris", "viridis", 1 << 26),
              ("C4 cs4 N=16384 (render_big_kernel)", "CS4", 16384, 1, "blackmanHarris", "viridis", 1 << 26),
              ("C4 cu12 N=65536 (render_big_kernel)", "CU12", 65536, 1, "blackmanHarris", "viridis", 1 << 26),
              ("C5 cf32 N=65536 Hann hop N, one GPU's shard of the 8 GSample capture", "CF32", 65536, 1, "hann", "viridis", 1 << 30)]
    # the four-step sizes exist in two forms (csrc/sp_engine.cu): the L2-ring kernel (1.0 x DRAM traffic; chosen by default for
    # these two long captures) and the round-1 HBM-scratch pair - both are reported
    cases += [("C3 cf32 N=32768 zoom x1, HBM-scratch form (SP_FOURSTEP=hbm)", "CF32", 32768, 1, "hann", "inferno", 1 << 30),
              ("C5 cf32 N=65536, HBM-scratch form (SP_FOURSTEP=hbm)", "CF32", 65536, 1, "hann", "viridis", 1 << 30)]
    out = []
    for c in cases:
        hbm = "SP_FOURSTEP=hbm" in c[0]
        if hbm:
            os.environ["SP_FOURSTEP"] = "hbm"
        try:
            out.append(run_config(eng, torch, stream, dev, *c))
        except Exception as ex:                              # a config must never take the headline down with it
            out.append({"case": c[0], "error": repr(ex)[:300]})
            torch.cuda.empty_cache()
        finally:
            if hbm:
                os.environ.pop("SP_FOURSTEP", None)
    return out


def c5_strong(eng, torch, dist, stream, dev, world, rank):
    """BASELINE.json config 5 as stated, strong scaling over the ranks of this run: ONE cf32 capture (2^30 samples per
    GPU, i.e. 2^33 at N=8), FFT N = 65536, hop N, contiguous frame ranges with a window-length halo, histograms and
    min / max merged by one NCCL all-gather.  Returns the record on rank 0."""
    from spectro_b200 import windows, sharding
    fmt, n, sw, seed = "CF32", 65536, 8, 0x5EC70005
    S = (1 << 30) * world
    W = S // n
    sh = sharding.plan_shards(S, n, W, world)[rank]
    width, nbytes = sh["width"], sh["sample_count"] * sw
    cm = viridis_cmap()
    wd = windows.hannWindow(n)
    ww, wt = np.array(wd["window"], np.float64), float(wd["weight"])
    d_in = torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)
    eng.synth_fill(d_in.data_ptr(), fmt, sh["sample_first"], sh["sample_count"], S, seed)
    d_img = torch.empty(4 * width * n, dtype=torch.uint8, device=dev)
    d_g = torch.empty(3 * width, dtype=torch.uint8, device=dev)
    d_stats, d_hist, d_mm, d_gath = sharding.stats_buffers(torch, 1000 + len(cm), world, dev)
    shard = sharding.shard_fields(sh, S, sw, W)

    def step():
        rq, keep = eng.make_request(d_in.data_ptr(), fmt, n, width, ww, 1.0 / wt, 6, 30, cm, byte_length=nbytes, shard=shard)
        rp = eng.render_enqueue(rq, d_img.data_ptr(), (d_g.data_ptr(), d_g.data_ptr() + width, d_g.data_ptr() + 2 * width),
                                d_hist.data_ptr(), d_hist.data_ptr() + 8000, d_mm.data_ptr())
        sharding.gather_stats(dist, d_stats, d_gath)
        return rp
    for _ in range(2):
        rp = step()
    dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = 3
    e0.record(stream)
    for _ in range(steps):
        rp = step()
    e1.record(stream)
    dist.barrier(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    eng.render_finish(rp)
    hist, mn, mx = sharding.fold_gathered(torch, d_gath, 1000 + len(cm))
    total = int(hist[1000:].sum().item())
    ms = float(t.item())
    del d_in, d_img, d_g
    torch.cuda.empty_cache()
    alg = S * sw + 4.0 * W * n
    peak, _ = measured_peaks()
    return {"case": "C5: ONE cf32 capture, FFT N=65536, hop N, frame-range shards with halo, strong scaling over the ranks",
            "samples": S, "n": n, "width": W, "gpus": world, "halo_samples": n, "ms_per_render": ms, "msamples_s": S / ms / 1e3,
            "frac_of_measured_hbm_per_gpu": alg / world / ms / 1e6 / peak, "c_hist_total": total, "hist_total_ok": total == W * n,
            "dBfs_min": mn, "dBfs_max": mx, "merge": "one NCCL all-gather of {cB_hist, c_hist, min, max} per render"}


# ----------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import spectro_b200
    from spectro_b200 import _lib, sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    eng = spectro_b200.Engine(local)
    # a real (non-default) stream shared by torch (events, NCCL) and the engine (kernels)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    eng.set_stream(stream.cuda_stream)

    total_samples = SAMPLES_PER_GPU * world
    total_width = total_samples // N_FFT                    # hop == N exactly
    sh = sharding.plan_shards(total_samples, N_FFT, total_width, world)[rank]
    width = sh["width"]
    nbytes_in = sh["sample_count"] * SW
    w, wt = window_f64()
    cm = viridis_cmap()

    # device-resident capture shard, generated on the device (bit-identical to the oracle's generator)
    d_in = torch.empty(nbytes_in + 256, dtype=torch.uint8, device=dev)
    eng.synth_fill(d_in.data_ptr(), FMT, sh["sample_first"], sh["sample_count"], total_samples, SEED)
    d_img = torch.empty(4 * width * N_FFT, dtype=torch.uint8, device=dev)
    d_g = torch.empty(3 * width, dtype=torch.uint8, device=dev)
    # cB_hist | c_hist (u64 counters) | dBfs_min, dBfs_max: one buffer, so the multi-GPU merge is ONE all-gather.
    # Two sets: the all-gather of message i runs on its own stream while message i+1 renders (nothing in a render
    # depends on the previous message's merged statistics); the timed region ends only when the last gather is done.
    stats = [sharding.stats_buffers(torch, 1000 + len(cm), world, dev) for _ in range(2)]
    coll_stream = torch.cuda.Stream(device=dev) if world > 1 else None
    ev_render = [torch.cuda.Event() for _ in range(2)]
    ev_coll = [torch.cuda.Event() for _ in range(2)]
    state = {"i": 0}
    shard = sharding.shard_fields(sh, total_samples, SW, total_width) if world > 1 else None

    def step():
        rq, keep = eng.make_request(d_in.data_ptr(), FMT, N_FFT, width, w, 1.0 / wt, GAIN, RANGE, cm,
                                    byte_length=nbytes_in, shard=shard)
        b = state["i"] & 1
        state["i"] += 1
        d_stats, d_hist, d_mm, d_gath = stats[b]
        if world > 1:
            stream.wait_event(ev_coll[b])                   # this buffer set was last gathered two messages ago
        rp = eng.render_enqueue(rq, d_img.data_ptr(), (d_g.data_ptr(), d_g.data_ptr() + width, d_g.data_ptr() + 2 * width),
                                d_hist.data_ptr(), d_hist.data_ptr() + 8000, d_mm.data_ptr())
        if world > 1:                                       # the exchange step: one ~10 KB all-gather over NVLink
            ev_render[b].record(stream)
            with torch.cuda.stream(coll_stream):
                coll_stream.wait_event(ev_render[b])
                sharding.gather_stats(dist, d_stats, d_gath)
                ev_coll[b].record(coll_stream)
        return rp

    def join_collectives():
        if world > 1:
            stream.wait_event(ev_coll[0]); stream.wait_event(ev_coll[1])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(3, args.warmup)):
        rp = step()
    barrier()
    eng.profile_enable(args.steps)
    prof_every = int(os.environ.get("SP_BENCH_PROF_EVERY", "4"))
    eng.profile_sample(prof_every)                          # every 4th timed launch carries the kernel's event pair
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    launches = 0
    for _ in range(args.steps):
        rp = step()
    join_collectives()
    e1.record(stream)
    barrier()
    ms_total = e0.elapsed_time(e1)
    kern_ms = eng.profile_read(args.steps)
    if args.dump_outputs and rank == 0:                     # before the untimed steps below reuse the buffers
        dump_outputs(args.dump_outputs, torch, d_img, d_g, stats[(state["i"] - 1) & 1], width, world, len(cm))
    # nvidia-smi samples every 100 ms and the timed region is a few ms: keep the SAME step running (untimed)
    # until the sampler has seen >= 0.7 s of this load, so the clock record describes the kernel under load
    t_load = time.perf_counter()
    while time.perf_counter() - t_load < max(0.0, 0.7 - ms_total * 1e-3):
        for _ in range(20):
            rp = step()
        torch.cuda.synchronize()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "warm-up + timed region + the same step repeated untimed to 0.7 s (nvidia-smi -lms 100)"
    eng.render_finish(rp)
    launches = rp.kernel_launches * args.steps
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = total_samples / (ms_step * 1e-3) / 1e6

    # sanity of the timed output: histogram totals (size-independent property)
    d_stats, d_hist, d_mm, d_gath = stats[(state["i"] - 1) & 1]        # the last message
    if world > 1:                                           # histograms add, min/max fold (lib/spectroplot.js:1229-1238)
        m_hist, m_min, m_max = sharding.fold_gathered(torch, d_gath, 1000 + len(cm))
    else:
        m_hist = d_hist
    c_total = int(m_hist[1000:].sum().item())
    if args.kernel_only:
        if rank == 0:
            kms = float(np.mean(kern_ms)) if len(kern_ms) else ms_step
            peak, _ = measured_peaks()
            emit({"lib": os.environ.get("SP_LIB", "default"), "ms_per_step": ms_step, "kernel_ms": kms,
                  "frac": ALG_BYTES_PER_SAMPLE * sh["sample_count"] / (kms * 1e-3) / 1e9 / peak, "value": value,
                  "hist_ok": c_total == total_width * N_FFT, "clocks": clocks})
        return 0
    assert c_total == total_width * N_FFT, (c_total, total_width * N_FFT)

    # ---- end to end through the host-buffer API (pinned host memory both ways)
    pin_in = spectro_b200.PinnedBuffer(nbytes_in)
    eng.d2h(pin_in.array, d_in.data_ptr())
    pin_img = spectro_b200.PinnedBuffer(4 * width * N_FFT)
    pin_img2 = spectro_b200.PinnedBuffer(4 * width * N_FFT)
    e2e_steps = args.steps
    eng.set_stream(None)
    out = None

    def merge(out):
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, dict(cB_hist=out["cB_hist"], c_hist=out["c_hist"], dBfs_min=out["dBfs_min"],
                                               dBfs_max=out["dBfs_max"]))
            sharding.merge_stats(parts)

    # (1) one message at a time: sp_render, the call of round 1
    for i in range(1 + e2e_steps):
        if i == 1:
            barrier(); t0 = time.perf_counter()
        out = eng.render(pin_in.array, FMT, N_FFT, width, w, 1.0 / wt, GAIN, RANGE, cm, shard=shard,
                         out_image=pin_img.array)
        merge(out)
    barrier()
    e2e_sync_ms = 1e3 * (time.perf_counter() - t0) / e2e_steps
    # (2) the same messages through sp_render_async / sp_render_wait, two in flight (as the reference keeps several worker
    # messages in flight): every step still copies its own input in and its own picture out; the copy-out tail of a step
    # overlaps the copy-in head of the next.  Two output pictures alternate.
    imgs = (pin_img, pin_img2)
    pend = None
    for i in range(2 + e2e_steps):
        if i == 2:                                          # two warm-up messages have been enqueued, one collected
            barrier(); t0 = time.perf_counter()
        h = eng.render_async(pin_in.array, FMT, N_FFT, width, w, 1.0 / wt, GAIN, RANGE, cm, shard=shard,
                             out_image=imgs[i & 1].array)
        if pend is not None:
            out = eng.wait(pend)
            merge(out)
        pend = h
    barrier()
    # steps 2 .. e2e_steps + 1 were enqueued inside the timed region and steps 1 .. e2e_steps collected: e2e_steps messages each way
    e2e_ms = 1e3 * (time.perf_counter() - t0) / e2e_steps
    out = eng.wait(pend)
    merge(out)
    assert int(out["c_hist"].sum()) == width * N_FFT
    te = torch.tensor([e2e_ms, e2e_sync_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms, e2e_sync_ms = float(te[0].item()), float(te[1].item())
    e2e_val = total_samples / (e2e_ms * 1e-3) / 1e6
    h2d = nbytes_in + 8 * N_FFT // 2 + 4 * len(cm)
    d2h = 4 * width * N_FFT + 3 * width + 8 * (1000 + len(cm)) + 16

    c5 = None
    if world > 1 and not args.no_configs:
        img_keep = d_img                                      # (the C2 buffers stay allocated: 1.3 GB of 180)
        eng.set_stream(stream.cuda_stream)
        eng.profile_enable(0)
        try:
            c5 = c5_strong(eng, torch, dist, stream, dev, world, rank)
        except Exception as ex:
            c5 = {"error": repr(ex)[:300]}
        eng.set_stream(None)

    if rank == 0:
        peak, how = measured_peaks()
        kms = float(np.mean(kern_ms)) if len(kern_ms) else ms_step
        alg_bytes = ALG_BYTES_PER_SAMPLE * sh["sample_count"]
        achieved = alg_bytes / (kms * 1e-3) / 1e9
        # DRAM traffic of the dominant kernel comes from an ncu --set full capture (profiles/latest_traffic.json); it is only
        # quoted when that capture was taken on THIS build of the kernels (sp_build_id), otherwise it is stale and left null
        traffic, kname, traffic_note = None, "render kernel of " + eng.kernel_plan(FMT, N_FFT), None
        try:
            with open(os.path.join(ROOT, "profiles", "latest_traffic.json")) as f:
                lt = json.load(f)
            if lt.get("build_id") == _lib.build_id():
                traffic, kname = lt.get("dram_bytes_per_launch"), lt.get("kernel", kname)
                traffic_note = lt.get("source")
            else:
                traffic_note = (f"profiles/latest_traffic.json was captured on build {lt.get('build_id')}, this library is "
                                f"{_lib.build_id()}: stale figure withheld")
        except Exception:
            pass
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": WORKLOAD.format(width=total_width // world),
                           "samples_total": total_samples, "frames_total": total_width, "sharding": f"frame-range x{world}", "numa_binding": numa,
                           "l2": "inputs (419 MB) and outputs (419 MB) per GPU exceed the 126 MB L2; no flush needed",
                           "kernel_plan": eng.kernel_plan(FMT, N_FFT)},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "traffic_source": traffic_note, "peak_source": how, "kernel": kname,
                             "kernel_build": _lib.build_id(),
                             "kernel_ms": kms, "algorithmic_bytes_per_launch": alg_bytes,
                             "kernel_ms_source": f"mean of the {len(kern_ms)} launches of the timed region that were bracketed by a CUDA event pair "
                                                 f"on the launching stream (every {prof_every}th launch: an event pair between dependent kernels "
                                                 "costs the step several microseconds)"},
                "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": e2e_ms, "steps": e2e_steps,
                        "api": "sp_render_async / sp_render_wait, two host-buffer messages in flight (every step copies its own input in "
                               "and its own picture out of pinned memory; the copy-out tail of a step overlaps the copy-in head of the next)",
                        "one_message_at_a_time": {"value": total_samples / (e2e_sync_ms * 1e-3) / 1e6, "ms_per_step": e2e_sync_ms,
                                                  "api": "sp_render"}},
                "gpu_launches": int(launches), "clocks": clocks,
                "parity_check": {"c_hist_total": c_total, "dBfs_min": m_min if world > 1 else rp.dBfs_min,
                                 "dBfs_max": m_max if world > 1 else rp.dBfs_max}}
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline_sample()
            line["parity_check"].update(oracle_parity_sample(eng, torch, d_img, width, total_samples, w, wt, cm))
        if world == 1 and not args.no_configs:
            eng.set_stream(stream.cuda_stream)
            eng.profile_enable(0)                             # no per-launch event pairs: these are whole-render timings
            line["configs"] = configs_block(eng, torch, stream, dev)
        if c5 is not None:
            line["c5_strong"] = c5
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


_RESULT_FD = None


def claim_stdout():
    """stdout carries exactly ONE JSON line: keep the real stdout for it and send everything else written to fd 1 by
    libraries (NCCL prints its version banner there) to stderr."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-configs", action="store_true", help="skip the `configs` block (N=1) / the `c5_strong` record (N>1)")
    ap.add_argument("--kernel-only", action="store_true",
                    help="development: device-resident leg only (no e2e, no cpu leg, no output check) - A/B runs of experiment builds ($SP_LIB)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of this repo's CUDA path computed as DIR/<name>.npy (float32 / float64, "
                         "sampled to <= 64 MB; at N > 1 rank 0's shard with the merged histograms)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to this repo's CUDA path only, not to --impl reference")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
