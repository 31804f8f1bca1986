#!/usr/bin/env python
"""Compressed -png files (vp8_gpu_set_png_deflate) against the stored ones, on the GPU. Writes profiles/pngz_bench.json
(or --out PATH) and prints a summary; the GPU's name and power limit are read in the same run.

  e2e      256 x 1080p compact frames of the bench mix (rgbgrad, checker, diag, noise) -> -png files in pinned host memory, ONE
           pipelined call (vp8_gpu_decode_compact); stored and deflate calls alternate. Median ms per call, file bytes (total
           and per content), d2h_bytes per call. Stored files are checked against the reference's digests, compressed ones
           decoded with PIL against the reference's pixels.
  kernels  1024 RGB images (the same mix) in HBM -> files in HBM: ms per batch of the launch (vp8_gpu_png_time), and
           (RGB bytes read + file bytes written) / time against the HBM copy bandwidth measured here (device-to-device copy
           of 4 GiB, read + write bytes). Per-kernel device times from torch.profiler in a pass of their own.

python tools/pngz_bench.py [--frames 256] [--kernel-frames 1024] [--rounds 5] [--calls 3] [--out PATH]"""
from __future__ import annotations

import argparse
import hashlib
import io
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

FRAMES_1080P = ["rgbgrad_1920x1080_q75.webp", "checker_1920x1080_q75.webp", "diag_1920x1080_q75.webp", "noise_1920x1080_q75.webp"]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()}"


def hbm_copy_gbs(torch):
    n = 4 << 30
    a = torch.empty(n, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    gbs = 2 * n * reps / (e0.elapsed_time(e1) / 1e3) / 1e9
    del a, b
    torch.cuda.empty_cache()
    return gbs


def ppm_digest(png: bytes) -> str:
    from PIL import Image
    im = Image.open(io.BytesIO(png))
    w, h = im.size
    return hashlib.sha256(b"P6\n%d %d\n255\n" % (w, h) + im.tobytes()).hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--kernel-frames", type=int, default=1024)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--calls", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "pngz_bench.json"))
    args = ap.parse_args()
    import torch
    import webp_decoder_b200 as W
    from webp_decoder_b200 import parse as P
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    dg = json.loads((ROOT / "bench_data" / "digests.json").read_text())
    res = {"gpu": gpu_info(), "torch_device": torch.cuda.get_device_name(0)}
    print("GPU (name, power limit, max SM clock):", res["gpu"], flush=True)
    ctx = W.Context(0)
    peak = hbm_copy_gbs(torch)
    res["hbm_copy_gbs_measured"] = peak

    # ---- e2e: one pipelined call, stored and deflate alternated
    n = args.frames
    cf = P.parse_batch_compact([(ROOT / "bench_data" / f).read_bytes() for f in FRAMES_1080P], pinned=True)
    idx = [i % cf.n for i in range(n)]
    cfrs = [cf.frame_list()[i] for i in idx]
    kfs = [cf.kfs[i] for i in idx]
    out = W.PinnedBuffer(ctx.decode_bytes(kfs, ppm="png"))
    modes = {"stored": False, "deflate": True}
    times = {m: [] for m in modes}
    stats = {}
    for r in range(args.rounds + 1):  # round 0 warms up and checks
        for mode, on in modes.items():
            ctx.set_png_deflate(on)
            for c in range(args.calls):
                d0 = ctx.d2h_bytes
                t0 = time.perf_counter()
                offs, sizes = ctx.decode_compact_into(cfrs, out.array, ppm="png")
                ms = (time.perf_counter() - t0) * 1e3
                if r:
                    times[mode].append(ms)
                elif c == 0:
                    files = [out.array[int(o):int(o) + int(s)].tobytes() for o, s in zip(offs, sizes)]
                    if on:
                        ok = all(ppm_digest(f) == dg[FRAMES_1080P[i]]["ppm"] for f, i in zip(files[:8], idx[:8]))
                    else:
                        ok = all(hashlib.sha256(f).hexdigest() == dg[FRAMES_1080P[i]]["png"] for f, i in zip(files, idx))
                    per = {FRAMES_1080P[i].split("_")[0]: len(f) for f, i in zip(files, idx)}
                    stats[mode] = {"file_bytes_total": int(sum(int(s) for s in sizes)), "file_bytes_per_content": per,
                                   "d2h_bytes_per_call": ctx.d2h_bytes - d0, "checked": ok}
    ctx.set_png_deflate(False)
    for mode in modes:
        stats[mode]["median_ms"] = statistics.median(times[mode])
        stats[mode]["ms_all"] = [round(t, 3) for t in times[mode]]
    res["e2e"] = {"frames": n, "what": "compact 1080p frames in pinned host memory -> -png files in pinned host memory, one "
                  "vp8_gpu_decode_compact call (default chunk), host clock around the blocking call", **stats}
    out.close()
    cf.free()
    ctx.trim()
    for mode in modes:
        s = stats[mode]
        print(f"e2e {mode:8s}: median {s['median_ms']:.2f} ms per {n} frames, {s['file_bytes_total'] / 1e6:.1f} MB of files, "
              f"d2h {s['d2h_bytes_per_call'] / 1e6:.1f} MB, per file {s['file_bytes_per_content']}, checked {s['checked']}", flush=True)

    # ---- kernels alone on RGB in HBM
    m = args.kernel_frames
    pf = P.parse_batch([(ROOT / "bench_data" / f).read_bytes() for f in FRAMES_1080P], pinned=True)
    order = [i % pf.n for i in range(m)]
    b = ctx.upload([pf.kfs[i] for i in order], [pf.frames[i] for i in order])
    ctx.run(b, True, W.TIGHT)
    ctx.rgb(b)
    rgb_bytes = sum(pf.kfs[i].width * pf.kfs[i].height * 3 for i in order)
    kern = {}
    for rnd in range(3):
        for mode, on in modes.items():
            ctx.set_png_deflate(on)
            ctx.png(b)
            ctx.png_time()
            for _ in range(5):
                ctx.png(b)
            ms, launches = ctx.png_time()
            kern.setdefault(mode, []).append(ms / launches)
    for mode, on in modes.items():
        ctx.set_png_deflate(on)
        ctx.png(b)
        buf, offs, sizes = ctx.download_png(b)
        fb = int(sum(int(s) for s in sizes))
        ms = statistics.median(kern[mode])
        gbs = (rgb_bytes + fb) / (ms / 1e3) / 1e9
        kern[mode] = {"ms_per_batch": ms, "ms_all": [round(t, 4) for t in kern[mode]], "rgb_bytes_read": rgb_bytes, "file_bytes_written": fb,
                      "gbs": gbs, "frac_of_measured_hbm_copy": gbs / peak}
        print(f"kernels {mode:8s}: {ms:.3f} ms per {m} images, {gbs:.0f} GB/s (RGB read + files written) = "
              f"{100 * gbs / peak:.1f} % of the measured {peak:.0f} GB/s", flush=True)
        del buf
    # per-kernel device times, profiler on, deflate
    ctx.set_png_deflate(True)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            ctx.png(b)
        ctx.sync()
    per_kernel = {}
    for ev in prof.key_averages():
        if "pngz" in ev.key or "Memset" in ev.key:
            per_kernel[ev.key.replace("(anonymous namespace)::", "").split("(")[0]] = round(getattr(ev, "device_time_total", getattr(ev, "cuda_time_total", 0)) / 1e3 / 3, 4)
    kern["deflate"]["per_kernel_ms"] = per_kernel
    print("deflate per kernel (ms per batch):", per_kernel, flush=True)
    ctx.set_png_deflate(False)
    res["kernels"] = {"images": m, **kern}
    b.free()
    pf.free()
    ctx.close()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
