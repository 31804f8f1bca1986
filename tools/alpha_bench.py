"""RGBA door vs -ppm door on the same colour data: vp8_gpu_decode_webp_rgba against vp8_gpu_decode_webp(ppm), alternated in one
process. The 256 inputs wrap the committed 1080p ALPH payloads (tests/golden/alpha/bench_alph_1920x1080_f*.bin, one per
filter, VP8L-compressed) around the 'VP8 ' chunks of the 1080p pictures of bench_data/; the -ppm door gets the same 'VP8 '
chunks as simple files. Needs no Pillow. Prints one JSON line (wall ms per call, host work ms, alpha kernel ms, GPU name and
power limit) and writes it under profiles/ unless --out says otherwise.

    python tools/alpha_bench.py [--frames 256] [--reps 5] [--out profiles/alpha_bench.json]
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:  # the numbers are reported without the card's description rather than not at all
        return {"gpu": f"unknown ({e})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "alpha_bench.json"))
    args = ap.parse_args()
    import alphafix as A
    import webp_decoder_b200 as W
    from webp_decoder_b200 import parse as P

    vp8s = []
    for p in sorted((ROOT / "bench_data").glob("*_1920x1080_q75.webp")):
        vp8s.append([d for t, d in A.chunks(p.read_bytes()) if t == b"VP8 "][0])
    alphs = [(ROOT / "tests" / "golden" / "alpha" / f"bench_alph_1920x1080_f{m}.bin").read_bytes() for m in range(4)]
    rgba_files, ppm_files = [], []
    for i in range(args.frames):
        vp8 = vp8s[i % len(vp8s)]
        rgba_files.append(A.wrap(vp8, 1920, 1080, alphs[(i // len(vp8s)) % 4]))
        ppm_files.append(A.riff(A.chunk(b"VP8 ", vp8)))
    want = json.loads((ROOT / "tests" / "golden" / "alpha.json").read_text())["bench_alph_1920x1080"]["alpha"]
    assert all(hashlib.sha256(P.alpha_plane(rgba_files[k]).tobytes()).hexdigest() == want for k in range(4 * len(vp8s)) if k % len(vp8s) == 0)

    ctx = W.Context(0)
    fa, fp = W.WebpFiles(rgba_files), W.WebpFiles(ppm_files)
    out_a = W.PinnedBuffer(ctx.decode_webp_rgba_bytes(fa))
    out_p = W.PinnedBuffer(ctx.decode_webp_bytes(fp, ppm=True))
    res = {"rgba": [], "ppm": []}
    for rep in range(args.reps + 1):  # the first round warms up both
        for kind in ("rgba", "ppm"):
            ctx.alpha_time()
            t0 = time.perf_counter()
            if kind == "rgba":
                offs, sizes = ctx.decode_webp_rgba_into(fa, out_a.array)
            else:
                offs, sizes = ctx.decode_webp_into(fp, out_p.array, ppm=True)
            wall = (time.perf_counter() - t0) * 1e3
            prof = ctx.last_call_profile()
            ams, alaunch = ctx.alpha_time()
            if rep:
                res[kind].append({"wall_ms": wall, "host_work_ms": prof["host_work_ms"], "alpha_kernel_ms": ams, "alpha_launches": alaunch})
    # same RGB on both doors
    offs_a, sizes_a = ctx.decode_webp_rgba_into(fa, out_a.array)
    offs_p, sizes_p = ctx.decode_webp_into(fp, out_p.array, ppm=True)
    same_rgb = True
    for i in range(0, args.frames, 37):
        pam = out_a.array[int(offs_a[i]):int(offs_a[i]) + int(sizes_a[i])].tobytes()
        ppm = out_p.array[int(offs_p[i]):int(offs_p[i]) + int(sizes_p[i])].tobytes()
        rgba = np.frombuffer(pam[pam.index(b"ENDHDR\n") + 7:], np.uint8).reshape(-1, 4)
        same_rgb &= np.ascontiguousarray(rgba[:, :3]).tobytes() == ppm[ppm.index(b"255\n") + 4:]

    def med(kind, key):
        return round(statistics.median(r[key] for r in res[kind]), 2)

    line = {"what": "tools/alpha_bench.py", "frames": args.frames, "size": "1920x1080", "reps": args.reps,
            "rgba_wall_ms": med("rgba", "wall_ms"), "ppm_wall_ms": med("ppm", "wall_ms"),
            "rgba_host_work_ms": med("rgba", "host_work_ms"), "ppm_host_work_ms": med("ppm", "host_work_ms"),
            "alpha_kernels_ms": med("rgba", "alpha_kernel_ms"), "alpha_launches": res["rgba"][0]["alpha_launches"],
            "rgba_out_bytes": int(sum(sizes_a)), "ppm_out_bytes": int(sum(sizes_p)), "same_rgb": bool(same_rgb),
            "host_cpus": os.cpu_count(), **gpu_info(), "runs": res}
    print(json.dumps({k: v for k, v in line.items() if k != "runs"}))
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(line) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
