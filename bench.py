#!/usr/bin/env python
"""Headline benchmark: decoded Mpixel/s for a batch of 1080p key frames through -yuvf (recon + loop filter -> I420).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload yuvf|yuv|ppm] [--batch B] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...      (one rank per GPU)
    python bench.py --impl reference ...                                              (reference CPU arm)

A step = one pass of the hot path over one batch (default 1024 frames per GPU: 256 each of the noise / rgbgrad /
checker / diag 1080p inputs under bench_data/, made offline by the reference's gen_ppm + encoder --q 75 --loopfilter).

  value            whole-job Mpixel/s with the parsed frames already resident in HBM (kernel stage only)
  roofline         algorithmic bytes (820 B/macroblock in + tight I420 out, SURVEY.md 8d) / device-timed kernel duration,
                   against the measured HBM copy bandwidth of MEASURED_PEAKS.json; `issue` = the same kernel against its
                   own bound, the instruction issue rate (executed warp instructions of the committed ncu capture /
                   (SMs x 4 schedulers x SM clock) / kernel time)
  e2e              same metric through the reference-facing call vp8_gpu_decode_i420: dense Vp8DecodedFrames in pinned
                   HOST memory in (every frame with its own 6.7 MB of arrays), I420 bytes in pinned host memory out
  e2e_compact      same through vp8_gpu_decode_compact: frames as the library's own parser emits them (compact wire
                   format, no host pass)
  e2e_from_webp    .webp bytes in host memory -> I420 bytes in host memory through vp8_gpu_decode_webp (host threads run
                   the bool decoder / token parser, chunk by chunk, while the GPU works); bounded batch
  cpu_baseline     the reference's own m06+m07 on the box's host cores (oracle/cpu_baseline.py), bounded sample, stage-matched
                   with `value` and `e2e`; cpu_baseline_whole = its whole decoder (m01..m07), the counterpart of e2e_from_webp
  configs          BASELINE.json configs 3-5 in small: -ppm batch, one 4K frame latency, mixed-size batch sharded by cost
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

FRAMES_1080P = ["noise_1920x1080_q75.webp", "rgbgrad_1920x1080_q75.webp", "checker_1920x1080_q75.webp", "diag_1920x1080_q75.webp"]
METRIC = "decoded Mpixel/s (1080p -yuvf batch)"
DATA = "synthetic (gen_ppm patterns through the reference encoder, --q 75 --loopfilter; no published dataset)"
SM_COUNT = 148


def workload_string(workload, batch):
    """The same on both arms: what one step decodes."""
    return (f"{batch} x 1920x1080 key frames per GPU, -{workload} "
            f"({'recon only' if workload == 'yuv' else 'recon + loop filter'}{' + fancy-upsampled RGB' if workload == 'ppm' else ''}), "
            "q75 --loopfilter level 8, mix noise/rgbgrad/checker/diag in equal parts, interleaved")


def algorithmic_bytes(w, h, workload):
    mb = ((w + 15) // 16) * ((h + 15) // 16)
    if workload == "ppm":
        return 820 * mb + 3 * w * h
    return 820 * mb + w * h + 2 * ((w + 1) // 2) * ((h + 1) // 2)


class ClockSampler:
    """nvidia-smi clocks and throttle reasons under load (profiling recipe's clocks line). Started before the warm-up;
    samples whose timestamp falls inside the timed region are preferred, else all samples since the warm-up began
    (the GPU runs the same kernel back to back through both)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc, self.t0, self.t1 = gpu_index, [], None, None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def mark_timed(self, t0, t1):
        self.t0, self.t1 = t0, t1

    def stop(self):
        if not self.proc:
            return None
        time.sleep(0.05)
        self.proc.terminate()
        self.t.join(timeout=2)
        ok = [(ts, r) for ts, r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        inside = [(ts, r) for ts, r in ok if self.t0 is not None and self.t0 <= ts <= self.t1]
        use, window = (inside, "timed region") if inside else (ok, "warm-up + timed region")
        if not use:
            return None
        sm = [float(r[1]) for _, r in use]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for _, r in use for n, v in zip(names, r[5:9]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(use[0][1][2]), "power_w_max": max(float(r[3]) for _, r in use),
                "samples": len(sm), "window": window, "reasons": reasons}


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_record(workload, kernel_name):
    """What the committed ncu capture of this kernel says per launch of the benchmark batch (profiles/current.json,
    written from the .ncu-rep by tools/ncu_summary.py): DRAM bytes and executed warp instructions."""
    p = ROOT / "profiles" / "current.json"
    if p.exists():
        return json.loads(p.read_text()).get(workload, {}).get(kernel_name)
    return None


def files_for(args):
    return [str(ROOT / "bench_data" / f) for f in FRAMES_1080P]


# The contract is ONE JSON line on stdout. Libraries print there too (NCCL announces its version on the first collective
# when NCCL_DEBUG says so), so the process's stdout is pointed at stderr for the whole run and the line goes out through a
# saved descriptor.
_JSON_FD = None


def claim_stdout():
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def cpu_arm(files, mode, seconds, whole=False):
    out = subprocess.run([sys.executable, str(ROOT / "oracle" / "cpu_baseline.py"), *files, "--mode", mode, "--seconds", str(seconds)] +
                         (["--whole"] if whole else []), capture_output=True, text=True)
    if out.returncode == 0:
        r = json.loads(out.stdout.strip().splitlines()[-1])
        return {"value": r["value"], "unit": "Mpixel/s", "cores": r["cores"], "kind": r["kind"], "flags": r.get("flags"), "sample": r["sample"]}
    return {"value": None, "unit": "Mpixel/s", "cores": 0, "kind": "unavailable", "sample": out.stderr[-300:]}


# ------------------------------------------------------------------------------------------------ reference arm
def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    files = files_for(args)
    # bounded sample: a "step" is ~2 s of decoding on every core at once; calibration pass = warm-up
    seconds = min(60.0, max(6.0, 2.0 * args.steps))
    t0 = time.perf_counter()
    r = cpu_arm(files, args.workload, seconds)
    whole = cpu_arm(files, args.workload, min(seconds, 12.0), whole=True)
    wall = time.perf_counter() - t0
    line = {
        "impl": "reference", "metric": METRIC if args.workload == "yuvf" else f"decoded Mpixel/s (1080p -{args.workload} batch)",
        "value": r["value"], "unit": "Mpixel/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": seconds * 1e3 / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8/int16", "data": DATA,
        "config": {"workload": workload_string(args.workload, args.batch),
                   "note": "reference m06+m07 CPU code on all host threads; one process per core; bounded sample of the same inputs",
                   "wall_s": round(wall, 1)},
        "cpu_baseline": r,
        "e2e": {"value": r["value"], "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "e2e_from_webp": {"value": whole["value"], "unit": "Mpixel/s", "cores": whole["cores"], "sample": whole["sample"],
                          "note": "the reference's whole decoder per frame (m01 + m02 + m05 + m06 + m07, main.c:630-702), one process per core"},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------------ host topology
def gpu_local_cpus(index):
    """CPUs local to GPU `index` (sysfs), or None."""
    try:
        import torch
        p = torch.cuda.get_device_properties(index)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        return Path(f"/sys/bus/pci/devices/{bdf}/local_cpulist").read_text().strip()
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------ GPU arm
def gpu_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)

    # CPU baselines first (rank 0, N=1 only): no GPU work competes for the host cores while they run
    cpu = cpu_whole = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_arm(files_for(args), args.workload, args.cpu_seconds)
        cpu_whole = cpu_arm(files_for(args), args.workload, min(args.cpu_seconds, 8.0), whole=True)

    import webp_decoder_b200 as W
    from webp_decoder_b200 import parse as P
    from webp_decoder_b200 import shard as S

    # a non-default torch stream: its handle is what the library launches on, so torch.cuda.Event sees our kernels
    stream = torch.cuda.Stream(device=local)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    ctx = W.Context(local, stream.cuda_stream)
    kernel_version = args.kernel or int(os.environ.get("VP8_GPU_KERNEL", "3") or 3)
    ctx.set_kernel(kernel_version)
    if args.warps or args.images_per_sm:
        ctx.set_tuning(args.warps, args.images_per_sm)
    # The ranks of one node share its cores and its memory: each rank binds itself (and the library's worker threads,
    # and thereby its pinned staging) to its share of the CPUs that are local to its GPU.
    host = {"cpus_visible": len(os.sched_getaffinity(0))}
    if world > 1 and not args.no_bind:
        lists = [gpu_local_cpus(i) for i in range(world)]
        mine = lists[local]
        sharers = [i for i in range(world) if lists[i] == mine]
        bound = ctx.bind_host(sharers.index(local), len(sharers)) if mine else 0
        host.update({"gpu_local_cpulist": mine, "ranks_sharing_it": len(sharers), "cpus_bound": bound})
    threads = len(os.sched_getaffinity(0)) if (world == 1 or host.get("cpus_bound")) else max(1, (os.cpu_count() or 1) // world)
    if os.environ.get("VP8_GPU_HOST_THREADS"):
        threads = int(os.environ["VP8_GPU_HOST_THREADS"])
    host["host_threads_per_gpu"] = threads

    # ---- inputs: parse the distinct frames once (host threads, pinned arenas)
    files = files_for(args)
    datas = [Path(f).read_bytes() for f in files]
    pf = P.parse_batch(datas, pinned=True)
    nd = pf.n
    order = [i % nd for i in range(args.batch)]  # interleaved mix
    kfs = [pf.kfs[i] for i in order]
    frs = [pf.frames[i] for i in order]
    w, h = pf.kfs[0].width, pf.kfs[0].height
    px_step = sum(pf.kfs[i].width * pf.kfs[i].height for i in order)
    alg_bytes = sum(algorithmic_bytes(pf.kfs[i].width, pf.kfs[i].height, args.workload) for i in order)
    filtered = args.workload != "yuv"
    ppm = args.workload == "ppm"
    dg = json.loads((ROOT / "bench_data" / "digests.json").read_text())
    key = "ppm" if ppm else ("yuvf" if filtered else "yuv")
    want = [dg[Path(files[i]).name][key] for i in order]

    def check(buf, offs, sizes, idx=None):
        idx = range(len(offs)) if idx is None else idx
        return all(hashlib.sha256(buf[int(offs[i]):int(offs[i]) + int(sizes[i])]).hexdigest() == want[i] for i in idx)

    def step_resident(b):
        ctx.run(b, filtered, W.TIGHT)
        if ppm:
            ctx.rgb(b)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def job_max(ms):
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- (1) kernel stage, inputs resident in HBM
    batch = ctx.upload(kfs, frs)
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(args.warmup):
        step_resident(batch)
    ctx.kernel_time()
    ctx.rgb_time()
    sync_all()
    l0 = ctx.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tw0 = time.perf_counter()
    e0.record(stream)
    for _ in range(args.steps):
        step_resident(batch)
    e1.record(stream)
    sync_all()
    sampler.mark_timed(tw0, time.perf_counter())
    elapsed_ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    launches = ctx.launches - l0
    kern_ms, kern_n = ctx.kernel_time()
    rgb_ms, rgb_n = ctx.rgb_time()
    cfg = ctx.last_launch_config()
    job_ms = job_max(elapsed_ms)
    value = world * px_step * args.steps / (job_ms / 1e3) / 1e6

    # every frame of the resident result against the reference decoder's digests (outside the timed region)
    if ppm:
        buf, offs, sizes = ctx.download_ppm(batch)
    else:
        buf, offs, sizes = ctx.download_i420(batch)
    parity = check(buf, offs, sizes)
    if args.dump_outputs and rank == 0:
        dump_outputs(Path(args.dump_outputs), args.workload, buf, offs, sizes)
    del buf
    batch.free()
    ctx.trim()

    # ---- (2) end to end: host buffers in, host buffers out, three input contracts
    e2e = e2e_compact = e2e_webp = None
    if not args.no_e2e:
        host_out = W.PinnedBuffer(ctx.decode_bytes(kfs, ppm=ppm))

        def timed_calls(fn, steps, warm):
            for _ in range(warm):
                fn()
            sync_all()
            h0, d0 = ctx.h2d_bytes, ctx.d2h_bytes
            e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e2.record(stream)
            prof = []
            for _ in range(steps):
                fn()
                prof.append(ctx.last_call_profile())
            e3.record(stream)
            sync_all()
            wall_ms = (time.perf_counter() - t0) * 1e3
            ms = job_max(max(wall_ms, e2.elapsed_time(e3)))
            return ms / steps, (ctx.h2d_bytes - h0) // steps, (ctx.d2h_bytes - d0) // steps, prof[-1]

        n_e2e = max(1, min(args.steps, args.e2e_steps))
        warm = max(1, min(args.warmup, 2))

        # (2a) the reference's contract: dense Vp8DecodedFrames, every frame with its own host memory
        dense = P.replicate_dense(pf, order)
        dkfs, dfrs = dense.kf_list(), dense.frame_list()
        # transport "auto": chunk by chunk, dense when the copy engine has run dry, compact (host threads drop the all-zero
        # blocks) otherwise - neither the link nor the host threads wait for the other
        ctx.set_transport({"auto": "auto", "compact": True, "dense": False}[args.transport], threads)
        ms, up, down, prof = timed_calls(lambda: ctx.decode_into(dkfs, dfrs, host_out.array, filtered=filtered, ppm=ppm, chunk=args.chunk), n_e2e, warm)
        ok = check(host_out.array, *_layout(ctx, dkfs, ppm), idx=_spot(args.batch))
        e2e = {"value": world * px_step / (ms / 1e3) / 1e6, "unit": "Mpixel/s", "h2d_bytes_per_step": up, "d2h_bytes_per_step": down,
               "steps": n_e2e, "ms_per_step": ms, "api": "vp8_gpu_decode_ppm" if ppm else "vp8_gpu_decode_i420",
               "transport": {"mode": args.transport, **ctx.last_transport(), "host_threads": threads},
               "host_bytes_in_per_step": dense.nbytes, "host_profile_ms": prof, "bit_exact_spot_check": ok,
               "note": "dense Vp8DecodedFrame arrays (the reference's m05 output layout) in pinned host memory, one private copy per "
                       "frame; token decode (m03/m05) not included"}
        dense.free()

        # (2b) the library's own parser output: compact frames, nothing to do on the host
        cf = P.parse_batch_compact(datas, pinned=True, replicate=args.batch // nd)
        cfrs = cf.frame_list()[:args.batch]
        ms, up, down, prof = timed_calls(lambda: ctx.decode_compact_into(cfrs, host_out.array, filtered=filtered, ppm=ppm, chunk=args.chunk), n_e2e, warm)
        ok = check(host_out.array, *_layout(ctx, kfs[:len(cfrs)], ppm), idx=_spot(len(cfrs)))
        e2e_compact = {"value": world * sum(f.width * f.height for f in cfrs) / (ms / 1e3) / 1e6, "unit": "Mpixel/s", "h2d_bytes_per_step": up,
                       "d2h_bytes_per_step": down, "steps": n_e2e, "ms_per_step": ms, "api": "vp8_gpu_decode_compact",
                       "host_bytes_in_per_step": cf.used, "host_profile_ms": prof, "bit_exact_spot_check": ok,
                       "note": "frames as vp8_parse_batch_compact emits them (per-macroblock mask + non-zero blocks), pinned, one private "
                               "copy per frame; token decode not included"}
        cf.free()

        # (2c) from .webp bytes: host threads parse chunk k while the GPU works on the chunks before it
        nw = max(nd, min(args.batch, args.webp_batch))
        wf = W.WebpFiles([datas[i % nd] for i in range(nw)])
        ctx.set_transport("auto", threads)
        steps_w = max(1, min(n_e2e, 2))
        ms, up, down, prof = timed_calls(lambda: ctx.decode_webp_into(wf, host_out.array, filtered=filtered, ppm=ppm, chunk=args.chunk), steps_w, 1)
        ok = check(host_out.array, *_layout(ctx, kfs[:nw], ppm), idx=_spot(nw))
        e2e_webp = {"value": world * (px_step * nw // args.batch) / (ms / 1e3) / 1e6, "unit": "Mpixel/s", "h2d_bytes_per_step": up,
                    "d2h_bytes_per_step": down, "steps": steps_w, "ms_per_step": ms, "frames_per_step": nw, "api": "vp8_gpu_decode_webp",
                    "host_threads": threads, "host_profile_ms": prof, "bit_exact_spot_check": ok,
                    "note": "container + header + bool decoder + token parsing on the host threads (serial per frame), everything "
                            "after it on the GPU; bound by the parser threads, not by the GPU stage"}
        host_out.close()
        ctx.trim()

    # ---- (3) BASELINE configs 3-5 in small (outside the headline's timed regions)
    configs = None
    if not args.no_configs:
        try:
            configs = other_configs(ctx, W, P, S, torch, dist, world, rank, local, stream, job_max, sync_all, ppm_done=ppm, args=args)
        except Exception as e:  # the headline above is measured already: a failing side leg is reported, not allowed to swallow the line
            import traceback
            traceback.print_exc()
            configs = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        peak, peak_src = measured_peak()
        k_ms = kern_ms / max(kern_n, 1)
        achieved = alg_bytes / (k_ms / 1e3) / 1e9 if kern_n else None
        kname = {2: "vp8_mb_pairs", 3: "vp8_mb_lockstep"}[kernel_version]
        rec = ncu_record("yuvf" if ppm else args.workload, kname) if args.batch == 1024 else None
        issue = None
        if rec and rec.get("inst_executed") and clocks:
            slots = SM_COUNT * 4 * clocks["sm_mhz"] * 1e6 * (k_ms / 1e3)
            issue = {"inst_executed_per_launch": rec["inst_executed"], "issue_slots": slots, "frac": rec["inst_executed"] / slots,
                     "per_macroblock": rec["inst_executed"] / (args.batch * 8160), "source": rec.get("file"),
                     "note": "executed warp instructions (ncu capture of this kernel on this batch) / (148 SMs x 4 schedulers x SM clock x "
                             "kernel time): how close the kernel is to its own bound, the issue rate"}
        line = {
            "metric": METRIC if args.workload == "yuvf" else f"decoded Mpixel/s (1080p -{args.workload} batch)",
            "value": value, "unit": "Mpixel/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": job_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/int16", "data": DATA,
            "config": {"workload": workload_string(args.workload, args.batch),
                       "images_per_s": value * 1e6 / (w * h), "batch_per_gpu": args.batch, "distinct_frames": nd,
                       "cache": f"inputs {sum(820 * pf.frames[i].mb_total for i in order) / 1e9:.2f} GB per step, far larger than the 126 MB L2",
                       "launch": cfg, "bit_exact_all_frames_vs_reference_digests": parity, "host": host},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                         "traffic": rec.get("dram_bytes") if rec else None, "traffic_source": rec.get("file") if rec else None,
                         "peak_source": peak_src, "kernel": kname, "kernel_ms": k_ms, "algorithmic_bytes_per_launch": alg_bytes,
                         "launches_timed": kern_n, "issue": issue,
                         "rgb_kernel": ({"kernel": "vp8_i420_to_rgb", "kernel_ms": rgb_ms / rgb_n, "algorithmic_bytes_per_launch": 4.5 * px_step,
                                         "achieved": 4.5 * px_step / (rgb_ms / rgb_n / 1e3) / 1e9,
                                         "frac": 4.5 * px_step / (rgb_ms / rgb_n / 1e3) / 1e9 / peak} if rgb_n else None)},
            "cpu_baseline": cpu,
            "cpu_baseline_whole": cpu_whole,
            "e2e": e2e,
            "e2e_compact": e2e_compact,
            "e2e_from_webp": e2e_webp,
            "configs": configs,
            "gpu_launches": launches,
            "clocks": clocks,
        }
        emit(line)
    pf.free()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


DUMP_BYTES = 64 << 20
DUMP_SAMPLES_PER_FRAME = 8192


def dump_outputs(out_dir, name, buf, offs, sizes):
    """Writes what the last timed step computed (frame i = buf[offs[i]:offs[i]+sizes[i]]) to out_dir, so that two builds can be
    compared output for output; the inputs are the same files on every run. At most DUMP_BYTES in all:
      <name>_frame0.npy       every byte of frame 0, float32
      <name>_sample.npy       (frames, K) float32: the bytes at K positions per frame, drawn with a fixed seed (the same
                              positions for every frame of one size)
      <name>_frame_sums.npy   float64 sum of every byte of each frame (exact), so that a change outside the sample shows too"""
    import numpy as np
    out_dir.mkdir(parents=True, exist_ok=True)
    offs, sizes = offs.astype(np.int64), sizes.astype(np.int64)
    n = len(offs)
    frame0 = buf[offs[0]:offs[0] + sizes[0]].astype(np.float32)
    payload = DUMP_BYTES - 3 * 4096  # room for the three .npy headers (128 bytes each as numpy writes them today)
    k = int(min(DUMP_SAMPLES_PER_FRAME, sizes.min(), (payload - frame0.nbytes - 8 * n) // (4 * n)))
    if k < 1:
        raise SystemExit(f"--dump-outputs: {n} frames do not fit {DUMP_BYTES >> 20} MB")
    positions = {}
    sample = np.empty((n, k), np.float32)
    sums = np.empty(n, np.float64)
    for i, (o, s) in enumerate(zip(offs, sizes)):
        if s not in positions:
            positions[s] = np.sort(np.random.default_rng(int(s)).choice(int(s), k, replace=False))
        frame = buf[o:o + s]
        sample[i] = frame[positions[s]]
        sums[i] = frame.sum(dtype=np.uint64)
    np.save(out_dir / f"{name}_frame0.npy", frame0)
    np.save(out_dir / f"{name}_sample.npy", sample)
    np.save(out_dir / f"{name}_frame_sums.npy", sums)


def _layout(ctx, kfs, ppm):
    """(offsets, sizes) of the frames inside the output buffer of a pipelined call (256-byte aligned slots)."""
    offs, sizes, at = [], [], 0
    for k in kfs:
        w, h = k.width, k.height
        if ppm:
            hdr = len(f"P6\n{w} {h}\n255\n")
            offs.append(at + 32 - hdr)
            sizes.append(hdr + w * h * 3)
            at += (32 + w * h * 3 + 255) // 256 * 256
        else:
            n = w * h + 2 * ((w + 1) // 2) * ((h + 1) // 2)
            offs.append(at)
            sizes.append(n)
            at += (n + 255) // 256 * 256
    return offs, sizes


def _spot(n):
    return sorted({0, 1, 2, 3, n // 2, n - 1} & set(range(n)))


def other_configs(ctx, W, P, S, torch, dist, world, rank, local, stream, job_max, sync_all, ppm_done, args):
    """BASELINE.json configs 3, 4, 5, each bounded to a few seconds; every result is byte-checked against the reference
    decoder's digests (bench_data/digests.json, bench_data/mixed/digests.json)."""
    import numpy as np
    out = {}
    dg = json.loads((ROOT / "bench_data" / "digests.json").read_text())
    peak, _ = measured_peak()

    def sha_all(buf, offs, sizes):
        return [hashlib.sha256(buf[int(o):int(o) + int(s)]).hexdigest() for o, s in zip(offs, sizes)]

    # ---- config 4: the 1080p batch through -ppm (recon + loop filter + RGB), kernel stage
    if not ppm_done:
        names = FRAMES_1080P
        pf = P.parse_batch([(ROOT / "bench_data" / n).read_bytes() for n in names], pinned=True)
        order = [i % pf.n for i in range(args.batch)]
        b = ctx.upload([pf.kfs[i] for i in order], [pf.frames[i] for i in order])
        for _ in range(2):
            ctx.run(b, True, W.TIGHT)
            ctx.rgb(b)
        ctx.kernel_time(), ctx.rgb_time()
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        e0.record(stream)
        for _ in range(reps):
            ctx.run(b, True, W.TIGHT)
            ctx.rgb(b)
        e1.record(stream)
        sync_all()
        ms = job_max(e0.elapsed_time(e1)) / reps
        k_ms, k_n = ctx.kernel_time()
        r_ms, r_n = ctx.rgb_time()
        buf, offs, sizes = ctx.download_ppm(b)
        ok = sha_all(buf, offs, sizes) == [dg[names[i]]["ppm"] for i in order]
        # m09 kernels on the same batch (RGB in HBM -> -png files in HBM)
        for _ in range(2):
            ctx.png(b)
        ctx.png_time()
        for _ in range(reps):
            ctx.png(b)
        p_ms, p_n = ctx.png_time()
        buf, offs, sizes = ctx.download_png(b)
        ok_png = sha_all(buf, offs, sizes) == [dg[names[i]]["png"] for i in order]
        png_bytes = 2 * int(sum(int(x) for x in sizes))  # every file byte read once (as RGB) and written once
        px = sum(pf.kfs[i].width * pf.kfs[i].height for i in order)
        algb = sum(algorithmic_bytes(pf.kfs[i].width, pf.kfs[i].height, "ppm") for i in order)
        out["ppm_1080p_batch"] = {"value": world * px / (ms / 1e3) / 1e6, "unit": "Mpixel/s", "ms_per_step": ms, "frames_per_gpu": args.batch,
                                  "wavefront_ms": k_ms / k_n, "rgb_ms": r_ms / r_n,
                                  "roofline": {"bound": "hbm", "achieved": algb / (ms / 1e3) / 1e9, "peak": peak, "frac": algb / (ms / 1e3) / 1e9 / peak,
                                               "algorithmic_bytes_per_step": algb,
                                               "rgb_kernel_frac": 4.5 * px / (r_ms / r_n / 1e3) / 1e9 / peak},
                                  "bit_exact_all_frames_vs_reference_digests": ok,
                                  "png_kernels": {"ms": p_ms / p_n, "algorithmic_bytes": png_bytes, "achieved_gbs": png_bytes / (p_ms / p_n / 1e3) / 1e9,
                                                  "frac": png_bytes / (p_ms / p_n / 1e3) / 1e9 / peak, "bit_exact_all_frames_vs_reference_digests": ok_png,
                                                  "note": "vp8_png_frame + vp8_png_finish on the 1024 RGB images in HBM (m09: stored-deflate framing, "
                                                          "Adler-32, CRC-32); CUDA events around the launch pair"}}
        del buf
        b.free()
        pf.free()
        ctx.trim()

    # ---- the -png path (m09, north_star: "-png is a drop-in"): compact frames in host memory -> the reference's -png files in host
    #      memory in ONE pipelined call; the PNG framing (stored deflate, Adler-32, CRC-32) happens in HBM (vp8_png_frame), the
    #      host only moves bytes. Every file checked against `decoder -png`. Beside it: the same job with the framing done on
    #      the host threads (vp8_gpu_png_frame per picture), which is what this path did before the kernel existed.
    if not args.no_e2e:
        from concurrent.futures import ThreadPoolExecutor
        names = FRAMES_1080P
        n_png = args.png_batch
        cf = P.parse_batch_compact([(ROOT / "bench_data" / names[i % len(names)]).read_bytes() for i in range(len(names))], pinned=True)
        cfrs = [cf.frame_list()[i % cf.n] for i in range(n_png)]
        kfs = [cf.kfs[i % cf.n] for i in range(n_png)]
        threads = max(1, len(os.sched_getaffinity(0)))
        host_png = W.PinnedBuffer(ctx.decode_bytes(kfs, ppm="png"))
        d2h0 = ctx.d2h_bytes
        offs, sizes = ctx.decode_compact_into(cfrs, host_png.array, ppm="png", chunk=args.chunk)
        d2h_png = ctx.d2h_bytes - d2h0
        sync_all()
        reps = 3
        t0 = time.perf_counter()
        for _ in range(reps):
            offs, sizes = ctx.decode_compact_into(cfrs, host_png.array, ppm="png", chunk=args.chunk)
        sync_all()
        ms = job_max((time.perf_counter() - t0) * 1e3) / reps
        ok = sha_all(host_png.array, offs, sizes) == [dg[names[i % len(names)]]["png"] for i in range(n_png)]
        host_png.close()
        # the host-framed variant
        host_ppm = W.PinnedBuffer(ctx.decode_bytes(kfs, ppm=True))
        L = W.load_library()
        L.vp8_gpu_png_bound.argtypes, L.vp8_gpu_png_bound.restype = [C.c_uint32, C.c_uint32], C.c_size_t
        L.vp8_gpu_png_frame.argtypes, L.vp8_gpu_png_frame.restype = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p], C.c_size_t
        png_out = np.empty((n_png, L.vp8_gpu_png_bound(1920, 1080)), np.uint8)

        def frame_png(i):
            o = int(offs[i]) + int(sizes[i]) - 1920 * 1080 * 3  # RGB behind the PPM header
            return L.vp8_gpu_png_frame(host_ppm.array[o:].ctypes.data, 1920, 1080, png_out[i].ctypes.data)

        def run_host_framed():
            nonlocal offs, sizes
            offs, sizes = ctx.decode_compact_into(cfrs, host_ppm.array, filtered=True, ppm=True, chunk=args.chunk)
            with ThreadPoolExecutor(threads) as ex:
                return list(ex.map(frame_png, range(n_png)))
        run_host_framed()
        sync_all()
        t0 = time.perf_counter()
        lens = run_host_framed()
        sync_all()
        ms_host = job_max((time.perf_counter() - t0) * 1e3)
        ok_host = all(hashlib.sha256(png_out[i, :lens[i]]).hexdigest() == dg[names[i % len(names)]]["png"] for i in range(n_png))
        out["png_1080p_batch"] = {"value": world * n_png * 1920 * 1080 / (ms / 1e3) / 1e6, "unit": "Mpixel/s", "ms_per_step": ms,
                                  "frames_per_gpu": n_png, "d2h_bytes_per_step": d2h_png, "bit_exact_all_frames_vs_reference_digests": ok,
                                  "api": "vp8_gpu_decode_compact(VP8_GPU_OUT_PNG)",
                                  "host_framed": {"ms_per_step": ms_host, "host_threads": threads, "bit_exact": ok_host},
                                  "note": "compact frames in host memory -> PNG files in host memory, one pipelined call; framing and both "
                                          "checksums on the device (vp8_png_frame / vp8_png_finish), bound by the device->host link; "
                                          "host_framed = the same job with vp8_gpu_png_frame per picture on the host threads"}
        host_ppm.close()
        cf.free()
        del png_out
        ctx.trim()

    # ---- config 3: one 3840x2160 frame, latency of recon + loop filter (one image per GPU: replicas, no split)
    lat = {}
    for name in ("checker_3840x2160_q75.webp", "rgbgrad_3840x2160_q75.webp"):
        pf = P.parse_batch([(ROOT / "bench_data" / name).read_bytes()], pinned=True)
        b = ctx.upload([pf.kfs[0]], [pf.frames[0]])
        for _ in range(3):
            ctx.run(b, True, W.TIGHT)
        ctx.kernel_time()
        for _ in range(20):
            ctx.run(b, True, W.TIGHT)
        ms, n = ctx.kernel_time()
        buf, offs, sizes = ctx.download_i420(b)
        lat[name] = {"latency_us": job_max(ms / n) * 1e3, "launch": ctx.last_launch_config(), "bit_exact": sha_all(buf, offs, sizes) == [dg[name]["yuvf"]]}
        b.free()
        pf.free()
    out["latency_4k_one_frame"] = {"unit": "us", "frames": lat, "value": max(v["latency_us"] for v in lat.values()),
                                   "note": "device time of one vp8_gpu_run (recon + loop filter) on one 3840x2160 frame resident in HBM; the frame "
                                           "is spread over a thread-block cluster of CTAs; under torchrun every rank decodes its own replica"}

    # ---- config 5: mixed sizes / qualities / modes, sharded over the ranks by cost (macroblocks), no collective
    mixed_dir = ROOT / "bench_data" / "mixed"
    if (mixed_dir / "digests.json").exists():
        mdg = json.loads((mixed_dir / "digests.json").read_text())
        names = sorted(mdg) * args.mixed_copies
        costs = [((mdg[n]["width"] + 15) // 16) * ((mdg[n]["height"] + 15) // 16) for n in names]
        mine = S.shard_by_cost(costs, world)[rank]
        wf = W.WebpFiles([(mixed_dir / names[i]).read_bytes() for i in mine])
        cf = P.parse_batch_compact([(mixed_dir / names[i]).read_bytes() for i in mine], pinned=True)
        cfrs = cf.frame_list()
        kfs = [cf.kfs[i] for i in range(cf.n)]
        host_out = W.PinnedBuffer(ctx.decode_bytes(kfs, ppm=False))

        def run_compact():
            return ctx.decode_compact_into(cfrs, host_out.array, filtered=True, chunk=args.chunk)

        def run_webp():
            return ctx.decode_webp_into(wf, host_out.array, filtered=True, chunk=args.chunk)
        res = {}
        for label, fn, reps in (("from_compact_frames", run_compact, 3), ("from_webp", run_webp, 1)):
            fn()
            sync_all()
            t0 = time.perf_counter()
            for _ in range(reps):
                offs, sizes = fn()
            sync_all()
            ms = job_max((time.perf_counter() - t0) * 1e3) / reps
            ok = sha_all(host_out.array, offs, sizes) == [mdg[names[i]]["yuvf"] for i in mine]
            res[label] = {"ms_per_step": ms, "bit_exact_all_frames_vs_reference_digests": ok}
        px = sum(mdg[n]["width"] * mdg[n]["height"] for n in names)
        flags = torch.tensor([float(all(r["bit_exact_all_frames_vs_reference_digests"] for r in res.values())), float(sum(costs[i] for i in mine))],
                             dtype=torch.float64, device="cuda")
        share = [flags.clone() for _ in range(world)]
        if world > 1:
            dist.all_gather(share, flags)
        out["mixed_batch"] = {"value": px / (res["from_compact_frames"]["ms_per_step"] / 1e3) / 1e6, "unit": "Mpixel/s", "frames_total": len(names),
                              "value_from_webp": px / (res["from_webp"]["ms_per_step"] / 1e3) / 1e6,
                              "ms_per_step": {k: v["ms_per_step"] for k, v in res.items()},
                              "sharding": "longest-first by macroblock count (webp-decoder_b200/shard.py), no data-path collective",
                              "macroblocks_per_rank": [int(s[1].item()) for s in share],
                              "bit_exact_all_ranks": all(bool(s[0].item()) for s in share),
                              "scaling": "strong (the same mixed batch whatever the GPU count)",
                              "sizes": sorted({f"{mdg[n]['width']}x{mdg[n]['height']}" for n in names}),
                              "note": "end to end (host buffers in and out), the whole job's pixels / slowest rank's wall time"}
        host_out.close()
        cf.free()
        ctx.trim()
        if rank == 0 and not args.no_cpu_baseline:
            # BASELINE config 5 asks for it "vs the reference CPU decoder on all host cores": the whole decoder, .webp bytes to pixels
            out["mixed_batch"]["cpu_baseline_whole"] = cpu_arm([str(mixed_dir / n) for n in sorted(mdg)], "yuvf", 4.0, whole=True)

    # ---- SURVEY 8(f) row 4: the encoder's in-loop reconstruction (whole-macroblock mode search), 1080p pictures per launch
    enc_gold = ROOT / "tests" / "golden" / "enc.json"
    if enc_gold.exists():
        sys.path.insert(0, str(ROOT / "tests"))
        from encfix import digest as enc_digest, picture as enc_picture
        from webp_decoder_b200 import enc as E
        gd = json.loads(enc_gold.read_text())
        base = [enc_picture(900, 1920, 1080, 0), enc_picture(901, 1920, 1080, 1)]
        keys = ["900_1920x1080_k0_q75_s1", "901_1920x1080_k1_q75_s1"]
        n_pic = args.enc_batch
        # every picture its own copy in pinned memory, results into pinned memory: the copies are asynchronous DMA
        pin_in = W.PinnedBuffer(n_pic * 3110400)
        pics = []
        for i in range(n_pic):
            yb, ub, vb = base[i % 2]
            o = i * 3110400
            y = pin_in.array[o:o + 2073600].reshape(1080, 1920)
            u = pin_in.array[o + 2073600:o + 2592000].reshape(540, 960)
            v = pin_in.array[o + 2592000:o + 3110400].reshape(540, 960)
            y[:], u[:], v[:] = yb, ub, vb
            pics.append((y, u, v))
        pin_out = W.PinnedBuffer(E.batch_out_bytes(pics))
        E.encode_batch(pics, 75, 1, device=local, out_buffer=pin_out.array)
        sync_all()
        t0 = time.perf_counter()
        outs, qi = E.encode_batch(pics, 75, 1, device=local, out_buffer=pin_out.array)
        sync_all()
        wall = job_max((time.perf_counter() - t0) * 1e3)
        k_ms = job_max(E.last_kernel_ms())
        ok = all(enc_digest(o["coeffs"], o["y_modes"], o["uv_modes"]) == gd[keys[i % 2]]["digest"] and qi == gd[keys[i % 2]]["qindex"]
                 for i, o in enumerate(outs))
        px = n_pic * 1920 * 1080
        out["encoder_inloop_i16"] = {"value": world * px / (k_ms / 1e3) / 1e6, "unit": "Mpixel/s", "kernel_ms": k_ms, "pictures_per_gpu": n_pic,
                                     "e2e": {"value": world * px / (wall / 1e3) / 1e6, "unit": "Mpixel/s", "ms_per_step": wall,
                                             "h2d_bytes_per_step": n_pic * 3110400, "d2h_bytes_per_step": n_pic * 8160 * 802,
                                             "note": "pinned planes in, coefficients and modes out into pinned memory (vp8_gpu_enc_i16_inloop)"},
                                     "bit_exact_all_pictures_vs_reference_digests": ok,
                                     "note": "enc_vp8_encode_i16x16_uv_sad_inloop (reference enc_recon.c:1189-1483) for 1920x1080 noise / gradient "
                                             "pictures, quality 75: mode search + forward transforms + quantisation + reconstruction, one kernel"}
        del outs
        # the 4x4 sub-block front end (--mode bpred) on the same pictures
        bkeys = ["900_1920x1080_k0_q75_s2", "901_1920x1080_k1_q75_s2"]
        pin_out2 = W.PinnedBuffer(E.batch_out_bytes(pics, bpred=True))
        E.encode_batch(pics, 75, "bpred", device=local, out_buffer=pin_out2.array)
        sync_all()
        t0 = time.perf_counter()
        outs, qi = E.encode_batch(pics, 75, "bpred", device=local, out_buffer=pin_out2.array)
        sync_all()
        wall_b = job_max((time.perf_counter() - t0) * 1e3)
        kb_ms = job_max(E.last_kernel_ms())
        ok_b = all(enc_digest(o["coeffs"], o["y_modes"], o["uv_modes"], o["b_modes"]) == gd[bkeys[i % 2]]["digest"] for i, o in enumerate(outs))
        out["encoder_inloop_bpred"] = {"value": world * px / (kb_ms / 1e3) / 1e6, "unit": "Mpixel/s", "kernel_ms": kb_ms, "pictures_per_gpu": n_pic,
                                       "e2e": {"value": world * px / (wall_b / 1e3) / 1e6, "unit": "Mpixel/s", "ms_per_step": wall_b},
                                       "bit_exact_all_pictures_vs_reference_digests": ok_b,
                                       "note": "enc_vp8_encode_bpred_uv_sad_inloop (reference enc_recon.c:1507-1831), same pictures"}
        del outs
        pin_out2.close()
        pin_in.close()
        pin_out.close()
        if rank == 0 and not args.no_cpu_baseline:
            r = subprocess.run([sys.executable, str(ROOT / "oracle" / "cpu_baseline.py"), "--encoder-bpred", "--seconds", "3"], capture_output=True, text=True)
            try:
                out["encoder_inloop_bpred"]["cpu_baseline"] = json.loads(r.stdout.strip().splitlines()[-1])
            except Exception:
                out["encoder_inloop_bpred"]["cpu_baseline"] = {"unavailable": (r.stderr or r.stdout)[-200:]}
        if rank == 0 and not args.no_cpu_baseline:
            r = subprocess.run([sys.executable, str(ROOT / "oracle" / "cpu_baseline.py"), "--encoder", "--seconds", "4"], capture_output=True, text=True)
            try:
                out["encoder_inloop_i16"]["cpu_baseline"] = json.loads(r.stdout.strip().splitlines()[-1])
            except Exception:
                out["encoder_inloop_i16"]["cpu_baseline"] = {"unavailable": (r.stderr or r.stdout)[-200:]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="yuvf", choices=["yuvf", "yuv", "ppm"])
    ap.add_argument("--batch", type=int, default=1024, help="frames per GPU per step")
    ap.add_argument("--kernel", type=int, default=0, help="2 = vp8_mb_pairs for every batch size, 3 = lockstep flavour for big batches (0 = library default)")
    ap.add_argument("--warps", type=int, default=0)
    ap.add_argument("--images-per-sm", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--chunk", type=int, default=0, help="frames per pipeline chunk of the end-to-end calls (0 = library default)")
    ap.add_argument("--transport", default="auto", choices=["auto", "compact", "dense"], help="how e2e (dense contract) crosses the link")
    ap.add_argument("--webp-batch", type=int, default=256, help="frames per step of the e2e_from_webp leg (parser-bound: seconds per step)")
    ap.add_argument("--mixed-copies", type=int, default=2, help="config 5: copies of the 48-file mixed set per step")
    ap.add_argument("--png-batch", type=int, default=256, help="-png leg: 1080p frames per GPU per step")
    ap.add_argument("--enc-batch", type=int, default=64, help="encoder row: 1080p pictures per GPU per launch")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--no-bind", action="store_true", help="do not bind ranks to the CPUs local to their GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (rank 0) as .npy files to DIR")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not (args.impl == "b200" and args.gpus > 1 and world == 1):  # (the relaunching parent just passes its children's output on)
        claim_stdout()
    if args.impl == "reference":
        return reference_arm(args)
    if args.gpus > 1 and world == 1:
        # convenience: relaunch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", "29517", str(Path(__file__).resolve())] + sys.argv[1:]
        return subprocess.call(cmd)
    return gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
