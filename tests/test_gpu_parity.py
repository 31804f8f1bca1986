"""Parity tests proper: the CUDA path, called through the C-ABI of libvp8gpu.so, against
   (1) digests of the unmodified reference decoder's -yuv/-yuvf/-ppm/-png bytes (tests/golden, bench_data),
   (2) the CPU oracle on seeded fuzz frames, and (3) size-independent properties at the benchmark sizes.
Bit-exact is the bar: every comparison is equality of bytes."""
import ctypes as C
import errno
import json

import numpy as np
import pytest

from vp8fix import GOLDEN, ROOT, fuzz_frame, sha

pytestmark = pytest.mark.gpu


def _slices(buf, offs, sizes):
    return [buf[int(o):int(o) + int(s)] for o, s in zip(offs, sizes)]


def test_golden_webp_batch_yuv_yuvf_ppm(gpu_ctx, golden, parsed_golden):
    """All 254 golden inputs (1x1 .. 960x1162, segmentation, i16/B_PRED mixes) as ONE mixed-size batch."""
    names = sorted(golden)
    kfs = [parsed_golden[n][0] for n in names]
    frs = [parsed_golden[n][1] for n in names]
    for filtered, key in ((False, "yuv"), (True, "yuvf")):
        outs = gpu_ctx.decode_i420(kfs, frs, filtered=filtered)
        bad = [n for n, o in zip(names, outs) if sha(o) != golden[n][key]]
        assert not bad, f"-{key}: {len(bad)} differ, e.g. {bad[:5]}"
    ppms = gpu_ctx.decode_ppm(kfs, frs)
    bad = [n for n, p in zip(names, ppms) if sha(p) != golden[n]["ppm"]]
    assert not bad, f"-ppm: {len(bad)} differ, e.g. {bad[:5]}"
    # the reference's dwebp-derived golden PNG pixels (libwebp itself)
    for n, p in zip(names, ppms):
        if "dwebp_rgb" in golden[n]:
            w, h = golden[n]["width"], golden[n]["height"]
            assert sha(p[len(p) - w * h * 3:]) == golden[n]["dwebp_rgb"], n


def test_reference_fuzz_digests(gpu_ctx):
    """120 struct-level fuzz frames whose digests came from the real reference hot path: simple filter,
    sharpness, lf deltas, absolute segment levels, int16 wrap of dequant/IDCT."""
    fz = json.loads((GOLDEN / "fuzz.json").read_text())
    seeds = sorted(fz, key=int)
    frames = [fuzz_frame(int(s), fz[s]["width"], fz[s]["height"], **fz[s]["kw"]) for s in seeds]
    kfs, ds = [f.header() for f in frames], [f.cstruct() for f in frames]
    for filtered, key in ((False, "yuv"), (True, "yuvf")):
        outs = gpu_ctx.decode_i420(kfs, ds, filtered=filtered)
        bad = [s for s, o in zip(seeds, outs) if sha(o) != fz[s][key]]
        assert not bad, f"{key}: seeds {bad[:8]}"
    ppms = gpu_ctx.decode_ppm(kfs, ds)
    assert not [s for s, p in zip(seeds, ppms) if sha(p) != fz[s]["ppm"]]


DEFAULT_KERNEL = 3  # what a fresh context runs (vp8_gpu.h: vp8_gpu_set_kernel)


@pytest.mark.parametrize("kernel,warps", [(2, 4), (2, 8), (2, 16), (3, 4), (3, 8), (3, 16)])
def test_fuzz_vs_oracle_all_kernels_and_warp_shapes(gpu_ctx, oracle, kernel, warps):
    """Both schedules of the wavefront kernel (warps spinning on progress stamps / warps of a CTA meeting at a barrier) in
    every CTA shape."""
    gpu_ctx.set_kernel(kernel)
    gpu_ctx.set_tuning(warps, 0)
    try:
        frames = []
        for s in range(48):
            rng = np.random.default_rng(s * 31 + warps)
            frames.append(fuzz_frame(9000 + s + 100 * warps, int(rng.integers(1, 400)), int(rng.integers(1, 400)),
                                     amp=[5, 40, 400, 2500][s % 4], density=[0.02, 0.2, 0.7][s % 3], raw=bool(s & 1)))
        kfs, ds = [f.header() for f in frames], [f.cstruct() for f in frames]
        for filtered in (False, True):
            outs = gpu_ctx.decode_i420(kfs, ds, filtered=filtered)
            for f, o in zip(frames, outs):
                assert np.array_equal(o, oracle.decode_i420(f, filtered)), (f.width, f.height, filtered)
    finally:
        gpu_ctx.set_tuning(0, 0)
        gpu_ctx.set_kernel(DEFAULT_KERNEL)


def test_edge_geometries(gpu_ctx, oracle):
    """1-pixel frames, single rows/columns of macroblocks, widths that break 4-byte store alignment."""
    dims = [(1, 1), (1, 40), (40, 1), (2, 2), (15, 15), (16, 16), (17, 17), (33, 16), (16, 33), (129, 129), (131, 67),
            (1000, 24), (24, 1000), (258, 30), (255, 255)]
    frames = [fuzz_frame(70 + i, w, h, density=0.3) for i, (w, h) in enumerate(dims)]
    kfs, ds = [f.header() for f in frames], [f.cstruct() for f in frames]
    for filtered in (False, True):
        for f, o in zip(frames, gpu_ctx.decode_i420(kfs, ds, filtered=filtered)):
            assert np.array_equal(o, oracle.decode_i420(f, filtered)), (f.width, f.height, filtered)
    for f, p in zip(frames, gpu_ctx.decode_ppm(kfs, ds)):
        yuvf = oracle.decode_i420(f, True)
        assert p == oracle.ppm(oracle.rgb(yuvf, f.width, f.height), f.width, f.height), (f.width, f.height)


@pytest.mark.parametrize("kernel", [2, 3])
def test_maximum_frame_dimensions(gpu_ctx, oracle, kernel):
    """VP8 dimensions are 14-bit (vp8_header.c:46-49): the widest (1024 macroblock columns: largest line buffers) and the
    tallest (1024 macroblock rows: longest wavefront, progress ring wrap-around) frames a bitstream can carry."""
    gpu_ctx.set_kernel(kernel)
    try:
        for w, h in ((16383, 33), (33, 16383), (4099, 257)):
            f = fuzz_frame(w + h, w, h, density=0.05, lf_level=24, lf_use_simple=0)
            for filtered in (False, True):
                got = gpu_ctx.decode_i420([f.header()], [f.cstruct()], filtered=filtered)[0]
                assert np.array_equal(got, oracle.decode_i420(f, filtered)), (w, h, filtered)
        f = fuzz_frame(77, 16383, 17, density=0.05)
        assert gpu_ctx.decode_ppm([f.header()], [f.cstruct()])[0] == oracle.ppm(oracle.rgb(oracle.decode_i420(f, True), 16383, 17), 16383, 17)
    finally:
        gpu_ctx.set_kernel(DEFAULT_KERNEL)


@pytest.mark.parametrize("per_cta", [2, 5, 7])
def test_lockstep_flavour_several_images_per_cta(gpu_ctx, oracle, per_cta):
    """Kernel 3, lockstep flavour: one CTA carries several images (4 warps each) and all its warps meet at a barrier once
    per macroblock step. Mixed sizes in one CTA, frames with a single row pair (three of the four warps never get work),
    frames taller than the progress ring (64 rows), more images than slots (every group takes several in turn), the
    stand-alone loop filter through the same schedule."""
    dims = [(64, 48), (129, 129), (300, 90), (17, 33), (48, 200), (1, 1), (33, 1100), (500, 16), (16, 16), (250, 250)]
    frames = [fuzz_frame(1200 + s, *dims[s % len(dims)], density=[0.3, 0.02, 0.9, 0.0][s % 4], amp=[40, 400, 2500][s % 3], raw=bool(s & 1))
              for s in range(43)]
    kfs, ds = [f.header() for f in frames], [f.cstruct() for f in frames]
    gpu_ctx.set_kernel(3)
    gpu_ctx.set_tuning(4, per_cta)
    try:
        for filtered in (False, True):
            outs = gpu_ctx.decode_i420(kfs, ds, filtered=filtered)
            assert gpu_ctx.last_launch_config()["images_per_cta"] == per_cta
            bad = [i for i, (f, o) in enumerate(zip(frames, outs)) if not np.array_equal(o, oracle.decode_i420(f, filtered))]
            assert not bad, (per_cta, filtered, bad)
        # staged: m06 into padded planes, m07 in place, both through the lockstep schedule
        b = gpu_ctx.recon(kfs[:12], ds[:12])
        gpu_ctx.filter(b)
        assert gpu_ctx.last_launch_config()["images_per_cta"] == per_cta
        for i in range(12):
            oy, ou, ov = oracle.recon_padded(frames[i])
            oracle.loopfilter_padded(frames[i], oy, ou, ov)
            y, u, v = gpu_ctx.download_padded(b, i)
            assert np.array_equal(y, oy) and np.array_equal(u, ou) and np.array_equal(v, ov), i
        b.free()
    finally:
        gpu_ctx.set_tuning(0, 0)
        gpu_ctx.set_kernel(DEFAULT_KERNEL)


def test_lockstep_is_what_big_batches_run_by_default(gpu_ctx, oracle):
    """No tuning: a batch of several images per SM takes the lockstep flavour on its own; very wide frames get fewer
    images per CTA (their line buffers fill the shared memory sooner)."""
    frames = [fuzz_frame(3000 + s, 32 + 16 * (s % 3), 32 + 16 * (s % 2), density=0.2) for s in range(720)]
    outs = gpu_ctx.decode_i420([f.header() for f in frames], [f.cstruct() for f in frames], filtered=True)
    cfg = gpu_ctx.last_launch_config()
    assert cfg["images_per_cta"] >= 2 and cfg["warps_per_image"] == 4, cfg
    bad = [i for i, (f, o) in enumerate(zip(frames, outs)) if not np.array_equal(o, oracle.decode_i420(f, True))]
    assert not bad, bad[:8]
    wide = [fuzz_frame(3900 + s, 16383, 17, density=0.05) for s in range(6)]
    gpu_ctx.set_tuning(4, 7)
    try:
        outs = gpu_ctx.decode_i420([f.header() for f in wide], [f.cstruct() for f in wide], filtered=True)
        cfg = gpu_ctx.last_launch_config()
        assert 2 <= cfg["images_per_cta"] < 7, cfg
        assert all(np.array_equal(o, oracle.decode_i420(f, True)) for f, o in zip(wide, outs))
    finally:
        gpu_ctx.set_tuning(0, 0)


def test_batch_of_more_than_a_wave_is_cut_into_segments(gpu_ctx, oracle):
    """148 SMs x 7 images is one lockstep wave; 1100 images = one full wave + 64 images that get their own launch shape."""
    frames = [fuzz_frame(5000 + s, 32 + 16 * (s % 2), 32 + 16 * (s % 3), density=0.15) for s in range(1100)]
    outs = gpu_ctx.decode_i420([f.header() for f in frames], [f.cstruct() for f in frames], filtered=True)
    cfg = gpu_ctx.last_launch_config()
    sms = cfg["grid"]  # one CTA per SM in the first segment
    assert cfg["images_per_cta"] == 7 and (cfg["segments"] == 2 or sms * 7 >= 1100), cfg
    bad = [i for i, (f, o) in enumerate(zip(frames, outs)) if not np.array_equal(o, oracle.decode_i420(f, True))]
    assert not bad, bad[:8]


@pytest.mark.parametrize("ctas,split", [(1, False), (2, False), (4, False), (8, False), (4, True), (8, True)])
def test_cluster_mode_one_image_over_several_ctas(gpu_ctx, oracle, ctas, split):
    """Few big frames: each image is decoded by a thread-block cluster (row pairs dealt to the warps of 2/4/8 co-scheduled
    CTAs, line buffers and progress stamps exchanged through L2). split: the fused mode on 4 / 8 CTAs runs vp8_mb_split (a
    reconstruction warp and a filter warp per row pair). Same bytes as the single-CTA path and the oracle."""
    gpu_ctx.set_cluster(ctas, split)
    try:
        frames = [fuzz_frame(600 + s, 400 + 64 * s, 1100 + 200 * s, density=0.15, lf_level=20 + s, lf_use_simple=0) for s in range(3)]
        # 250 macroblock rows, 4 columns: the only frame that gives rows to CTAs 4..8; pinned so that it really filters
        frames.append(fuzz_frame(610, 64, 4000, density=0.2, lf_level=40, lf_delta_enabled=0, lf_use_simple=0))
        frames.append(fuzz_frame(611, 2500, 600, density=0.1, lf_use_simple=1, lf_level=33))
        kfs, ds = [f.header() for f in frames], [f.cstruct() for f in frames]
        for filtered in (False, True):
            outs = gpu_ctx.decode_i420(kfs, ds, filtered=filtered)
            for f, o in zip(frames, outs):
                assert np.array_equal(o, oracle.decode_i420(f, filtered)), (ctas, f.width, f.height, filtered)
        cfg = gpu_ctx.last_launch_config()
        assert cfg["ctas_per_image"] == ctas and cfg["grid"] == len(frames) * ctas and cfg["split"] == split, cfg
        # stand-alone loop filter (stage API) through the cluster path as well
        b = gpu_ctx.recon(kfs[:2], ds[:2])
        gpu_ctx.filter(b)
        for i in range(2):
            y, u, v = oracle.recon_padded(frames[i])
            oracle.loopfilter_padded(frames[i], y, u, v)
            for got, want in zip(gpu_ctx.download_padded(b, i), (y, u, v)):
                assert np.array_equal(got, want)
        b.free()
    finally:
        gpu_ctx.set_cluster(0, True)


def test_all_zero_and_saturated_inputs(gpu_ctx, oracle):
    a = fuzz_frame(1, 96, 80, density=0.0)                          # prediction only, every IDCT short-circuits
    b = fuzz_frame(2, 96, 80, density=1.0, amp=2047, q_index=127)   # every coefficient set, maximal quantiser
    c = fuzz_frame(3, 96, 80, density=1.0, amp=32767)               # beyond any bitstream: pure int16 wrap behaviour
    for f in (a, b, c):
        for filtered in (False, True):
            got = gpu_ctx.decode_i420([f.header()], [f.cstruct()], filtered=filtered)[0]
            assert np.array_equal(got, oracle.decode_i420(f, filtered))


def test_has_coeff_may_be_null(gpu_ctx, oracle):
    f = fuzz_frame(11, 120, 90, lf_level=30, lf_use_simple=0)
    got = gpu_ctx.decode_i420([f.header()], [f.cstruct(drop_has_coeff=True)], filtered=True)[0]
    assert np.array_equal(got, oracle.decode_i420(f, True, drop_has_coeff=True))


def test_staged_entry_points_recon_filter_rgb(gpu_ctx, oracle):
    """vp8_gpu_recon -> vp8_gpu_filter -> vp8_gpu_rgb on macroblock-aligned planes, checked after every stage."""
    frames = [fuzz_frame(300 + s, 40 + 23 * s, 200 - 17 * s, density=0.25) for s in range(8)]
    b = gpu_ctx.recon([f.header() for f in frames], [f.cstruct() for f in frames])
    want = [oracle.recon_padded(f) for f in frames]
    for i, f in enumerate(frames):
        for got, w in zip(gpu_ctx.download_padded(b, i), want[i]):
            assert np.array_equal(got, w), ("recon", i)
    gpu_ctx.filter(b)
    for i, f in enumerate(frames):
        oracle.loopfilter_padded(f, *want[i])
        for got, w in zip(gpu_ctx.download_padded(b, i), want[i]):
            assert np.array_equal(got, w), ("filter", i)
    with pytest.raises(OSError):  # filtering twice is a caller error
        gpu_ctx.filter(b)
    gpu_ctx.rgb(b)
    buf, offs, sizes = gpu_ctx.download_ppm(b)
    for f, p in zip(frames, _slices(buf, offs, sizes)):
        yuvf = oracle.decode_i420(f, True)
        assert p.tobytes() == oracle.ppm(oracle.rgb(yuvf, f.width, f.height), f.width, f.height)
    b.free()


def test_reference_module_interfaces(lib, gpu_ctx, oracle):
    """The seven symbols main.c binds, used the way main.c uses them (main.c:591,665,742,758,811,827)."""
    f = fuzz_frame(21, 150, 70, density=0.3, lf_level=25, lf_use_simple=0)
    kf, d = f.header(), f.cstruct()
    yuv = lib.vp8_reconstruct_keyframe_yuv(kf, d)
    yuvf = lib.vp8_reconstruct_keyframe_yuv_filtered(kf, d)
    assert np.array_equal(yuv, oracle.decode_i420(f, False))
    assert np.array_equal(yuvf, oracle.decode_i420(f, True))
    rgb = oracle.rgb(yuvf, f.width, f.height)
    assert lib.yuv420_write_ppm(yuvf, f.width, f.height) == oracle.ppm(rgb, f.width, f.height)
    assert lib.yuv420_write_png(yuvf, f.width, f.height) == oracle.png(rgb, f.width, f.height)
    # in-place loop filter on a host image with padded dims (vp8_loopfilter.h:10-14)
    y, u, v = oracle.recon_padded(f)
    wy, wu, wv = y.copy(), u.copy(), v.copy()
    oracle.loopfilter_padded(f, wy, wu, wv)
    lib.vp8_loopfilter_apply_keyframe(y, u, v, d)
    assert np.array_equal(y, wy) and np.array_equal(u, wu) and np.array_equal(v, wv)
    # dims that are not the macroblock grid are rejected like the reference does (vp8_loopfilter.c:206-209)
    with pytest.raises(OSError) as e:
        lib.vp8_loopfilter_apply_keyframe(y[:-16], u[:-8], v[:-8], d)
    assert e.value.errno == errno.EINVAL


def test_simple_filter_and_level_zero_paths(gpu_ctx, oracle):
    frames = [fuzz_frame(400, 100, 60, lf_use_simple=1, lf_level=40, segmentation_enabled=0, lf_delta_enabled=0),
              fuzz_frame(401, 100, 60, lf_use_simple=1),
              fuzz_frame(402, 100, 60, lf_level=0, segmentation_enabled=0, lf_delta_enabled=0),          # no filtering at all
              fuzz_frame(403, 100, 60, lf_level=0, segmentation_enabled=1, segmentation_abs=0,
                         seg_lf_level=[0, 20, 0, 63], lf_delta_enabled=0)]                                # level 0 in some segments only
    outs = gpu_ctx.decode_i420([f.header() for f in frames], [f.cstruct() for f in frames], filtered=True)
    for f, o in zip(frames, outs):
        assert np.array_equal(o, oracle.decode_i420(f, True))


def test_pinned_and_pageable_inputs_agree(lib, gpu_ctx, golden):
    from webp_decoder_b200 import parse as P
    names = [n for n in sorted(golden) if golden[n]["width"] >= 100][:24]
    datas = [(GOLDEN / "webp" / n).read_bytes() for n in names]
    h2d0 = gpu_ctx.h2d_bytes
    for pinned in (False, True):
        pf = P.parse_batch(datas, pinned=pinned)
        outs = gpu_ctx.decode_i420(pf.kf_list(), pf.frame_list(), filtered=True)
        assert [sha(o) for o in outs] == [golden[n]["yuvf"] for n in names], pinned
        pf.free()
    assert gpu_ctx.h2d_bytes > h2d0


def test_bench_inputs_full_size_parity_and_replication(lib, gpu_ctx):
    """BASELINE.json sizes: 1080p / 512x512 / 4K inputs against the reference decoder's digests, then the
    size-independent properties a big batch offers: replicas of one frame decode identically wherever they sit
    in the batch, and a batch result equals the frame-at-a-time result."""
    from webp_decoder_b200 import parse as P
    dg = json.loads((ROOT / "bench_data" / "digests.json").read_text())
    names = sorted(dg)
    pf = P.parse_batch([(ROOT / "bench_data" / n).read_bytes() for n in names], pinned=True)
    kfs, frs = pf.kf_list(), pf.frame_list()
    for filtered, key in ((False, "yuv"), (True, "yuvf")):
        outs = gpu_ctx.decode_i420(kfs, frs, filtered=filtered)
        assert [sha(o) for o in outs] == [dg[n][key] for n in names], key
    ppms = gpu_ctx.decode_ppm(kfs, frs)
    assert [sha(p) for p in ppms] == [dg[n]["ppm"] for n in names]
    # 96 replicas of the four 1080p frames, interleaved
    idx = [i for i, n in enumerate(names) if "1920x1080" in n]
    order = [idx[k % len(idx)] for k in range(96)]
    outs = gpu_ctx.decode_i420([kfs[i] for i in order], [frs[i] for i in order], filtered=True)
    for k, o in zip(order, outs):
        assert sha(o) == dg[names[k]]["yuvf"]
    single = gpu_ctx.decode_i420([kfs[idx[0]]], [frs[idx[0]]], filtered=True)[0]
    assert sha(single) == dg[names[idx[0]]]["yuvf"]
    pf.free()


def test_pipelined_decode_matches_digests(lib, gpu_ctx, golden, parsed_golden):
    """vp8_gpu_decode_i420 / _ppm: chunks overlapped on internal streams; many small chunks, pinned and pageable output."""
    names = sorted(golden)
    kfs = [parsed_golden[n][0] for n in names]
    frs = [parsed_golden[n][1] for n in names]
    try:
        for compact in (True, False, "auto"):  # zero blocks dropped on the host / arrays as they are / chosen per chunk
            gpu_ctx.set_transport(compact, 3)
            h2d0 = gpu_ctx.h2d_bytes
            for ppm, key, filtered in ((False, "yuvf", True), (False, "yuv", False), (True, "ppm", True)):
                need = gpu_ctx.decode_bytes(kfs, ppm=ppm)
                pinned = lib.PinnedBuffer(need)
                for out in (pinned.array, np.empty(need, np.uint8)):
                    out[:] = 0xAA
                    offs, sizes = gpu_ctx.decode_into(kfs, frs, out, filtered=filtered, ppm=ppm, chunk=7)
                    bad = [n for n, o, s in zip(names, offs, sizes) if sha(out[int(o):int(o) + int(s)]) != golden[n][key]]
                    assert not bad, (compact, key, len(bad), bad[:4])
                pinned.close()
            moved = gpu_ctx.h2d_bytes - h2d0
            t = gpu_ctx.last_transport()
            if compact is True:
                compact_bytes = moved
                assert t["dense_chunks"] == 0 and t["compact_chunks"] > 0
            elif compact is False:
                assert compact_bytes < 0.6 * moved, (compact_bytes, moved)  # the corpus is mostly sparse
                assert t["compact_chunks"] == 0 and t["dense_chunks"] > 0
            else:
                assert t["compact_chunks"] + t["dense_chunks"] > 0
    finally:
        gpu_ctx.set_transport("auto", 0)
    with pytest.raises(OSError):
        gpu_ctx.decode_into(kfs, frs, np.empty(10, np.uint8))


@pytest.mark.parametrize("storage", ["pinned", "pageable", "separate"])
def test_compact_frames_pipelined_decode(lib, gpu_ctx, golden, storage):
    """vp8_gpu_decode_compact: frames the parser emitted in the compact wire format (no dense arrays anywhere, nothing
    re-scanned on the host). pinned: one contiguous pinned buffer, read by the copy engine in runs; pageable: the same
    layout in pageable memory, gathered through staging; separate: one allocation per frame."""
    from webp_decoder_b200 import parse as P
    names = sorted(golden)
    datas = [(GOLDEN / "webp" / n).read_bytes() for n in names]
    cf = P.parse_batch_compact(datas, threads=4, pinned=(storage == "pinned"), contiguous=(storage != "separate"))
    frs = cf.frame_list()
    kfs = [cf.kfs[i] for i in range(cf.n)]
    h2d0 = gpu_ctx.h2d_bytes
    for ppm, key, filtered in ((False, "yuvf", True), (False, "yuv", False), (True, "ppm", True)):
        need = gpu_ctx.decode_bytes(kfs, ppm=ppm)
        out = lib.PinnedBuffer(need)
        for chunk in (9, 0):
            out.array[:] = 0x55
            offs, sizes = gpu_ctx.decode_compact_into(frs, out.array, filtered=filtered, ppm=ppm, chunk=chunk)
            bad = [n for n, o, s in zip(names, offs, sizes) if sha(out.array[int(o):int(o) + int(s)]) != golden[n][key]]
            assert not bad, (storage, key, chunk, len(bad), bad[:4])
        out.close()
    assert gpu_ctx.h2d_bytes > h2d0
    # a frame that is not standalone / inconsistent is refused
    broken = P.CompactFrame.from_buffer_copy(frs[0])
    broken.bytes += 32
    with pytest.raises(OSError):
        gpu_ctx.decode_compact_into([broken], np.empty(1 << 20, np.uint8))
    cf.free()


def test_png_framed_on_the_device(lib, gpu_ctx, golden, parsed_golden, oracle):
    """m09 on the GPU (vp8_png_frame / vp8_png_finish): the reference decoder's -png bytes, checksums included, for all 254
    golden inputs as one mixed-size batch (1x1 .. 960x1162: files of one partial span up to 51 spans), through the staged
    calls and through every pipelined door; then frame geometries around the segment / scanline / stored-block boundaries
    against the oracle's writer; then the 1080p / 4K bench inputs (95 / 380 CTAs per file)."""
    from webp_decoder_b200 import parse as P
    names = sorted(golden)
    kfs = [parsed_golden[n][0] for n in names]
    frs = [parsed_golden[n][1] for n in names]
    pngs = gpu_ctx.decode_png(kfs, frs)
    bad = [n for n, p in zip(names, pngs) if sha(p) != golden[n]["png"]]
    assert not bad, f"-png: {len(bad)} differ, e.g. {bad[:5]}"
    ms, pairs = gpu_ctx.png_time()
    assert pairs >= 1 and ms > 0
    # dense frames, pipelined
    need = gpu_ctx.decode_bytes(kfs, ppm="png")
    out = lib.PinnedBuffer(need)
    out.array[:] = 0x77
    offs, sizes = gpu_ctx.decode_into(kfs, frs, out.array, ppm="png", chunk=11)
    bad = [n for n, o, s in zip(names, offs, sizes) if sha(out.array[int(o):int(o) + int(s)]) != golden[n]["png"]]
    assert not bad, ("decode_png", len(bad), bad[:4])
    # compact frames and .webp bytes
    datas = [(GOLDEN / "webp" / n).read_bytes() for n in names]
    cf = P.parse_batch_compact(datas, threads=4, pinned=True, contiguous=True)
    for chunk in (9, 0):
        out.array[:] = 0x55
        offs, sizes = gpu_ctx.decode_compact_into(cf.frame_list(), out.array, ppm="png", chunk=chunk)
        bad = [n for n, o, s in zip(names, offs, sizes) if sha(out.array[int(o):int(o) + int(s)]) != golden[n]["png"]]
        assert not bad, ("compact", chunk, len(bad), bad[:4])
    cf.free()
    files = lib.WebpFiles(datas)
    assert gpu_ctx.decode_webp_bytes(files, ppm="png") == need
    out.array[:] = 0x33
    offs, sizes = gpu_ctx.decode_webp_into(files, out.array, ppm="png", chunk=16)
    bad = [n for n, o, s in zip(names, offs, sizes) if sha(out.array[int(o):int(o) + int(s)]) != golden[n]["png"]]
    assert not bad, ("webp", len(bad), bad[:4])
    out.close()
    # geometries: 3*w+1 around multiples of 16, scanlines longer than a stored block, a block boundary inside a filter byte
    dims = [(1, 1), (1, 40), (40, 1), (2, 2), (5, 5), (15, 15), (16, 16), (21, 13), (85, 3), (341, 64), (1365, 48), (1366, 49),
            (129, 129), (1000, 24), (24, 1000), (255, 255), (16383, 4), (7, 9000)]
    frames = [fuzz_frame(170 + i, w, h, density=0.2 if w * h < 100000 else 0.02) for i, (w, h) in enumerate(dims)]
    for f, p in zip(frames, gpu_ctx.decode_png([f.header() for f in frames], [f.cstruct() for f in frames])):
        yuvf = oracle.decode_i420(f, True)
        assert p == bytes(oracle.png(oracle.rgb(yuvf, f.width, f.height), f.width, f.height)), (f.width, f.height)
    # bench inputs, each several times in one batch
    dg = json.loads((ROOT / "bench_data" / "digests.json").read_text())
    bnames = sorted(dg)
    pf = P.parse_batch([(ROOT / "bench_data" / n).read_bytes() for n in bnames], pinned=True)
    order = [k % len(bnames) for k in range(3 * len(bnames))]
    pngs = gpu_ctx.decode_png([pf.kf_list()[k] for k in order], [pf.frame_list()[k] for k in order])
    assert [sha(p) for p in pngs] == [dg[bnames[k]]["png"] for k in order]
    pf.free()


@pytest.mark.parametrize("threads,chunk", [(1, 5), (3, 16), (0, 0)])
def test_webp_bytes_to_pixels_in_one_call(lib, gpu_ctx, golden, threads, chunk):
    """vp8_gpu_decode_webp: .webp bytes in, -yuv/-yuvf/-ppm bytes out; host threads parse chunk k straight into the pinned
    arena while the GPU works on the chunks before it. Same bytes as the reference decoder's files."""
    names = sorted(golden)
    files = lib.WebpFiles([(GOLDEN / "webp" / n).read_bytes() for n in names])
    gpu_ctx.set_transport(True, threads)
    try:
        for ppm, key, filtered in ((False, "yuvf", True), (False, "yuv", False), (True, "ppm", True)):
            need = gpu_ctx.decode_webp_bytes(files, ppm=ppm)
            out = lib.PinnedBuffer(need)
            out.array[:] = 0x33
            offs, sizes = gpu_ctx.decode_webp_into(files, out.array, filtered=filtered, ppm=ppm, chunk=chunk)
            bad = [n for n, o, s in zip(names, offs, sizes) if sha(out.array[int(o):int(o) + int(s)]) != golden[n][key]]
            assert not bad, (key, len(bad), bad[:4])
            out.close()
        prof = gpu_ctx.last_call_profile()
        assert prof["total_ms"] > 0 and prof["host_work_ms"] > 0
    finally:
        gpu_ctx.set_transport("auto", 0)
    # a broken file fails the whole call with the parser's errno
    junk = lib.WebpFiles([(GOLDEN / "webp" / names[0]).read_bytes(), b"RIFF\x04\x00\x00\x00WEBP"])
    assert gpu_ctx.decode_webp_bytes(junk) == 0
    with pytest.raises(OSError):
        gpu_ctx.decode_webp_into(junk, np.empty(1 << 20, np.uint8))


def test_host_binding_reports_local_cpus(gpu_ctx):
    """vp8_gpu_bind_host: the GPU's local CPU list from sysfs (0 = topology unreadable: nothing changed)."""
    import os
    before = os.sched_getaffinity(0)
    try:
        n = gpu_ctx.bind_host(0, 1)
        assert n >= 0
        if n:
            assert len(os.sched_getaffinity(0)) == n
    finally:
        os.sched_setaffinity(0, before)


@pytest.mark.parametrize("chunk", [1, 2, 5, 16, 1000])
def test_pipelined_chunk_schedule_and_arena_granules(gpu_ctx, oracle, chunk):
    """The pipelined call ramps its chunk sizes (chunk/4, chunk/4, chunk/2, chunk ..., short last chunk) and several
    host threads compact a chunk into one arena in 64 KiB granules: dense frames that span many granules, sparse ones
    that fit in one, odd sizes, every chunk size against the oracle."""
    frames = [fuzz_frame(900 + s, [300, 64, 129, 17, 400][s % 5], [280, 48, 129, 33, 90][s % 5],
                         density=[0.9, 0.02, 0.3, 0.0][s % 4], amp=[40, 400, 2500][s % 3], raw=bool(s & 1)) for s in range(23)]
    kfs = [f.header() for f in frames]
    frs = [f.cstruct() for f in frames]
    want = [oracle.decode_i420(f, True) for f in frames]
    try:
        for threads in (1, 4):
            gpu_ctx.set_transport(True, threads)
            out = np.full(gpu_ctx.decode_bytes(kfs), 0x55, np.uint8)
            offs, sizes = gpu_ctx.decode_into(kfs, frs, out, filtered=True, chunk=chunk)
            bad = [i for i, (o, s) in enumerate(zip(offs, sizes)) if not np.array_equal(out[int(o):int(o) + int(s)], want[i])]
            assert not bad, (chunk, threads, bad)
    finally:
        gpu_ctx.set_transport("auto", 0)


def test_dense_frames_pass_through_compact_chunks(lib, gpu_ctx, golden):
    """Compact transport of dense Vp8DecodedFrames: frames from pinned parser arenas whose blocks are mostly non-zero are not
    compacted but shipped as they are, next to compacted ones in the same chunk and the same launch."""
    from vp8fix import GOLDEN
    from webp_decoder_b200 import parse as P
    names = sorted(n for n in golden if "noise" in n and golden[n]["width"] >= 32)[:6] + sorted(n for n in golden if "noise" not in n)[:14]
    pf = P.parse_batch([(GOLDEN / "webp" / n).read_bytes() for n in names], pinned=True)
    kfs, frs = [pf.kfs[i] for i in range(pf.n)], [pf.frames[i] for i in range(pf.n)]
    try:
        gpu_ctx.set_transport(True, 3)
        for filtered, key in ((True, "yuvf"), (False, "yuv")):
            out = np.full(gpu_ctx.decode_bytes(kfs), 0x33, np.uint8)
            offs, sizes = gpu_ctx.decode_into(kfs, frs, out, filtered=filtered, chunk=8)
            bad = [n for n, o, s in zip(names, offs, sizes) if sha(out[int(o):int(o) + int(s)]) != golden[n][key]]
            assert not bad, (key, bad)
            passed = gpu_ctx.last_dense_frames()
            assert 0 < passed < len(names), passed  # some crossed dense, some compact
    finally:
        gpu_ctx.set_transport("auto", 0)
        pf.free()


def test_argument_errors(lib, gpu_ctx):
    f = fuzz_frame(5, 64, 64)
    kf, d = f.header(), f.cstruct()
    kf.width = 100  # macroblock grid no longer matches the frame size
    with pytest.raises(OSError) as e:
        gpu_ctx.decode_i420([kf], [d])
    assert e.value.errno == errno.EINVAL
    d2 = f.cstruct()
    d2.coeff_y = C.POINTER(C.c_int16)()
    with pytest.raises(OSError) as e:
        gpu_ctx.decode_i420([f.header()], [d2])
    assert e.value.errno == errno.EINVAL
    with pytest.raises(OSError):
        gpu_ctx.set_tuning(5, 0)


def test_kernels_really_launch(gpu_ctx, oracle):
    f = fuzz_frame(8, 64, 64, lf_level=20)
    n0 = gpu_ctx.launches
    gpu_ctx.decode_ppm([f.header()], [f.cstruct()])
    assert gpu_ctx.launches - n0 == 2  # fused recon+filter wavefront, RGB
    cfg = gpu_ctx.last_launch_config()
    assert cfg["warps_per_image"] in (4, 8, 16, 32) and cfg["grid"] >= 1 and cfg["smem_bytes"] > 0
