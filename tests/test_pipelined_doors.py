"""Output layout of the pipelined calls (vp8_gpu_decode_i420 / _ppm / _png, _compact, _webp, _webp_rgba). A call whose frames
differ by 2x or more in pixel count lays its slots out biggest first (stable by pixel count), back to back and 256-byte
aligned, and reports offsets[i] / sizes[i] for the caller's frame i; within 2x the caller's order stays. The call's *_bytes is
exactly what it used. Compressed -png files lie back to back in the same order."""
import hashlib
import json
import struct
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
MIXED = ROOT / "bench_data" / "mixed"
DIGESTS = json.loads((MIXED / "digests.json").read_text())
PPM_ARG = {"i420": False, "ppm": True, "png": "png"}


def ppm_header(w, h):
    return f"P6\n{w} {h}\n255\n".encode()


def pam_header(w, h):
    return f"P7\nWIDTH {w}\nHEIGHT {h}\nDEPTH 4\nMAXVAL 255\nTUPLTYPE RGB_ALPHA\nENDHDR\n".encode()


def file_bytes(fmt, w, h):
    if fmt == "i420":
        return w * h + 2 * ((w + 1) // 2) * ((h + 1) // 2)
    if fmt == "ppm":
        return len(ppm_header(w, h)) + 3 * w * h
    if fmt == "pam":
        return len(pam_header(w, h)) + 4 * w * h
    raw = (3 * w + 1) * h  # stored -png: signature, IHDR, one IDAT of stored blocks, IEND
    return 57 + 2 + raw + 5 * ((raw + 65534) // 65535) + 4


def align(v):
    return (v + 255) // 256 * 256


def geometry(name):
    return DIGESTS[name]["width"], DIGESTS[name]["height"]


def processing_order(names):
    px = [w * h for w, h in map(geometry, names)]
    if max(px) < 2 * min(px):
        return list(range(len(names)))
    return sorted(range(len(names)), key=lambda i: -px[i])  # stable


def check_layout(names, fmt, out, offs, sizes, need, packed=False):
    """Slots in processing order, back to back from 0, each file where offsets / sizes say and of the caller's frame."""
    order = processing_order(names)
    assert sorted(range(len(names)), key=lambda i: int(offs[i])) == order
    end = 0
    for i in order:
        w, h = geometry(names[i])
        o, s = int(offs[i]), int(sizes[i])
        f = out[o:o + s]
        if packed:
            assert o == end, (names[i], o, end)
        else:
            assert s == file_bytes(fmt, w, h), names[i]
            assert o // 256 * 256 == align(end), (names[i], o, end)  # the slot right behind the one before
        end = o + s
        if fmt == "i420":
            assert hashlib.sha256(f).hexdigest() == DIGESTS[names[i]]["yuvf"], names[i]
        elif fmt == "ppm":
            assert hashlib.sha256(f).hexdigest() == DIGESTS[names[i]]["ppm"], names[i]
        elif fmt == "pam":
            hl = len(pam_header(w, h))
            assert f[:hl].tobytes() == pam_header(w, h), names[i]
            px = f[hl:].reshape(-1, 4)
            assert (px[:, 3] == 255).all(), names[i]
            rgb = ppm_header(w, h) + px[:, :3].tobytes()
            assert hashlib.sha256(rgb).hexdigest() == DIGESTS[names[i]]["ppm"], names[i]
        else:
            assert f[:8].tobytes() == b"\x89PNG\r\n\x1a\n" and struct.unpack(">II", f[16:24].tobytes()) == (w, h), names[i]
    if not packed:
        assert align(end) == need  # *_bytes is what the call used


@pytest.fixture(scope="module")
def mixed(lib):
    """bench_data/mixed (129x129 .. 3840x2160) shuffled with a fixed seed, as dense frames, compact frames and .webp bytes."""
    from webp_decoder_b200 import parse as P
    names = sorted(DIGESTS)
    names = [names[k] for k in np.random.default_rng(20261022).permutation(len(names))]
    datas = [(MIXED / n).read_bytes() for n in names]
    pf = P.parse_batch(datas, pinned=True)
    cf = P.parse_batch_compact(datas, pinned=True)
    yield names, datas, pf, cf, lib.WebpFiles(datas)
    cf.free()
    pf.free()


def call(lib, ctx, door, fmt, kfs, frs, cfs, wf, chunk):
    """One pipelined call into a buffer of exactly its *_bytes: (buffer, offsets, sizes, bytes)."""
    if door == "rgba":
        need = ctx.decode_webp_rgba_bytes(wf)
    elif door == "webp":
        need = ctx.decode_webp_bytes(wf, ppm=PPM_ARG[fmt])
    else:
        need = ctx.decode_bytes(kfs, ppm=PPM_ARG[fmt])
    assert need > 0
    out = lib.PinnedBuffer(need)
    out.array[:] = 0x5A
    if door == "dense":
        offs, sizes = ctx.decode_into(kfs, frs, out.array, filtered=True, ppm=PPM_ARG[fmt], chunk=chunk)
    elif door == "compact":
        offs, sizes = ctx.decode_compact_into(cfs, out.array, filtered=True, ppm=PPM_ARG[fmt], chunk=chunk)
    elif door == "webp":
        offs, sizes = ctx.decode_webp_into(wf, out.array, filtered=True, ppm=PPM_ARG[fmt], chunk=chunk)
    else:
        offs, sizes = ctx.decode_webp_rgba_into(wf, out.array, chunk=chunk)
    return out, offs, sizes, need


DOORS = [("dense", "i420"), ("dense", "ppm"), ("dense", "png"), ("compact", "i420"), ("compact", "ppm"), ("compact", "png"),
         ("webp", "i420"), ("webp", "ppm"), ("webp", "png"), ("rgba", "pam")]


@pytest.mark.parametrize("door,fmt", DOORS)
def test_mixed_sizes_biggest_first(lib, gpu_ctx, mixed, door, fmt):
    names, _, pf, cf, wf = mixed
    out, offs, sizes, need = call(lib, gpu_ctx, door, fmt, pf.kf_list(), pf.frame_list(), cf.frame_list(), wf, chunk=7)
    try:
        check_layout(names, fmt, out.array, offs, sizes, need)
    finally:
        out.close()
        gpu_ctx.trim()


@pytest.mark.parametrize("door", ["dense", "webp"])
def test_mixed_sizes_deflate_png_back_to_back(lib, gpu_ctx, mixed, door):
    """Compressed -png: the files back to back from 0 in processing order, each no longer than its stored file."""
    names, _, pf, cf, wf = mixed
    try:
        gpu_ctx.set_png_deflate(True)
        out, offs, sizes, need = call(lib, gpu_ctx, door, "png", pf.kf_list(), pf.frame_list(), cf.frame_list(), wf, chunk=7)
    finally:
        gpu_ctx.set_png_deflate(False)
    try:
        check_layout(names, "png", out.array, offs, sizes, need, packed=True)
        assert all(int(s) <= file_bytes("png", *geometry(n)) for n, s in zip(names, sizes))
    finally:
        out.close()
        gpu_ctx.trim()


@pytest.mark.parametrize("door,fmt", [("dense", "ppm"), ("compact", "i420"), ("webp", "i420"), ("rgba", "pam")])
def test_sizes_within_2x_keep_the_callers_order(lib, gpu_ctx, mixed, door, fmt):
    """1920x1080 and 2560x1440 frames (1.8x apart), shuffled: slots in the caller's order."""
    names, _, pf, cf, wf = mixed
    keep = [i for i, n in enumerate(names) if geometry(n) in ((1920, 1080), (2560, 1440))]
    sub = [names[i] for i in keep]
    assert len({geometry(n) for n in sub}) == 2 and processing_order(sub) == list(range(len(sub)))
    kfs, frs, cfs = pf.kf_list(), pf.frame_list(), cf.frame_list()
    sub_wf = lib.WebpFiles([mixed[1][i] for i in keep])
    out, offs, sizes, need = call(lib, gpu_ctx, door, fmt, [kfs[i] for i in keep], [frs[i] for i in keep], [cfs[i] for i in keep],
                                  sub_wf, chunk=3)
    try:
        assert list(offs) == sorted(int(o) for o in offs)
        check_layout(sub, fmt, out.array, offs, sizes, need)
    finally:
        out.close()
        gpu_ctx.trim()
