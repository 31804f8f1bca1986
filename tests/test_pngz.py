"""Compressed -png files (vp8_gpu_set_png_deflate; webp-decoder_b200/csrc/vp8_pngz.cuh / vp8_pngz.cu): per-row PNG filters
and run-length fixed-Huffman deflate, framed on the device.

On the host: tests/native/pngz_check.cpp replays the kernels' grid from vp8_pngz.cuh against an independent byte-at-a-time
writer of the format, and one replayed file is taken apart here with zlib and PIL. On the GPU: every -png door with the
setting on gives files that decode to the reference's pixels, the same bytes through every door, the host writer's bytes
on frame geometries around the piece and scanline boundaries, and fewer bytes over the link than the stored files."""
import hashlib
import io
import json
import shutil
import struct
import subprocess
import zlib
from pathlib import Path

import numpy as np
import pytest

from vp8fix import GOLDEN, ROOT, fuzz_frame, sha


@pytest.fixture(scope="module")
def pngz_check(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    exe = tmp_path_factory.mktemp("pngz") / "pngz_check"
    subprocess.run([gxx, "-O2", "-std=c++17", "-o", str(exe), str(ROOT / "tests" / "native" / "pngz_check.cpp")], check=True)
    return exe


def chunks_of(png: bytes):
    assert png[:8] == b"\x89PNG\r\n\x1a\n"
    pos, out = 8, []
    while pos < len(png):
        n, = struct.unpack(">I", png[pos:pos + 4])
        kind, data = png[pos + 4:pos + 8], png[pos + 8:pos + 8 + n]
        crc, = struct.unpack(">I", png[pos + 8 + n:pos + 12 + n])
        assert zlib.crc32(kind + data) == crc, kind
        out.append((kind, data))
        pos += 12 + n
    assert pos == len(png)
    return out


def unfilter(raw: bytes, w: int, h: int) -> np.ndarray:
    """The PNG reader's side (PNG spec 9.2-9.4, bpp 3), written out here in numpy."""
    lines = np.frombuffer(raw, np.uint8).reshape(h, 3 * w + 1)
    assert lines[:, 0].max() <= 4
    out = np.zeros((h, 3 * w), np.int32)
    prev = np.zeros(3 * w, np.int32)
    for y in range(h):
        f, cur = int(lines[y, 0]), lines[y, 1:].astype(np.int32)
        if f in (0, 2):
            row = (cur + (prev if f == 2 else 0)) & 255
        else:
            row = np.zeros(3 * w, np.int32)
            for i in range(3 * w):
                a = row[i - 3] if i >= 3 else 0
                b, c = prev[i], prev[i - 3] if i >= 3 else 0
                if f == 1:
                    pred = a
                elif f == 3:
                    pred = (a + b) >> 1
                else:
                    p = a + b - c
                    pa, pb, pc = abs(p - a), abs(p - b), abs(p - c)
                    pred = a if pa <= pb and pa <= pc else b if pb <= pc else c
                row[i] = (cur[i] + pred) & 255
        out[y], prev = row, row
    return out.astype(np.uint8)


def test_pngz_arithmetic_replayed_on_the_host(pngz_check):
    """The kernels' grid in plain loops against the independent writer: 121 images of 18 sizes (1x1; 3w+1 just under and
    over 65535; a piece that ends in front of a filter byte; runs of 255..262 and 515..518 bytes; flat, gradient, noise and
    mixed content, noise over flat and flat over noise), byte for byte, none longer than its stored file; both kinds of
    piece occur, in the middle and at the end of a file."""
    out = subprocess.run([str(pngz_check)], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.startswith("ok 121 "), out.stdout + out.stderr
    stored, fixed, last_stored, last_fixed = map(int, out.stdout.split()[3:7])
    assert stored > 0 and fixed > 0 and last_stored > 0 and last_fixed > 0, out.stdout


def test_replayed_file_taken_apart(pngz_check, tmp_path):
    """One replayed file of mixed content: chunk CRCs (zlib.crc32), the zlib stream inflates (Adler-32 checked by zlib), the
    scanlines unfilter to the RGB, and PIL reads the same RGB."""
    from PIL import Image
    w, h = 487, 301  # 440062 filtered bytes: 6 full pieces and a partial one
    png_path, rgb_path = tmp_path / "replayed.png", tmp_path / "replayed.rgb"
    assert subprocess.run([str(pngz_check), "dump", str(w), str(h), str(png_path), str(rgb_path)]).returncode == 0
    png, rgb = png_path.read_bytes(), rgb_path.read_bytes()
    chunks = chunks_of(png)
    assert [k for k, _ in chunks] == [b"IHDR", b"IDAT", b"IEND"]
    assert chunks[0][1] == struct.pack(">IIBBBBB", w, h, 8, 2, 0, 0, 0)
    idat = chunks[1][1]
    assert idat[:2] == b"\x78\x01"
    raw = zlib.decompress(idat)
    assert len(raw) == (3 * w + 1) * h
    assert len({raw[y * (3 * w + 1)] for y in range(h)}) > 1  # several filters in use
    assert unfilter(raw, w, h).tobytes() == rgb
    assert Image.open(io.BytesIO(png)).tobytes() == rgb
    assert len(png) < 57 + 2 + len(raw) + 5 * 7 + 4  # smaller than the stored file


# ------------------------------------------------------------------------------------------------------------ GPU
def pixels_of(png: bytes):
    from PIL import Image
    im = Image.open(io.BytesIO(png))
    assert im.mode == "RGB"
    return im.size, im.tobytes()


def ppm_digest_of(png: bytes) -> str:
    (w, h), rgb = pixels_of(png)
    return hashlib.sha256(b"P6\n%d %d\n255\n" % (w, h) + rgb).hexdigest()


def stored_len(w: int, h: int) -> int:
    raw = (3 * w + 1) * h
    return 57 + 2 + raw + 5 * ((raw + 65534) // 65535) + 4


@pytest.mark.gpu
def test_deflate_every_door_golden(lib, gpu_ctx, golden, parsed_golden):
    """All 254 golden inputs as one mixed-size batch with the setting on, through the staged calls, the dense pipelined call,
    compact frames (chunks 9 and 0) and .webp bytes: every file decodes (PIL) to the RGB behind the reference's -ppm digest,
    and every door gives the same bytes. Turned off again, the same context gives the reference's -png bytes."""
    from webp_decoder_b200 import parse as P
    names = sorted(golden)
    kfs = [parsed_golden[n][0] for n in names]
    frs = [parsed_golden[n][1] for n in names]
    try:
        gpu_ctx.set_png_deflate(True)
        staged = gpu_ctx.decode_png(kfs, frs)
        bad = [n for n, p in zip(names, staged) if ppm_digest_of(p) != golden[n]["ppm"]]
        assert not bad, ("staged", len(bad), bad[:4])
        assert all(len(p) <= stored_len(golden[n]["width"], golden[n]["height"]) for n, p in zip(names, staged))
        need = gpu_ctx.decode_bytes(kfs, ppm="png")
        out = lib.PinnedBuffer(need)

        def same(what, offs, sizes):
            got = [out.array[int(o):int(o) + int(s)].tobytes() for o, s in zip(offs, sizes)]
            bad = [n for n, g, s in zip(names, got, staged) if g != s]
            assert not bad, (what, len(bad), bad[:4])
            spans = sorted((int(o), int(o) + int(s)) for o, s in zip(offs, sizes))
            assert spans[0][0] == 0 and all(a[1] == b[0] for a, b in zip(spans, spans[1:]))  # back to back

        out.array[:] = 0x77
        same("decode_png", *gpu_ctx.decode_into(kfs, frs, out.array, ppm="png", chunk=11))
        datas = [(GOLDEN / "webp" / n).read_bytes() for n in names]
        cf = P.parse_batch_compact(datas, threads=4, pinned=True, contiguous=True)
        for chunk in (9, 0):
            out.array[:] = 0x55
            same(("compact", chunk), *gpu_ctx.decode_compact_into(cf.frame_list(), out.array, ppm="png", chunk=chunk))
        cf.free()
        files = lib.WebpFiles(datas)
        assert gpu_ctx.decode_webp_bytes(files, ppm="png") == need
        out.array[:] = 0x33
        same("webp", *gpu_ctx.decode_webp_into(files, out.array, ppm="png", chunk=16))
        out.close()
    finally:
        gpu_ctx.set_png_deflate(False)
    pngs = gpu_ctx.decode_png(kfs, frs)
    bad = [n for n, p in zip(names, pngs) if sha(p) != golden[n]["png"]]
    assert not bad, ("stored after deflate", len(bad), bad[:4])


@pytest.mark.gpu
def test_deflate_geometries_and_bench_inputs(lib, gpu_ctx, oracle, pngz_check, tmp_path):
    """The frame geometries of the stored framing's test (3w+1 around multiples of 16, scanlines longer than a piece, a piece
    boundary inside a filter byte) give the host writer's bytes for the oracle's RGB; the 1080p / 4K bench inputs decode to the
    reference's pixels, and the flat and smooth contents (rgbgrad, checker, diag) come out smaller than stored."""
    dims = [(1, 1), (1, 40), (40, 1), (2, 2), (5, 5), (15, 15), (16, 16), (21, 13), (85, 3), (341, 64), (1365, 48), (1366, 49),
            (129, 129), (1000, 24), (24, 1000), (255, 255), (16383, 4), (7, 9000)]
    frames = [fuzz_frame(170 + i, w, h, density=0.2 if w * h < 100000 else 0.02) for i, (w, h) in enumerate(dims)]
    from webp_decoder_b200 import parse as P
    try:
        gpu_ctx.set_png_deflate(True)
        pngs = gpu_ctx.decode_png([f.header() for f in frames], [f.cstruct() for f in frames])
        for f, p in zip(frames, pngs):
            rgb = oracle.rgb(oracle.decode_i420(f, True), f.width, f.height)
            (tmp_path / "in.rgb").write_bytes(rgb.tobytes())
            r = subprocess.run([str(pngz_check), "write", str(f.width), str(f.height), str(tmp_path / "in.rgb"), str(tmp_path / "out.png")],
                               capture_output=True, text=True)
            assert r.returncode == 0, r.stdout + r.stderr
            assert p == (tmp_path / "out.png").read_bytes(), (f.width, f.height)
        dg = json.loads((ROOT / "bench_data" / "digests.json").read_text())
        bnames = sorted(dg)
        pf = P.parse_batch([(ROOT / "bench_data" / n).read_bytes() for n in bnames], pinned=True)
        order = [k % len(bnames) for k in range(2 * len(bnames))]
        pngs = gpu_ctx.decode_png([pf.kf_list()[k] for k in order], [pf.frame_list()[k] for k in order])
        pf.free()
    finally:
        gpu_ctx.set_png_deflate(False)
    for k, p in zip(order, pngs):
        n = bnames[k]
        assert ppm_digest_of(p) == dg[n]["ppm"], n
        (w, h), _ = pixels_of(p)
        if not n.startswith("noise"):
            assert len(p) < stored_len(w, h), (n, len(p))
    first = {bnames[k]: p for k, p in zip(order, pngs)}
    assert all(first[bnames[k]] == p for k, p in zip(order, pngs))  # the same picture, the same bytes


@pytest.mark.gpu
def test_deflate_pipelined_link_bytes(lib, gpu_ctx):
    """A pipelined deflate call moves each file's bytes and 4 bytes of length per file over the link, strictly fewer than
    the stored files."""
    from webp_decoder_b200 import parse as P
    dg = json.loads((ROOT / "bench_data" / "digests.json").read_text())
    bnames = sorted(dg)
    order = [k % len(bnames) for k in range(4 * len(bnames))]
    pf = P.parse_batch([(ROOT / "bench_data" / bnames[k]).read_bytes() for k in order], pinned=True)
    kfs, frs = pf.kf_list(), pf.frame_list()
    need = gpu_ctx.decode_bytes(kfs, ppm="png")
    out = lib.PinnedBuffer(need)
    try:
        gpu_ctx.set_png_deflate(True)
        d0 = gpu_ctx.d2h_bytes
        offs, sizes = gpu_ctx.decode_into(kfs, frs, out.array, ppm="png", chunk=8)
        moved = gpu_ctx.d2h_bytes - d0
    finally:
        gpu_ctx.set_png_deflate(False)
    total = int(sizes.sum())
    assert moved == total + 4 * len(order), (moved, total)
    assert total < sum(stored_len(k.width, k.height) for k in kfs)
    for k, o, s in zip(order, offs, sizes):
        assert ppm_digest_of(out.array[int(o):int(o) + int(s)].tobytes()) == dg[bnames[k]]["ppm"], bnames[k]
    out.close()
    pf.free()


@pytest.mark.gpu
def test_batch_cli_deflate(lib, golden, tmp_path):
    """vp8gpu_batch -png --deflate writes .png files that decode to the reference's pixels; --deflate with another mode is a
    usage error."""
    exe = ROOT / "webp-decoder_b200" / "vp8gpu_batch"
    assert exe.exists(), "run `python __graft_entry__.py build`"
    names = sorted(golden)[::7]
    files = [str(GOLDEN / "webp" / n) for n in names]
    out = tmp_path / "z"
    r = subprocess.run([str(exe), "-png", str(out), "--deflate", "--threads", "4", "--chunk", "9", *files], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    for n in names:
        data = (out / (n[:-5] + ".png")).read_bytes()
        assert ppm_digest_of(data) == golden[n]["ppm"], n
        assert len(data) <= stored_len(golden[n]["width"], golden[n]["height"])
    r = subprocess.run([str(exe), "-ppm", str(tmp_path / "p"), "--deflate", *files[:2]], capture_output=True, text=True)
    assert r.returncode == 2 and "--deflate" in r.stderr
