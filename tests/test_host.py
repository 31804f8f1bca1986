"""Host-side logic and the C-ABI surface, no GPU needed: the library loads and exports every declared symbol,
derives per-frame parameters like the oracle, parses .webp files like the reference's m01/m02/m05, and fails
loudly (no CPU fallback) when there is no CUDA device."""
import ctypes as C
import errno
import re
from pathlib import Path

import numpy as np
import pytest

from vp8fix import GOLDEN, I16_ARRAYS, SCALARS, U8_ARRAYS, VEC4, fuzz_frame, sha

ROOT = Path(__file__).resolve().parent.parent


def declared_symbols(header: Path):
    text = re.sub(r"/\*.*?\*/", "", header.read_text(), flags=re.S)
    return sorted(set(re.findall(r"\b((?:vp8_gpu|vp8_parse|yuv420|vp8_reconstruct|vp8_loopfilter|enc_vp8)\w*)\s*\(", text)))


def test_library_exports_every_declared_symbol(lib):
    L = lib.load_library()
    syms = (declared_symbols(ROOT / "include" / "vp8_gpu.h") + declared_symbols(ROOT / "include" / "vp8_parse.h")
            + declared_symbols(ROOT / "include" / "vp8_enc.h"))
    assert len(syms) >= 44
    missing = [s for s in syms if not hasattr(L, s)]
    assert not missing, missing
    assert set(lib.EXPORTS) <= set(syms)
    # the seven symbols the reference's main.c / main_ultra.c bind from m06..m09 (SURVEY.md 8b)
    for s in ("yuv420_alloc", "yuv420_free", "vp8_reconstruct_keyframe_yuv", "vp8_reconstruct_keyframe_yuv_filtered",
              "vp8_loopfilter_apply_keyframe", "yuv420_write_ppm_fd", "yuv420_write_png_fd"):
        assert s in syms


def test_struct_layouts_match_the_reference_abi(lib):
    from webp_decoder_b200.abi import DecodedFrame, KeyFrameHeader, Yuv420Image
    assert (C.sizeof(KeyFrameHeader), C.sizeof(DecodedFrame), C.sizeof(Yuv420Image)) == (28, 320, 40)
    assert KeyFrameHeader.width.offset == 20 and KeyFrameHeader.height.offset == 22
    assert DecodedFrame.segment_id.offset == 40 and DecodedFrame.coeff_v.offset == 112 and DecodedFrame.stats_opaque.offset == 120
    assert Yuv420Image.y.offset == 16 and Yuv420Image.v.offset == 32


def test_yuv420_alloc_free_contract(lib):
    from webp_decoder_b200.abi import Yuv420Image
    L = lib.load_library()
    img = Yuv420Image()
    assert L.yuv420_alloc(C.addressof(img), 5, 3) == 0
    assert (img.width, img.height, img.stride_y, img.stride_uv) == (5, 3, 5, 3)
    assert bytes(np.ctypeslib.as_array(img.y, (15,))) == b"\0" * 15           # vp8_recon.c:381
    assert bytes(np.ctypeslib.as_array(img.u, (6,))) == b"\x80" * 6            # vp8_recon.c:382
    L.yuv420_free(C.addressof(img))
    assert not img.y and img.width == 0
    C.set_errno(0)
    assert L.yuv420_alloc(C.addressof(img), 0, 3) == -1 and C.get_errno() == errno.EINVAL
    L.yuv420_free(None)


@pytest.mark.parametrize("seed", range(40))
def test_frame_params_match_oracle(lib, oracle, seed):
    fr = fuzz_frame(seed, 32, 32)
    dq, lf = lib.frame_params(fr.cstruct())
    odq, olf = oracle.frame_params(fr)
    assert np.array_equal(dq, odq) and np.array_equal(lf, olf)


def test_no_device_means_error_not_fallback(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(lib.Vp8GpuError) as e:
        lib.Context(0)
    assert e.value.errno == errno.EIO
    fr = fuzz_frame(1, 16, 16)
    with pytest.raises(lib.Vp8GpuError):
        lib.vp8_reconstruct_keyframe_yuv_filtered(fr.header(), fr.cstruct())


def test_legacy_entry_points_reject_bad_arguments(lib):
    L = lib.load_library()
    C.set_errno(0)
    assert L.vp8_reconstruct_keyframe_yuv(None, None, None) == -1 and C.get_errno() == errno.EINVAL
    assert L.vp8_loopfilter_apply_keyframe(None, None) == -1 and C.get_errno() == errno.EINVAL
    assert L.yuv420_write_ppm_fd(-1, None) == -1 and C.get_errno() == errno.EINVAL
    assert L.yuv420_write_png_fd(-1, None) == -1 and C.get_errno() == errno.EINVAL


# ---------------------------------------------------------------------------------------------- host front end
def parsed_fields(kf, d, pf, i):
    """What the product parser made of golden input i: {field: sha256}, the arrays at their element type."""
    out = {"size": sha(np.array([kf.width, kf.height], np.int64))}
    out.update({k: sha(np.array([int(getattr(d, k))], np.int64)) for k in SCALARS})
    out.update({k: sha(np.array([int(getattr(d, k)[j]) for j in range(4)], np.int64)) for k in VEC4})
    out.update({k: sha(np.ascontiguousarray(pf.array(i, k), np.uint8)) for k in U8_ARRAYS})
    out.update({k: sha(np.ascontiguousarray(pf.array(i, k), np.int16)) for k in I16_ARRAYS})
    return out


def reference_fields(ref):
    """The same for the original's m01..m05 (a Frame from Reference.parse_webp)."""
    out = {"size": sha(np.array([ref.width, ref.height], np.int64))}
    out.update({k: sha(np.array([ref.params[k]], np.int64)) for k in SCALARS})
    out.update({k: sha(np.array(ref.params[k], np.int64)) for k in VEC4})
    out.update({k: sha(np.ascontiguousarray(ref.arrays[k], np.uint8)) for k in U8_ARRAYS})
    out.update({k: sha(np.ascontiguousarray(ref.arrays[k], np.int16)) for k in I16_ARRAYS})
    return out


def fields_digest(fields):
    """One sha256 over all fields of one input (what tests/golden/ref_checks.json stores per input)."""
    return sha("".join(f"{k}={fields[k]};" for k in sorted(fields)).encode())


def test_parser_matches_reference_m05_on_golden_inputs(lib, reference, ref_digests, golden, parsed_golden):
    names = sorted(golden)
    assert len(names) == len(ref_digests["parser"])
    for i, name in enumerate(names):
        kf, d, pf = parsed_golden[name]
        got = parsed_fields(kf, d, pf, i)
        if reference is not None:
            want = reference_fields(reference.parse_webp((GOLDEN / "webp" / name).read_bytes()))
            assert [k for k in want if got[k] != want[k]] == [], name
        else:
            assert fields_digest(got) == ref_digests["parser"][name], name


def test_parser_is_reentrant_across_threads(lib, golden):
    from webp_decoder_b200 import parse as P
    names = sorted(golden)[:64]
    datas = [(GOLDEN / "webp" / n).read_bytes() for n in names]
    a = P.parse_batch(datas, threads=1)
    b = P.parse_batch(datas * 3, threads=8)
    for i in range(len(names)):
        for k in ("coeff_y", "coeff_y2", "bmode", "ymode", "has_coeff"):
            for rep in range(3):
                assert np.array_equal(a.array(i, k), b.array(i + rep * len(names), k)), (names[i], k)


def test_parser_rejects_what_the_reference_rejects(lib):
    from webp_decoder_b200 import parse as P
    good = (GOLDEN / "webp" / "enc_noise_16x16_q10_rdo_nolf.webp").read_bytes()
    bad_cases = {
        "truncated": good[:-3],
        "not riff": b"RIFX" + good[4:],
        "not webp": good[:8] + b"WEBX" + good[12:],
        "vp8l chunk": good[:12] + b"VP8L" + good[16:],
        "inter frame": good[:20] + bytes([good[20] | 1]) + good[21:],
        "bad start code": good[:23] + b"\x00\x01\x2a" + good[26:],
        "empty": b"",
    }
    for what, data in bad_cases.items():
        with pytest.raises(OSError) as e:
            P.parse_batch([data], threads=1)
        assert e.value.errno == errno.EINVAL, what
    assert P.webp_size(good) == (16, 16)


def test_rgb_tile_arithmetic_on_the_host(tmp_path):
    """webp-decoder_b200/csrc/vp8_rgb.cuh (the arithmetic of the m08 kernel: U|V packed upsampler over 2x16-pixel tiles,
    mult_hi as IMAD.HI, fused clip) also compiles for the host with each device instruction emulated;
    tests/native/rgb_check.cpp runs 263 images (all edge geometries, three content flavours) through it against the
    oracle's orc_i420_to_rgb and checks the clamped-index identity behind the row-end cases exhaustively."""
    import shutil
    import subprocess
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    root = Path(__file__).resolve().parent.parent
    exe = tmp_path / "rgb_check"
    subprocess.run([gxx, "-O2", "-std=c++17", "-o", str(exe), str(root / "tests" / "native" / "rgb_check.cpp"), f"-L{root / 'oracle'}",
                    "-loracle", f"-Wl,-rpath,{root / 'oracle'}"], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.startswith("ok "), out.stdout + out.stderr


def test_png_framing_arithmetic_on_the_host(tmp_path):
    """webp-decoder_b200/csrc/vp8_png.cuh (the arithmetic of the m09 kernels: byte-shifted copy with scanline / stored-block
    boundaries, Adler-32 from weighted partial sums, CRC-32 pieces combined by multiplication mod the CRC polynomial) also
    compiles for the host; tests/native/png_check.cpp replays the kernels' whole grid - every CTA, thread, reduction and the
    finish step - for 76 images against an independent byte-at-a-time writer. One replayed file is then taken apart here
    with zlib (chunk CRCs, inflate, Adler-32) and compared with the host framing the library exports
    (vp8_gpu_png_frame, itself pinned by the reference decoder's -png digests)."""
    import shutil
    import struct
    import subprocess
    import zlib
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    root = Path(__file__).resolve().parent.parent
    exe = tmp_path / "png_check"
    subprocess.run([gxx, "-O2", "-std=c++17", "-o", str(exe), str(root / "tests" / "native" / "png_check.cpp")], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.startswith("ok 76 "), out.stdout + out.stderr
    w, h = 487, 301  # 3 * w + 1 = 1462; 440062 scanline bytes = 6 full stored blocks + a partial one, 7 spans
    dump = tmp_path / "replayed.png"
    assert subprocess.run([str(exe), "dump", str(w), str(h), str(dump)]).returncode == 0
    png = dump.read_bytes()
    assert png[:8] == b"\x89PNG\r\n\x1a\n"
    pos, chunks = 8, []
    while pos < len(png):
        n, = struct.unpack(">I", png[pos:pos + 4])
        kind, data = png[pos + 4:pos + 8], png[pos + 8:pos + 8 + n]
        crc, = struct.unpack(">I", png[pos + 8 + n:pos + 12 + n])
        assert zlib.crc32(kind + data) == crc, kind
        chunks.append((kind, data))
        pos += 12 + n
    assert [k for k, _ in chunks] == [b"IHDR", b"IDAT", b"IEND"]
    assert chunks[0][1] == struct.pack(">IIBBBBB", w, h, 8, 2, 0, 0, 0)
    raw = zlib.decompress(chunks[1][1])  # checks the Adler-32 too
    lines = np.frombuffer(raw, np.uint8).reshape(h, 3 * w + 1)
    assert not lines[:, 0].any()
    import webp_decoder_b200 as lib
    L = lib.load_library()
    L.vp8_gpu_png_bound.argtypes, L.vp8_gpu_png_bound.restype = [C.c_uint32, C.c_uint32], C.c_size_t
    L.vp8_gpu_png_frame.argtypes, L.vp8_gpu_png_frame.restype = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p], C.c_size_t
    rgb = np.ascontiguousarray(lines[:, 1:])
    host = np.empty(L.vp8_gpu_png_bound(w, h), np.uint8)
    n = L.vp8_gpu_png_frame(rgb.ctypes.data, w, h, host.ctypes.data)
    assert host[:n].tobytes() == png


def _dense_to_compact(pf, i):
    """What the compact wire format of parsed frame i must hold, from its dense arrays (numpy restatement of
    include/vp8_parse.h: mask bit b = block b non-zero; 0..15 luma, 16..19 U, 20..23 V, 24 Y2; blocks in bit order)."""
    mb = pf.frames[i].mb_total
    blocks = np.concatenate([pf.array(i, "coeff_y").reshape(mb, 16, 16), pf.array(i, "coeff_u").reshape(mb, 4, 16),
                             pf.array(i, "coeff_v").reshape(mb, 4, 16), pf.array(i, "coeff_y2").reshape(mb, 1, 16)], axis=1)
    nz = (blocks != 0).any(axis=2)
    mask = (nz.astype(np.uint64) << np.arange(25, dtype=np.uint64)).sum(axis=1).astype(np.uint32)
    counts = nz.sum(axis=1)
    first = np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.uint32)
    return mask, first, blocks[nz]


@pytest.mark.parametrize("contiguous", [False, True])
def test_compact_parser_equals_dense_parser(lib, golden, contiguous):
    """vp8_parse_webp_compact / vp8_parse_batch_compact emit the wire format directly while decoding tokens; it must say
    exactly what compacting the dense arrays of the same file says (which the GPU tests pin against the reference), and
    carry the same scalars and modes."""
    from webp_decoder_b200 import parse as P
    from vp8fix import GOLDEN
    names = sorted(golden)[::3]
    datas = [(GOLDEN / "webp" / n).read_bytes() for n in names]
    pf = P.parse_batch(datas, threads=4)
    cf = P.parse_batch_compact(datas, threads=4, contiguous=contiguous)
    scalars = ["mb_cols", "mb_rows", "mb_total", "q_index", "y1_dc_delta_q", "y2_dc_delta_q", "y2_ac_delta_q", "uv_dc_delta_q", "uv_ac_delta_q",
               "segmentation_enabled", "segmentation_abs", "lf_use_simple", "lf_level", "lf_sharpness", "lf_delta_enabled"]
    prev_end = None
    for i, n in enumerate(names):
        d, c = pf.frames[i], cf.frames[i]
        for s in scalars:
            assert getattr(d, s) == getattr(c.f, s), (n, s)
        for s in ("seg_quant_idx", "seg_lf_level", "lf_ref_delta", "lf_mode_delta"):
            assert list(getattr(d, s)) == list(getattr(c.f, s)), (n, s)
        assert (c.width, c.height) == (pf.kfs[i].width, pf.kfs[i].height) == (cf.kfs[i].width, cf.kfs[i].height)
        mb = d.mb_total
        for name, per in (("ymode", 1), ("uv_mode", 1), ("segment_id", 1), ("has_coeff", 1), ("bmode", 16)):
            got = np.ctypeslib.as_array(getattr(c.f, name), shape=(mb * per,))
            assert np.array_equal(got, pf.array(i, name)), (n, name)
        mask, first, blocks = cf.head(i)
        wmask, wfirst, wblocks = _dense_to_compact(pf, i)
        assert np.array_equal(mask, wmask), n
        assert np.array_equal(first, wfirst), n
        assert c.n_blocks == len(wblocks) and np.array_equal(blocks, wblocks), n
        assert c.bytes == (28 * mb + 31) // 32 * 32 + 32 * c.n_blocks and c.head_off == 0
        if contiguous:  # back to back in index order, 256-byte aligned: one transfer per chunk
            assert c.base % 256 == 0 and (prev_end is None or c.base == prev_end), n
            prev_end = c.base + (c.bytes + 255) // 256 * 256
    if contiguous:
        assert cf.used == prev_end - cf.frames[0].base
    # replication gives every copy its own bytes and self-consistent pointers
    rep = P.parse_batch_compact(datas[:3], threads=2, contiguous=True, replicate=3)
    for k in range(9):
        m0, f0, b0 = cf.head(k % 3)
        m1, f1, b1 = rep.head(k)
        assert np.array_equal(m0, m1) and np.array_equal(f0, f1) and np.array_equal(b0, b1)
        assert rep.frames[k].f.ymode and C.addressof(rep.frames[k].f.ymode.contents) == rep.frames[k].base + 8 * rep.frames[k].f.mb_total
    assert len({rep.frames[k].base for k in range(9)}) == 9
    pf.free()


def test_compact_parser_rejects_what_the_dense_one_rejects(lib):
    from webp_decoder_b200 import parse as P
    with pytest.raises(OSError):
        P.parse_batch_compact([b"RIFF\x04\x00\x00\x00WEBP"], threads=1)
