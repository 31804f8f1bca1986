"""Lossy WebP with alpha (VP8X + ALPH + 'VP8 '): the container walk and ALPH decode on the host (vp8_parse_webp_info,
vp8_parse_alpha, webp_alpha.cpp), the device unfilter grid replayed on the host, the VP8L decoder under sanitizers on
damaged payloads, and on the GPU the RGBA door vp8_gpu_decode_webp_rgba and vp8gpu_batch -pam. The committed fixtures
(tests/golden/alpha, tools/make_alpha_fixtures.py) carry libwebp's answers as digests, so Pillow is only needed for the
tests that make fresh files."""
import errno
import hashlib
import json
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

import alphafix as A
from vp8fix import GOLDEN

ROOT = Path(__file__).resolve().parent.parent
ALPHA = GOLDEN / "alpha"
META = json.loads((GOLDEN / "alpha.json").read_text())
NAMES = sorted(k for k in META if k.endswith(".webp"))


def sha(b) -> str:
    return hashlib.sha256(bytes(b)).hexdigest()


def pillow():
    try:
        from PIL import features
        return features.check("webp")
    except ImportError:
        return False


@pytest.fixture(scope="module")
def P(lib):
    from webp_decoder_b200 import parse
    return parse


# ------------------------------------------------------------------------------------------------ host
def test_fixtures_cover_the_grid():
    seen = {(m["filter"], m["compression"]) for m in META.values() if m.get("filter") is not None}
    assert seen == {(f, c) for f in range(4) for c in range(2)}
    assert any(m.get("preprocessing") == 1 for m in META.values())
    assert sum(p.stat().st_size for p in ALPHA.iterdir()) < 4_000_000


@pytest.mark.parametrize("name", NAMES)
def test_host_alpha_plane_matches_libwebp(P, name):
    data = (ALPHA / name).read_bytes()
    m = META[name]
    w, h, has_alpha = P.webp_info(data)
    assert (w, h) == (m["width"], m["height"])
    plane = P.alpha_plane(data)
    if m["alpha"] is None:
        assert plane is None and not has_alpha
    else:
        assert has_alpha and plane.shape == (h, w) and sha(plane.tobytes()) == m["alpha"]


@pytest.mark.skipif(not pillow(), reason="Pillow with WebP support is not installed")
@pytest.mark.parametrize("kind", ["const", "levels", "ramp", "noise", "runs", "mixed"])
def test_host_alpha_plane_matches_pillow_on_fresh_files(P, kind):
    for (w, h) in ((1, 1), (3, 2), (33, 17), (71, 40)):
        vp8 = A.vp8_chunk_of(A.picture(w, h, w + h))
        a = A.alpha_content(kind, w, h, 31 * w + h)
        for m in range(4):
            for comp in (0, 1):
                f = A.wrap(vp8, w, h, A.alph_payload(a, m, comp))
                want = A.pillow_rgba(f)[..., 3]
                assert np.array_equal(want, a)
                assert np.array_equal(P.alpha_plane(f), want), (w, h, kind, m, comp)


def _base():
    return (ALPHA / "grid_37x23_mixed_f3_c1.webp").read_bytes()


def _rewrap(data, mutate):
    """Apply mutate(list of (tag, payload)) and rebuild the file."""
    cs = mutate(A.chunks(data))
    return A.riff(b"".join(A.chunk(t, d) for t, d in cs))


def _errno(P, data):
    with pytest.raises(OSError) as e:
        P.webp_info(data)
    return e.value.errno


def test_container_rules(P):
    base = _base()
    vp8x, alph, vp8 = A.chunks(base)
    assert P.webp_info(base) == (37, 23, True)
    anim_flag = A.riff(A.vp8x(37, 23, True, flags=0x02) + A.chunk(*alph) + A.chunk(*vp8))
    assert _errno(P, anim_flag) == errno.ENOTSUP
    assert _errno(P, _rewrap(base, lambda cs: [cs[0], (b"ANIM", b"\0" * 6)] + cs[1:])) == errno.ENOTSUP
    assert _errno(P, _rewrap(base, lambda cs: cs + [(b"ANMF", b"\0" * 16)])) == errno.ENOTSUP
    assert _errno(P, _rewrap(base, lambda cs: [cs[0], (b"VP8L", b"\x2f" + b"\0" * 8)])) == errno.ENOTSUP
    assert _errno(P, A.riff(A.chunk(b"VP8L", b"\x2f" + b"\0" * 8))) == errno.ENOTSUP
    assert _errno(P, _rewrap(base, lambda cs: [cs[0], cs[2], cs[1]])) == errno.EINVAL            # ALPH after 'VP8 '
    assert _errno(P, _rewrap(base, lambda cs: [cs[0], cs[1], cs[1], cs[2]])) == errno.EINVAL     # two ALPH
    assert _errno(P, _rewrap(base, lambda cs: [cs[0], cs[1]])) == errno.EINVAL                   # no image
    assert _errno(P, A.riff(A.vp8x(38, 23) + A.chunk(*alph) + A.chunk(*vp8))) == errno.EINVAL    # canvas mismatch
    assert _errno(P, A.riff(A.vp8x(37, 24) + A.chunk(*alph) + A.chunk(*vp8))) == errno.EINVAL
    for hdr in (0x40, 0x80, 0x02, 0x03, 0x20, 0x30):  # reserved bits, compression > 1, pre-processing > 1
        bad = _rewrap(base, lambda cs: [cs[0], (b"ALPH", bytes([hdr]) + cs[1][1][1:]), cs[2]])
        assert _errno(P, bad) == errno.EINVAL, hex(hdr)
    for cut in (1, 9, 30, len(base) // 2, len(base) - 1):
        assert _errno(P, base[:cut]) == errno.EINVAL, cut


def test_truncated_and_damaged_payloads_fail_with_einval(P):
    base = _base()
    vp8x, alph, vp8 = A.chunks(base)
    for keep in (1, 2, 5, len(alph[1]) // 2, len(alph[1]) - 1):
        f = A.riff(A.chunk(*vp8x) + A.chunk(b"ALPH", alph[1][:keep]) + A.chunk(*vp8))
        with pytest.raises(OSError) as e:
            P.alpha_plane(f)
        assert e.value.errno == errno.EINVAL, keep
    raw = (ALPHA / "grid_37x23_mixed_f3_c0.webp").read_bytes()
    cs = A.chunks(raw)
    f = A.riff(A.chunk(*cs[0]) + A.chunk(b"ALPH", cs[1][1][:-1]) + A.chunk(*cs[2]))  # raw plane one byte short
    with pytest.raises(OSError) as e:
        P.alpha_plane(f)
    assert e.value.errno == errno.EINVAL


def test_existing_calls_still_reject_extended_files(P):
    base = _base()
    with pytest.raises(OSError) as e:
        P.webp_size(base)
    assert e.value.errno == errno.EINVAL
    with pytest.raises(OSError) as e:
        P.parse_batch([base], threads=1)
    assert e.value.errno == errno.EINVAL
    with pytest.raises(OSError) as e:
        P.parse_batch_compact([base], threads=1)
    assert e.value.errno == errno.EINVAL
    from webp_decoder_b200 import WebpFiles, load_library
    files = WebpFiles([base])
    assert load_library().vp8_gpu_decode_webp_bytes(files.ptrs, files.sizes, 1, 1) == 0


def test_simple_files_are_opaque(P):
    data = (GOLDEN / "webp" / "enc_noise_16x16_q10_rdo_nolf.webp").read_bytes()
    assert P.webp_info(data) == (16, 16, False)
    assert P.alpha_plane(data) is None


def _gxx():
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    return gxx


def test_unfilter_grid_replayed_on_the_host(tmp_path):
    """tests/native/alpha_check.cpp emulates every warp and lane of the unfilter kernel - the shuffle scans, and the gradient
    wavefront's skew, band chaining through progress stamps (warps interleaved in a seeded random order) and warp tails - and
    compares with plain row-by-row unfiltering."""
    exe = tmp_path / "alpha_check"
    subprocess.run([_gxx(), "-O2", "-std=c++17", "-o", str(exe), str(ROOT / "tests" / "native" / "alpha_check.cpp")], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.startswith("ok 153 "), out.stdout + out.stderr


def test_vp8l_decoder_under_sanitizers(tmp_path):
    """The ALPH decoder built with -fsanitize=address,undefined on truncated and bit-flipped payloads (seeded): each one
    decodes or fails with EINVAL, and no sanitizer reports anything."""
    exe = tmp_path / "alpha_fuzz"
    csrc = ROOT / "webp-decoder_b200" / "csrc"
    build = subprocess.run([_gxx(), "-O1", "-g", "-std=c++17", "-pthread", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined",
                            "-o", str(exe), str(ROOT / "tests" / "native" / "alpha_fuzz.cpp"), str(csrc / "webp_alpha.cpp"), str(csrc / "vp8_parse.cpp")],
                           capture_output=True, text=True)
    if build.returncode != 0 and "asan" in build.stderr.lower():
        pytest.skip("no sanitizer runtime: " + build.stderr[-300:])
    assert build.returncode == 0, build.stderr
    inputs = [str(ALPHA / n) for n in NAMES if META[n]["compression"] == 1 and META[n]["width"] * META[n]["height"] <= 200_000]
    out = subprocess.run([str(exe), *inputs], capture_output=True, text=True, env={"ASAN_OPTIONS": "detect_leaks=1:abort_on_error=0"})
    assert out.returncode == 0 and out.stdout.startswith("ok ") and "runtime error" not in out.stderr, out.stdout + out.stderr[-2000:]
    payloads, decoded, rejected = map(int, out.stdout.split()[1:4])
    assert payloads == 160 * len(inputs) and rejected > 0


# ------------------------------------------------------------------------------------------------ GPU
def _decode(ctx, datas, chunk=0):
    from webp_decoder_b200 import WebpFiles
    files = WebpFiles(datas)
    cap = ctx.decode_webp_rgba_bytes(files)
    assert cap > 0
    out = np.zeros(cap, np.uint8)
    offs, sizes = ctx.decode_webp_rgba_into(files, out, chunk=chunk)
    return [out[int(o):int(o) + int(s)].tobytes() for o, s in zip(offs, sizes)]


def _pam_parts(pam: bytes):
    hdr_end = pam.index(b"ENDHDR\n") + 7
    head = pam[:hdr_end].decode().split("\n")
    w, h = int(head[1].split()[1]), int(head[2].split()[1])
    return w, h, np.frombuffer(pam[hdr_end:], np.uint8).reshape(h, w, 4)


@pytest.mark.gpu
def test_gpu_rgba_matches_libwebp_on_every_fixture(gpu_ctx):
    datas = [(ALPHA / n).read_bytes() for n in NAMES]
    pams = _decode(gpu_ctx, datas)
    bad = [n for n, p in zip(NAMES, pams) if sha(p) != META[n]["pam"]]
    assert not bad, bad
    ms, launches = gpu_ctx.alpha_time()
    assert launches >= 2 and ms > 0


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", [1, 3, 0])
def test_gpu_mixed_batch(gpu_ctx, golden, chunk):
    """Simple golden files and alpha fixtures of several sizes in one call: a simple file gives exactly its golden -ppm RGB with
    alpha 255, an alpha file its libwebp digest."""
    simple = sorted(golden)[::9]
    alpha = NAMES[::2]
    names = [("s", n) for n in simple] + [("a", n) for n in alpha]
    order = list(range(len(names)))
    np.random.default_rng(chunk).shuffle(order)
    names = [names[i] for i in order]
    datas = [(GOLDEN / "webp" / n).read_bytes() if k == "s" else (ALPHA / n).read_bytes() for k, n in names]
    for (kind, n), p in zip(names, _decode(gpu_ctx, datas, chunk)):
        if kind == "a":
            assert sha(p) == META[n]["pam"], n
            continue
        w, h, rgba = _pam_parts(p)
        assert (w, h) == (golden[n]["width"], golden[n]["height"]) and (rgba[..., 3] == 255).all(), n
        ppm = f"P6\n{w} {h}\n255\n".encode() + np.ascontiguousarray(rgba[..., :3]).tobytes()
        assert sha(ppm) == golden[n]["ppm"], n


@pytest.mark.gpu
def test_gpu_alpha_planes_equal_the_host_decoder(gpu_ctx, P):
    datas = [(ALPHA / n).read_bytes() for n in NAMES]
    for n, d, p in zip(NAMES, datas, _decode(gpu_ctx, datas, chunk=5)):
        plane = P.alpha_plane(d)
        _, _, rgba = _pam_parts(p)
        assert np.array_equal(rgba[..., 3], plane if plane is not None else np.full(rgba.shape[:2], 255, np.uint8)), n


@pytest.mark.gpu
def test_gpu_rgba_rejects_what_the_host_rejects(gpu_ctx):
    from webp_decoder_b200 import Vp8GpuError, WebpFiles
    base = _base()
    bad = A.riff(A.vp8x(38, 23) + b"".join(A.chunk(t, d) for t, d in A.chunks(base)[1:]))
    files = WebpFiles([base, bad])
    out = np.zeros(1 << 20, np.uint8)
    with pytest.raises(Vp8GpuError) as e:
        gpu_ctx.decode_webp_rgba_into(files, out)
    assert e.value.errno == errno.EINVAL
    # a payload that only the worker's VP8L decode finds broken fails the call too
    cs = A.chunks(base)
    trunc = A.riff(A.chunk(*cs[0]) + A.chunk(b"ALPH", cs[1][1][:8]) + A.chunk(*cs[2]))
    with pytest.raises(Vp8GpuError) as e:
        gpu_ctx.decode_webp_rgba_into(WebpFiles([base, trunc]), out)
    assert e.value.errno == errno.EINVAL
    assert sha(_decode(gpu_ctx, [base])[0]) == META["grid_37x23_mixed_f3_c1.webp"]["pam"]  # the context is still usable


@pytest.mark.gpu
def test_cli_pam_writes_the_same_bytes(lib, tmp_path):
    exe = ROOT / "webp-decoder_b200" / "vp8gpu_batch"
    names = [n for n in NAMES if META[n]["width"] * META[n]["height"] < 50_000][:6] + ["vp8x_flag_without_alph.webp"]
    paths = [str(ALPHA / n) for n in names] + [str(GOLDEN / "webp" / "enc_noise_16x16_q10_rdo_nolf.webp")]
    out = subprocess.run([str(exe), "-pam", str(tmp_path), *paths], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    for n in names:
        assert sha((tmp_path / (n[:-5] + ".pam")).read_bytes()) == META[n]["pam"], n
    _, _, rgba = _pam_parts((tmp_path / "enc_noise_16x16_q10_rdo_nolf.pam").read_bytes())
    assert (rgba[..., 3] == 255).all()
