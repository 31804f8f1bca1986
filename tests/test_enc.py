"""Encoder in-loop reconstruction (SURVEY.md 8(f) row 4; include/vp8_enc.h).

CPU (-m "not gpu"): the oracle restatement (oracle/vp8_enc_oracle.c) against the reference encoder library on fresh seeded
pictures (where oracle/_ref is built, else its digests in tests/golden/ref_checks.json) and against the committed digests of
that reference; the library exports the symbols.
GPU (-m gpu): the CUDA path through the C-ABI - the reference's own entry points and the batch call - against the oracle
and the digests, bit for bit: coefficients, modes, qindex and the reconstruction planes."""
import json
import re
from pathlib import Path

import numpy as np
import pytest

from encfix import GOLDEN, EncOracle, EncReference, cases, digest, picture, same

ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def enc_oracle():
    return EncOracle()


@pytest.fixture(scope="module")
def enc_golden():
    return json.loads((GOLDEN / "enc.json").read_text())


def parse_key(k):
    """-> seed, w, h, kind, quality, search (0 DC, 1 whole-macroblock modes, "bpred")"""
    seed, size, kind, q, s = k.split("_")
    w, h = size.split("x")
    return int(seed), int(w), int(h), int(kind[1:]), int(q[1:]), {0: 0, 1: 1, 2: "bpred"}[int(s[1:])]


def key_digest(r, s):
    if s == "bpred":
        return digest(r["coeffs"], r["y_modes"], r["uv_modes"], r["b_modes"])
    z = np.zeros_like(r["y_modes"])
    return digest(r["coeffs"], r["y_modes"] if s else z, r["uv_modes"] if s else z)


def test_oracle_matches_reference_encoder_digests(enc_oracle, enc_golden):
    assert len(enc_golden) >= 150
    for k, g in enc_golden.items():
        seed, w, h, kind, q, s = parse_key(k)
        if w * h > 1280 * 720:
            continue  # the 1080p entries are for the GPU tests; the scalar oracle takes seconds on each
        r = enc_oracle.run(*picture(seed, w, h, kind), q, s)
        assert r["qindex"] == g["qindex"] and key_digest(r, s) == g["digest"], k


def library_key(seed, w, h, kind, q, s):
    return f"{seed}_{w}x{h}_k{kind}_q{q}_s{2 if s == 'bpred' else s}"


def test_oracle_matches_reference_encoder_library(enc_oracle):
    """Fresh seeded pictures against the original encoder's modules (oracle/_ref/libref_enc.so) where they are built, else
    against their digests (tests/golden/ref_checks.json)."""
    ref = EncReference() if EncReference.available() else None
    stored = json.loads((GOLDEN / "ref_checks.json").read_text())["encoder"]
    for seed, w, h, kind, q in cases(40, seed0=5000):
        y, u, v = picture(seed, w, h, kind)
        for s in (0, 1, "bpred"):
            got = enc_oracle.run(y, u, v, q, s)
            if ref is not None:
                assert same(ref.run(y, u, v, q, s), got, s), (seed, w, h, kind, q, s)
            else:
                g = stored[library_key(seed, w, h, kind, q, s)]
                assert got["qindex"] == g["qindex"] and key_digest(got, s) == g["digest"], (seed, w, h, kind, q, s)


def test_oracle_honours_strides(enc_oracle):
    y, u, v = picture(7, 37, 21, 0)
    yp, up, vp = np.zeros((21, 64), np.uint8), np.zeros((11, 32), np.uint8), np.zeros((11, 32), np.uint8)
    yp[:, :37], up[:, :19], vp[:, :19] = y, u, v
    assert same(enc_oracle.run(y, u, v, 60, 1), enc_oracle.run(yp[:, :37], up[:, :19], vp[:, :19], 60, 1), 1)


def test_library_exports_the_encoder_symbols(lib):
    L = lib.load_library()
    text = re.sub(r"/\*.*?\*/", "", (ROOT / "include" / "vp8_enc.h").read_text(), flags=re.S)
    syms = sorted(set(re.findall(r"\b((?:enc_vp8|vp8_gpu_enc)\w*)\s*\(", text)))
    assert len(syms) == 8, syms
    assert not [s for s in syms if not hasattr(L, s)]
    from webp_decoder_b200.enc import EncYuv420Image
    import ctypes as C
    assert C.sizeof(EncYuv420Image) == 40 and EncYuv420Image.y.offset == 16  # reference enc_rgb_to_yuv.h:9-17


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_gpu_reference_entry_points_match_oracle(lib, enc_oracle):
    from webp_decoder_b200 import enc
    for seed, w, h, kind, q in cases(24, seed0=100):
        y, u, v = picture(seed, w, h, kind)
        co, qi = enc.encode_dc_pred_inloop(y, u, v, q)
        o = enc_oracle.run(y, u, v, q, 0)
        assert qi == o["qindex"] and np.array_equal(co, o["coeffs"]), ("dc", seed, w, h, kind, q)
        ym, cm, co, qi = enc.encode_i16x16_uv_sad_inloop(y, u, v, q)
        o = enc_oracle.run(y, u, v, q, 1)
        assert same({"coeffs": co, "y_modes": ym, "uv_modes": cm, "qindex": qi}, o, 1), ("i16", seed, w, h, kind, q)
        ym, bm, cm, co, qi = enc.encode_bpred_uv_sad_inloop(y, u, v, q)
        o = enc_oracle.run(y, u, v, q, "bpred")
        assert same({"coeffs": co, "y_modes": ym, "uv_modes": cm, "b_modes": bm, "qindex": qi}, o, "bpred"), ("bpred", seed, w, h, kind, q)
        assert (ym == 4).all()


@pytest.mark.gpu
def test_gpu_batch_matches_oracle_with_reconstruction_planes(lib, enc_oracle):
    from webp_decoder_b200 import enc
    cs = cases(40, seed0=300, max_w=260, max_h=200)
    pics = [picture(seed, w, h, kind) for seed, w, h, kind, _ in cs]
    for s in (0, 1, "bpred"):
        outs, qi = enc.encode_batch(pics, 63, s, want_recon=True)
        for (seed, w, h, kind, _), p, g in zip(cs, pics, outs):
            o = enc_oracle.run(*p, 63, s, want_recon=True)
            g["qindex"] = qi
            assert same(g, o, s), (seed, w, h, kind, s)
            for k in ("rec_y", "rec_u", "rec_v"):
                assert np.array_equal(g[k], o[k]), (k, seed, w, h, kind, s)


@pytest.mark.gpu
def test_gpu_more_pictures_than_resident_ctas(lib, enc_oracle):
    """A launch holds 4 CTAs per SM; with more pictures than that every CTA walks several (stamps and shared state are reset
    in between), and a wide flat picture exercises the longest rows."""
    from webp_decoder_b200 import enc
    pics = [picture(2000 + i, 16 + 16 * (i % 3), 16 + 16 * (i % 2), i % 4) for i in range(1300)] + [picture(9, 4000, 16, 0)]
    for s in (1, "bpred"):
        outs, qi = enc.encode_batch(pics, 40, s)
        for i in list(range(0, 1300, 37)) + [1299, 1300]:
            o = enc_oracle.run(*pics[i], 40, s)
            outs[i]["qindex"] = qi
            assert same(outs[i], o, s), (i, s)


@pytest.mark.gpu
def test_gpu_matches_reference_encoder_digests(lib, enc_golden):
    from webp_decoder_b200 import enc
    for k, g in enc_golden.items():
        seed, w, h, kind, q, s = parse_key(k)
        outs, qi = enc.encode_batch([picture(seed, w, h, kind)], q, s)
        assert qi == g["qindex"] and key_digest(outs[0], s) == g["digest"], k


@pytest.mark.gpu
def test_gpu_strided_planes_and_bad_arguments(lib, enc_oracle):
    from webp_decoder_b200 import Vp8GpuError, enc
    y, u, v = picture(7, 37, 21, 0)
    yp, up, vp = np.zeros((21, 64), np.uint8), np.zeros((11, 32), np.uint8), np.zeros((11, 32), np.uint8)
    yp[:, :37], up[:, :19], vp[:, :19] = y, u, v
    ym, cm, co, qi = enc.encode_i16x16_uv_sad_inloop(yp[:, :37], up[:, :19], vp[:, :19], 60)
    assert same({"coeffs": co, "y_modes": ym, "uv_modes": cm, "qindex": qi}, enc_oracle.run(y, u, v, 60, 1), 1)
    import ctypes as C
    L = lib.load_library()
    co_p, n, q8 = C.c_void_p(), C.c_size_t(), C.c_uint8()
    assert L.enc_vp8_encode_dc_pred_inloop(None, 50, C.byref(co_p), C.byref(n), C.byref(q8)) == -1  # reference: EINVAL (enc_recon.c:867-870)
    assert C.get_errno() == 22 and co_p.value is None and n.value == 0
    with pytest.raises(Vp8GpuError):
        enc.encode_batch([], 50, 0)
