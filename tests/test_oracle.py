"""The CPU oracle (oracle/vp8_oracle.c) against everything that pins it:
   - digests produced by the UNMODIFIED reference decoder binary on 254 .webp inputs (tests/golden/digests.json),
   - RGB pixels of the reference's dwebp-derived golden PNGs (149 of those inputs), i.e. libwebp itself,
   - digests of the reference hot path on 120 struct-level fuzz frames (simple filter, sharpness, lf deltas, int16 wrap),
   - and the reference library called directly on fresh fuzz frames where oracle/_ref is built, else its digests
     (tests/golden/ref_checks.json)."""
import ctypes as C
import json

import numpy as np
import pytest

from vp8fix import GOLDEN, Frame, fuzz_frame, sha


class ParsedAsFrame:
    """Adapter: a (kf, DecodedFrame) pair from the product parser with the Frame interface Oracle expects."""

    def __init__(self, kf, d):
        self.width, self.height, self._d = kf.width, kf.height, d
        self.mb_cols, self.mb_rows = d.mb_cols, d.mb_rows

    def cstruct(self, drop_has_coeff=False):
        from vp8fix import DecodedFrame
        c = DecodedFrame.from_buffer_copy(bytes(self._d))
        c._keep = self._d
        return c

    @property
    def i420_size(self):
        return self.width * self.height + 2 * ((self.width + 1) // 2) * ((self.height + 1) // 2)


def test_oracle_matches_reference_decoder_digests(oracle, golden, parsed_golden):
    assert len(golden) >= 250
    for name, g in golden.items():
        kf, d, _ = parsed_golden[name]
        fr = ParsedAsFrame(kf, d)
        w, h = g["width"], g["height"]
        assert (fr.width, fr.height) == (w, h), name
        yuv, yuvf = oracle.decode_i420(fr, False), oracle.decode_i420(fr, True)
        assert sha(yuv) == g["yuv"], f"{name}: -yuv"
        assert sha(yuvf) == g["yuvf"], f"{name}: -yuvf"
        rgb = oracle.rgb(yuvf, w, h)
        assert sha(oracle.ppm(rgb, w, h)) == g["ppm"], f"{name}: -ppm"
        assert sha(oracle.png(rgb, w, h)) == g["png"], f"{name}: -png"
        if "dwebp_rgb" in g:
            assert sha(rgb) == g["dwebp_rgb"], f"{name}: libwebp golden PNG"


def test_golden_corpus_covers_the_branches(golden):
    infos = [g["info"] for g in golden.values()]
    assert sum(i["Use segment"] == "1" for i in infos) >= 40
    assert sum(i["Level"] == "0" for i in infos) >= 5
    assert sum(int(i["MB B_PRED"]) > 0 for i in infos) >= 60
    assert sum(0 < int(i["MB B_PRED"]) < int(i["MB total"]) for i in infos) >= 20  # mixed i16 / B_PRED frames
    assert sum("dwebp_rgb" in g for g in golden.values()) == 149


def test_oracle_matches_reference_fuzz_digests(oracle):
    fz = json.loads((GOLDEN / "fuzz.json").read_text())
    assert len(fz) == 120
    seen = dict(simple=0, sharp=0, delta=0, seg=0)
    for seed, g in fz.items():
        fr = fuzz_frame(int(seed), g["width"], g["height"], **g["kw"])
        seen["simple"] += fr.params["lf_use_simple"]
        seen["sharp"] += fr.params["lf_sharpness"] != 0
        seen["delta"] += fr.params["lf_delta_enabled"]
        seen["seg"] += fr.params["segmentation_enabled"]
        yuvf = oracle.decode_i420(fr, True)
        assert sha(oracle.decode_i420(fr, False)) == g["yuv"], seed
        assert sha(yuvf) == g["yuvf"], seed
        assert sha(oracle.ppm(oracle.rgb(yuvf, fr.width, fr.height), fr.width, fr.height)) == g["ppm"], seed
    assert min(seen.values()) >= 30, seen  # the branches no bitstream fixture reaches are exercised


def library_case(seed):
    rng = np.random.default_rng(seed + 777)
    w, h = int(rng.integers(1, 120)), int(rng.integers(1, 120))
    return fuzz_frame(seed + 5000, w, h, amp=[5, 40, 400, 2500][seed % 4], density=[0.05, 0.2, 0.6][seed % 3], raw=bool(seed % 2))


def library_outputs(checker, oracle, fr):
    """sha256 of what `checker` (the oracle or the reference library) computes for one fuzz frame."""
    w, h = fr.width, fr.height
    out = {"yuv": checker.decode_i420(fr, False), "yuvf": checker.decode_i420(fr, True),
           # has_coeff == NULL is legal input (vp8_loopfilter.c:226)
           "yuvf_no_has_coeff": checker.decode_i420(fr, True, drop_has_coeff=True)}
    yuvf = out["yuvf"]
    if checker is oracle:
        rgb = oracle.rgb(yuvf, w, h)
        out["ppm"], out["png"] = oracle.ppm(rgb, w, h), oracle.png(rgb, w, h)
    else:
        out["ppm"], out["png"] = checker.ppm_bytes(yuvf, w, h), checker.png_bytes(yuvf, w, h)
    # stand-alone loop filter on padded planes (the oracle's reconstruction as input for both)
    y, u, v = oracle.recon_padded(fr)
    checker.loopfilter_padded(fr, y, u, v)
    out.update(lf_y=y, lf_u=u, lf_v=v)
    return {k: sha(v) for k, v in out.items()}


def rgb_cases():
    rng = np.random.default_rng(5)
    for w, h in [(1, 1), (2, 2), (3, 5), (16, 16), (17, 9), (18, 10), (31, 32), (64, 7), (2, 1), (1, 2), (5, 1)]:
        yield f"{w}x{h}", w, h, rng.integers(0, 256, w * h + 2 * ((w + 1) // 2) * ((h + 1) // 2)).astype(np.uint8)


def png_cases():
    # raw scanline stream sizes around the 65535-byte stored-block limit
    rng = np.random.default_rng(9)
    for w, h in [(21845, 1), (150, 145), (149, 146), (2731, 8), (300, 73)]:
        yield f"{w}x{h}", w, h, rng.integers(0, 256, w * h + 2 * ((w + 1) // 2) * ((h + 1) // 2)).astype(np.uint8)


@pytest.mark.parametrize("seed", range(0, 60))
def test_oracle_vs_reference_library(oracle, reference, ref_digests, seed):
    fr = library_case(seed)
    want = library_outputs(reference, oracle, fr) if reference is not None else ref_digests["library"][str(seed)]
    assert library_outputs(oracle, oracle, fr) == want


def test_rgb_closed_form_on_tiny_and_odd_sizes(oracle, reference, ref_digests):
    for key, w, h, i420 in rgb_cases():
        want = sha(reference.rgb(i420, w, h)) if reference is not None else ref_digests["rgb"][key]
        assert sha(oracle.rgb(i420, w, h)) == want, (w, h)


def test_png_block_boundaries(oracle, reference, ref_digests):
    for key, w, h, i420 in png_cases():
        want = sha(reference.png_bytes(i420, w, h)) if reference is not None else ref_digests["png"][key]
        assert sha(oracle.png(oracle.rgb(i420, w, h), w, h)) == want, (w, h)
