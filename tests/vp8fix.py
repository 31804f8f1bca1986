"""Test-side helpers: ctypes mirrors of the boundary structs, the CPU checkers (oracle/ and
oracle/_ref), a struct-level frame fuzzer, and fixture (de)serialisation.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import io
import os
import subprocess
from dataclasses import dataclass, field
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
ORACLE_DIR = ROOT / "oracle"
REF_DIR = ORACLE_DIR / "_ref"
GOLDEN = ROOT / "tests" / "golden"

u8p = C.POINTER(C.c_uint8)
i16p = C.POINTER(C.c_int16)


class KeyFrameHeader(C.Structure):
    """reference src/m02_vp8_header/vp8_header.h:7-18"""
    _fields_ = [
        ("is_key_frame", C.c_int), ("profile", C.c_uint8), ("show_frame", C.c_int),
        ("first_partition_len", C.c_uint32), ("start_code_ok", C.c_int),
        ("width", C.c_uint16), ("height", C.c_uint16), ("x_scale", C.c_uint8), ("y_scale", C.c_uint8),
    ]


class DecodedFrame(C.Structure):
    """reference src/m05_tokens/vp8_tokens.h:52-99"""
    _fields_ = [
        ("mb_cols", C.c_uint32), ("mb_rows", C.c_uint32), ("mb_total", C.c_uint32),
        ("q_index", C.c_uint8), ("y1_dc_delta_q", C.c_int8), ("y2_dc_delta_q", C.c_int8),
        ("y2_ac_delta_q", C.c_int8), ("uv_dc_delta_q", C.c_int8), ("uv_ac_delta_q", C.c_int8),
        ("segmentation_enabled", C.c_uint8), ("segmentation_abs", C.c_uint8),
        ("seg_quant_idx", C.c_int8 * 4), ("seg_lf_level", C.c_int8 * 4),
        ("lf_use_simple", C.c_uint8), ("lf_level", C.c_uint8), ("lf_sharpness", C.c_uint8),
        ("lf_delta_enabled", C.c_uint8), ("lf_ref_delta", C.c_int8 * 4), ("lf_mode_delta", C.c_int8 * 4),
        ("segment_id", u8p), ("skip_coeff", u8p), ("has_coeff", u8p), ("ymode", u8p), ("uv_mode", u8p),
        ("bmode", u8p),
        ("coeff_y2", i16p), ("coeff_y", i16p), ("coeff_u", i16p), ("coeff_v", i16p),
        ("stats_opaque", C.c_uint64 * 25),
    ]


class Yuv420Image(C.Structure):
    """reference src/m06_recon/vp8_recon.h:10-18"""
    _fields_ = [
        ("width", C.c_uint32), ("height", C.c_uint32), ("stride_y", C.c_uint32), ("stride_uv", C.c_uint32),
        ("y", u8p), ("u", u8p), ("v", u8p),
    ]


class ByteSpan(C.Structure):
    _fields_ = [("data", u8p), ("size", C.c_size_t)]


assert C.sizeof(KeyFrameHeader) == 28 and C.sizeof(DecodedFrame) == 320 and C.sizeof(Yuv420Image) == 40

SCALARS = ["q_index", "y1_dc_delta_q", "y2_dc_delta_q", "y2_ac_delta_q", "uv_dc_delta_q", "uv_ac_delta_q",
           "segmentation_enabled", "segmentation_abs", "lf_use_simple", "lf_level", "lf_sharpness",
           "lf_delta_enabled"]
VEC4 = ["seg_quant_idx", "seg_lf_level", "lf_ref_delta", "lf_mode_delta"]
U8_ARRAYS = ["segment_id", "skip_coeff", "has_coeff", "ymode", "uv_mode", "bmode"]
I16_ARRAYS = ["coeff_y2", "coeff_y", "coeff_u", "coeff_v"]


@dataclass
class Frame:
    """A decoded key frame held in numpy arrays (the host-side input of the pixel path)."""
    width: int
    height: int
    params: dict
    arrays: dict = field(default_factory=dict)

    @property
    def mb_cols(self):
        return (self.width + 15) // 16

    @property
    def mb_rows(self):
        return (self.height + 15) // 16

    @property
    def mb_total(self):
        return self.mb_cols * self.mb_rows

    def cstruct(self, drop_has_coeff: bool = False) -> DecodedFrame:
        d = DecodedFrame()
        d.mb_cols, d.mb_rows, d.mb_total = self.mb_cols, self.mb_rows, self.mb_total
        for k in SCALARS:
            setattr(d, k, int(self.params[k]))
        for k in VEC4:
            arr = getattr(d, k)
            for i in range(4):
                arr[i] = int(self.params[k][i])
        for k in U8_ARRAYS:
            a = self.arrays[k]
            assert a.dtype == np.uint8 and a.flags.c_contiguous
            setattr(d, k, a.ctypes.data_as(u8p))
        if drop_has_coeff:
            d.has_coeff = u8p()
        for k in I16_ARRAYS:
            a = self.arrays[k]
            assert a.dtype == np.int16 and a.flags.c_contiguous
            setattr(d, k, a.ctypes.data_as(i16p))
        d._keep = self  # noqa: keep numpy buffers alive
        return d

    def header(self) -> KeyFrameHeader:
        h = KeyFrameHeader()
        h.is_key_frame, h.show_frame, h.start_code_ok = 1, 1, 1
        h.width, h.height = self.width, self.height
        return h

    @property
    def i420_size(self):
        cw, ch = (self.width + 1) // 2, (self.height + 1) // 2
        return self.width * self.height + 2 * cw * ch

    # ---- fixtures -------------------------------------------------------------------------
    def save(self, path):
        meta = {k: np.array(self.params[k]) for k in SCALARS + VEC4}
        np.savez_compressed(path, width=self.width, height=self.height, **meta, **self.arrays)

    @staticmethod
    def load(path) -> "Frame":
        z = np.load(path)
        params = {k: int(z[k]) for k in SCALARS}
        params.update({k: [int(x) for x in z[k]] for k in VEC4})
        arrays = {k: np.ascontiguousarray(z[k]) for k in U8_ARRAYS + I16_ARRAYS}
        return Frame(int(z["width"]), int(z["height"]), params, arrays)


def default_params(**over):
    p = dict(q_index=40, y1_dc_delta_q=0, y2_dc_delta_q=0, y2_ac_delta_q=0, uv_dc_delta_q=0, uv_ac_delta_q=0,
             segmentation_enabled=0, segmentation_abs=0, lf_use_simple=0, lf_level=0, lf_sharpness=0,
             lf_delta_enabled=0, seg_quant_idx=[0] * 4, seg_lf_level=[0] * 4, lf_ref_delta=[0] * 4,
             lf_mode_delta=[0] * 4)
    p.update(over)
    return p


def fuzz_frame(seed: int, width: int, height: int, *, density: float = 0.2, amp: int = 40,
               bpred_frac: float = 0.5, raw: bool = False, **over) -> Frame:
    """Random-but-valid decoded frame: random modes, sparse random coefficients, random header knobs.
    Anything in `over` pins a header parameter; amp is the coefficient magnitude bound (the token
    alphabet allows |c| <= 2048+; large amp exercises the int16 wrap of dequant/IDCT)."""
    rng = np.random.default_rng(seed)
    cols, rows = (width + 15) // 16, (height + 15) // 16
    n = cols * rows
    p = default_params(
        q_index=int(rng.integers(0, 128)),
        y1_dc_delta_q=int(rng.integers(-15, 16)), y2_dc_delta_q=int(rng.integers(-15, 16)),
        y2_ac_delta_q=int(rng.integers(-15, 16)), uv_dc_delta_q=int(rng.integers(-15, 16)),
        uv_ac_delta_q=int(rng.integers(-15, 16)),
        segmentation_enabled=int(rng.integers(0, 2)), segmentation_abs=int(rng.integers(0, 2)),
        lf_use_simple=int(rng.integers(0, 2)), lf_level=int(rng.integers(0, 64)),
        lf_sharpness=int(rng.integers(0, 8)), lf_delta_enabled=int(rng.integers(0, 2)),
        seg_lf_level=[int(x) for x in rng.integers(-63, 64, 4)],
        lf_ref_delta=[int(x) for x in rng.integers(-63, 64, 4)],
        lf_mode_delta=[int(x) for x in rng.integers(-63, 64, 4)],
    )
    p["seg_quant_idx"] = [int(x) for x in (rng.integers(0, 128, 4) if p["segmentation_abs"] else rng.integers(-40, 41, 4))]
    if p["segmentation_abs"]:
        p["seg_lf_level"] = [int(x) for x in rng.integers(0, 64, 4)]
    p.update(over)

    def coeffs(count):
        c = rng.integers(-amp, amp + 1, count).astype(np.int16)
        c[rng.random(count) >= density] = 0
        return c

    a = {
        "segment_id": rng.integers(0, 4, n).astype(np.uint8),
        "skip_coeff": np.zeros(n, np.uint8),
        "ymode": np.where(rng.random(n) < bpred_frac, 4, rng.integers(0, 4, n)).astype(np.uint8),
        "uv_mode": rng.integers(0, 4, n).astype(np.uint8),
        "bmode": rng.integers(0, 10, n * 16).astype(np.uint8),
        "coeff_y2": coeffs(n * 16), "coeff_y": coeffs(n * 256), "coeff_u": coeffs(n * 64), "coeff_v": coeffs(n * 64),
    }
    # whole macroblocks with no residual at all, so the loop filter's inner-edge skip is exercised
    empty = rng.random(n) < 0.25
    for k, per in (("coeff_y2", 16), ("coeff_y", 256), ("coeff_u", 64), ("coeff_v", 64)):
        a[k].reshape(n, per)[empty] = 0
    if raw:
        # not expressible by a bitstream: coded-looking data in the slots the pixel path must ignore
        # (Y2 of B_PRED macroblocks, luma DC of i16 macroblocks) and an arbitrary has_coeff map
        a["has_coeff"] = rng.integers(0, 2, n).astype(np.uint8)
    else:
        a["has_coeff"] = compute_has_coeff(a, n)
    return Frame(width, height, p, a)


def stress_frame(recipe: str, seed: int, width: int, height: int) -> Frame:
    """A frame whose reconstruction drives the loop filter into particular arms. Content is made of i16 macroblocks
    with Y2 DC/AC (flat 4x4 blocks: steps at block edges), one low-frequency luma AC term per block (ramps: hev),
    textured macroblocks (dense coefficients: interior-limit failures) and macroblocks without coefficients."""
    rng = np.random.default_rng(seed)
    n = ((width + 15) // 16) * ((height + 15) // 16)
    p = default_params(q_index=int(rng.integers(0, 8)), lf_level=int(rng.integers(20, 64)))
    # Y2 DC / Y2 AC / luma AC bounds, share of B_PRED, textured and empty macroblocks, Y2 DC offset of every macroblock
    y2dc, y2ac, ac, bpred, tex, empty, bias = 60, 0, 0, 0.0, 0.0, 0.1, 0
    if recipe == "smooth":      # small steps between flat blocks: the 27/18/9 arm
        y2dc, y2ac = 40, 6
    elif recipe == "ramp":      # gradients inside the blocks: hev, at the levels where the hev threshold changes
        y2dc, ac = 40, 12
        p["lf_level"] = int(rng.choice([15, 16, 39, 40, 63]))
    elif recipe == "steps63":   # large steps, the widest limits: w and a saturate
        y2dc, y2ac, ac = 400, 30, 4
        p.update(lf_level=63, lf_sharpness=0)
    elif recipe == "extremes":  # content pushed to 0 or 255 with texture next to it: clip255 clips
        y2dc, y2ac, ac, tex, bias = 300, 40, 10, 0.3, int(rng.choice([-600, 600]))
        p.update(lf_level=63, lf_sharpness=0)
    elif recipe == "textured":  # smooth macroblocks next to textured partners, every sharpness: interior limit
        y2dc, ac, tex = 60, 8, 0.5
        p.update(lf_sharpness=int(rng.integers(0, 8)), lf_level=int(rng.integers(8, 40)))
    elif recipe == "simple":
        y2dc, y2ac, ac, tex = 60, 8, 8, 0.2
        p.update(lf_use_simple=1, lf_level=int(rng.integers(10, 64)), lf_sharpness=int(rng.integers(0, 8)))
    elif recipe == "segments":  # per-segment levels (some 0), B_PRED mode delta, B_PRED without coefficients
        y2dc, y2ac, ac, tex, bpred, empty = 60, 8, 8, 0.2, 0.4, 0.3
        p.update(segmentation_enabled=1, segmentation_abs=int(rng.integers(0, 2)), lf_delta_enabled=1, lf_sharpness=4,
                 lf_ref_delta=[int(rng.integers(-10, 10)), 0, 0, 0], lf_mode_delta=[int(rng.integers(-20, 21)), 0, 0, 0])
        p["seg_lf_level"] = [0, 15, 40, 63] if p["segmentation_abs"] else [-63, -5, 0, 20]
    else:
        raise ValueError(recipe)
    a = {
        "segment_id": rng.integers(0, 4, n).astype(np.uint8),
        "skip_coeff": np.zeros(n, np.uint8),
        "ymode": np.where(rng.random(n) < bpred, 4, rng.integers(0, 4, n)).astype(np.uint8),
        "uv_mode": rng.integers(0, 4, n).astype(np.uint8),
        "bmode": rng.integers(0, 10, n * 16).astype(np.uint8),
    }
    y2 = np.zeros((n, 16), np.int16)
    y2[:, 0] = bias + rng.integers(-y2dc, y2dc + 1, n)
    y2[:, 1:] = rng.integers(-y2ac, y2ac + 1, (n, 15)) * (rng.random((n, 15)) < 0.3)
    yy = np.zeros((n, 16, 16), np.int16)
    yy[:, :, 0] = rng.integers(-y2dc // 4, y2dc // 4 + 1, (n, 16))  # DC of B_PRED blocks (compute_has_coeff clears it for i16)
    term = np.where(rng.random((n, 16)) < 0.5, 1, 4)                  # first horizontal or first vertical AC term
    np.put_along_axis(yy, term[..., None], rng.integers(-ac, ac + 1, (n, 16, 1)), axis=2)
    t = rng.random(n) < tex
    yy[t] = rng.integers(-60, 61, (int(t.sum()), 16, 16))
    uv = [np.zeros((n, 4, 16), np.int16) for _ in range(2)]
    for c in uv:
        c[:, :, 0] = rng.integers(-20, 21, (n, 4))
        c[t] = rng.integers(-40, 41, (int(t.sum()), 4, 16))
    e = rng.random(n) < empty
    y2[e], yy[e], uv[0][e], uv[1][e] = 0, 0, 0, 0
    a.update(coeff_y2=y2.reshape(-1), coeff_y=yy.reshape(-1), coeff_u=uv[0].reshape(-1), coeff_v=uv[1].reshape(-1))
    a["has_coeff"] = compute_has_coeff(a, n)
    return Frame(width, height, p, a)


RECIPES = ("smooth", "ramp", "steps63", "extremes", "textured", "simple", "segments")
# widths that are not a multiple of 16, single macroblock columns and rows, a frame wider than 1000 px
SIZES = ((160, 96), (100, 72), (16, 200), (9, 130), (300, 16), (200, 12), (1040, 40), (96, 160))
# 512 macroblock rows, 2 columns: the 8 CTAs x 16 warps of a fused cluster of 8 deal 2-row pairs round-robin, so every
# CTA gets rows and every warp takes a second pair (more than 2 * 255 rows); every 16-row band must really filter
TALL = ("ramp", 999, 24, 8192)
# the loop-filter stress set (tests/test_loopfilter_arms.py), its tall frame last
STRESS = tuple((r, 100 * i + j, *SIZES[(4 * i + j) % len(SIZES)]) for i, r in enumerate(RECIPES) for j in range(4)) + (TALL,)


def compute_has_coeff(a, n):
    """has_coeff as the host token parser defines it (reference vp8_tokens.c:331-339,604): any decoded
    coefficient of the macroblock non-zero. Y2 only counts where it is coded (ymode != B_PRED), and for
    those macroblocks the luma DC slots are never coded."""
    y2 = a["coeff_y2"].reshape(n, 16)
    yy = a["coeff_y"].reshape(n, 16, 16)
    not_b = a["ymode"] != 4
    # keep the arrays consistent with what a bitstream can express
    y2[~not_b] = 0
    yy[not_b, :, 0] = 0
    nz = (y2 != 0).any(1) | (yy != 0).any((1, 2)) | (a["coeff_u"].reshape(n, 64) != 0).any(1) | \
        (a["coeff_v"].reshape(n, 64) != 0).any(1)
    return nz.astype(np.uint8)


def first_difference(f, got, want, padded=False):
    """plane / x / y / macroblock of the first differing byte of an I420 buffer, or of padded (y, u, v) planes."""
    if padded:
        planes = list(zip("yuv", got, want))
    else:
        w, h, cw, ch = f.width, f.height, (f.width + 1) // 2, (f.height + 1) // 2
        cut = lambda b: (b[:w * h].reshape(h, w), b[w * h:w * h + cw * ch].reshape(ch, cw), b[w * h + cw * ch:].reshape(ch, cw))
        planes = list(zip("yuv", cut(got), cut(want)))
    for name, g, wnt in planes:
        bad = np.argwhere(g != wnt)
        if len(bad):
            y, x = (int(v) for v in bad[0])
            mb = 16 if name == "y" else 8
            return f"plane {name} x={x} y={y} macroblock ({x // mb}, {y // mb}): got {g[y, x]} want {wnt[y, x]}"
    return "no difference"


# ---------------------------------------------------------------------------- wavefront kernel shapes
DEFAULT_KERNEL = 3  # what a fresh context runs (vp8_gpu.h: vp8_gpu_set_kernel)

# (kernel, warps, images per SM, CTAs per image, split): set_kernel / set_tuning / set_cluster of a context
SHAPES = [(2, w, 0, 1, False) for w in (4, 8, 16)]  # vp8_mb_pairs<NW, ..., LS=false>
# kernel 3 + 8 warps + images_per_cta == 0 is the 8-warp lockstep-small pairs shape, vp8_mb_pairs<8, ..., LS=true>; no
# field of the launch config reports LS itself
SHAPES += [(3, 8, 0, 1, False)]
# g = 1: vp8_mb_pairs<4>; g >= 2: vp8_mb_lockstep with g images per CTA
SHAPES += [(3, 4, g, 1, False) for g in range(1, 8)]
SHAPES += [(3, 16, 0, c, False) for c in (2, 4, 8)] + [(3, 16, 0, c, True) for c in (4, 8)]


def set_shape(ctx, shape):
    kernel, warps, per_sm, ctas, split = shape
    ctx.set_kernel(kernel)
    ctx.set_tuning(warps, per_sm)
    ctx.set_cluster(ctas, split)


def reset_shape(ctx):
    ctx.set_cluster(0, True)
    ctx.set_tuning(0, 0)
    ctx.set_kernel(DEFAULT_KERNEL)


def expected_launch(shape, staged_filter=False):
    """(warps_per_image, ctas_per_image, split, images_per_cta) that last_launch_config reports for a launch in `shape`
    (the stand-alone filter never runs the split flavour)."""
    kernel, warps, per_sm, ctas, split = shape
    return warps, ctas, split and not staged_filter, per_sm if per_sm >= 2 else 0


def launch_of(cfg):
    return cfg["warps_per_image"], cfg["ctas_per_image"], cfg["split"], cfg["images_per_cta"]


def shape_batches(n, tall, ctas):
    """Index batches of n frames for one shape: all at once, or for clusters batches of up to 7 frames that each hold
    frame `tall` (enough macroblock rows that every CTA of the cluster gets some; at most 7 frames, so that all the
    clusters are resident at once and the planner keeps the cluster size)."""
    if ctas <= 1:
        return [list(range(n))]
    rest = [i for i in range(n) if i != tall]
    return [rest[i:i + 6] + [tall] for i in range(0, len(rest), 6)]


# ---------------------------------------------------------------------------- CPU checkers
def build_oracle():
    subprocess.run(["make", "-s", "-C", str(ORACLE_DIR), "all"], check=True)


class Checker:
    """Common face of the two CPU checkers so tests can parametrise over them."""

    def decode_i420(self, fr: Frame, filtered: bool) -> np.ndarray: ...
    def rgb(self, i420: np.ndarray, w: int, h: int) -> np.ndarray: ...


# orc_loopfilter_census cells (oracle/vp8_oracle.h): one named field per cell block, the labels of each axis below
LF_AXES = {
    "kind": ("mb", "inner", "simple"),
    "dir": ("vert", "horz"),
    "plane": ("y", "uv"),
    "outcome": ("fail_edge", "fail_interior", "no_hev", "hev", "simple"),
    "sat": ("w", "a", "a_round", "clip"),
    "hev_thr": (0, 1, 2),
    "parity": ("even", "odd"),
}
LF_FIELDS = {"outcome": ("kind", "dir", "plane", "outcome"), "sat": ("kind", "sat"), "hev_thr": ("kind", "hev_thr"),
             "parity": ("parity", "outcome")}
LF_CENSUS = np.dtype([(k, np.uint64, tuple(len(LF_AXES[a]) for a in axes)) for k, axes in LF_FIELDS.items()])


def census_sum(censuses):
    """Cell-wise sum of loopfilter_census results."""
    flat = sum(np.asarray(c).reshape(1).view(np.uint64) for c in censuses)
    return flat.view(LF_CENSUS)[0]


class Oracle(Checker):
    """oracle/liboracle.so: our C restatement (or a library built from a copy of its source: so)."""
    name = "oracle"

    def __init__(self, so=None):
        if so is None:
            so = ORACLE_DIR / "liboracle.so"
            if not so.exists():
                build_oracle()
        L = self.lib = C.CDLL(str(so))
        L.orc_decode_i420.argtypes = [C.POINTER(DecodedFrame), C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]
        L.orc_recon_padded.argtypes = [C.POINTER(DecodedFrame)] + [C.c_void_p] * 3
        L.orc_loopfilter_padded.argtypes = [C.POINTER(DecodedFrame)] + [C.c_void_p] * 3
        L.orc_loopfilter_census.argtypes = [C.POINTER(DecodedFrame)] + [C.c_void_p] * 4
        L.orc_loopfilter_census_cells.restype = C.c_size_t
        assert L.orc_loopfilter_census_cells() * 8 == LF_CENSUS.itemsize
        L.orc_i420_to_rgb.argtypes = [C.c_void_p] * 3 + [C.c_uint32] * 4 + [C.c_void_p]
        L.orc_i420_to_rgb.restype = None
        L.orc_ppm.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
        L.orc_ppm.restype = C.c_size_t
        L.orc_png_bound.argtypes = [C.c_uint32, C.c_uint32]
        L.orc_png_bound.restype = C.c_size_t
        L.orc_png.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
        L.orc_png.restype = C.c_size_t
        L.orc_frame_params.argtypes = [C.POINTER(DecodedFrame), C.c_void_p, C.c_void_p]
        L.orc_frame_params.restype = None

    def decode_i420(self, fr, filtered, drop_has_coeff=False):
        out = np.empty(fr.i420_size, np.uint8)
        d = fr.cstruct(drop_has_coeff)
        rc = self.lib.orc_decode_i420(C.byref(d), fr.width, fr.height, int(filtered), out.ctypes.data)
        assert rc == 0
        return out

    def frame_params(self, fr):
        dq, lf = np.zeros((4, 6), np.int16), np.zeros((4, 2, 4), np.uint8)
        d = fr.cstruct()
        self.lib.orc_frame_params(C.byref(d), dq.ctypes.data, lf.ctypes.data)
        return dq, lf

    def recon_padded(self, fr):
        pw, ph = fr.mb_cols * 16, fr.mb_rows * 16
        y, u, v = np.zeros((ph, pw), np.uint8), np.full((ph // 2, pw // 2), 128, np.uint8), np.full((ph // 2, pw // 2), 128, np.uint8)
        d = fr.cstruct()
        assert self.lib.orc_recon_padded(C.byref(d), y.ctypes.data, u.ctypes.data, v.ctypes.data) == 0
        return y, u, v

    def loopfilter_padded(self, fr, y, u, v):
        d = fr.cstruct()
        assert self.lib.orc_loopfilter_padded(C.byref(d), y.ctypes.data, u.ctypes.data, v.ctypes.data) == 0

    def loopfilter_census(self, fr):
        """Counts of the loop filter's arms over one frame (recon_padded, then the filter): a record of dtype LF_CENSUS."""
        y, u, v = self.recon_padded(fr)
        out = np.zeros((), LF_CENSUS)
        d = fr.cstruct()
        assert self.lib.orc_loopfilter_census(C.byref(d), y.ctypes.data, u.ctypes.data, v.ctypes.data, out.ctypes.data) == 0
        return out

    def rgb(self, i420, w, h):
        cw, ch = (w + 1) // 2, (h + 1) // 2
        i420 = np.ascontiguousarray(i420)
        base = i420.ctypes.data
        out = np.empty(w * h * 3, np.uint8)
        self.lib.orc_i420_to_rgb(base, base + w * h, base + w * h + cw * ch, w, h, w, cw, out.ctypes.data)
        return out

    def ppm(self, rgb, w, h):
        out = np.empty(32 + w * h * 3, np.uint8)
        n = self.lib.orc_ppm(np.ascontiguousarray(rgb).ctypes.data, w, h, out.ctypes.data)
        return out[:n].tobytes()

    def png(self, rgb, w, h):
        out = np.empty(self.lib.orc_png_bound(w, h), np.uint8)
        n = self.lib.orc_png(np.ascontiguousarray(rgb).ctypes.data, w, h, out.ctypes.data)
        return out[:n].tobytes()


def _plane(ptr, n):
    return np.ctypeslib.as_array(ptr, shape=(n,)).copy()


class Reference(Checker):
    """oracle/_ref/libref_decode.so: the unmodified reference sources compiled by oracle/Makefile."""
    name = "reference"

    @staticmethod
    def available():
        return (REF_DIR / "libref_decode.so").exists()

    def __init__(self, lib_path=None):
        L = self.lib = C.CDLL(str(lib_path or REF_DIR / "libref_decode.so"))
        for fn in ("vp8_reconstruct_keyframe_yuv", "vp8_reconstruct_keyframe_yuv_filtered"):
            getattr(L, fn).argtypes = [C.POINTER(KeyFrameHeader), C.POINTER(DecodedFrame), C.POINTER(Yuv420Image)]
        L.vp8_loopfilter_apply_keyframe.argtypes = [C.POINTER(Yuv420Image), C.POINTER(DecodedFrame)]
        L.yuv420_free.argtypes = [C.POINTER(Yuv420Image)]
        L.yuv420_free.restype = None
        L.yuv420_write_ppm_fd.argtypes = [C.c_int, C.POINTER(Yuv420Image)]
        L.yuv420_write_png_fd.argtypes = [C.c_int, C.POINTER(Yuv420Image)]
        L.vp8_decode_decoded_frame.argtypes = [ByteSpan, C.POINTER(DecodedFrame)]
        L.vp8_decoded_frame_free.argtypes = [C.POINTER(DecodedFrame)]
        L.vp8_decoded_frame_free.restype = None
        L.vp8_parse_keyframe_header.argtypes = [ByteSpan, C.POINTER(KeyFrameHeader)]

    def decode_i420(self, fr, filtered, drop_has_coeff=False):
        d, h, img = fr.cstruct(drop_has_coeff), fr.header(), Yuv420Image()
        fn = self.lib.vp8_reconstruct_keyframe_yuv_filtered if filtered else self.lib.vp8_reconstruct_keyframe_yuv
        assert fn(C.byref(h), C.byref(d), C.byref(img)) == 0
        cw, ch = (fr.width + 1) // 2, (fr.height + 1) // 2
        out = np.concatenate([_plane(img.y, fr.width * fr.height), _plane(img.u, cw * ch), _plane(img.v, cw * ch)])
        self.lib.yuv420_free(C.byref(img))
        return out

    def loopfilter_padded(self, fr, y, u, v):
        img = Yuv420Image(y.shape[1], y.shape[0], y.shape[1], u.shape[1], y.ctypes.data_as(u8p),
                          u.ctypes.data_as(u8p), v.ctypes.data_as(u8p))
        d = fr.cstruct()
        assert self.lib.vp8_loopfilter_apply_keyframe(C.byref(img), C.byref(d)) == 0

    def _write(self, fn, i420, w, h):
        cw, ch = (w + 1) // 2, (h + 1) // 2
        i420 = np.ascontiguousarray(i420)
        base = i420.ctypes.data
        img = Yuv420Image(w, h, w, cw, C.cast(base, u8p), C.cast(base + w * h, u8p), C.cast(base + w * h + cw * ch, u8p))
        r, wfd = os.pipe()
        import threading
        buf = io.BytesIO()

        def drain():
            with os.fdopen(r, "rb") as fp:
                buf.write(fp.read())
        t = threading.Thread(target=drain)
        t.start()
        rc = fn(wfd, C.byref(img))
        os.close(wfd)
        t.join()
        assert rc == 0
        return buf.getvalue()

    def ppm_bytes(self, i420, w, h):
        return self._write(self.lib.yuv420_write_ppm_fd, i420, w, h)

    def png_bytes(self, i420, w, h):
        return self._write(self.lib.yuv420_write_png_fd, i420, w, h)

    def rgb(self, i420, w, h):
        ppm = self.ppm_bytes(i420, w, h)
        return np.frombuffer(ppm[len(ppm) - w * h * 3:], np.uint8).copy()

    # ---- .webp -> Frame through the reference's own m01..m05 (fixture generation only)
    def parse_webp(self, data: bytes) -> Frame:
        assert data[:4] == b"RIFF" and data[8:16] == b"WEBPVP8 "
        size = int.from_bytes(data[16:20], "little")
        payload = (C.c_uint8 * size).from_buffer_copy(data[20:20 + size])
        span = ByteSpan(C.cast(payload, u8p), size)
        kf, d = KeyFrameHeader(), DecodedFrame()
        assert self.lib.vp8_parse_keyframe_header(span, C.byref(kf)) == 0
        assert self.lib.vp8_decode_decoded_frame(span, C.byref(d)) == 0
        n = d.mb_total
        params = {k: int(getattr(d, k)) for k in SCALARS}
        params.update({k: [int(getattr(d, k)[i]) for i in range(4)] for k in VEC4})
        sizes = dict(segment_id=n, skip_coeff=n, has_coeff=n, ymode=n, uv_mode=n, bmode=n * 16, coeff_y2=n * 16,
                     coeff_y=n * 256, coeff_u=n * 64, coeff_v=n * 64)
        arrays = {k: _plane(getattr(d, k), sizes[k]) for k in U8_ARRAYS + I16_ARRAYS}
        self.lib.vp8_decoded_frame_free(C.byref(d))
        return Frame(kf.width, kf.height, params, arrays)


def sha(b) -> str:
    return hashlib.sha256(bytes(b)).hexdigest()
