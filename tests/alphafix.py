"""Lossy WebP files with alpha for the tests: the extended container (VP8X + ALPH + 'VP8 ', RFC 9649), the alpha filters
written plainly in numpy, and seeded picture / alpha contents. Pillow (libwebp) encodes the colour and the VP8L payloads
and is the judge of what a file decodes to; it is only needed where fixtures are made (tools/make_alpha_fixtures.py) or
where a test makes fresh ones."""
from __future__ import annotations

import io
import struct

import numpy as np

FILTERS = ("none", "horizontal", "vertical", "gradient")


def chunks(data: bytes):
    """[(tag, payload)] of a RIFF/WEBP file."""
    assert data[:4] == b"RIFF" and data[8:12] == b"WEBP"
    out, p = [], 12
    while p + 8 <= len(data):
        tag, n = data[p:p + 4], struct.unpack("<I", data[p + 4:p + 8])[0]
        out.append((tag, data[p + 8:p + 8 + n]))
        p += 8 + n + (n & 1)
    return out


def chunk(tag: bytes, payload: bytes) -> bytes:
    return tag + struct.pack("<I", len(payload)) + payload + (b"\0" if len(payload) & 1 else b"")


def riff(body: bytes) -> bytes:
    return b"RIFF" + struct.pack("<I", len(body) + 4) + b"WEBP" + body


def vp8x(w: int, h: int, alpha: bool = True, flags: int = 0) -> bytes:
    return chunk(b"VP8X", bytes([(0x10 if alpha else 0) | flags, 0, 0, 0]) + (w - 1).to_bytes(3, "little") + (h - 1).to_bytes(3, "little"))


def wrap(vp8: bytes, w: int, h: int, alph: bytes | None, extra_before=(), extra_after=(), alpha_flag: bool | None = None) -> bytes:
    """VP8X [+ extra chunks] [+ ALPH] + 'VP8 ' [+ trailing chunks]."""
    body = vp8x(w, h, alph is not None if alpha_flag is None else alpha_flag)
    body += b"".join(chunk(t, d) for t, d in extra_before)
    if alph is not None:
        body += chunk(b"ALPH", alph)
    body += chunk(b"VP8 ", vp8) + b"".join(chunk(t, d) for t, d in extra_after)
    return riff(body)


def filter_plane(a: np.ndarray, method: int) -> np.ndarray:
    """The encoder side of the ALPH filters: F = A - pred mod 256 (pred as in vp8_alpha.cuh)."""
    a = a.astype(np.int32)
    h, w = a.shape
    pred = np.zeros_like(a)
    if method == 0:
        return a.astype(np.uint8)
    pred[0, 1:] = a[0, :-1]
    if h > 1:
        pred[1:, 0] = a[:-1, 0]
        if method == 1:
            pred[1:, 1:] = a[1:, :-1]
        elif method == 2:
            pred[1:, :] = a[:-1, :]
        else:
            pred[1:, 1:] = np.clip(a[1:, :-1] + a[:-1, 1:] - a[:-1, :-1], 0, 255)
    return ((a - pred) & 255).astype(np.uint8)


def unfilter_plane(f: np.ndarray, method: int) -> np.ndarray:
    """Plain row-by-row inverse (slow; small planes only)."""
    a = f.astype(np.int32).copy()
    h, w = a.shape
    for y in range(h):
        for x in range(w):
            if method == 0:
                p = 0
            elif y == 0:
                p = a[0, x - 1] if x else 0
            elif x == 0 or method == 2:
                p = a[y - 1, x]
            elif method == 1:
                p = a[y, x - 1]
            else:
                p = min(255, max(0, a[y, x - 1] + a[y - 1, x] - a[y - 1, x - 1]))
            a[y, x] = (a[y, x] + p) & 255
    return a.astype(np.uint8)


def alpha_content(kind: str, w: int, h: int, seed: int) -> np.ndarray:
    """Alpha planes that drive different VP8L tools."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    if kind == "const":
        return np.full((h, w), 200, np.uint8)
    if kind == "levels":  # <= 16 levels: colour indexing with pixel bundling
        return (((xx // 5 + yy // 3) % 4) * 85).astype(np.uint8)
    if kind == "ramp":  # smooth: the predictor transform
        return ((xx * 3 + yy * 2) % 256).astype(np.uint8)
    if kind == "noise":
        return rng.integers(0, 256, (h, w), dtype=np.uint8)
    if kind == "runs":  # long runs and repeats: LZ77 and the colour cache
        row = rng.integers(0, 256, (w,), dtype=np.uint8)
        a = np.repeat(row[None, :], h, 0)
        a[:, w // 3:w // 2] = 0
        a[h // 2:, :] = np.roll(a[h // 2:, :], 7, axis=1)
        return a
    if kind == "mixed":
        a = ((xx * 7 + yy * 5) % 256).astype(np.uint8)
        a[h // 4:h // 2, w // 8:w // 2] = rng.integers(0, 256, (h // 2 - h // 4, w // 2 - w // 8), dtype=np.uint8)
        return a
    raise KeyError(kind)


def picture(w: int, h: int, seed: int, noise: int = 12) -> np.ndarray:
    rng = np.random.default_rng(1000 + seed)
    yy, xx = np.mgrid[0:h, 0:w]
    rgb = np.stack([(xx * 255 // max(w - 1, 1)), (yy * 255 // max(h - 1, 1)), ((xx + yy) % 64) * 4], -1).astype(np.int32)
    rgb += rng.integers(-noise, noise + 1, rgb.shape)
    return np.clip(rgb, 0, 255).astype(np.uint8)


# ---------------------------------------------------------------------------------------------------- needs Pillow
def vp8_chunk_of(rgb: np.ndarray, quality: int = 80) -> bytes:
    from PIL import Image
    buf = io.BytesIO()
    Image.fromarray(rgb, "RGB").save(buf, "WEBP", quality=quality)
    return [d for t, d in chunks(buf.getvalue()) if t == b"VP8 "][0]


def vp8l_payload(plane: np.ndarray) -> bytes:
    """The VP8L image stream (without its 5-byte header) of an image whose green channel is `plane`."""
    from PIL import Image
    g = np.zeros(plane.shape + (3,), np.uint8)
    g[..., 1] = plane
    buf = io.BytesIO()
    Image.fromarray(g, "RGB").save(buf, "WEBP", lossless=True)
    vl = [d for t, d in chunks(buf.getvalue()) if t == b"VP8L"][0]
    return vl[5:]


def alph_payload(a: np.ndarray, method: int, compression: int) -> bytes:
    f = filter_plane(a, method)
    body = f.tobytes() if compression == 0 else vp8l_payload(f)
    return bytes([(method << 2) | compression]) + body


def make_file(rgb: np.ndarray, a: np.ndarray, method: int, compression: int, quality: int = 80) -> bytes:
    h, w = a.shape
    return wrap(vp8_chunk_of(rgb, quality), w, h, alph_payload(a, method, compression))


def pillow_rgba(data: bytes) -> np.ndarray:
    from PIL import Image
    return np.asarray(Image.open(io.BytesIO(data)).convert("RGBA"))


def pam(rgba: np.ndarray) -> bytes:
    """dwebp -pam: the header, then RGBA."""
    h, w = rgba.shape[:2]
    return f"P7\nWIDTH {w}\nHEIGHT {h}\nDEPTH 4\nMAXVAL 255\nTUPLTYPE RGB_ALPHA\nENDHDR\n".encode() + np.ascontiguousarray(rgba, np.uint8).tobytes()
