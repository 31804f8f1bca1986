"""Writes tests/golden/alpha/*.webp and tests/golden/alpha.json: lossy WebP files with alpha (VP8X + ALPH + 'VP8 '), with the
sha256 of what libwebp (through Pillow) decodes them to - the RGBA as a dwebp -pam file, and the alpha plane - plus each
file's ALPH filter and compression. Also the 1080p ALPH payloads tools/alpha_bench.py wraps around bench_data/ (one per
filter). Seeded: running it again gives the same files. Needs Pillow built with libwebp; the tests that read the result do not.

    python tools/make_alpha_fixtures.py
"""
from __future__ import annotations

import hashlib
import io
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tests"))
import alphafix as A  # noqa: E402

OUT = ROOT / "tests" / "golden" / "alpha"


def sha(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


def pillow_rgba_file(rgb, a, quality, alpha_quality) -> bytes:
    from PIL import Image
    buf = io.BytesIO()
    Image.fromarray(np.dstack([rgb, a]), "RGBA").save(buf, "WEBP", quality=quality, alpha_quality=alpha_quality, method=4)
    return buf.getvalue()


def main():
    OUT.mkdir(parents=True, exist_ok=True)
    for old in OUT.glob("*"):
        old.unlink()
    files = {}

    def add(name, data):
        files[name] = data

    # every filter x compression, two sizes and contents
    for (w, h, kind) in ((37, 23, "mixed"), (129, 129, "ramp")):
        vp8 = A.vp8_chunk_of(A.picture(w, h, w))
        a = A.alpha_content(kind, w, h, w * h)
        for m in range(4):
            for comp in (0, 1):
                add(f"grid_{w}x{h}_{kind}_f{m}_c{comp}", A.wrap(vp8, w, h, A.alph_payload(a, m, comp)))
    # Pillow's own RGBA files at two alpha qualities (below 100 sets the pre-processing bit)
    for (w, h, kind) in ((37, 23, "mixed"), (129, 129, "noise"), (200, 120, "ramp")):
        rgb, a = A.picture(w, h, 7), A.alpha_content(kind, w, h, 11)
        for aq in (100, 50):
            add(f"pillow_{w}x{h}_{kind}_aq{aq}", pillow_rgba_file(rgb, a, 80, aq))
    # contents that drive different VP8L tools, each through the gradient filter and unfiltered
    w, h = 15, 70
    vp8 = A.vp8_chunk_of(A.picture(w, h, 3))
    for kind in ("const", "levels", "ramp", "noise", "runs"):
        for m in (0, 3):
            add(f"content_{w}x{h}_{kind}_f{m}_c1", A.wrap(vp8, w, h, A.alph_payload(A.alpha_content(kind, w, h, 5), m, 1)))
    # sizes: tiny, odd chroma, warp and band edges, a wide one, big ones
    for (w, h, kind, m, comp) in ((1, 1, "noise", 3, 1), (1, 1, "noise", 1, 0), (2, 3, "ramp", 3, 1), (2, 3, "noise", 2, 0),
                                  (129, 129, "mixed", 3, 1), (1, 2000, "ramp", 2, 1), (1, 2000, "noise", 3, 0), (4000, 3, "runs", 3, 1),
                                  (4000, 3, "mixed", 1, 0), (33, 65, "noise", 3, 0), (1000, 700, "levels", 3, 1),
                                  (1000, 700, "ramp", 1, 1), (1920, 1080, "runs", 3, 1)):
        vp8 = A.vp8_chunk_of(A.picture(w, h, 9, noise=2 if w * h > 100000 else 12), 60 if w * h > 100000 else 80)
        add(f"size_{w}x{h}_{kind}_f{m}_c{comp}", A.wrap(vp8, w, h, A.alph_payload(A.alpha_content(kind, w, h, w + h), m, comp)))
    # containers without an ALPH chunk: metadata chunks only, and the alpha flag set with no ALPH
    w, h = 37, 23
    vp8 = A.vp8_chunk_of(A.picture(w, h, 4))
    add("vp8x_iccp_exif_noalpha", A.wrap(vp8, w, h, None, extra_before=[(b"ICCP", b"\0" * 13)], extra_after=[(b"EXIF", b"Exif\0\0x"), (b"XMP ", b"<x/>")]))
    add("vp8x_flag_without_alph", A.wrap(vp8, w, h, None, alpha_flag=True))
    add("vp8x_unknown_chunks", A.wrap(vp8, w, h, A.alph_payload(A.alpha_content("ramp", w, h, 1), 3, 1),
                                      extra_before=[(b"ABCD", b"123")], extra_after=[(b"WXYZ", b"")]))

    meta = {}
    for name, data in sorted(files.items()):
        (OUT / f"{name}.webp").write_bytes(data)
        rgba = A.pillow_rgba(data)
        alph = [d for t, d in A.chunks(data) if t == b"ALPH"]
        h, w = rgba.shape[:2]
        meta[name + ".webp"] = {
            "width": w, "height": h,
            "pam": sha(A.pam(rgba)),
            "alpha": sha(np.ascontiguousarray(rgba[..., 3]).tobytes()) if alph else None,
            "filter": (alph[0][0] >> 2) & 3 if alph else None,
            "compression": alph[0][0] & 3 if alph else None,
            "preprocessing": (alph[0][0] >> 4) & 3 if alph else None,
        }
    # the benchmark's ALPH payloads (1080p, VP8L, one per filter)
    a = A.alpha_content("mixed", 1920, 1080, 2024)
    for m in range(4):
        (OUT / f"bench_alph_1920x1080_f{m}.bin").write_bytes(A.alph_payload(a, m, 1))
    meta["bench_alph_1920x1080"] = {"alpha": sha(a.tobytes())}
    (ROOT / "tests" / "golden" / "alpha.json").write_text(json.dumps(meta, indent=1, sort_keys=True) + "\n")
    total = sum(p.stat().st_size for p in OUT.iterdir())
    print(f"{len(files)} files + 4 bench payloads, {total / 1e6:.2f} MB in {OUT}")


if __name__ == "__main__":
    main()
