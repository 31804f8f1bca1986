#!/usr/bin/env python
"""Writes tests/golden/ref_checks.json: sha256 digests of what the original decoder and encoder compute in the tests that call
them directly (oracle/_ref, built by `make -C oracle ref REF=<checkout of the original>`), so that those tests compare with
the original on machines where it is not built:

  library   per seed of tests/test_oracle.py::test_oracle_vs_reference_library: -yuv, -yuvf, -yuvf without has_coeff, -ppm,
            -png and the stand-alone loop filter on padded planes
  rgb, png  tests/test_oracle.py::test_rgb_closed_form_on_tiny_and_odd_sizes / test_png_block_boundaries
  parser    per golden input: one digest over every field of the m05 output
            (tests/test_host.py::test_parser_matches_reference_m05_on_golden_inputs)
  encoder   per case of tests/test_enc.py::test_oracle_matches_reference_encoder_library: qindex and digest

    python tools/make_ref_checks.py                 from the original (oracle/_ref must be built)
    python tools/make_ref_checks.py --from-oracle   from what the tests compare with it (the oracle, the product parser);
                                                    only where the original cannot be built. "source" in the file says which.
"""
from __future__ import annotations

import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]

from encfix import EncOracle, EncReference, cases, picture  # noqa: E402
from vp8fix import GOLDEN, Oracle, Reference, sha  # noqa: E402
import test_enc  # noqa: E402
import test_host  # noqa: E402
import test_oracle  # noqa: E402

SOURCES = {
    "original": "the original decoder and encoder (oracle/_ref, built from their unmodified sources)",
    "oracle": "oracle/liboracle.so and the product parser, recorded where the original could not be built; these tests had "
              "compared them with the original bit for bit. Regenerate from the original when it is at hand",
}


def main():
    from_oracle = "--from-oracle" in sys.argv
    if not from_oracle and not (Reference.available() and EncReference.available()):
        sys.exit("oracle/_ref is not built: run `make -C oracle ref REF=<checkout of the original>` (or pass --from-oracle)")
    oracle = Oracle()
    ref = oracle if from_oracle else Reference()
    enc = EncOracle() if from_oracle else EncReference()
    out = {"source": SOURCES["oracle" if from_oracle else "original"]}
    out["library"] = {str(s): test_oracle.library_outputs(ref, oracle, test_oracle.library_case(s)) for s in range(60)}
    out["rgb"] = {k: sha(ref.rgb(i420, w, h)) for k, w, h, i420 in test_oracle.rgb_cases()}
    png = (lambda i420, w, h: oracle.png(oracle.rgb(i420, w, h), w, h)) if from_oracle else ref.png_bytes
    out["png"] = {k: sha(png(i420, w, h)) for k, w, h, i420 in test_oracle.png_cases()}

    golden = json.loads((GOLDEN / "digests.json").read_text())
    names = sorted(golden)
    datas = [(GOLDEN / "webp" / n).read_bytes() for n in names]
    if from_oracle:
        import webp_decoder_b200  # noqa: F401  (the in-tree library; only its host parser runs here)
        from webp_decoder_b200 import parse as P
        pf = P.parse_batch(datas)
        out["parser"] = {n: test_host.fields_digest(test_host.parsed_fields(pf.kfs[i], pf.frames[i], pf, i)) for i, n in enumerate(names)}
    else:
        out["parser"] = {n: test_host.fields_digest(test_host.reference_fields(ref.parse_webp(d))) for n, d in zip(names, datas)}

    out["encoder"] = {}
    for seed, w, h, kind, q in cases(40, seed0=5000):
        y, u, v = picture(seed, w, h, kind)
        for s in (0, 1, "bpred"):
            r = enc.run(y, u, v, q, s)
            out["encoder"][test_enc.library_key(seed, w, h, kind, q, s)] = {"qindex": int(r["qindex"]), "digest": test_enc.key_digest(r, s)}
    (GOLDEN / "ref_checks.json").write_text(json.dumps(out, indent=0, sort_keys=True))
    print({k: len(v) for k, v in out.items() if isinstance(v, dict)}, out["source"][:40])


if __name__ == "__main__":
    main()
