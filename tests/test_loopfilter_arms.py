"""The loop filter's arms, reached on purpose.

Whether a filter position is modified, and by which arm, depends on the pixels, and the fuzz frames are mostly dense
random content on which most positions fail the edge or the interior limit. The stress set (vp8fix.stress_frame) is
built recipe by recipe so that every arm of the filter runs many times: both hev outcomes of macroblock and inner edges, the simple
filter, the clamps of w and a, clip255 at 0 and 255, every hev threshold, skipped inner edges next to filtered ones.
- CPU: the oracle's arm census (orc_loopfilter_census) of the set stays above a stated floor in every reachable cell,
  and twelve one-line mutants of the oracle's filter each change some output byte of the set.
- GPU: every wavefront kernel shape decodes the set (fused and stand-alone filter) to the oracle's bytes."""
import shutil
import subprocess

import numpy as np
import pytest

from vp8fix import (LF_AXES, ORACLE_DIR, SHAPES, STRESS, TALL, Oracle, census_sum, expected_launch, first_difference, launch_of,
                    reset_shape, set_shape, shape_batches, stress_frame)


@pytest.fixture(scope="module")
def stress():
    return [stress_frame(*s) for s in STRESS]


# ------------------------------------------------------------------------------------------------------- census floor
# Minimum count of every cell of the census over STRESS, about half of what it measured when the set was made. 0 marks
# a cell no position can reach (no W clamp outside the 27/18/9 arm, no interior test or hev in the simple filter, no
# simple filter on U/V): those must stay 0.
OUTCOME_FLOOR = {"mb": (2000, 700, 4000, 150, 0), "inner": (4000, 400, 6000, 1500, 0), "simple": (1500, 0, 0, 0, 5000)}
SAT_FLOOR = {"mb": (100, 50, 30, 100), "inner": (0, 150, 100, 300), "simple": (0, 20, 15, 100)}
HEV_FLOOR = {"mb": (250, 20000, 10000), "inner": (500, 50000, 25000), "simple": (0, 0, 0)}
PARITY_FLOOR = {"even": (3000, 800, 6000, 2500, 400), "odd": (3000, 800, 6000, 2500, 400)}


def census_rows(census):
    """(cell name, count, floor) for every cell of a census, floors from the tables above."""
    rows = []
    for ki, kind in enumerate(LF_AXES["kind"]):
        for di, d in enumerate(LF_AXES["dir"]):
            for pi, plane in enumerate(LF_AXES["plane"]):
                for oi, o in enumerate(LF_AXES["outcome"]):
                    floor = OUTCOME_FLOOR[kind][oi] if not (kind == "simple" and plane == "uv") else 0
                    rows.append((f"outcome {kind} {d} {plane} {o}", int(census["outcome"][ki, di, pi, oi]), floor))
        for si, s in enumerate(LF_AXES["sat"]):
            rows.append((f"sat {kind} {s}", int(census["sat"][ki, si]), SAT_FLOOR[kind][si]))
        for ti, thr in enumerate(LF_AXES["hev_thr"]):
            rows.append((f"hev_thr {kind} {thr}", int(census["hev_thr"][ki, ti]), HEV_FLOOR[kind][ti]))
    for pi, par in enumerate(LF_AXES["parity"]):
        for oi, o in enumerate(LF_AXES["outcome"]):
            rows.append((f"mb-row top edge {par} {o}", int(census["parity"][pi, oi]), PARITY_FLOOR[par][oi]))
    return rows


def census_table(census) -> str:
    return "\n".join(f"{name:40s} {count:10d}  floor {floor}" for name, count, floor in census_rows(census))


def test_census_of_the_stress_set_reaches_every_arm(oracle, stress):
    census = census_sum(oracle.loopfilter_census(f) for f in stress)
    low = [(name, count, floor) for name, count, floor in census_rows(census) if count < floor or (floor == 0 and count)]
    assert not low, f"cells below their floor (or unreachable cells counted): {low}\n{census_table(census)}"


def test_census_counts_every_position_once(oracle, stress):
    """One outcome per filter position: the count of positions follows from the macroblock levels and edges alone."""
    for f in stress:
        _, lf = oracle.frame_params(f)
        cols, rows = f.mb_cols, f.mb_rows
        seg = f.arrays["segment_id"] & 3 if f.params["segmentation_enabled"] else np.zeros(f.mb_total, np.uint8)
        bpred = f.arrays["ymode"] == 4
        level = lf[seg, bpred.astype(int), 0].reshape(rows, cols)
        inner = ((f.arrays["has_coeff"] != 0) | bpred).reshape(rows, cols)
        left = np.arange(cols)[None, :] > 0
        top = np.arange(rows)[:, None] > 0
        # per macroblock edge: 16 positions of Y (+ 2 x 8 of U/V); per direction of inner edges: 3 x 16 of Y (+ 2 x 8)
        simple = f.params["lf_use_simple"]
        per_edge, per_inner = (16, 48) if simple else (32, 64)
        want = int(((level > 0) * (per_edge * (left.astype(int) + top) + 2 * per_inner * inner)).sum())
        census = oracle.loopfilter_census(f)
        assert int(census["outcome"].sum()) == want, (f.width, f.height)
        assert int(census["parity"].sum()) == int(((level > 0) * per_edge * top).sum())


def test_tall_frame_filters_every_band(oracle, stress):
    """The tall frame gives the deep CTAs of a cluster filtered rows: every band of 16 macroblock rows changes."""
    f = stress[-1]
    assert (f.width, f.height) == TALL[2:] and f.mb_rows > 256
    y0 = oracle.decode_i420(f, False)[:f.width * f.height].reshape(f.height, f.width)
    y1 = oracle.decode_i420(f, True)[:f.width * f.height].reshape(f.height, f.width)
    bands = [b for b in range(0, f.height, 256) if np.array_equal(y0[b:b + 256], y1[b:b + 256])]
    assert not bands, f"unfiltered bands starting at pixel rows {bands}"


# ------------------------------------------------------------------------------------------------------------ mutants
# One textual change each to oracle/vp8_oracle.c's loop filter: (anchor, replacement). Every anchor occurs exactly once,
# so an edit of the oracle that moves one fails here loudly instead of testing nothing.
_INTERIOR = ("if (iabs(p3 - p2) > interior || iabs(p2 - p1) > interior || iabs(p1 - p0) > interior ||\n"
             "\t\t    iabs(q3 - q2) > interior || iabs(q2 - q1) > interior || iabs(q1 - q0) > interior)")
MUTANTS = {
    "edge limit > to >=": ("(iabs(p1 - q1) >> 1) > lim)", "(iabs(p1 - q1) >> 1) >= lim)"),
    "interior > to >=": (_INTERIOR, _INTERIOR.replace("> interior", ">= interior")),
    "hev > to >=": ("hev = iabs(p1 - p0) > hev_thr || iabs(q1 - q0) > hev_thr;",
                    "hev = iabs(p1 - p0) >= hev_thr || iabs(q1 - q0) >= hev_thr;"),
    "27 * w + 64": ("(27 * w + 63)", "(27 * w + 64)"),
    "third tap c = 0": ("c = (9 * w + 63) >> 7", "c = 0"),
    "a + 4 unclamped": ("sclamp(a + 4)", "(a + 4)"),
    "f1 >> 1 for (f1 + 1) >> 1": ("(f1 + 1) >> 1", "f1 >> 1"),
    "outer ignores hev": ("int outer = (kind != EDGE_INNER) || hev;", "int outer = (kind != EDGE_INNER);"),
    "hev threshold lvl > 15": ("(lvl >= 15) + (lvl >= 40)", "(lvl > 15) + (lvl >= 40)"),
    "sharpness shift >= 4": ("(f->lf_sharpness > 4) ? 2 : 1", "(f->lf_sharpness >= 4) ? 2 : 1"),
    "B_PRED does not force inner edges": ("(f->has_coeff && f->has_coeff[mb]) || f->ymode[mb] == 4;",
                                          "(f->has_coeff && f->has_coeff[mb]);"),
    "MB arm p2 + c truncated": ("clip255_n(p2 + c, &clips)", "(uint8_t)(p2 + c)"),
}


def test_every_filter_mutant_changes_the_stress_set(oracle, stress, tmp_path):
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("no g++")
    src = (ORACLE_DIR / "vp8_oracle.c").read_text()
    builds = {}
    for i, (name, (anchor, repl)) in enumerate(MUTANTS.items()):
        assert src.count(anchor) == 1, f"mutant {name!r}: its anchor occurs {src.count(anchor)} times in vp8_oracle.c"
        c = tmp_path / f"m{i}.c"
        c.write_text(src.replace(anchor, repl))
        builds[name] = subprocess.Popen([gxx, "-x", "c", "-std=c11", "-O1", "-shared", "-fPIC", "-I", str(ORACLE_DIR),
                                         "-o", str(tmp_path / f"m{i}.so"), str(c)])
    mutants = {}
    for i, (name, proc) in enumerate(builds.items()):
        assert proc.wait() == 0, name
        mutants[name] = Oracle(tmp_path / f"m{i}.so")
    changed = dict.fromkeys(MUTANTS, 0)
    for f in stress:
        recon = oracle.recon_padded(f)
        want = [p.copy() for p in recon]
        oracle.loopfilter_padded(f, *want)
        for name, m in mutants.items():
            got = [p.copy() for p in recon]
            m.loopfilter_padded(f, *got)
            changed[name] += sum(int((g != w).sum()) for g, w in zip(got, want))
    survivors = [name for name, n in changed.items() if n == 0]
    assert not survivors, f"mutants the stress set does not tell from the oracle: {survivors} (bytes changed: {changed})"


# ---------------------------------------------------------------------------------------- GPU: every wavefront shape
@pytest.fixture(scope="module")
def oracle_out(oracle, stress):
    """The oracle's I420 (unfiltered, filtered) and padded planes (reconstructed + filtered) of every stress frame."""
    out = []
    for f in stress:
        planes = oracle.recon_padded(f)
        oracle.loopfilter_padded(f, *planes)
        out.append({False: oracle.decode_i420(f, False), True: oracle.decode_i420(f, True), "padded": planes})
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,warps,per_sm,ctas,split", SHAPES)
def test_every_wavefront_shape_on_the_stress_set(gpu_ctx, stress, oracle_out, kernel, warps, per_sm, ctas, split):
    """Fused recon + filter (filtered and not) and the staged recon() -> filter() in one launch shape, against the oracle.
    Clusters run in batches of up to 7 frames that each hold the tall frame, so that they stay clusters (as many as are
    resident at once) and every CTA of a cluster gets filtered rows."""
    shape = (kernel, warps, per_sm, ctas, split)
    set_shape(gpu_ctx, shape)
    try:
        for batch in shape_batches(len(stress), len(stress) - 1, ctas):
            frames = [stress[i] for i in batch]
            kfs, ds = [f.header() for f in frames], [f.cstruct() for f in frames]
            for filtered in (False, True):
                outs = gpu_ctx.decode_i420(kfs, ds, filtered=filtered)
                cfg = gpu_ctx.last_launch_config()
                assert launch_of(cfg) == expected_launch(shape), (shape, cfg)
                for i, f, o in zip(batch, frames, outs):
                    want = oracle_out[i][filtered]
                    assert np.array_equal(o, want), (f"shape {shape} filtered={filtered} recipe {STRESS[i][0]} "
                                                     f"{f.width}x{f.height}: {first_difference(f, o, want)}")
            # staged: reconstruction, then the stand-alone filter (VP8_K_FILTER), which never runs the split flavour
            b = gpu_ctx.recon(kfs, ds)
            try:
                gpu_ctx.filter(b)
                cfg = gpu_ctx.last_launch_config()
                assert launch_of(cfg) == expected_launch(shape, staged_filter=True), (shape, cfg)
                for k, (i, f) in enumerate(zip(batch, frames)):
                    got, want = gpu_ctx.download_padded(b, k), oracle_out[i]["padded"]
                    assert all(np.array_equal(g, w) for g, w in zip(got, want)), (
                        f"shape {shape} staged filter recipe {STRESS[i][0]} {f.width}x{f.height}: "
                        f"{first_difference(f, got, want, padded=True)}")
            finally:
                b.free()
    finally:
        reset_shape(gpu_ctx)
