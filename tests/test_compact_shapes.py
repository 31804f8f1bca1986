"""The compact transport, in every wavefront kernel shape, on frames built for their block-presence masks.

A compact frame (vp8_parse_internal.h) hands the kernels a 25-bit presence mask and a first-block index per macroblock.
Each of the 13 lane roles of a half-warp fetches its one or two blocks through them (fetch_compact, vp8_pairs.cu), and
which blocks arrived gates the WHT and every IDCT. The mask-edge set below is built recipe by recipe so that every
role sees each of its presence patterns. It also holds Y2-only and AC-without-Y2 macroblocks, single blocks at the ends
of each plane's bit range, full macroblocks next to empty ones at row starts and ends, data the pixel path must ignore,
and frames whose blocks span many 64 KiB granules.
- CPU: a mask census of the set stays above stated floors. The shared-arena parse of the host front end stops writing
  when its capacity runs out (tests/native/parse_arena_check.cpp).
- GPU: every shape decodes through every compact producer, filtered and not, to the oracle's (or the reference
  decoder's) bytes. The producers are host compaction of dense frames, the parser's compact frames, and one launch that
  mixes dense pass-through frames with compacted ones. Each call is a single launch in the requested shape."""
import json
import shutil
import subprocess

import numpy as np
import pytest

from vp8fix import (GOLDEN, I16_ARRAYS, ROOT, SCALARS, SHAPES, STRESS, U8_ARRAYS, VEC4, Frame, compute_has_coeff, default_params,
                    expected_launch, first_difference, launch_of, reset_shape, set_shape, shape_batches, sha,
                    stress_frame)

GRANULE = 64 << 10  # vp8c::kGranule
# lane role -> (mask bit of its first block, blocks): luma pairs 2h, 2h+1; U 16..19 and V 20..23 in pairs; Y2 alone
LANE_BITS = [(2 * h, 2) for h in range(8)] + [(16, 2), (18, 2), (20, 2), (22, 2), (24, 1)]


# ------------------------------------------------------------------------------------------------- mask-edge frames
def _nonzero(rng, shape, amp):
    return (rng.integers(1, amp + 1, shape) * rng.choice([-1, 1], shape)).astype(np.int16)


def mask_frame(recipe: str, seed: int, width: int, height: int) -> Frame:
    """A frame whose blocks are present (some coefficient non-zero) or absent by recipe; presence is what host compaction
    turns into the mask. Present blocks carry a random sparse residual with at least one coefficient that counts (an AC
    term for luma, so that i16 macroblocks keep it)."""
    rng = np.random.default_rng(seed)
    cols, rows = (width + 15) // 16, (height + 15) // 16
    n = cols * rows
    p = default_params(q_index=int(rng.integers(0, 128)), lf_level=int(rng.integers(0, 64)), lf_sharpness=int(rng.integers(0, 8)),
                       lf_use_simple=int(rng.random() < 0.25))
    ymode = np.where(rng.random(n) < 0.3, 4, rng.integers(0, 4, n)).astype(np.uint8)
    i16 = lambda: rng.integers(0, 4, n).astype(np.uint8)
    present = np.zeros((n, 25), bool)
    dc_only = np.zeros((n, 16), bool)  # raw: luma blocks of i16 macroblocks whose only coefficient is the (ignored) DC
    raw = False
    if recipe == "lanes":      # every role with each presence pattern: none, first only, second only, both
        for b0, w in LANE_BITS:
            nz = rng.integers(0, 2 * w, n)
            present[:, b0] = nz & 1
            if w == 2:
                present[:, b0 + 1] = nz >> 1
        present[rng.random(n) < 0.1] = False
    elif recipe == "y2only":   # i16 with nothing but Y2: every luma DC comes from the WHT, every luma lane has nz = 0
        ymode = i16()
        present[:, 24] = rng.random(n) < 0.85
    elif recipe == "acnoy2":   # i16 whose luma blocks hold AC terms but whose Y2 is absent: the WHT gets nothing
        ymode = i16()
        present[:, :16] = rng.random((n, 16)) < 0.6
        present[:, 16:24] = rng.random((n, 8)) < 0.3
    elif recipe == "single":   # one block per macroblock, mostly at the ends of each plane's bit range
        bit = np.where(rng.random(n) < 0.8, rng.choice([0, 15, 16, 23, 24], n), rng.integers(0, 25, n))
        present[np.arange(n), bit] = True
        present[rng.random(n) < 0.15] = False
        ymode[bit == 24] = i16()[bit == 24]
    elif recipe == "rowedges": # all 25 blocks at the first and last column of a row, empty neighbours; odd rows shifted in by one
        full = np.zeros((rows, cols), bool)
        inset = 1 if cols >= 3 else 0
        full[0::2, [0, -1]] = True
        full[1::2, [inset, cols - 1 - inset]] = True
        full = full.reshape(-1)
        present[full] = True
        ymode[full] = i16()[full]
    elif recipe == "raw":      # not expressible by a bitstream: Y2 at B_PRED, lone luma DC at i16, has_coeff at random
        raw = True
        present = rng.random((n, 25)) < 0.4
        dc_only = (ymode != 4)[:, None] & present[:, :16] & (rng.random((n, 16)) < 0.5)
    elif recipe == "dense":    # every block present: packed blocks span several granules
        present[:] = True
    else:
        raise ValueError(recipe)
    if not raw:
        present[ymode == 4, 24] = False
    amp = int(rng.choice([6, 40, 300]))
    dens = float(rng.choice([0.05, 0.3]))

    def blocks(count, first_pos):
        c = rng.integers(-amp, amp + 1, (n, count, 16)).astype(np.int16) * (rng.random((n, count, 16)) < dens)
        pos = rng.integers(first_pos, 16, (n, count))
        np.put_along_axis(c, pos[..., None], _nonzero(rng, (n, count, 1), amp), axis=2)
        return c

    yy, uu, vv, y2 = blocks(16, 1), blocks(4, 0), blocks(4, 0), blocks(1, 0)[:, 0]
    if recipe == "y2only":
        y2[rng.random(n) < 0.7, 1:] = 0  # mostly DC only: the override without any AC term
    yy[dc_only] = 0
    yy[dc_only, 0] = _nonzero(rng, int(dc_only.sum()), amp)
    yy[~present[:, :16]] = 0
    uu[~present[:, 16:20]] = 0
    vv[~present[:, 20:24]] = 0
    y2[~present[:, 24]] = 0
    a = {
        "segment_id": rng.integers(0, 4, n).astype(np.uint8),
        "skip_coeff": np.zeros(n, np.uint8),
        "ymode": ymode,
        "uv_mode": rng.integers(0, 4, n).astype(np.uint8),
        "bmode": rng.integers(0, 10, n * 16).astype(np.uint8),
        "coeff_y": yy.reshape(-1), "coeff_u": uu.reshape(-1), "coeff_v": vv.reshape(-1), "coeff_y2": y2.reshape(-1),
    }
    a["has_coeff"] = rng.integers(0, 2, n).astype(np.uint8) if raw else compute_has_coeff(a, n)
    return Frame(width, height, p, a)


MASK_SET = (("lanes", 1, 160, 96), ("lanes", 2, 100, 72), ("lanes", 3, 16, 200), ("lanes", 4, 9, 130), ("lanes", 5, 300, 16),
            ("y2only", 11, 200, 12), ("y2only", 12, 96, 400), ("y2only", 13, 17, 33),
            ("acnoy2", 21, 100, 72), ("acnoy2", 22, 1, 1), ("acnoy2", 23, 48, 200),
            ("single", 31, 160, 320), ("single", 32, 16, 16), ("single", 33, 9, 130), ("single", 34, 300, 16),
            ("rowedges", 41, 160, 96), ("rowedges", 42, 33, 300), ("rowedges", 43, 48, 400), ("rowedges", 44, 1040, 40),
            ("rowedges", 45, 40, 1),
            ("raw", 51, 160, 240), ("raw", 52, 100, 72), ("raw", 53, 16, 200),
            ("dense", 61, 1040, 48), ("dense", 62, 333, 100),
            ("lanes", 99, 24, 8192))  # 512 macroblock rows, last: the frame that gives every CTA of a cluster rows
# the widest frame a bitstream can carry (1024 macroblock columns), every block present: 13 granules per row
WIDE = ("dense", 71, 16383, 33)


def block_masks(f: Frame) -> np.ndarray:
    """Per macroblock: bit b set when block b has a non-zero coefficient - the mask host compaction packs."""
    n = f.mb_total
    nz = np.concatenate([(f.arrays["coeff_y"].reshape(n, 16, 16) != 0).any(2), (f.arrays["coeff_u"].reshape(n, 4, 16) != 0).any(2),
                         (f.arrays["coeff_v"].reshape(n, 4, 16) != 0).any(2), (f.arrays["coeff_y2"].reshape(n, 1, 16) != 0).any(2)], 1)
    return (nz.astype(np.uint32) << np.arange(25, dtype=np.uint32)).sum(1, dtype=np.uint32)


def granules(masks) -> int:
    """64 KiB granules one frame's packed blocks take (compact_frame: a new one when fewer than 800 bytes are left)."""
    count, left = 0, 0
    for m in masks:
        if left < 800:
            count, left = count + 1, GRANULE
        left -= 32 * bin(int(m)).count("1")
    return count


def mask_census(frames):
    """role x nz (nz = which of the lane's blocks are present: 0, 1 first, 2 second, 3 both), macroblocks by block count
    (0, 1, 24, 25, other), frames by granules (1, 2, 3..9, 10+) and the edge cases the recipes aim at."""
    c = {"role": np.zeros((13, 4), np.int64), "blocks": dict.fromkeys((0, 1, 24, 25, "other"), 0),
         "granules": dict.fromkeys(("1", "2", "3-9", "10+"), 0), "edge": {}}
    edge = c["edge"]

    def add(name, k):
        edge[name] = edge.get(name, 0) + int(k)

    for f in frames:
        m = block_masks(f)
        for r, (b0, w) in enumerate(LANE_BITS):
            c["role"][r] += np.bincount((m >> b0) & (2 ** w - 1), minlength=4)
        pc = np.array([bin(int(x)).count("1") for x in m])
        for k in (0, 1, 24, 25):
            c["blocks"][k] += int((pc == k).sum())
        c["blocks"]["other"] += int((~np.isin(pc, (0, 1, 24, 25))).sum())
        g = granules(m)
        c["granules"]["1" if g == 1 else "2" if g == 2 else "3-9" if g < 10 else "10+"] += 1
        bpred = f.arrays["ymode"] == 4
        for b in (0, 15, 16, 23, 24):
            add(f"single block at bit {b}", (m == (1 << b)).sum())
        add("i16 with Y2 only", (~bpred & (m == 1 << 24)).sum())
        add("i16 with luma AC, no Y2", (~bpred & ((m & 0xFFFF) != 0) & ((m >> 24) == 0)).sum())
        grid = m.reshape(f.mb_rows, f.mb_cols)
        full, empty = grid == (1 << 25) - 1, grid == 0
        if f.mb_cols > 1:
            add("all 25 at a row start, empty right neighbour", (full[:, 0] & empty[:, 1]).sum())
            add("all 25 at a row end, empty left neighbour", (full[:, -1] & empty[:, -2]).sum())
            add("empty row start, full right neighbour", (empty[:, 0] & full[:, 1]).sum())
        add("Y2 block at B_PRED", (bpred & ((m >> 24) & 1 == 1)).sum())
        add("lone luma DC at i16", (~bpred[:, None] & ((f.arrays["coeff_y"].reshape(-1, 16, 16)[:, :, 1:] == 0).all(2))
                                    & (f.arrays["coeff_y"].reshape(-1, 16, 16)[:, :, 0] != 0)).sum())
        add("has_coeff disagrees with the blocks", ((f.arrays["has_coeff"] != 0) != (m != 0)).sum())
    return c


def census_rows(c, floors=None):
    """(cell name, count, floor) of every census cell; floors default to the mask-edge set's."""
    role_floor, block_floor, gran_floor, edge_floor = floors or (ROLE_FLOOR, BLOCKS_FLOOR, GRANULES_FLOOR, EDGE_FLOOR)
    names = [f"luma {2 * h},{2 * h + 1}" for h in range(8)] + ["U 16,17", "U 18,19", "V 20,21", "V 22,23", "Y2 24"]
    rows = [(f"role {names[r]} nz={k}", int(c["role"][r, k]), role_floor[r][k]) for r in range(13) for k in range(4)]
    rows += [(f"macroblocks with {k} blocks", v, block_floor[k]) for k, v in c["blocks"].items()]
    rows += [(f"frames over {k} granules", v, gran_floor[k]) for k, v in c["granules"].items()]
    rows += [(k, v, edge_floor.get(k, 0)) for k, v in c["edge"].items()]
    return rows


def census_table(c, floors=None) -> str:
    return "\n".join(f"{name:48s} {count:9d}  floor {floor}" for name, count, floor in census_rows(c, floors))


# Floors: about half of what the set measured when it was made. Y2 is one block: its nz = 2 / 3 cannot occur (floor 0,
# must stay 0).
ROLE_FLOOR = [(500, 150, 150, 1800)] * 12 + [(1200, 1400, 0, 0)]
BLOCKS_FLOOR = {0: 250, 1: 130, 24: 500, 25: 1200, "other": 650}
GRANULES_FLOOR = {"1": 10, "2": 1, "3-9": 2, "10+": 1}
EDGE_FLOOR = {"single block at bit 0": 15, "single block at bit 15": 15, "single block at bit 16": 15, "single block at bit 23": 15,
              "single block at bit 24": 50, "i16 with Y2 only": 50, "i16 with luma AC, no Y2": 300,
              "all 25 at a row start, empty right neighbour": 15, "all 25 at a row end, empty left neighbour": 15,
              "empty row start, full right neighbour": 12, "Y2 block at B_PRED": 10, "lone luma DC at i16": 200,
              "has_coeff disagrees with the blocks": 40}


@pytest.fixture(scope="module")
def mask_set():
    return [mask_frame(*s) for s in MASK_SET]


@pytest.fixture(scope="module")
def wide():
    return mask_frame(*WIDE)


def test_mask_census_of_the_mask_edge_set(mask_set, wide):
    c = mask_census(mask_set + [wide])
    low = [(name, count, floor) for name, count, floor in census_rows(c) if count < floor or (floor == 0 and count)]
    assert not low, f"cells below their floor (or unreachable cells counted): {low}\n{census_table(c)}"
    assert granules(block_masks(wide)) >= 10 and wide.mb_cols == 1024


def test_mask_edge_frames_are_what_the_recipes_say(mask_set):
    """Spot checks of the recipes: presence is exactly what the mask reports, whole planes are empty where they must be."""
    for (recipe, *_), f in zip(MASK_SET, mask_set):
        m = block_masks(f)
        pc = np.array([bin(int(x)).count("1") for x in m])
        if recipe == "y2only":
            assert ((m & ~np.uint32(1 << 24)) == 0).all() and (m != 0).any()
        elif recipe == "acnoy2":
            assert ((m >> 24) == 0).all() and ((m & 0xFFFF) != 0).any()
        elif recipe == "single":
            assert (pc <= 1).all()
        elif recipe == "rowedges":
            assert np.isin(m, (0, (1 << 25) - 1)).all()
        elif recipe == "dense":
            bpred = f.arrays["ymode"] == 4
            assert (m[~bpred] == (1 << 25) - 1).all() and (m[bpred] == (1 << 24) - 1).all()


@pytest.fixture(scope="module")
def parse_arena_check(tmp_path_factory):
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("no g++")
    exe = tmp_path_factory.mktemp("native") / "parse_arena_check"
    subprocess.run([gxx, "-O1", "-std=c++17", "-pthread", "-o", str(exe), str(ROOT / "tests" / "native" / "parse_arena_check.cpp"),
                    str(ROOT / "webp-decoder_b200" / "csrc" / "vp8_parse.cpp")], check=True)
    return exe


def test_shared_arena_parse_stops_at_its_capacity(parse_arena_check):
    """vp8_simple_chunk + vp8_parse_payload_shared with capacities from just past the frame's head up to its bound: every
    one that cannot hold the frame (8 granules) fails with ENOSPC and writes nothing past the capacity; the rest, and two
    frames sharing a cursor at exactly their summed bounds, give the standalone parse's masks and blocks."""
    webp = GOLDEN / "webp"
    r = subprocess.run([str(parse_arena_check), str(webp / "ref_generated_gen_noise_400x416_q10.webp"),
                        str(webp / "enc_noise_200x120_q75_i16_lf.webp")], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.startswith("ok "), r.stdout + r.stderr[-3000:]


# ------------------------------------------------------------------------------------------------ GPU: shapes x producers
def launch_fits(cfg, shape, exact):
    """The launch ran in `shape`. Not `exact`: a batch with frames wider than the stress set's 1040 px may get fewer images
    per CTA (line buffers take the shared memory) or a smaller cluster, but never another number of warps per image."""
    if exact:
        return launch_of(cfg) == expected_launch(shape)
    _, warps, per_sm, ctas, split = shape
    w, c, s, g = launch_of(cfg)
    return w == warps and 1 <= c <= ctas and (not s or split) and (2 <= g <= per_sm if g else True)


def check_outputs(tag, frames, out, offs, sizes, want):
    for i, (f, o, s) in enumerate(zip(frames, offs, sizes)):
        got = out[int(o):int(o) + int(s)]
        assert np.array_equal(got, want[i]), f"{tag} frame {i} {f.width}x{f.height}: {first_difference(f, got, want[i])}"


@pytest.fixture(scope="module")
def synthetic(mask_set):
    """Mask-edge set + loop-filter stress set, the 512-row mask frame last; with the oracle's bytes."""
    from vp8fix import Oracle
    orc = Oracle()
    frames = mask_set[:-1] + [stress_frame(*s) for s in STRESS] + mask_set[-1:]
    return frames, [{False: orc.decode_i420(f, False), True: orc.decode_i420(f, True)} for f in frames]


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,warps,per_sm,ctas,split", SHAPES)
def test_host_compaction_every_shape(gpu_ctx, oracle, synthetic, wide, kernel, warps, per_sm, ctas, split):
    """Dense frames compacted by one and by eight host threads into one arena (mb_first counted from the arena, blocks in
    granules shared between frames), decoded in one launch of the shape. The 16383-wide frame goes with the tall frame."""
    shape = (kernel, warps, per_sm, ctas, split)
    frames, want = synthetic
    batches = [(b, True) for b in shape_batches(len(frames), len(frames) - 1, ctas)]
    wide_want = {False: oracle.decode_i420(wide, False), True: oracle.decode_i420(wide, True)}
    set_shape(gpu_ctx, shape)
    try:
        for threads in (1, 8):
            gpu_ctx.set_transport(True, threads)
            for batch, exact in batches + [(None, False)]:
                fs = [frames[i] for i in batch] if batch else [wide, frames[-1]] + frames[:5 if ctas == 1 else 0]
                ws = [want[i] for i in batch] if batch else [wide_want, want[-1]] + want[:5 if ctas == 1 else 0]
                kfs, ds = [f.header() for f in fs], [f.cstruct() for f in fs]
                for filtered in (False, True):
                    out = np.full(gpu_ctx.decode_bytes(kfs), 0x55, np.uint8)
                    n0 = gpu_ctx.launches
                    offs, sizes = gpu_ctx.decode_into(kfs, ds, out, filtered=filtered, chunk=4 * len(fs))
                    cfg = gpu_ctx.last_launch_config()
                    assert gpu_ctx.launches - n0 == 1 and launch_fits(cfg, shape, exact), (shape, len(fs), cfg)
                    assert gpu_ctx.last_transport() == {"dense_chunks": 0, "compact_chunks": 1} and gpu_ctx.last_dense_frames() == 0
                    check_outputs(f"shape {shape} threads {threads} filtered={filtered}", fs, out, offs, sizes,
                                  [w[filtered] for w in ws])
    finally:
        gpu_ctx.set_transport("auto", 0)
        reset_shape(gpu_ctx)


def _parsed_frame(data: bytes) -> Frame:
    """The product's dense parse of one file as a Frame (for the oracle)."""
    from webp_decoder_b200 import parse as P
    pf = P.parse_batch([data], threads=1)
    d = pf.frames[0]
    params = {k: int(getattr(d, k)) for k in SCALARS}
    params.update({k: [int(getattr(d, k)[i]) for i in range(4)] for k in VEC4})
    f = Frame(pf.kfs[0].width, pf.kfs[0].height, params, {k: pf.array(0, k).copy() for k in U8_ARRAYS + I16_ARRAYS})
    pf.free()
    return f


@pytest.fixture(scope="module")
def parser_files(lib, golden):
    """Golden and bench_data/mixed files with their reference digests, the one with the most macroblock rows last, and
    their compact frames from the parser (one contiguous pinned buffer)."""
    from webp_decoder_b200 import parse as P
    mdir = ROOT / "bench_data" / "mixed"
    mixed = json.loads((mdir / "digests.json").read_text())
    files = [((GOLDEN / "webp" / n).read_bytes(), golden[n]) for n in sorted(golden)]
    files += [((mdir / n).read_bytes(), mixed[n]) for n in sorted(mixed)]
    files.sort(key=lambda t: t[1]["height"])
    cf = P.parse_batch_compact([d for d, _ in files], threads=8, pinned=True)
    yield files, cf
    cf.free()


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,warps,per_sm,ctas,split", SHAPES)
def test_parser_compact_frames_every_shape(lib, gpu_ctx, oracle, parser_files, kernel, warps, per_sm, ctas, split):
    """The parser's compact frames (one contiguous pinned buffer, mb_first counted per frame) of every golden and mixed
    file, decoded in one launch of the shape, against the reference decoder's digests; a mismatch is reported at its first
    differing byte against the oracle's decode of the same file."""
    shape = (kernel, warps, per_sm, ctas, split)
    files, cf = parser_files
    frames = cf.frame_list()
    set_shape(gpu_ctx, shape)
    try:
        for batch in shape_batches(len(frames), len(frames) - 1, ctas):
            fs = [frames[i] for i in batch]
            kfs = [cf.kfs[i] for i in batch]
            for filtered, key in ((False, "yuv"), (True, "yuvf")):
                out = np.full(gpu_ctx.decode_bytes(kfs), 0x55, np.uint8)
                n0 = gpu_ctx.launches
                offs, sizes = gpu_ctx.decode_compact_into(fs, out, filtered=filtered, chunk=4 * len(fs))
                cfg = gpu_ctx.last_launch_config()
                assert gpu_ctx.launches - n0 == 1 and launch_fits(cfg, shape, False), (shape, len(fs), cfg)
                for i, o, s in zip(batch, offs, sizes):
                    got = out[int(o):int(o) + int(s)]
                    if sha(got) != files[i][1][key]:
                        f = _parsed_frame(files[i][0])
                        assert False, (f"shape {shape} filtered={filtered} file {i} {f.width}x{f.height}: "
                                       f"{first_difference(f, got, oracle.decode_i420(f, filtered))}")
    finally:
        reset_shape(gpu_ctx)


@pytest.fixture(scope="module")
def passthrough_mix(lib, golden, synthetic):
    """Golden noise files (mostly non-zero blocks: they cross as they are) and sparse golden files (compacted) from
    pinned parser arenas, and the 512-row mask frame (numpy memory: compacted)."""
    from webp_decoder_b200 import parse as P
    noise = sorted(n for n in golden if "noise" in n and golden[n]["width"] >= 32)[:6]
    sparse = sorted(n for n in golden if "noise" not in n and golden[n]["width"] >= 16)[:14]
    names = noise + sparse
    pf = P.parse_batch([(GOLDEN / "webp" / n).read_bytes() for n in names], pinned=True)
    frames, want = synthetic
    yield pf, names, frames[-1], want[-1]
    pf.free()


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,warps,per_sm,ctas,split", SHAPES)
def test_dense_and_compact_frames_in_one_launch_every_shape(gpu_ctx, golden, passthrough_mix, kernel, warps, per_sm, ctas, split):
    """One launch in which some images read the dense layout (Vp8ImgDesc::compact = 0) and the others the compact one."""
    shape = (kernel, warps, per_sm, ctas, split)
    pf, names, tall, tall_want = passthrough_mix
    n = len(names)
    if ctas == 1:
        batches = [list(range(n))]
    else:  # up to 6 files, noise and sparse, and the tall frame
        batches = [[k % 6, 6 + k, 6 + (k + 1) % 14, (k + 3) % 6, 6 + (k + 2) % 14, 6 + (k + 3) % 14] for k in range(0, 14, 4)]
    set_shape(gpu_ctx, shape)
    gpu_ctx.set_transport(True, 4)
    try:
        for batch in batches:
            kfs = [pf.kfs[i] for i in batch] + [tall.header()]
            ds = [pf.frames[i] for i in batch] + [tall.cstruct()]
            for filtered, key in ((False, "yuv"), (True, "yuvf")):
                out = np.full(gpu_ctx.decode_bytes(kfs), 0x33, np.uint8)
                n0 = gpu_ctx.launches
                offs, sizes = gpu_ctx.decode_into(kfs, ds, out, filtered=filtered, chunk=4 * len(kfs))
                cfg = gpu_ctx.last_launch_config()
                assert gpu_ctx.launches - n0 == 1 and launch_fits(cfg, shape, True), (shape, cfg)
                assert gpu_ctx.last_transport() == {"dense_chunks": 0, "compact_chunks": 1}
                passed = gpu_ctx.last_dense_frames()
                assert 0 < passed < len(kfs), (shape, batch, passed)
                bad = [names[i] for i, o, s in zip(batch, offs, sizes) if sha(out[int(o):int(o) + int(s)]) != golden[names[i]][key]]
                assert not bad, (shape, filtered, bad)
                got = out[int(offs[-1]):int(offs[-1]) + int(sizes[-1])]
                assert np.array_equal(got, tall_want[filtered]), f"shape {shape} tall frame: {first_difference(tall, got, tall_want[filtered])}"
    finally:
        gpu_ctx.set_transport("auto", 0)
        reset_shape(gpu_ctx)
