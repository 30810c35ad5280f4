"""The TMA-staged kernels past their first tile.  Each case of one table is planned by tests/c/plan_driver.cpp (the
library's own planner, compiled without a GPU) and claims the regimes it reaches -- a stage ring that goes round twice,
row segments, multi-row flex tiles and their dealing modes, tall batches whose tiles span frames of odd height, the
pooling kernel's producer layouts and consumer specialisations -- so that a planner change which stops a case from
reaching its regime fails on a machine without a GPU, naming the case and the label.  On the GPU every case runs with
its options and must equal the CPU oracle on every frame (each frame holds different bytes: a stale stage shows up as
another tile's data) and the generic gather kernel on the whole batch, and leave every byte around its output untouched
(except the row padding the pooling kernel writes on ragged rows, which must be zero for bundle formats)."""
import itertools
import os
import subprocess
from collections import namedtuple

import numpy as np
import pytest

import oracle
from conftest import ROOT

CSRC = os.path.join(ROOT, "chroma-subsampling-image-compressor_b200", "csrc")
B200 = (148, 232448)
FIELDS = ("family", "grid", "stages", "ctas_per_sm", "tile_rows", "nsplit", "tile_px", "n_tiles", "block_threads",
          "smem_bytes", "Ho", "n_frames", "tall_ho", "slots_per_row", "in_dense", "out_dense")
GENERIC, ROWS, POOL, FLEX = 1, 2, 3, 4
YCC888, RGB888, BUNDLE64, BUNDLE128, PLANAR = 0, 1, 2, 3, 4
OPT = {"family": 0, "ctas": 2, "stages": 3, "tile": 4, "threads": 5}     # csic_option
ORD = {"S": 1, "Q": 2, "C": 3}

# One case: parameters, launch path, context options, the kernel family it must take and the regimes it claims.
#   path   "dense": csic_process_device; "offset": the same with input / output bases at byte offsets 1-15 (`at`);
#          "pitched": csic_process_device_pitched with the layout `at` = (in_pitch, in_frame, out_pitch, out_frame);
#          "band": csic_process_band of output rows `at` = (row0, rows)
#   opts   family, stages, tile (bytes), threads (per CTA), ctas (per SM); absent: the planner's choice
# The plan driver takes each case's bit depths q, which set the bundle slot width (1, 2 or 4 bytes).
Case = namedtuple("Case", "name W H a b f order fmt q inf rm pool n path at opts kernel labels")


def case(name, W, H, a, b, f, n, kernel, labels, order="CSQ", fmt=YCC888, q=(8, 8, 8), inf=0, rm=0, pool=0,
         path="dense", at=None, **opts):
    return Case(name, W, H, a, b, f, order, fmt, q, inf, rm, pool, n, path, at, opts, kernel, frozenset(labels.split()))


CASES = [
    # ---- row kernel: forced depths with laps (1024-pixel rows in 4 segments: 4:2:0 held chroma from aux windows)
    case("rows_s2", 1024, 40, 2, 0, 1, 31, ROWS, "laps segments", stages=2, tile=1024, ctas=1),
    case("rows_s3_rgb_trunc", 1024, 40, 2, 0, 1, 31, ROWS, "laps segments", fmt=RGB888, q=(6, 5, 5), rm=1, stages=3,
         tile=1024, ctas=1),
    case("rows_s4_planar", 1024, 40, 2, 0, 1, 31, ROWS, "laps segments", fmt=PLANAR, stages=4, tile=1024, ctas=1),
    case("rows_s5_b128_rgba", 1024, 40, 2, 0, 1, 31, ROWS, "laps segments", fmt=BUNDLE128, inf=1, stages=5, tile=1024,
         ctas=1),
    case("rows_s8", 1024, 40, 2, 0, 1, 31, ROWS, "laps segments", q=(5, 4, 3), stages=8, tile=1024, ctas=1),
    case("rows_s16", 1024, 40, 2, 0, 1, 31, ROWS, "laps segments", fmt=RGB888, stages=16, tile=1024, ctas=1),
    # case B (spatial first, 4:2:0, f = 2) in segments: the held pixel of an odd counter line is fetched per segment
    case("rows_caseb_seg", 512, 64, 2, 0, 2, 64, ROWS, "laps segments", order="SQC", fmt=BUNDLE128, inf=1, tile=1024,
         ctas=1),
    # multi-row tiles, the held row inside the tile (4:2:0, f = 1); staged and direct output
    case("rows_multi_ycc", 256, 64, 2, 0, 1, 90, ROWS, "laps multirow", stages=3, tile=4096, ctas=1),
    case("rows_multi_b64", 512, 64, 2, 0, 2, 80, ROWS, "laps multirow", fmt=BUNDLE64, stages=3, tile=4096, ctas=1),
    # ---- pooling kernel (depth 2): 4x4 AVERAGE rows in two segments, pooling first and chroma first
    case("pool_seg_sqc", 4096, 32, 2, 0, 4, 48, POOL, "laps pool_seg pool_first held_block mode3", order="SQC", pool=1,
         ctas=1),
    case("pool_seg_csq", 4096, 32, 2, 0, 4, 48, POOL, "laps pool_seg held_aux mode1", order="CSQ", fmt=RGB888,
         q=(6, 5, 5), pool=1, ctas=1),
    # every factor with every output format, 4-byte input, each consumer specialisation (mode0-3, trunc) and hold
    # width, and every producer layout: one copy or one copy per input row, ragged rows, bands, held pixels
    # f = 2
    case("p2_ycc_multi_held", 256, 64, 2, 0, 2, 100, POOL, "laps one_load multirow held_in_tile mode1", pool=1,
         ctas=1),
    case("p2_ycc_ragged_one_load", 200, 32, 2, 0, 2, 120, POOL, "laps one_load multirow ragged held_in_tile mode1",
         pool=1, path="pitched", at=(672, 672 * 32, 336, 336 * 16), ctas=1),
    # two-row tiles of an 8-row band from row 3: one held line per tile, four tiles per band, so (148 CTAs) every CTA
    # reduces the held block of the same line in frame after frame
    case("p2_rgba_band_first", 128, 64, 2, 0, 2, 200, POOL, "laps band multirow pool_first held_block mode3",
         order="SQC", fmt=RGB888, inf=1, pool=1, path="band", at=(3, 8), ctas=1),
    case("p2_slot8_ragged_rows", 200, 32, 4, 4, 2, 50, POOL, "laps row_loads ragged mode2", fmt=BUNDLE64,
         q=(3, 3, 2), pool=1, path="pitched", at=(688, 688 * 32 + 48, 128, 128 * 16 + 16), ctas=1),
    case("p2_bgra_slot16_q_first", 512, 32, 2, 2, 2, 60, POOL, "laps one_load mode0", order="QCS", fmt=BUNDLE128,
         q=(6, 5, 5), inf=2, pool=1, threads=96, ctas=1),
    case("p2_slot32_trunc_hf4", 256, 64, 1, 0, 2, 60, POOL, "laps one_load held_in_tile trunc", fmt=BUNDLE128, rm=1,
         pool=1, ctas=1),
    case("p2_first_hf4", 256, 64, 1, 1, 2, 60, POOL, "laps one_load pool_first mode3", order="SQC", pool=1, ctas=1),
    case("p2_first_hf1_held", 256, 64, 4, 0, 2, 60, POOL, "laps one_load pool_first held_block mode3", order="SCQ",
         pool=1, ctas=1),
    case("p2_rgb_ragged_rows_64", 232, 32, 1, 0, 2, 50, POOL, "laps row_loads ragged held_in_tile mode1", fmt=RGB888,
         pool=1, path="pitched", at=(784, 784 * 32 + 16, 400, 400 * 16 + 32), threads=64, ctas=1),
    case("p2_slot32_b64_ragged_first", 216, 32, 2, 0, 2, 50, POOL, "laps one_load ragged pool_first held_block mode3",
         order="SQC", fmt=BUNDLE64, pool=1, path="pitched", at=(672, 672 * 32, 464, 464 * 16), ctas=1),
    case("p2_slot32_b64_band_held", 256, 64, 2, 0, 2, 150, POOL, "laps band held_in_tile mode1", fmt=BUNDLE64,
         pool=1, path="band", at=(3, 20), ctas=1),
    # f = 4
    case("p4_ycc_96", 512, 64, 2, 2, 4, 100, POOL, "laps one_load mode2", pool=1, threads=96, ctas=1),
    case("p4_rgba_slot16_band_first", 128, 64, 1, 0, 4, 250, POOL, "laps band pool_first held_block mode3",
         order="SCQ", fmt=BUNDLE64, q=(6, 5, 5), inf=1, pool=1, path="band", at=(5, 8), ctas=1),
    case("p4_ycc_band", 256, 64, 4, 4, 4, 150, POOL, "laps band one_load mode2", pool=1, path="band", at=(5, 9),
         ctas=1),
    case("p4_rgb_q_first", 256, 64, 2, 2, 4, 100, POOL, "laps one_load mode0", order="QCS", fmt=RGB888, q=(5, 6, 4),
         pool=1, ctas=1),
    case("p4_slot8_hf4_512", 512, 64, 1, 0, 4, 100, POOL, "laps one_load held_in_tile mode1", fmt=BUNDLE128,
         q=(3, 3, 2), pool=1, threads=512, ctas=1),
    case("p4_rgba_slot16_trunc_first", 256, 64, 2, 0, 4, 150, POOL, "laps one_load pool_first held_block trunc",
         order="SQC", fmt=BUNDLE64, q=(6, 5, 5), inf=1, rm=1, pool=1, ctas=1),
    case("p4_bgra_slot32_ragged", 200, 32, 2, 0, 4, 100, POOL, "laps row_loads ragged pool_first held_block mode0",
         order="QSC", fmt=BUNDLE128, q=(7, 7, 7), inf=2, pool=1, path="pitched", at=(1088, 1088 * 32, 272, 272 * 8),
         ctas=1),
    # f = 8
    case("p8_ycc_small_cta", 256, 64, 2, 0, 8, 100, POOL, "laps one_load held_in_tile small_cta mode1", pool=1,
         ctas=1),
    case("p8_rgba_first_hf4_64", 256, 64, 1, 0, 8, 100, POOL, "laps one_load pool_first held_block mode3",
         order="SQC", fmt=RGB888, inf=1, pool=1, threads=64, ctas=1),
    case("p8_slot8_rows", 256, 64, 2, 2, 8, 100, POOL, "laps row_loads mode2", fmt=BUNDLE64, q=(3, 3, 2), pool=1,
         path="pitched", at=(800, 800 * 64 + 32, 64, 64 * 8 + 16), ctas=1),
    case("p8_bgra_slot16_band", 128, 128, 2, 0, 8, 125, POOL, "laps band held_in_tile mode0", order="CQS",
         fmt=BUNDLE128, q=(6, 5, 5), inf=2, pool=1, path="band", at=(9, 6), ctas=1),
    case("p8_ycc_ragged_first", 320, 64, 2, 0, 8, 100, POOL, "laps one_load ragged pool_first held_block mode3",
         order="SQC", pool=1, path="pitched", at=(1152, 1152 * 64, 160, 160 * 8), ctas=1),
    case("p8_ycc_band_first", 128, 128, 2, 0, 8, 250, POOL, "laps band pool_first held_block mode3", order="SQC",
         pool=1, path="band", at=(9, 6), ctas=1),
    case("p8_rgb_q_first_512", 512, 64, 2, 2, 8, 100, POOL, "laps one_load mode0", order="QCS", fmt=RGB888,
         q=(5, 6, 4), pool=1, threads=512, ctas=1),
    case("p8_slot32_trunc_aux", 2048, 16, 4, 0, 8, 185, POOL, "laps pool_seg held_aux trunc", fmt=BUNDLE128, rm=1,
         pool=1, ctas=1),
    # ---- flex kernel: odd width in 1024-byte segments, forced depths with laps
    case("flex_s2_seg", 1001, 13, 2, 0, 1, 30, FLEX, "laps segments", family=2, stages=2, tile=1024, ctas=1),
    case("flex_s3_seg", 1001, 13, 2, 0, 1, 40, FLEX, "laps segments", fmt=RGB888, family=2, stages=3, tile=1024, ctas=1),
    case("flex_s5_seg_rgba", 1001, 13, 2, 0, 1, 60, FLEX, "laps segments", inf=1, family=2, stages=5, tile=1024, ctas=1),
    case("flex_s8_seg_trunc", 1001, 13, 2, 0, 1, 80, FLEX, "laps segments", rm=1, family=2, stages=8, tile=1024, ctas=1),
    case("flex_planar_seg", 1000, 20, 2, 0, 1, 20, FLEX, "laps segments planar_seg", fmt=PLANAR, family=2, tile=1024,
         ctas=1),
    # multi-row tiles: dealing modes 0, 2 and 3; one packed span; direct stores
    case("flex_mode0", 700, 30, 2, 0, 1, 104, FLEX, "laps multirow mode0", family=2, stages=3, tile=8192, ctas=1),
    case("flex_mode2_out_one", 128, 40, 2, 0, 1, 420, FLEX, "laps multirow mode2 out_one", family=2, stages=3, tile=6144,
         ctas=1),
    case("flex_mode3_direct", 37, 40, 2, 0, 1, 750, FLEX, "laps multirow mode3 direct", fmt=RGB888, family=2, stages=5,
         tile=2048, ctas=1),
    case("flex_nw3", 128, 40, 2, 0, 1, 300, FLEX, "laps multirow mode2 nw3", family=2, tile=6144, threads=96, ctas=1),
    case("flex_nw2_direct_b64", 100, 40, 2, 0, 2, 500, FLEX, "laps multirow direct", fmt=BUNDLE64, family=2, tile=4096,
         threads=64, ctas=1),
    # unaligned bases, dense rows
    case("flex_offset", 333, 24, 2, 0, 1, 180, FLEX, "laps multirow", path="offset", at=(7, 13), family=2, stages=3,
         tile=4096, ctas=1),
    # >= 2048-byte rows on odd pitches, several per tile: per-row spans by the whole CTA
    case("flex_span_rows", 700, 30, 2, 0, 1, 104, FLEX, "laps multirow span_rows", path="pitched",
         at=(2107, 2107 * 30 + 41, 2113, 2113 * 30 + 29), family=2, stages=3, tile=8192, ctas=1),
    # natural tall plans (tiles span frames) of odd frame height: chroma first at f = 1, and case B
    case("flex_tall_odd", 333, 51, 2, 0, 1, 700, FLEX, "laps multirow tall_odd", family=2, ctas=1),
    case("flex_tall_odd_rgb", 37, 9, 2, 0, 1, 4000, FLEX, "laps multirow tall_odd direct", fmt=RGB888, family=2, ctas=1),
    case("flex_tall_caseb", 256, 38, 2, 0, 2, 900, FLEX, "laps multirow tall_caseb", order="SQC", family=2, ctas=1),
    # a middle band of a multi-row plan
    case("flex_band", 333, 51, 2, 0, 1, 90, FLEX, "laps multirow", path="band", at=(3, 45), family=2, stages=3,
         tile=4096, ctas=1),
]


# ---- the plan driver and the producer's rules ---------------------------------------------------------------------
@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("plandrv") / "plan_driver")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", f"-I{ROOT}/include",
                           os.path.join(ROOT, "tests", "c", "plan_driver.cpp"), os.path.join(CSRC, "csic_plan.cpp"),
                           os.path.join(CSRC, "csic_params.cpp"), "-o", exe])
    return exe


def driver_line(c):
    ops = "".join(str(ORD[ch]) for ch in c.order)
    row0, rows = c.at if c.path == "band" else (0, -1)
    o = c.opts
    line = (f"F {c.W} {c.H} {c.a} {c.b} {c.f} {ops} {c.fmt} {c.inf} {c.pool} {c.n} {row0} {rows} 0 "
            f"{o.get('family', 0)} {o.get('stages', 0)} {o.get('tile', 0)} {o.get('threads', 0)} {o.get('ctas', 0)}")
    return line + " %d %d %d %d" % (c.at if c.path == "pitched" else (0, 0, 0, 0)) + " %d %d %d" % c.q


def plan_cases(driver, limits):
    r = subprocess.run([driver, *map(str, limits)], input="".join(driver_line(c) + "\n" for c in CASES),
                       capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stderr
    out = r.stdout.splitlines()
    assert len(out) == len(CASES)
    plans = {}
    for c, line in zip(CASES, out):
        assert not line.startswith("error"), (c.name, line)
        plans[c.name] = dict(zip(FIELDS, map(int, line.split())))
    return plans


def flex_mode(nrows, ncols, consumers):
    """FlexDesc::mode, how flex_consume deals a tile's granules to the consumer warps: the producer's rule,
    csrc/csic_flex_kernel.cu:419-435."""
    nw, gpr = consumers // 32, (ncols + 3) // 4
    parts = nw // nrows if nrows <= nw else 0
    if parts and parts & (parts - 1) == 0:
        lanes = parts * 32
        if gpr * 5 >= -(-gpr // lanes) * lanes * 4:
            return 0
    if gpr >= 4 * consumers:
        return 1
    if nrows > nw and nrows * 5 >= -(-nrows // nw) * nw * 4 and gpr * 5 >= -(-gpr // 32) * 32 * 4:
        return 2
    return 3


def flex_stores(c, k):
    """(direct, out_one, output bytes per row) of a flex launch: narrow rows leave from registers (the consumers'
    launch-wide `direct`, csrc/csic_flex_kernel.cu:477-479); whole dense rows leave as one packed span (the producer's
    `out_one`, :422).  Output bytes per slot and per 4-slot granule: 3 / 12, PLANAR's Y plane 1 / 4, 8-bit bundles
    4 / 16."""
    opx, unit = {YCC888: (3, 12), RGB888: (3, 12), PLANAR: (1, 4)}.get(c.fmt, (4, 16))
    ncols = min(k["tile_px"], k["slots_per_row"])
    out_one = bool(k["out_dense"]) and k["nsplit"] == 1 and ncols * opx == (ncols + 3) // 4 * unit
    direct = c.fmt != PLANAR and k["nsplit"] == 1 and not out_one and ncols * opx < 257
    return direct, out_one, ncols * opx


def hold(c):
    """(hf, vf): the chroma stage's horizontal hold width and vertical factor (ChromaSubsampler.scala:17-18)."""
    return 4 // c.a, 2 if c.b == 0 else 1


def pool_first(c):
    """Spatial before chroma with a chroma stage that holds anything: the plan's case_b (csic_plan.cpp:418)."""
    hf, vf = hold(c)
    return c.f > 1 and c.order.index("S") < c.order.index("C") and hf * vf > 1


def kformat(c):
    """The pooling kernel's output format: "ycc", "rgb" or the bundle slot width "slot8" / "slot16" / "slot32"."""
    if c.fmt in (YCC888, RGB888):
        return "ycc" if c.fmt == YCC888 else "rgb"
    t = sum(c.q)
    return "slot8" if t <= 8 else ("slot16" if t <= 16 else "slot32")


def pool_mode(c):
    """The pool_tile specialisation the consumers run, csrc/csic_pool_kernel.cu:422-446: the quantiser's masks apply
    before the pooling when it comes first; without chroma pre-masks the sums run in the complement domain."""
    quant_first = c.order.index("Q") < c.order.index("S")
    pre = [((0xFF << (8 - bits)) & 0xFF) if quant_first else 0xFF for bits in c.q]
    linear = pre[1] == 0xFF and pre[2] == 0xFF
    if c.rm:
        return "trunc"
    if linear and pre[0] == 0xFF:
        return "mode3" if pool_first(c) else ("mode1" if hold(c)[1] == 2 else "mode2")
    return "mode0"


def regimes(c, k):
    """The labels the plan `k` of case `c` reaches."""
    got = set()
    if k["n_tiles"] // k["grid"] >= 2 * k["stages"] + 1:      # the CTA with the fewest tiles laps the ring twice
        got.add("laps")
    if k["nsplit"] > 1:
        got.add("pool_seg" if k["family"] == POOL else "segments")
        if c.fmt == PLANAR and k["family"] == FLEX:
            got.add("planar_seg")
    if k["tile_rows"] > 1:
        got.add("multirow")
    if k["family"] == FLEX:
        band = k["Ho"] if c.path != "band" else c.at[1]        # rows of one band (a tall batch: of the whole batch)
        rows = {min(k["tile_rows"], band), band - (-(-band // k["tile_rows"]) - 1) * k["tile_rows"]}
        last = k["slots_per_row"] - (k["nsplit"] - 1) * k["tile_px"]
        for nr, nc in itertools.product(rows, {min(k["tile_px"], k["slots_per_row"]), last}):
            got.add(f"mode{flex_mode(nr, nc, k['block_threads'])}")
        direct, out_one, row_out = flex_stores(c, k)
        if direct:
            got.add("direct")
        elif k["tile_rows"] > 1 and out_one:
            got.add("out_one")
        elif k["tile_rows"] > 1 and row_out >= 2048:
            got.add("span_rows")
        if k["block_threads"] == 96:
            got.add("nw3")
        # a tall batch of odd frame height whose tiles start inside frames
        if k["tall_ho"] % 2 == 1 and k["tall_ho"] % k["tile_rows"]:
            case_b = c.f > 1 and c.order.index("S") < c.order.index("C")
            got.add("tall_caseb" if case_b else "tall_odd")
    if k["family"] == POOL:
        if k["nsplit"] == 1:     # one TMA load per input row, or the tile's F * rows input rows as one copy
            # (csrc/csic_pool_kernel.cu:405-410)
            got.add("one_load" if k["in_dense"] else "row_loads")
        wo = -(-c.W // c.f)
        if -(-wo // 16) * 16 != wo:
            got.add("ragged")    # rows padded to Wp: bundle slots past Wo are zeroed (csic_pool_kernel.cu:283-287)
        if c.path == "band":
            got.add("band")
        hf, vf = hold(c)
        if pool_first(c):
            got.add("pool_first")
            if vf == 2:
                got.add("held_block")                # the producer reduces the block an odd line replays (:350-381)
        elif vf == 2:
            got.add("held_in_tile" if k["nsplit"] == 1 else "held_aux")    # (:383-398)
        if c.f == 8 and "threads" not in c.opts and k["block_threads"] < 192:
            got.add("small_cta")
        got.add(pool_mode(c))
    return got


def check_plans(plans):
    wrong = []
    for c in CASES:
        k = plans[c.name]
        if k["family"] != c.kernel:
            wrong.append(f"{c.name}: family {k['family']}, not {c.kernel}: {k}")
        elif c.labels - regimes(c, k):
            wrong.append(f"{c.name} no longer reaches {sorted(c.labels - regimes(c, k))}: {k}")
    assert not wrong, "\n".join(wrong)


def test_cases_reach_their_regimes(driver):
    """Every case still takes its kernel family and reaches every regime it claims under the B200 limits."""
    check_plans(plan_cases(driver, B200))


def test_table_covers_every_depth_and_regime():
    """The table's coverage, as the kernels' tests need it: forced row-kernel depths 2 - 16 and flex depths 2 - 8 that
    each lap the ring, and every flex regime."""
    def depths(family):
        return {c.opts.get("stages") for c in CASES if c.kernel == family and "laps" in c.labels}
    assert {2, 3, 4, 5, 8, 16} <= depths(ROWS) and {2, 3, 5, 8} <= depths(FLEX)
    flex = set().union(*(c.labels for c in CASES if c.kernel == FLEX))
    assert {"segments", "planar_seg", "mode0", "mode2", "mode3", "direct", "out_one", "span_rows", "nw3", "tall_odd",
            "tall_caseb"} <= flex
    assert {c.path for c in CASES if c.kernel == FLEX} == {"dense", "offset", "pitched", "band"}
    assert {64, 96} <= {c.opts.get("threads") for c in CASES if c.kernel == FLEX}
    # the pooling kernel (depth 2 always): every consumer instance pool_tile<F, FMT, IN4, HF, TRUNC, MODE> that matters,
    # and every layout branch of its producer, in cases that lap the ring
    pool = [c for c in CASES if c.kernel == POOL and "laps" in c.labels]
    modes = ("mode0", "mode1", "mode2", "mode3", "trunc")
    assert {(c.f, kformat(c)) for c in pool} >= set(itertools.product((2, 4, 8), ("ycc", "rgb", "slot8", "slot16",
                                                                                "slot32")))
    assert {BUNDLE64, BUNDLE128} <= {c.fmt for c in pool}
    assert {(c.f, c.inf) for c in pool} >= set(itertools.product((2, 4, 8), (1, 2)))
    assert {(c.f, m) for c in pool for m in c.labels & set(modes)} >= set(itertools.product((2, 4, 8), modes))
    held = {(hold(c)[0], m) for c in pool for m in c.labels & {"mode1", "mode2", "mode3"}}
    assert all({(hf, "mode1"), (hf, "mode2")} & held and (hf, "mode3") in held for hf in (1, 2, 4)), held
    assert {"row_loads", "one_load", "multirow", "pool_seg", "ragged", "band", "pool_first", "held_block",
            "held_in_tile", "held_aux", "small_cta"} <= set().union(*(c.labels for c in pool))
    assert {64, 96, 512} <= {c.opts.get("threads") for c in pool}
    assert any(c.f == 8 and c.opts.get("threads") == 64 for c in pool)
    assert {"dense", "pitched", "band"} <= {c.path for c in pool}
    # bands start inside a counter line of f output rows, on an odd one; pooling first, one of them over more frames
    # than CTAs: a CTA's next tile is then the same line of another frame (the held-block cache, DESIGN.md section 3)
    bands = [c for c in pool if c.path == "band"]
    assert all(c.at[0] % c.f and (c.at[0] // c.f) % 2 for c in bands), [c.name for c in bands]
    assert any("held_block" in c.labels and c.opts.get("ctas") == 1 and c.n > B200[0] for c in bands)


# ---- on the GPU -----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def csic():
    import csic_b200
    return csic_b200


@pytest.fixture(scope="module")
def gctx(csic):
    c = csic.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def live_plans(driver):
    """The plans for this device's limits: the two values csic_create reads."""
    import torch
    prop = torch.cuda.get_device_properties(0)
    plans = plan_cases(driver, (prop.multi_processor_count, prop.shared_memory_per_block_optin))
    check_plans(plans)
    return plans


def launch(ctx, c, p, d_in, n, fb, oh, orb):
    """Runs case `c` on d_in into a fresh output buffer with 0xA5 canaries on both sides -> (the whole buffer, the
    output rows as [n, oh, row pitch])."""
    import torch
    G = 4096
    S = torch.cuda.current_stream().cuda_stream or 1
    oi, oo = c.at if c.path == "offset" else (0, 0)
    if c.path == "pitched":
        in_pitch, in_frame, out_pitch, out_frame = c.at
        size = n * out_frame
    else:
        out_pitch, out_frame, size = orb, fb, n * fb
    buf = torch.full((G + oo + size + G,), 0xA5, dtype=torch.uint8, device="cuda")
    out = buf.data_ptr() + G + oo
    if c.path == "pitched":
        ctx.process_device_pitched(p, d_in.data_ptr(), in_pitch, in_frame, n, out, out_pitch, out_frame, S)
    elif c.path == "band":
        ctx.process_band(p, d_in.data_ptr(), n, out, c.at[0], c.at[1], S)
    else:
        ctx.process_device(p, d_in.data_ptr() + oi, n, out, S)
    torch.cuda.synchronize()
    frames = buf[G + oo:G + oo + size].view(n, out_frame)
    return buf, frames[:, :out_pitch * oh].view(n, oh, out_pitch)


def run_case(csic, ctx, c):
    """Runs case `c` with its options and checks it: the kernel family, every frame against the oracle, the bytes
    around the output, and the whole buffer against the generic gather kernel."""
    import torch
    ops = tuple(ORD[ch] for ch in c.order)
    p = csic.make_params(c.W, c.H, c.a, c.b, *c.q, c.f, ops, c.rm, c.pool, c.fmt, c.inf)
    po = oracle.make_params(c.W, c.H, c.a, c.b, c.q, c.f, c.order, c.rm, c.pool, c.fmt, c.inf)
    ipb = 3 if c.inf == 0 else 4
    _, oh, orb, fb = csic.out_shape(p)
    if c.fmt == PLANAR:
        oh, orb = 1, fb                       # three planes per frame: compared as one row
    rgb = np.random.default_rng(sum(map(ord, c.name))).integers(0, 256, size=(c.n, c.H, c.W, ipb), dtype=np.uint8)
    want = oracle.process(po, rgb, threads=8).reshape(c.n, oh, orb)
    # the input: dense at byte offset `oi` (0 unless the case says), or pitched rows with 0x5A in the padding and gaps
    if c.path == "pitched":
        in_pitch, in_frame = c.at[:2]
        assert in_pitch >= c.W * ipb and in_frame >= in_pitch * c.H and c.at[2] >= orb and c.at[3] >= c.at[2] * oh
        d_in = torch.full((c.n * in_frame,), 0x5A, dtype=torch.uint8, device="cuda")
        rows_in = d_in.view(c.n, in_frame)[:, :in_pitch * c.H].view(c.n, c.H, in_pitch)
        rows_in[:, :, :c.W * ipb] = torch.from_numpy(rgb.reshape(c.n, c.H, c.W * ipb)).cuda()
    else:
        oi = c.at[0] if c.path == "offset" else 0
        d_in = torch.empty((oi + rgb.size + 64,), dtype=torch.uint8, device="cuda")
        d_in[oi:oi + rgb.size] = torch.from_numpy(rgb.reshape(-1)).cuda()
    r0, r1 = (c.at[0], c.at[0] + c.at[1]) if c.path == "band" else (0, oh)
    # The pooling kernel writes whole rows of Wp = Wo rounded up to 16 output pixels (csic.h: columns beyond the frame
    # are written into the row padding), so on ragged rows the bytes [orb, Wp * opx) are the kernel's, not canaries;
    # bundle slots there are zero.  Every other byte keeps its check.
    pad_end = orb
    if "ragged" in c.labels:
        opx = {"slot8": 1, "slot16": 2, "slot32": 4}.get(kformat(c), 3)
        wo = -(-c.W // c.f)
        pad_end = (wo + 15) // 16 * 16 * opx
    try:
        for name, v in c.opts.items():
            ctx.set_option(OPT[name], v)
        buf, rows = launch(ctx, c, p, d_in, c.n, fb, oh, orb)
        got = rows[:, :, :orb]
        assert ctx.last_kernel()[0] == c.kernel, (c.name, ctx.last_kernel())
        # every frame against the oracle; outside a band the rows keep their canaries
        g = got.cpu().numpy()
        bad = [k for k in range(c.n) if not np.array_equal(g[k, r0:r1], want[k, r0:r1])]
        if bad:
            k = bad[0]
            diff = np.flatnonzero(g[k, r0:r1] != want[k, r0:r1])
            pytest.fail(f"{c.name}: {len(bad)} of {c.n} frames differ from the oracle; frame {k}: {diff.size} bytes, "
                        f"first at byte {diff[0]} of rows {r0}..{r1} ({diff[0] // orb + r0}, {diff[0] % orb})")
        assert (g[:, :r0] == 0xA5).all() and (g[:, r1:] == 0xA5).all(), c.name
        pad = rows[:, r0:r1, orb:pad_end]
        if c.fmt in (BUNDLE64, BUNDLE128):
            assert not bool(pad.any()), f"{c.name}: bundle slots past the frame's width are not zero"
        # nothing else in the buffer changed: canaries, pitch padding and the bytes between frames
        got.fill_(0xA5)
        pad.fill_(0xA5)
        assert bool((buf == 0xA5).all()), f"{c.name}: a write outside the output rows"
        # the generic gather kernel, byte for byte over the whole buffer
        ctx.set_option(OPT["family"], 1)
        buf_gen, _ = launch(ctx, c, p, d_in, c.n, fb, oh, orb)
        assert ctx.last_kernel()[0] == GENERIC
        got.copy_(torch.from_numpy(g))
        assert torch.equal(buf, buf_gen), f"{c.name}: differs from the generic kernel"
    finally:
        for name in OPT:
            ctx.set_option(OPT[name], 0)


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=[c.name for c in CASES])
def test_tile_walk_on_gpu(csic, gctx, live_plans, c):
    run_case(csic, gctx, c)


# Pooling with an input or output base 1 - 15 bytes off a 16-byte boundary: the TMA pooling kernel does not take it
# (csic.h, csic_process_device_pitched), the gather kernel does.  Not in CASES: the plan driver plans aligned bases.
OFFSET_CASES = [
    case("pool_offset_in", 256, 64, 2, 0, 2, 6, GENERIC, "", order="SQC", pool=1, path="offset", at=(7, 0)),
    case("pool_offset_out", 256, 64, 2, 0, 4, 6, GENERIC, "", fmt=BUNDLE128, q=(6, 5, 5), inf=1, pool=1,
         path="offset", at=(0, 5)),
    case("pool_offset_both", 512, 32, 1, 0, 8, 6, GENERIC, "", fmt=RGB888, pool=1, path="offset", at=(13, 15)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("c", OFFSET_CASES, ids=[c.name for c in OFFSET_CASES])
def test_pool_offset_bases_take_the_gather_kernel(csic, gctx, c):
    run_case(csic, gctx, c)
