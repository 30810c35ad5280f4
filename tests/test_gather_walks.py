"""The two kernels of csrc/csic_kernels.cu that are not TMA-staged, past their first row group.

Gather kernel (csic_generic_kernel, family 1): the independent implementation every other kernel is compared with, and
the only kernel for spatial-before-chroma ("case B") shapes whose counter lines are not whole output rows and for
AVERAGE on dense widths that break the pooling kernel's 16-byte rules -- shapes users hit at 1366x768 and 1918x1078.
Each case of one table is planned by tests/c/plan_driver.cpp (the library's own planner, compiled without a GPU) and
claims the regimes it reaches: warps that take two row groups or more, narrow rows shared by a warp (rows of two frames
in one warp, idle lanes), several 32-granule trips per row, the 12-byte load path, held lines, and the per-row case-B and
AVERAGE branches, restated below from the kernel's own rules.  So a planner change that stops a case from reaching a
regime fails on a machine without a GPU, naming the case and the label.  On the GPU every case must take the gather
kernel, equal the C oracle on every frame (each frame holds different bytes), leave every byte around its output alone,
and equal any other family that runs the same parameters.

LDG decoder (csic_expand_planar_any_kernel): what plan_decode declines in production -- rows narrower than a granule,
chroma rows too wide for a stage -- and shapes the TMA decoder would take, run under CSIC_DEC_NO_TMA, at batches where
every block takes two rows or more."""
import ctypes
import itertools
import json
import subprocess
from collections import namedtuple

import numpy as np
import pytest

import oracle
import test_decode_walks as dw
import test_tile_walks as tw
from test_tile_walks import ORD, OPT, case, driver  # noqa: F401  (driver: the plan driver fixture)

B200 = tw.B200
GENERIC, POOL = 1, 3
YCC888, RGB888, BUNDLE64, BUNDLE128, PLANAR = 0, 1, 2, 3, 4
KFORMATS = ("ycc", "rgb", "slot8", "slot16", "slot32", "planar")
OPT_CHUNK_BYTES = 1                          # csic_option CSIC_OPT_HOST_CHUNK_BYTES
HOST_PATHS = ("host", "host_band")

# Launch paths, beyond test_tile_walks.case's dense / offset / pitched / band:
#   "host"       csic_process_host with one chunk for the whole batch (DECIMATE at f > 1 ships every f-th row only)
#   "host_band"  csic_process_host_band of each band `at` = ((row0, rows), ...), one call per band
CASES = [
    # ---- the shapes users hit: bench-size frames only the gather kernel runs (no option forces it)
    case("bench_1366_420_f2_sqc", 1366, 768, 2, 0, 2, 50, GENERIC, "laps trips trips_ragged held_l0 back_row back_prev",
         order="SQC", path="host"),
    case("bench_1918_410_f4_scq_b128", 1918, 1078, 1, 0, 4, 72, GENERIC,
         "laps trips two_lines held_l0 held_l1 back_row", order="SCQ", fmt=BUNDLE128),
    case("bench_1918_avg_f2_rgb", 1918, 1078, 2, 0, 2, 40, GENERIC, "laps trips af2 held_lines", fmt=RGB888, pool=1),
    case("bench_1366_avg_410_f2_b128", 1366, 768, 1, 0, 2, 50, GENERIC, "laps trips af2 hold_inside_block held_lines",
         fmt=BUNDLE128, pool=1),
    case("bench_1366_avg_f2_sqc", 1366, 768, 2, 0, 2, 50, GENERIC, "laps trips af2 pool_first", order="SQC", pool=1),
    # ---- DECIMATE: every output format, narrow rows, held lines, both roundings, four-byte input
    # 13 x 9 at f = 2: 7-pixel rows, sixteen to a warp, rows of two frames in one warp; every case-B branch but the
    # division fallback; input bases 7 and output bases 13 bytes off 16
    case("n13_420_f2_sqc", 13, 9, 2, 0, 2, 100000, GENERIC,
         "laps narrow frames_in_warp two_lines held_l0 held_l1 back_row back_prev", order="SQC", path="offset",
         at=(7, 13)),
    # f = 1 RGB24 (12-byte loads) with held lines, truncating rounding; 250 granules: eight trips, the last partial
    case("d_rgb_trunc_f1_held", 1000, 40, 2, 0, 1, 480, GENERIC, "laps trips trips_ragged f1_fast held_row",
         fmt=RGB888, rm=1, family=1),
    case("d_planar_narrow_held", 20, 50, 2, 0, 1, 2300, GENERIC,
         "laps narrow frames_in_warp idle_lanes f1_fast held_row", fmt=PLANAR, family=1),
    case("d_slot8_rgba_411_f2_band", 27, 38, 1, 1, 2, 10200, GENERIC, "laps narrow frames_in_warp back_row back_prev",
         order="SQC", fmt=BUNDLE64, q=(3, 3, 2), inf=1, path="band", at=(3, 15)),
    case("d_slot16_bgra_422_f2_pitched", 333, 24, 2, 2, 2, 1600, GENERIC, "laps trips trips_ragged back_row back_prev",
         order="QSC", fmt=BUNDLE128, q=(6, 5, 5), inf=2, path="pitched", at=(1344, 1344 * 24 + 48, 352, 352 * 12 + 16)),
    # ---- AVERAGE, f = 2: the two slot widths the bench cases leave, narrow rows, four-byte input, truncation
    case("a2_slot8_trunc_narrow", 24, 40, 2, 0, 2, 9500, GENERIC,
         "laps narrow frames_in_warp af2 held_lines quant_first", order="QCS", fmt=BUNDLE64, q=(3, 3, 2),
         rm=1, pool=1),
    case("a2_slot16_rgba_first", 250, 40, 1, 1, 2, 1000, GENERIC, "laps af2 pool_first", order="SCQ", fmt=BUNDLE64,
         q=(6, 5, 5), inf=1, pool=1),
    # ---- AVERAGE, f = 4 (every format; rows of 40 - 100 output pixels, several to a warp or one)
    case("a4_ycc_first", 200, 64, 2, 0, 4, 2400, GENERIC, "laps narrow af4 pool_first", order="SQC", pool=1),
    case("a4_rgb_trunc_hold", 400, 32, 1, 0, 4, 2400, GENERIC, "laps af4 held_lines", fmt=RGB888, rm=1, pool=1),
    case("a4_slot8_bgra_q_first", 168, 36, 2, 2, 4, 4300, GENERIC, "laps narrow frames_in_warp af4 pool_first "
         "quant_first", order="QSC", fmt=BUNDLE64, q=(3, 3, 2), inf=2, pool=1),
    case("a4_slot16_band", 360, 64, 4, 4, 4, 2600, GENERIC, "laps af4", fmt=BUNDLE64, q=(6, 5, 5), pool=1, path="band",
         at=(1, 14)),
    case("a4_slot32_pitched", 200, 48, 1, 1, 4, 3200, GENERIC, "laps narrow af4 pool_first", order="SCQ",
         fmt=BUNDLE128, pool=1, path="pitched", at=(2432, 2432 * 48 + 16, 240, 240 * 12 + 32)),
    # ---- AVERAGE, f = 8: 16- and 17-pixel rows, several to a warp (the cheapest lapping batches: ~0.4 GB of input)
    case("a8_ycc_first", 136, 64, 2, 0, 8, 14300, GENERIC, "laps narrow frames_in_warp idle_lanes af8 pool_first",
         order="SQC", pool=1),
    case("a8_rgb_rgba", 136, 64, 4, 0, 8, 14300, GENERIC, "laps narrow af8 held_lines", fmt=RGB888, inf=1, pool=1),
    case("a8_slot8_trunc", 128, 64, 2, 2, 8, 19000, GENERIC, "laps narrow af8", fmt=BUNDLE128, q=(3, 3, 2), rm=1,
         pool=1, family=1),
    case("a8_slot16_bgra_q_first", 136, 64, 1, 0, 8, 14300, GENERIC, "laps narrow af8 held_lines quant_first",
         order="QCS", fmt=BUNDLE64, q=(6, 5, 5), inf=2, pool=1),
    case("a8_slot32_trunc_first", 136, 64, 1, 1, 8, 14300, GENERIC, "laps narrow af8 pool_first", order="SCQ",
         fmt=BUNDLE128, rm=1, pool=1),
    # ---- case B at every hold and factor: small frames, host bands that start at every phase of the counter line
    # (the band's buffer holds only its own rows), and rows narrower than the hold (the division fallback)
    case("hb_420_f2", 13, 40, 2, 0, 2, 3, GENERIC, "two_lines held_l0 held_l1 back_row back_prev", order="SQC",
         path="host_band", at=tuple((r, k) for r in range(9) for k in (1, 3)) + ((11, 5), (15, 5))),
    case("hb_410_f4_rgb", 31, 96, 1, 0, 4, 3, GENERIC, "two_lines held_l0 held_l1 back_row back_prev", order="SCQ",
         fmt=RGB888, path="host_band", at=tuple((r, k) for r in range(17) for k in (1, 2)) + ((19, 5),)),
    case("hb_422_f8_b64", 100, 192, 2, 2, 8, 3, GENERIC, "two_lines back_row back_prev", order="QSC", fmt=BUNDLE64,
         path="host_band", at=tuple((r, 1) for r in range(17)) + ((18, 5),)),
    case("hb_411_f2_b128", 21, 36, 1, 1, 2, 3, GENERIC, "two_lines back_row back_prev", order="SQC",
         fmt=BUNDLE128, q=(6, 5, 5), path="host_band", at=tuple((r, 2) for r in range(7)) + ((10, 8),)),
    case("cb_422_f4", 30, 40, 2, 2, 4, 20, GENERIC, "two_lines back_row", order="SQC", fmt=RGB888),
    case("cb_411_f4_trunc", 31, 44, 1, 1, 4, 20, GENERIC, "two_lines back_row back_prev", order="SCQ", rm=1),
    case("cb_420_f4", 30, 40, 2, 0, 4, 20, GENERIC, "two_lines held_l0 held_l1 back_row", order="SQC"),
    case("cb_420_f8", 60, 128, 2, 0, 8, 20, GENERIC, "two_lines held_l0 held_l1 back_row", order="SCQ", fmt=BUNDLE64,
         q=(6, 5, 5)),
    case("cb_410_f2", 27, 30, 1, 0, 2, 20, GENERIC, "two_lines held_l0 held_l1 back_row back_prev", order="SQC",
         fmt=BUNDLE64, q=(3, 3, 2)),
    # one-pixel rows, 32 to a warp: every hold group of a sampled line starts one or more rows above (the division
    # fallback), at a lapping batch
    case("cb_410_f8_far", 7, 128, 1, 0, 8, 40000, GENERIC, "laps narrow frames_in_warp held_l0 back_far",
         order="SQC"),
    case("cb_411_f8_far", 7, 24, 1, 1, 8, 2000, GENERIC, "narrow back_far", order="SCQ", fmt=BUNDLE128),
    case("cb_422_f2_band", 33, 30, 2, 2, 2, 20, GENERIC, "two_lines back_row back_prev", order="SQC", path="band",
         at=(5, 7)),
]


# ---- the plan driver and the gather kernel's per-row rules -----------------------------------------------------------
def launches(c):
    """(row0, rows) of each launch of case `c`; rows -1: the whole frame."""
    if c.path == "band":
        return [c.at]
    if c.path == "host_band":
        return list(c.at)
    return [(0, -1)]


def compact(c):
    """csic_process_host stores every f-th input row only: DECIMATE, f > 1, H a multiple of f (plan_host,
    csrc/csic_plan.cpp:554)."""
    return c.path in HOST_PATHS and not c.pool and c.f > 1 and c.H % c.f == 0


def plan_gather(driver, limits, cases=CASES):
    """{case name: [(row0, rows, the F line's plan) per launch]}."""
    jobs, lines = [], []
    for c in cases:
        for row0, rows in launches(c):
            t = c._replace(path="band", at=(row0, rows)) if rows > 0 else c
            if c.path in HOST_PATHS and rows < 0:
                t = t._replace(path="dense")
            tok = tw.driver_line(t).split()
            tok[13] = str(int(compact(c)))                     # the F line's `compact`
            jobs.append((c.name, row0, rows))
            lines.append(" ".join(tok) + "\n")
    r = subprocess.run([driver, *map(str, limits)], input="".join(lines), capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stderr
    out = r.stdout.splitlines()
    assert len(out) == len(jobs)
    plans = {}
    for (name, row0, rows), line in zip(jobs, out):
        assert not line.startswith("error"), (name, row0, rows, line)
        plans.setdefault(name, []).append((row0, rows, dict(zip(tw.FIELDS, map(int, line.split())))))
    return plans


def geometry(c):
    """(Wo, Ho, hf, vf, case_b, AF): case B is spatial before a chroma stage that holds anything (csic_plan.cpp:418);
    AF the AVERAGE factor of the kernel instance, 0 for DECIMATE (csic_kernels.cu:488)."""
    hf, vf = tw.hold(c)
    return -(-c.W // c.f), -(-c.H // c.f), hf, vf, tw.pool_first(c), c.f if c.pool and c.f > 1 else 0


def kformat(c):
    return "planar" if c.fmt == PLANAR else tw.kformat(c)


def gather_regimes(c, k, row0, rows):
    """The labels one launch (plan `k`, output rows [row0, row0 + rows)) of case `c` reaches."""
    Wo, Ho, hf, vf, case_b, af = geometry(c)
    rows = Ho if rows < 0 else rows
    got = set()
    # lanes -> rows, csrc/csic_kernels.cu:121-125: a warp per row, or 32 / gpr whole rows per warp under 32 granules;
    # four warps per CTA, grid-stride over the row groups
    gpr = -(-k["slots_per_row"] // 4)
    rpw = 32 // gpr if gpr < 32 else 1
    if -(-k["n_frames"] * rows // rpw) // (4 * k["grid"]) >= 2:
        got.add("laps")
    if gpr < 32:
        got.add("narrow")
        if rows % rpw:
            got.add("frames_in_warp")
        if 32 % gpr:
            got.add("idle_lanes")
    if gpr > 32:                                             # 32-granule trips through the warp's slot (:184)
        got.add("trips")
        if gpr % 32:
            got.add("trips_ragged")
    ipb = 3 if c.inf == 0 else 4
    ro = np.arange(row0, row0 + rows, dtype=np.int64)
    if not af:
        if c.f * ipb == 3 and Wo > 3:                        # twelve consecutive bytes (:192)
            got.add("f1_fast")
        if not case_b and vf == 2 and ((ro * c.f) & 1).any():
            got.add("held_row")                              # (:143-151)
        if case_b:
            got |= case_b_regimes(c, ro)
    else:
        got.add(f"af{af}")
        if not case_b and hf > c.f and Wo > 1:               # block columns co * f inside a hold group (:255)
            got.add("hold_inside_block")
        if not case_b and vf == 2:                           # odd block lines replay the held pair (:152-158, :253)
            got.add("held_lines")
        if case_b:
            got.add("pool_first")                            # (:267-281)
        if c.order.index("Q") < c.order.index("S"):
            got.add("quant_first")                           # (:244)
    return got


def case_b_regimes(c, ro):
    """The case-B DECIMATE branches rows `ro` reach, csrc/csic_kernels.cu:164-233: the row's two counter lines, their
    held pairs, and where each sampled pixel's hold group begins."""
    Wo, _, hf, vf, _, _ = geometry(c)
    got = set()
    m0 = ro * Wo                                             # (:168)
    line0 = m0 // c.W
    col0 = m0 - line0 * c.W
    split = c.W - col0                                       # first column in line0 + 1 (:169)
    two = split < Wo
    held0 = (vf == 2) & (line0 & 1 == 1)                     # (:174)
    held1 = (vf == 2) & ((line0 + 1) & 1 == 1) & two
    if two.any():
        got.add("two_lines")
    if held0.any():
        got.add("held_l0")
    if held1.any():
        got.add("held_l1")
    co = np.arange(Wo, dtype=np.int64)[None, :]
    second = co >= split[:, None]                            # (:215)
    sampled = ~np.where(second, held1[:, None], held0[:, None])
    back = np.where(second, co - split[:, None], co + (col0 & (hf - 1))[:, None]) & (hf - 1)     # (:221)
    live = sampled & (back > 0)
    if (live & (back <= co)).any():
        got.add("back_row")                                  # (:224)
    if (live & (back > co) & (Wo + co >= back)).any():
        got.add("back_prev")                                 # the group starts in the row above (:225)
    if (live & (Wo + co < back)).any():
        got.add("back_far")                                  # chroma_src_case_b (:226-229)
    return got


def regimes(c, launched):
    return set().union(*(gather_regimes(c, k, row0, rows) for row0, rows, k in launched))


def check_gather_plans(plans):
    wrong = []
    for c in CASES:
        for row0, rows, k in plans[c.name]:
            if rows > 0 and not (0 <= row0 and row0 + rows <= k["Ho"]):      # csic_process_band's bounds (csic_api.cu:100)
                wrong.append(f"{c.name}: band {row0}+{rows} outside the frame's {k['Ho']} output rows")
            if k["family"] != GENERIC:
                wrong.append(f"{c.name} (rows {row0}+{rows}): family {k['family']}, not the gather kernel: {k}")
        lost = c.labels - regimes(c, plans[c.name])
        if lost:
            wrong.append(f"{c.name} no longer reaches {sorted(lost)}: {[k for _, _, k in plans[c.name]]}")
    assert not wrong, "\n".join(wrong)


def host_plan(driver, limits, c, row0=0, rows=-1, chunk=0):
    """plan_host of case `c` through the H line (bit depths 8, which only the bundle slot width depends on)."""
    ops = "".join(str(ORD[ch]) for ch in c.order)
    line = f"H {c.W} {c.H} {c.a} {c.b} {c.f} {ops} {c.fmt} {c.inf} {c.pool} {c.n} {row0} {rows} 0 {chunk} 0\n"
    r = subprocess.run([driver, *map(str, limits)], input=line, capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and not r.stdout.startswith("error"), (c.name, r.stdout, r.stderr)
    return json.loads(r.stdout)


def chunk_bytes(c):
    """The host chunk size that holds the whole batch: one launch, so the plan of the F line is the one that runs."""
    return c.n * c.W * c.H * (3 if c.inf == 0 else 4)


def repitched_family(driver, limits, c):
    """The family csic_process_host's staging layout (csic_plan.cpp:530-544) gives case `c`'s parameters, or None when
    the staging buffers stay dense."""
    h = host_plan(driver, limits, c)
    if not h["lay"][0]:
        return None
    tok = tw.driver_line(c._replace(path="pitched", at=tuple(h["lay"][:4]))).split()
    r = subprocess.run([driver, *map(str, limits)], input=" ".join(tok) + "\n", capture_output=True, text=True,
                       timeout=60)
    return int(r.stdout.split()[0])


def test_gather_cases_reach_their_regimes(driver):
    """Every case takes the gather kernel on every launch and reaches every regime it claims under the B200 limits; a
    case that forces the gather kernel is one another family takes by itself."""
    check_gather_plans(plan_gather(driver, B200))
    forced = [c for c in CASES if c.opts.get("family") == GENERIC]
    auto = plan_gather(driver, B200, [c._replace(opts={}) for c in forced])
    assert forced and all(k["family"] != GENERIC for c in forced for _, _, k in auto[c.name]), auto


def test_host_cases_stage_what_they_claim(driver):
    """The host cases' staging: one chunk for the batch, compact rows, band buffers that start at the band's first input
    row; and the odd-width AVERAGE bench case re-pitched onto the pooling kernel."""
    for c in CASES:
        if c.path not in HOST_PATHS:
            continue
        for row0, rows in launches(c):
            h = host_plan(driver, B200, c, row0, rows, chunk_bytes(c))
            assert h["per"] == c.n and h["compact"] == int(compact(c)) == 1, (c.name, row0, h)
            assert h["in_rows"][0] // c.f == h["first_stored"], (c.name, row0, h)
    assert repitched_family(driver, B200, next(c for c in CASES if c.name == "bench_1918_avg_f2_rgb")) == POOL


def test_gather_table_covers_every_instance_and_regime(driver):
    """The table's coverage, as the gather kernel's tests need it: every csic_generic_kernel<TRUNC, FMT, AF> the planner
    selects, each in a case that laps, both roundings under every AF, four-byte input under DECIMATE and AVERAGE, every
    label with laps, narrow lapping rows for PLANAR, a bundle format and AVERAGE, every
    hold of case B at f = 2, 4 and 8, bench-size generic-only frames, every launch path, and host bands from every phase
    of the counter line."""
    lapping = [c for c in CASES if "laps" in c.labels]
    inst = {(kformat(c), geometry(c)[5]) for c in lapping}
    want = {(k, af) for k in KFORMATS for af in (0, 2, 4, 8) if k != "planar" or af == 0}
    assert len(want) == 21 and inst >= want, sorted(want - inst)
    assert {(geometry(c)[5], c.rm) for c in lapping} >= set(itertools.product((0, 2, 4, 8), (0, 1)))
    assert {(bool(geometry(c)[5]), c.inf) for c in lapping} >= set(itertools.product((False, True), (1, 2)))
    labels = {"laps", "narrow", "frames_in_warp", "idle_lanes", "trips", "trips_ragged", "f1_fast", "held_row",
              "two_lines", "held_l0", "held_l1", "back_row", "back_prev", "back_far", "af2", "af4", "af8",
              "hold_inside_block", "held_lines", "pool_first", "quant_first"}
    claimed = set().union(*(c.labels for c in CASES))
    assert labels <= claimed, labels - claimed
    with_laps = set().union(*(c.labels for c in lapping))
    assert labels <= with_laps, labels - with_laps
    narrow = [c for c in lapping if "narrow" in c.labels]
    assert any(c.fmt == PLANAR for c in narrow) and any(c.fmt in (BUNDLE64, BUNDLE128) for c in narrow)
    assert any(c.pool for c in narrow)
    holds = {((c.a, c.b), c.f) for c in CASES if geometry(c)[4] and not c.pool}
    assert holds >= set(itertools.product(((2, 0), (1, 0), (2, 2), (1, 1)), (2, 4, 8))), sorted(holds)
    bench = [c for c in lapping if (c.W, c.H) in ((1366, 768), (1918, 1078)) and "family" not in c.opts]
    assert len(bench) >= 4
    assert {c.path for c in CASES} == {"dense", "offset", "pitched", "band", "host", "host_band"}
    assert any(compact(c) for c in CASES if c.path == "host")
    # host bands: a first row at every phase of the counter line (W / Wo output rows), twice round the held-line
    # period, and bands deeper in the frame
    for c in (c for c in CASES if c.path == "host_band"):
        Wo, Ho, _, vf, case_b, _ = geometry(c)
        first = {r for r, _ in c.at}
        phases = 2 * vf * -(-c.W // Wo) + 1
        assert case_b and compact(c) and Ho > phases, c.name
        assert set(range(phases)) <= first and max(first) >= phases, (c.name, phases, sorted(first))


# ---- the gather kernel on the GPU -----------------------------------------------------------------------------------
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
def limits():
    """This device's limits: the two values csic_create reads."""
    import torch
    prop = torch.cuda.get_device_properties(0)
    return prop.multi_processor_count, prop.shared_memory_per_block_optin


@pytest.fixture(scope="module")
def live_gather_plans(driver, limits):
    plans = plan_gather(driver, limits)
    check_gather_plans(plans)
    return plans


def first_difference(c, got, want, r0):
    """Fails naming the first frame, row and column (byte of the row) where `got` differs from `want` ([n, rows, row
    bytes], output rows from r0)."""
    bad = np.flatnonzero((got != want).reshape(got.shape[0], -1).any(1))
    if bad.size:
        k = int(bad[0])
        r, col = (int(v[0]) for v in np.nonzero(got[k] != want[k]))
        pytest.fail(f"{c.name}: {bad.size} of {got.shape[0]} frames differ from the oracle; first: frame {k}, row "
                    f"{r + r0}, byte {col} of the row")


def run_device(csic, ctx, c, p, rgb, want, oh, orb, fb):
    """Case `c` on a device path: the oracle on every frame, the rows outside a band, every byte around the output, and,
    when the case forces the gather kernel, the automatic choice byte for byte over the whole buffer.  -> the output."""
    import torch
    ipb = rgb.shape[-1]
    if c.path == "pitched":
        in_pitch, in_frame = c.at[:2]
        d_in = torch.full((c.n * in_frame,), 0x5A, dtype=torch.uint8, device="cuda")
        rows_in = d_in.view(c.n, in_frame)[:, :in_pitch * c.H].view(c.n, c.H, in_pitch)
        rows_in[:, :, :c.W * ipb] = torch.from_numpy(rgb.reshape(c.n, c.H, c.W * ipb)).cuda()
    else:
        oi = c.at[0] if c.path == "offset" else 0
        d_in = torch.empty((oi + rgb.size + 64,), dtype=torch.uint8, device="cuda")
        d_in[oi:oi + rgb.size] = torch.from_numpy(rgb.reshape(-1)).cuda()
    r0, r1 = (c.at[0], c.at[0] + c.at[1]) if c.path == "band" else (0, oh)
    buf, rows = tw.launch(ctx, c, p, d_in, c.n, fb, oh, orb)
    assert ctx.last_kernel()[0] == GENERIC, (c.name, ctx.last_kernel())
    got = rows[:, :, :orb]
    g = got.cpu().numpy()
    first_difference(c, g[:, r0:r1], want[:, r0:r1], r0)
    assert (g[:, :r0] == 0xA5).all() and (g[:, r1:] == 0xA5).all(), f"{c.name}: a write outside the band"
    got.fill_(0xA5)
    assert bool((buf == 0xA5).all()), f"{c.name}: a write outside the output rows (canaries, padding, frame gaps)"
    got.copy_(torch.from_numpy(g))
    if c.opts.get("family") == GENERIC:
        ctx.set_option(OPT["family"], 0)
        auto, _ = tw.launch(ctx, c, p, d_in, c.n, fb, oh, orb)
        assert ctx.last_kernel()[0] != GENERIC, c.name
        assert torch.equal(buf, auto), f"{c.name}: family {ctx.last_kernel()[0]} differs from the gather kernel"
    return g


def run_host(csic, ctx, c, p, rgb, want, oh, orb, fb):
    """Case `c` on a host path, one chunk per call: the family, the bytes shipped (compact staging), the oracle on every
    frame, the rows outside each band and canaries on both sides of the caller's output array."""
    G, rb, ipb = 4096, fb // oh, rgb.shape[-1]
    ctx.set_option(OPT_CHUNK_BYTES, chunk_bytes(c))
    for row0, rows in launches(c):
        r0, r1 = (row0, row0 + rows) if rows > 0 else (0, oh)
        big = np.full(G + c.n * fb + G, 0xA5, np.uint8)
        out = big[G:G + c.n * fb].reshape(c.n, fb)
        before = ctx.host_bytes()
        if c.path == "host":
            ctx.process_host(p, rgb, out=out)
            stored = c.H // c.f if compact(c) else c.H
        else:
            ctx.process_host_band(p, rgb, out, r0, r1 - r0)
            in_row0, _ = csic.band_input_rows(p, r0, r1 - r0)
            stored = r1 - in_row0 // c.f
        assert ctx.last_kernel()[0] == GENERIC, (c.name, r0, ctx.last_kernel())
        assert ctx.host_bytes() - before == c.n * stored * c.W * ipb, (c.name, r0, "bytes shipped")
        o = out.reshape(c.n, oh, rb)[:, :, :orb]
        first_difference(c, o[:, r0:r1], want[:, r0:r1], r0)
        o[:, r0:r1] = 0xA5
        assert (big == 0xA5).all(), f"{c.name}: band {r0}..{r1}: a write outside the band's rows"


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=[c.name for c in CASES])
def test_gather_walk_on_gpu(csic, gctx, live_gather_plans, c):
    ops = tuple(ORD[ch] for ch in c.order)
    p = csic.make_params(c.W, c.H, c.a, c.b, *c.q, c.f, ops, c.rm, c.pool, c.fmt, c.inf)
    po = oracle.make_params(c.W, c.H, c.a, c.b, c.q, c.f, c.order, c.rm, c.pool, c.fmt, c.inf)
    ipb = 3 if c.inf == 0 else 4
    _, oh, orb, fb = csic.out_shape(p)
    if c.fmt == PLANAR:
        oh, orb = 1, fb                                      # three planes per frame: compared as one row
    rgb = np.random.default_rng(sum(map(ord, c.name))).integers(0, 256, size=(c.n, c.H, c.W, ipb), dtype=np.uint8)
    want = oracle.process(po, rgb, threads=8).reshape(c.n, oh, orb)
    try:
        for name, v in c.opts.items():
            gctx.set_option(OPT[name], v)
        if c.path in HOST_PATHS:
            run_host(csic, gctx, c, p, rgb, want, oh, orb, fb)
            return
        got = run_device(csic, gctx, c, p, rgb, want, oh, orb, fb)
        if c.pool and c.path == "dense" and "family" not in c.opts:
            # csic_process_host re-pitches an odd AVERAGE width onto the pooling kernel where it can
            gctx.set_option(OPT_CHUNK_BYTES, 0)
            host = gctx.process_host(p, rgb)
            fam = gctx.last_kernel()[0]
            assert np.array_equal(host.reshape(got.shape), got), f"{c.name}: family {fam} on the host path differs"
    finally:
        for opt in (*OPT.values(), OPT_CHUNK_BYTES):
            gctx.set_option(opt, 0)


# ---- the LDG decoder past its first row -----------------------------------------------------------------------------
# One case: W x H of 4:a:b at factor f (planes Wo x Ho), n frames, to RGB888 or YCC888, CSIC_DEC_NO_TMA (`ldg`: a shape
# plan_decode takes, run on the LDG decoder), the output `at` bytes past a 16-byte boundary.
Ldg = namedtuple("Ldg", "name W H a b f n rgb tile ldg at labels")


def ldg(name, W, H, a, b, f, n, labels, rgb=0, forced=False, at=0):
    return Ldg(name, W, H, a, b, f, n, rgb, 0, forced, at, frozenset(labels.split()))


LDG_CASES = [
    # production declines: rows narrower than a granule; 4:4:4 chroma rows too wide for a stage (eight 4096-pixel
    # segments per row, the last one partial)
    ldg("narrow_420", 3, 40, 2, 0, 1, 1000, "declined laps narrow held", rgb=1, at=5),
    ldg("narrow_f2", 6, 80, 2, 0, 2, 1000, "declined laps narrow f2"),
    ldg("wide_444", 30000, 2, 4, 4, 1, 2400, "declined laps segments partial_seg", at=3),
    # shapes the TMA decoder takes, on the LDG decoder: held lines, hs = 4, f = 2
    ldg("held_420_rgb", 333, 50, 2, 0, 1, 130, "forced laps held", rgb=1, forced=True, at=9),
    ldg("hs4_410", 1001, 30, 1, 0, 1, 160, "forced laps held hs4", forced=True),
    ldg("f2_411_rgb", 666, 100, 1, 1, 2, 130, "forced laps f2", rgb=1, forced=True, at=2),
]


def ldg_launch(c, sms):
    """(threads, grid) of launch_expand_planar, csrc/csic_kernels.cu:422-431: a warp per 32 granules of a row up to four
    warps, a block per row, at most 2048 threads per SM."""
    Wo, Ho = dw.out_wh(c)
    threads = min(128, (-(-Wo // 4) + 31) // 32 * 32)
    return threads, min(c.n * Ho, sms * (2048 // threads))


def ldg_regimes(c, P, sms):
    Wo, Ho = dw.out_wh(c)
    got = {"declined" if P is None else "forced"}
    _, grid = ldg_launch(c, sms)
    if c.n * Ho // grid >= 2:                                 # every block takes two rows or more
        got.add("laps")
    if Wo < 4:
        got.add("narrow")
    if Wo > 4096:                                             # 4096-pixel segments per row (:373)
        got.add("segments")
        if Wo % 4096:
            got.add("partial_seg")
    hf, vf = 4 // c.a, 2 if c.b == 0 else 1
    if vf == 2 and c.f == 1:
        got.add("held")                                       # odd lines replay the line above (:358, :366)
    if max(1, hf // c.f) == 4:
        got.add("hs4")
    if c.f == 2:
        got.add("f2")
    return got


def check_ldg_plans(plans, sms):
    wrong = []
    for c in LDG_CASES:
        lost = c.labels - ldg_regimes(c, plans[c.name], sms)
        if lost:
            wrong.append(f"{c.name} no longer reaches {sorted(lost)}: {plans[c.name]}")
        if (plans[c.name] is None) == c.ldg:
            wrong.append(f"{c.name}: plan_decode {'declines' if c.ldg else 'takes'} it: {plans[c.name]}")
    assert not wrong, "\n".join(wrong)


def test_ldg_cases_reach_their_regimes(driver):
    """plan_decode declines the production cases and takes the forced ones; every case laps its grid."""
    check_ldg_plans(dw.plan_decoders(driver, B200, LDG_CASES), B200[0])
    labels = set().union(*(c.labels for c in LDG_CASES))
    assert {"declined", "forced", "narrow", "segments", "partial_seg", "held", "hs4", "f2"} <= labels
    assert all("laps" in c.labels for c in LDG_CASES)
    assert {c.rgb for c in LDG_CASES if c.ldg} == {0, 1} and {c.f for c in LDG_CASES if "narrow" in c.labels} == {1, 2}


def decode_ref(csic, p, planar, n):
    """The replay rule as a torch gather on the device (tests/test_gpu_parity.py::_planar_decode_ref): pixel (r, c)
    shows chroma sample (r // vs, c // hs); the odd lines of a vertically held stream replay the line above's last
    sample.  -> [n, h * w * 3] YCC888."""
    import torch
    w, h, _, _ = csic.out_shape(p)
    cw, chh, ob, orr = csic.planar_shape(p)
    hf, vf = 4 // p.chroma_a, (2 if p.chroma_b == 0 else 1)
    hs, vs = max(1, hf // p.factor), max(1, vf // p.factor)
    last_c = (((p.width - 1) // hf) * hf // p.factor) // hs
    rows = torch.arange(h, device="cuda")
    held = (rows & 1).bool() if vs == 2 else torch.zeros(h, dtype=torch.bool, device="cuda")
    crow = (rows - held.long()) // vs
    ccol = (torch.arange(w, device="cuda") // hs)[None, :].expand(h, w).clone()
    ccol[held] = last_c
    idx = (crow[:, None] * cw + ccol).reshape(-1)
    return torch.stack([planar[:, :w * h], planar[:, ob:ob + cw * chh][:, idx],
                        planar[:, orr:orr + cw * chh][:, idx]], -1).reshape(n, -1)


@pytest.mark.gpu
@pytest.mark.parametrize("c", LDG_CASES, ids=[c.name for c in LDG_CASES])
def test_ldg_decoder_walk_on_gpu(csic, gctx, driver, limits, c, monkeypatch):
    """Case `c` on the LDG decoder: every frame against the replay rule, the canaries on both sides of the output."""
    import torch
    from csic_b200 import _ffi
    from csic_b200.api import check
    check_ldg_plans(dw.plan_decoders(driver, limits, LDG_CASES), limits[0])
    monkeypatch.delenv("CSIC_DEC_TILE", raising=False)
    if c.ldg:
        monkeypatch.setenv("CSIC_DEC_NO_TMA", "1")
    else:
        monkeypatch.delenv("CSIC_DEC_NO_TMA", raising=False)
    p = dw.planar_params(csic, c.W, c.H, c.a, c.b, c.f)
    w, h, _, fb = csic.out_shape(p)
    g = torch.Generator(device="cuda").manual_seed(sum(map(ord, c.name)))
    planar = torch.randint(0, 256, (c.n, fb), dtype=torch.uint8, device="cuda", generator=g)   # every frame differs
    want = decode_ref(csic, p, planar, c.n)
    if c.rgb:
        want = torch.from_numpy(oracle.ycbcr2rgb_array(want.cpu().numpy().reshape(-1, 3)).reshape(c.n, -1)).cuda()
    G, size = 4096, c.n * w * h * 3
    buf = torch.full((G + c.at + size + G,), 0xA5, dtype=torch.uint8, device="cuda")
    check(_ffi.lib().csic_expand_planar_device(gctx._h, ctypes.byref(p), planar.data_ptr(), c.n,
                                               buf.data_ptr() + G + c.at, c.rgb, torch.cuda.current_stream().cuda_stream
                                               or 1))
    torch.cuda.synchronize()
    got = buf[G + c.at:G + c.at + size].view(c.n, -1)
    bad = torch.nonzero((got != want).any(1)).flatten().tolist()
    if bad:
        k = bad[0]
        i = int(torch.nonzero(got[k] != want[k])[0])
        pytest.fail(f"{c.name}: {len(bad)} of {c.n} frames differ from the replay rule; frame {k} first at row "
                    f"{i // 3 // w}, column {i // 3 % w}, channel {i % 3}")
    assert bool((buf[:G + c.at] == 0xA5).all()) and bool((buf[G + c.at + size:] == 0xA5).all()), \
        f"{c.name}: a write outside the output"
