"""The TMA-staged kernels past their first tile.  Each case of one table is planned by tests/c/plan_driver.cpp (the
library's own planner, compiled without a GPU) and claims the regimes it reaches -- a stage ring that goes round twice,
row segments, multi-row flex tiles and their dealing modes, tall batches whose tiles span frames of odd height -- so
that a planner change which stops a case from reaching its regime fails on a machine without a GPU, naming the case and
the label.  On the GPU every case runs with its options and must equal the CPU oracle on every frame (each frame holds
different bytes: a stale stage shows up as another tile's data) and the generic gather kernel on the whole batch, and
leave every byte around its output untouched."""
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
# The plan driver plans 8-bit channels, so bundle cases keep q = (8, 8, 8) (4-byte slots).
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
    case("pool_seg_sqc", 4096, 32, 2, 0, 4, 48, POOL, "laps pool_seg", order="SQC", pool=1, ctas=1),
    case("pool_seg_csq", 4096, 32, 2, 0, 4, 48, POOL, "laps pool_seg", order="CSQ", fmt=RGB888, q=(6, 5, 5), pool=1,
         ctas=1),
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
    return line + (" %d %d %d %d" % c.at if c.path == "pitched" else "")


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
    assert {"laps", "pool_seg"} <= set().union(*(c.labels for c in CASES if c.kernel == POOL))
    assert {c.path for c in CASES if c.kernel == FLEX} == {"dense", "offset", "pitched", "band"}
    assert {64, 96} <= {c.opts.get("threads") for c in CASES if c.kernel == FLEX}


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
    output rows as [n, oh, orb])."""
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
    return buf, frames[:, :out_pitch * oh].view(n, oh, out_pitch)[:, :, :orb]


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=[c.name for c in CASES])
def test_tile_walk_on_gpu(csic, gctx, live_plans, c):
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
    try:
        for name, v in c.opts.items():
            gctx.set_option(OPT[name], v)
        buf, got = launch(gctx, c, p, d_in, c.n, fb, oh, orb)
        assert gctx.last_kernel()[0] == c.kernel, (c.name, gctx.last_kernel())
        # every frame against the oracle; outside a band the rows keep their canaries
        g = got.cpu().numpy()
        bad = [k for k in range(c.n) if not np.array_equal(g[k, r0:r1], want[k, r0:r1])]
        if bad:
            k = bad[0]
            diff = np.flatnonzero(g[k, r0:r1] != want[k, r0:r1])
            pytest.fail(f"{c.name}: {len(bad)} of {c.n} frames differ from the oracle; frame {k}: {diff.size} bytes, "
                        f"first at byte {diff[0]} of rows {r0}..{r1} ({diff[0] // orb + r0}, {diff[0] % orb})")
        assert (g[:, :r0] == 0xA5).all() and (g[:, r1:] == 0xA5).all(), c.name
        # nothing else in the buffer changed: canaries, pitch padding and the bytes between frames
        got.fill_(0xA5)
        assert bool((buf == 0xA5).all()), f"{c.name}: a write outside the output rows"
        # the generic gather kernel, byte for byte over the whole buffer
        gctx.set_option(OPT["family"], 1)
        buf_gen, _ = launch(gctx, c, p, d_in, c.n, fb, oh, orb)
        assert gctx.last_kernel()[0] == GENERIC
        got.copy_(torch.from_numpy(g))
        assert torch.equal(buf, buf_gen), f"{c.name}: differs from the generic kernel"
    finally:
        for name in OPT:
            gctx.set_option(OPT[name], 0)
