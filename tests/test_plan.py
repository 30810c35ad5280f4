"""The kernel planners (csrc/csic_plan.cpp) without a GPU.  tests/c/plan_driver.cpp, built with g++ from the planner and
the parameter sources, prints the kernel family and the key fields of each plan.  The pinned values are the plans the
tuned rules of DESIGN.md section 5 give on a B200 (148 SMs, 232448 bytes of opt-in shared memory per block): a change
to a tuned rule shows up here before any benchmark runs."""
import itertools
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

CSRC = os.path.join(ROOT, "chroma-subsampling-image-compressor_b200", "csrc")
B200 = ("148", "232448")
SMEM_LIMIT = 232448
FIELDS = ("family", "grid", "stages", "ctas_per_sm", "tile_rows", "nsplit", "tile_px", "n_tiles", "block_threads",
          "smem_bytes", "Ho", "n_frames", "tall_ho")
GENERIC, ROWS, POOL, FLEX = 1, 2, 3, 4


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("plandrv") / "plan_driver")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", f"-I{ROOT}/include",
                           os.path.join(ROOT, "tests", "c", "plan_driver.cpp"), os.path.join(CSRC, "csic_plan.cpp"),
                           os.path.join(CSRC, "csic_params.cpp"), "-o", exe])
    return exe


def run(driver, lines, limits=B200, env=None):
    r = subprocess.run([driver, *limits], input="\n".join(lines) + "\n", capture_output=True, text=True, timeout=300,
                       env=env)
    assert r.returncode == 0, r.stderr
    out = r.stdout.splitlines()
    assert len(out) == len(lines)
    return out


def fwd(W, H, a, b, f, ops=312, fmt=0, in_fmt=0, pool=0, n=1, row0=0, rows=-1, compact=0, family=0, stages=0,
        tile_bytes=0, block_threads=0, ctas_per_sm=0):
    """One forward case: dense, 4 KiB aligned buffers, 8/8/8 bits; ops 312 = chroma, spatial, colour."""
    return (f"F {W} {H} {a} {b} {f} {ops} {fmt} {in_fmt} {pool} {n} {row0} {rows} {compact} {family} {stages} "
            f"{tile_bytes} {block_threads} {ctas_per_sm}")


def plan(driver, line):
    vals = run(driver, [line])[0].split()
    assert vals[0] != "error", vals
    return dict(zip(FIELDS, map(int, vals)))


# (case, expected family, expected fields)
CASES = [
    # BASELINE workloads (bench.py cfg2 - cfg5, cfg4avg): the row kernel with 2 stages x 2 CTAs (cfg5: a third stage at
    # f = 4), the pooling kernel with 4 CTAs of 256 consumer threads
    ("cfg2", fwd(512, 512, 2, 2, 2, n=4096), ROWS,
     dict(stages=2, ctas_per_sm=2, tile_rows=16, nsplit=1, block_threads=256, grid=296, n_tiles=65536, smem_bytes=75424)),
    ("cfg3", fwd(1920, 1080, 2, 0, 1, n=256), ROWS,
     dict(stages=2, ctas_per_sm=2, tile_rows=4, nsplit=1, block_threads=256, grid=296, n_tiles=69120, smem_bytes=93088)),
    ("cfg4", fwd(3840, 2160, 2, 0, 2, fmt=3, n=1024), ROWS,
     dict(stages=2, ctas_per_sm=2, tile_rows=2, nsplit=1, block_threads=256, grid=296, n_tiles=552960, smem_bytes=47008)),
    ("cfg5", fwd(7680, 4320, 2, 0, 4, fmt=1, n=64), ROWS,
     dict(stages=3, ctas_per_sm=2, tile_rows=1, nsplit=1, block_threads=128, grid=296, n_tiles=69120, smem_bytes=81968)),
    ("cfg4avg", fwd(3840, 2160, 2, 0, 2, fmt=3, pool=1, n=1024), POOL,
     dict(stages=2, ctas_per_sm=4, tile_rows=1, nsplit=1, block_threads=256, grid=592, n_tiles=1105920, smem_bytes=47392)),
    # equal tiles: a band of 96 rows is two tiles of 48, not 64 + 32
    ("rows96", fwd(96, 192, 4, 4, 1, n=1024, rows=96), ROWS,
     dict(tile_rows=48, n_tiles=2048, stages=2, ctas_per_sm=3, Ho=192, n_frames=1024)),
    # tall image: 32x32 frames are one image of 4096 * 32 rows, 64-row tiles across frames; tiny tiles, 128-thread CTAs
    ("tall32", fwd(32, 32, 2, 0, 1, n=4096), ROWS,
     dict(tile_rows=64, n_tiles=2048, Ho=131072, n_frames=1, block_threads=128, ctas_per_sm=7, grid=1036)),
    # 1080p 8x8 pooling: the CTA is sized to the tile (96 consumer threads), five of them resident
    ("pool1080p8", fwd(1920, 1080, 2, 0, 8, pool=1, n=256), POOL,
     dict(block_threads=96, ctas_per_sm=5, nsplit=3, tile_px=80, tile_rows=1, grid=740)),
    # the flex row score (DESIGN.md 5.3): 1366x768 f = 1 RGB888 -> 4, 1080x1920 YCC888 -> 7, 1918x1078 -> 4,
    # 3838x2158 f = 2 -> 2; tiles across frames (tall_ho = rows of one frame)
    ("flex1366", fwd(1366, 768, 4, 4, 1, fmt=1, n=256), FLEX, dict(tile_rows=4, ctas_per_sm=4, tall_ho=768, n_frames=1)),
    ("flex1080x1920", fwd(1080, 1920, 4, 4, 1, fmt=0, n=256), FLEX, dict(tile_rows=7, tall_ho=1920)),
    ("flex1918", fwd(1918, 1078, 2, 0, 1, n=256), FLEX, dict(tile_rows=4, ctas_per_sm=3, tall_ho=1078)),
    ("flex3838", fwd(3838, 2158, 2, 0, 2, fmt=3, n=256), FLEX, dict(tile_rows=2, ctas_per_sm=3, tall_ho=1079)),
    # AVERAGE on dense odd widths: the generic kernel
    ("avg_odd", fwd(1918, 1078, 2, 0, 2, fmt=1, pool=1, n=256), GENERIC, dict(grid=2368)),
    # CSIC_OPT_KERNEL_FAMILY 1 (generic only) and 2 (no TMA row / pooling kernel) on cfg4
    ("cfg4_family1", fwd(3840, 2160, 2, 0, 2, fmt=3, n=1024, family=1), GENERIC, dict(grid=2368)),
    ("cfg4_family2", fwd(3840, 2160, 2, 0, 2, fmt=3, n=1024, family=2), FLEX,
     dict(tile_rows=2, ctas_per_sm=3, grid=444, tall_ho=1080)),
]


@pytest.mark.parametrize("line,family,want", [c[1:] for c in CASES], ids=[c[0] for c in CASES])
def test_plan_pins_design_cases(driver, line, family, want):
    got = plan(driver, line)
    assert got["family"] == family, got
    assert {k: got[k] for k in want} == want, got


def dec(W, H, a, b, f, n=1, to_rgb=0, tile=0):
    return f"D {W} {H} {a} {b} {f} {n} {to_rgb} {tile}"


def test_plan_decoder_tile_and_stages(driver):
    lines = [dec(1920, 1080, 2, 0, 1, 256), dec(1920, 1080, 2, 0, 1, 256, to_rgb=1), dec(333, 500, 2, 0, 1, 256),
             dec(3, 8, 2, 0, 1, 16), dec(4, 8, 2, 0, 1, 16), dec(1920, 1080, 2, 0, 1, 256, tile=1000)]
    got = [tuple(map(int, s.split())) for s in run(driver, lines)]
    # (ok, tile_px, stages, threads, grid, smem): 8192-pixel tiles made equal; two stages for the 16-pixel YCC888 path,
    # three for RGB888 and for widths that are not a multiple of 16; rows narrower than 4 pixels decline (the LDG
    # decoder runs); the tile option (CSIC_DEC_TILE) sets the tile
    assert got == [(1, 8176, 2, 288, 296, 81344), (1, 8176, 3, 288, 296, 97408), (1, 7936, 3, 288, 296, 88480), (0,),
                   (1, 32, 3, 96, 16, 1024), (1, 992, 2, 96, 1184, 16064)]


def grid_lines():
    lines = []
    for W, H in [(1, 1), (3, 5), (4, 4), (5, 3), (17, 16), (32, 32), (96, 96), (333, 500), (1366, 768), (1918, 1078),
                 (1920, 1080), (3840, 2160), (7680, 4320)]:
        for (a, b), f, fmt, pool, n in itertools.product([(4, 4), (2, 0), (1, 1)], [1, 2, 8], [0, 1, 3, 4], [0, 1],
                                                         [1, 7, 1024]):
            for ops in (312, 123):
                lines.append(fwd(W, H, a, b, f, ops=ops, fmt=fmt, pool=pool, n=n))
            lines.append(fwd(W, H, a, b, f, fmt=fmt, pool=pool, n=n, stages=4, tile_bytes=8192, block_threads=128,
                             ctas_per_sm=3))
        for (a, b), f, n, rgb in itertools.product([(4, 4), (2, 0), (1, 0)], [1, 2], [1, 64], [0, 1]):
            lines.append(dec(W, H, a, b, f, n, to_rgb=rgb))
    return lines


def test_plan_invariants_over_grid(driver):
    lines = grid_lines()
    out = run(driver, lines)
    planned = 0
    for line, res in zip(lines, out):
        vals = res.split()
        if vals[0] == "error":
            continue
        v = list(map(int, vals))
        if line.startswith("F"):
            p = dict(zip(FIELDS, v))
            assert p["grid"] > 0, (line, res)
            if p["family"] != GENERIC:
                planned += 1
                assert p["smem_bytes"] <= SMEM_LIMIT and p["ctas_per_sm"] >= 1 and p["n_tiles"] > 0, (line, res)
                assert p["grid"] <= p["n_tiles"], (line, res)
        elif v[0] == 1:
            assert v[5] <= SMEM_LIMIT and v[3] >= 96 and v[4] > 0, (line, res)
    assert planned > 1000


def test_plan_depends_only_on_arguments(driver):
    """Same plans in another order and under the environment switches the planners used to read."""
    lines = grid_lines()
    base = run(driver, lines)
    env = dict(os.environ, CSIC_ROWS_NO_TALL="1", CSIC_FLEX_NO_TALL="1", CSIC_FLEX_ROWS="3", CSIC_DEC_STAGES="4",
               CSIC_DEC_THREADS="64", CSIC_DEC_TILE="1000", CSIC_DEC_NO_TMA="1")
    assert run(driver, lines[::-1], env=env)[::-1] == base


# ---- host staging (plan_host, frame_copies, band_split) ----------------------------------------------------------------
MIB = 1 << 20


def host(W, H, a, b, f, ops=312, fmt=0, in_fmt=0, pool=0, n=1, row0=0, rows=-1, full=0, chunk=16 * MIB, gpus=0):
    return f"H {W} {H} {a} {b} {f} {ops} {fmt} {in_fmt} {pool} {n} {row0} {rows} {full} {chunk} {gpus}"


def host_plans(driver, lines):
    return [None if r.startswith("error") else json.loads(r) for r in run(driver, lines)]


def copy_kind(copies):
    """one 1-D copy, one 2-D copy over all frames, or one 2-D copy per frame"""
    if len(copies) == 1:
        return "1d" if copies[0][1] == 0 else "2d"
    return "frame"


# (case, line, compact, first stored, rows stored, in pitch, out pitch, device in / out frame, frames per chunk, H2D, D2H)
# 148 SMs, 16 MiB chunks, pinned buffers.  The last case's H2D was one 2-D copy per frame before the copy rule; its band
# input is the whole frame.
HOST_CASES = [
    ("4k_bundle128", host(3840, 2160, 2, 0, 2, fmt=3, n=128), 1, 0, 1080, 11520, 7680, 12441600, 8294400, 1, "2d", "1d"),
    ("w1000_f4", host(1000, 16, 2, 0, 4, n=2), 1, 0, 4, 3072, 768, 12288, 3072, 2, "2d", "2d"),
    ("band_5_20", host(256, 64, 2, 0, 2, n=3, row0=5, rows=15), 1, 5, 15, 768, 384, 11520, 5760, 3, "frame", "frame"),
    ("band_case_b", host(128, 48, 2, 0, 2, ops=123, n=2, row0=3, rows=10), 1, 1, 12, 384, 192, 4608, 1920, 2, "frame",
     "frame"),
    ("planar1080p", host(1920, 1080, 2, 0, 1, fmt=4, n=8), 0, 0, 1080, 5760, 1920, 6220800, 3110400, 2, "1d", "1d"),
    ("rgb1366", host(1366, 768, 2, 0, 1, fmt=1, n=4), 0, 0, 768, 4128, 4128, 3170304, 3170304, 4, "2d", "2d"),
    ("avg4k", host(3840, 2160, 2, 0, 2, fmt=3, pool=1, n=16), 0, 0, 2160, 11520, 7680, 24883200, 8294400, 1, "1d", "1d"),
    ("band_whole_input", host(64, 32, 2, 0, 1, n=3, row0=1, rows=31), 0, 0, 32, 192, 192, 6144, 5952, 3, "1d", "frame"),
]


@pytest.mark.parametrize("case", HOST_CASES, ids=[c[0] for c in HOST_CASES])
def test_host_plan_pins_cases(driver, case):
    _, line, compact, first, rows_stored, in_pitch, out_pitch, in_frame, out_frame, per, h2d, d2h = case
    h = host_plans(driver, [line])[0]
    assert h is not None
    got = (h["compact"], h["first_stored"], h["in_shape"][1], h["in_pitch"], h["out_pitch"], h["in_staging"][2],
           h["out_staging"][2], h["per"])
    assert got == (compact, first, rows_stored, in_pitch, out_pitch, in_frame, out_frame, per), h
    c0 = h["chunks"][0]
    assert (copy_kind(c0["h2d"]), copy_kind(c0["d2h"])) == (h2d, d2h), c0


def covered(copies, side, size, frame_bytes=None):
    """Bytes each copy touches on one side ("dst" or "src") as a count per byte of a buffer of `size` bytes; every range
    must lie inside the buffer."""
    off, pitch = (0, 1) if side == "dst" else (2, 3)
    diff = np.zeros(size + 1, dtype=np.int64)
    for c in copies:
        width, height = (c[4], 1) if c[1] == 0 else (c[4], c[5])
        starts = c[off] + np.arange(height, dtype=np.int64) * (c[pitch] if c[1] else 0)
        assert starts.min() >= 0 and starts.max() + width <= size, (c, size)
        np.add.at(diff, starts, 1)
        np.add.at(diff, starts + width, -1)
    return np.cumsum(diff[:-1])


def host_grid_lines():
    lines = []
    sizes = [(3, 5), (6, 4), (17, 16), (64, 32), (96, 64), (128, 48), (333, 120)]
    for (W, H), (a, b), f, fmt, pool, ops in itertools.product(sizes, [(4, 4), (2, 0), (1, 0)], [1, 2, 4],
                                                                 [0, 1, 3, 4], [0, 1], [312, 123]):
        Ho = -(-H // f)
        bands = [(0, -1), (1, Ho - 1), (Ho // 3, max(1, Ho // 3))]
        for (row0, rows), (chunk, gpus) in itertools.product(bands, [(64 << 10, 0), (96 << 10, 2), (16 * MIB, 3),
                                                                     (64 << 10, 1)]):
            if rows == 0 or (row0, rows) == (0, Ho):
                continue
            lines.append(host(W, H, a, b, f, ops=ops, fmt=fmt, pool=pool, n=7, row0=row0, rows=rows, chunk=chunk,
                              gpus=gpus, full=int(W == 17)))
    return lines


def test_host_copies_over_grid(driver):
    """The copies of every chunk: D2H writes exactly the band's output rows of every frame, each byte once; H2D reads
    exactly the rows csic_band_input_rows names (every f-th when compact), each once, and ships what csic_host_bytes
    counts; staging and bounce sides stay inside their buffers.  Direct and bounce paths alike."""
    lines = host_grid_lines()
    planned = 0
    for line, h in zip(lines, host_plans(driver, lines)):
        if h is None:
            continue
        planned += 1
        t = line.split()
        H, f, n, row0, rows = int(t[2]), int(t[5]), int(t[10]), int(t[11]), int(t[12])
        irb, in_frame = h["in_shape"][0], h["in_caller"][2]
        out_frame, (ow, orows) = h["out_caller"][2], h["out_shape"]
        per, compact = h["per"], h["compact"]
        if rows < 0:
            row0, rows, lo, n_in = 0, orows, 0, H
        else:
            lo, n_in = h["in_rows"]
        # expected caller bytes: output rows [row0, row0 + rows) of every frame (a PLANAR frame is one row)
        want_out = np.zeros(n * out_frame, dtype=np.int64)
        want_in = np.zeros(n * in_frame, dtype=np.int64)
        for k in range(n):
            want_out[k * out_frame + row0 * ow: k * out_frame + (row0 + orows) * ow] = 1
            for r in range(lo, lo + n_in):
                if not compact or r % f == 0:
                    want_in[k * in_frame + r * irb: k * in_frame + (r + 1) * irb] = 1
        for path in (("h2d", "d2h"), ("gather", "scatter")):
            reads, writes = [], []
            for c in h["chunks"]:
                reads += c[path[0]]
                writes += c[path[1]]
            assert np.array_equal(covered(writes, "dst", n * out_frame), want_out), (line, path)
            assert np.array_equal(covered(reads, "src", n * in_frame), want_in), (line, path)
            shipped = sum(c[4] * (1 if c[1] == 0 else c[5]) for c in reads)
            assert shipped == n * h["in_shape"][1] * irb == int(want_in.sum()), line
        for c in h["chunks"]:
            assert c["nf"] <= per
            for name, side, buf in (("h2d", "dst", "in_staging"), ("d2h", "src", "out_staging"),
                                    ("gather", "dst", "in_bounce"), ("scatter", "src", "out_bounce"),
                                    ("b2d", "dst", "in_staging"), ("b2d", "src", "in_bounce"),
                                    ("d2b", "dst", "out_bounce"), ("d2b", "src", "out_staging")):
                width, nrows = h["in_shape"] if buf.startswith("in") else h["out_shape"]
                cov = covered(c[name], side, per * h[buf][2])
                assert cov.max() <= 1 and cov.sum() == c["nf"] * width * nrows, (line, name, side)
    assert planned > 3000


def test_band_split_matches_sharding(driver):
    import csic_b200 as csic
    cases = []
    for (a, b), f, ops, H, G in itertools.product([(4, 4), (4, 2), (2, 2), (2, 0), (1, 1), (1, 0)], [1, 2, 4, 8],
                                                  [312, 123, 231, 132], [1, 7, 16, 33, 100, 1080], [1, 2, 3, 5, 8]):
        cases.append((f"B {8 * f} {H} {a} {b} {f} {ops} {G}", (a, b, f, ops, H, G)))
    out = run(driver, [c[0] for c in cases])
    checked = 0
    for (line, (a, b, f, ops, H, G)), res in zip(cases, out):
        if res.startswith("error"):
            continue
        digits = [ops // 100, ops // 10 % 10, ops % 10]
        chroma_first = digits.index(3) < digits.index(1)   # csic_step: 3 chroma, 1 spatial
        v = list(map(int, res.split()))
        got = [(v[2 * i], v[2 * i + 1] - v[2 * i]) for i in range(G)]
        assert got == csic.sharding.band_plan(-(-H // f), G, f, a, b, chroma_first), line
        checked += 1
    assert checked > 1000
