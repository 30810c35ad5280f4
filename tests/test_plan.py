"""The kernel planners (csrc/csic_plan.cpp) without a GPU.  tests/c/plan_driver.cpp, built with g++ from the planner and
the parameter sources, prints the kernel family and the key fields of each plan.  The pinned values are the plans the
tuned rules of DESIGN.md section 5 give on a B200 (148 SMs, 232448 bytes of opt-in shared memory per block): a change
to a tuned rule shows up here before any benchmark runs."""
import itertools
import os
import subprocess

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
