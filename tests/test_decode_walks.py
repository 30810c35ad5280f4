"""The PLANAR format past its first tile, both ways.

Decoder: one table of csic_expand_planar_device cases, each planned by tests/c/plan_driver.cpp (the library's own
plan_decode, compiled without a GPU) and claiming the regimes its tiles reach -- a stage ring that goes round twice,
the three compute paths of csic_decode_kernel (16 pixels per thread, 4 with a fixed hold pattern, 4 by column phase
with the row-end clean-up pass) and per-tile switching between them, both store paths, tiles that start or end on a held
line, every consumer count, and the two ways plan_decode declines -- so that a planner change which stops a case from
reaching a regime fails on a machine without a GPU, naming the case and the label.  On the GPU every case must equal a
numpy restatement of the replay rule on every frame, leave the bytes around its output alone, and equal the LDG decoder
byte for byte.

Forward: PLANAR row bands on the row, flex and gather kernels.  A band of output rows [r0, r1) owns its Y rows and,
in each chroma plane, the chroma rows rc with r0 <= rc * vs < r1; bands that tile a frame must rebuild it, and one
band must write exactly the bytes it owns."""
import ctypes
from collections import namedtuple

import numpy as np
import pytest

import oracle
import test_tile_walks as tw
from test_tile_walks import driver  # noqa: F401  (the plan driver fixture)

B200 = tw.B200
PLANAR = 4
GENERIC, ROWS, FLEX = 1, 2, 4
CSQ = (3, 1, 2)
CSIC_EINVAL_MODE = -8
DFIELDS = ("ok", "tile_px", "stages", "threads", "grid", "smem", "tiles_per_frame", "n_tiles", "A", "cw", "hs_sh",
           "vhold", "last_c", "y_slot", "c_slot", "frame_bytes", "cb_off", "cr_off")

# One decoder case: W x H input of 4:a:b at factor f (so the planes are Wo x Ho), n frames, decoded to RGB888 or
# YCC888, CSIC_DEC_TILE (0: the planner's tile), the planes `at[0]` and the output `at[1]` bytes past a 16-byte boundary.
Dec = namedtuple("Dec", "name W H a b f n rgb tile at labels")


def dec(name, W, H, a, b, f, n, labels, rgb=0, tile=0, at=(0, 0)):
    return Dec(name, W, H, a, b, f, n, rgb, tile, at, frozenset(labels.split()))


DEC_CASES = [
    # ---- the 16-pixel path at every hold width and both outputs, every tile on its phase: ring laps at depth 2 (YCC)
    # and 3 (RGB); 400-pixel rows in 256-pixel tiles start and end tiles on held lines
    dec("w16_444", 512, 64, 4, 4, 1, 50, "laps wide nc64", tile=256),
    dec("w16_444_rgb", 512, 64, 4, 4, 1, 69, "laps wide nc64", rgb=1, tile=256),
    dec("w16_420", 400, 64, 2, 0, 1, 63, "laps wide held_first held_last_multi nc64", tile=256),
    dec("w16_420_rgb", 400, 64, 2, 0, 1, 88, "laps wide held_first held_last_multi nc64", rgb=1, tile=256),
    dec("w16_410", 400, 64, 1, 0, 1, 63, "laps wide held_first held_last_multi nc64", tile=256),
    dec("w16_410_rgb", 400, 64, 1, 0, 1, 88, "laps wide held_first held_last_multi nc64", rgb=1, tile=256),
    dec("w16_440_rgb", 512, 64, 4, 0, 1, 69, "laps wide held_first nc64", rgb=1, tile=256),
    dec("w16_422_rgb", 512, 64, 2, 2, 1, 69, "laps wide nc64", rgb=1, tile=256),
    dec("w16_411_rgb", 512, 64, 1, 1, 1, 69, "laps wide nc64", rgb=1, tile=256),
    # ---- one launch, two paths: 4:1:x frames of 8 mod 16 bytes, so the planes of every other frame are off their
    # 16-byte phase; the same with 2-byte output phase (span stores on the 16-pixel path)
    dec("mixed_411", 272, 33, 1, 1, 1, 346, "laps wide al4 mixed", tile=512),
    dec("mixed_410_rgb", 272, 34, 1, 0, 1, 459, "laps wide al4 mixed held_first held_last_multi", rgb=1, tile=512),
    dec("mixed_411_span", 272, 33, 1, 1, 1, 346, "laps wide al4 mixed span_store", tile=512, at=(0, 2)),
    # ---- AL4: rows a multiple of 4 but not of 16, or 16-pixel rows with the output (word aligned: bulk stores with a
    # head) or the planes off their 16-byte phase
    dec("al4_w16_out4_rgb", 256, 33, 2, 2, 1, 513, "laps al4 head_tail", rgb=1, tile=512, at=(0, 4)),
    dec("al4_w16_off_440", 512, 48, 4, 0, 1, 131, "laps al4 held_first", tile=512, at=(4, 0)),
    dec("al4_444", 1000, 40, 4, 4, 1, 56, "laps al4 head_tail", tile=256, at=(0, 8)),
    dec("al4_420_rgb", 1000, 40, 2, 0, 1, 186, "laps al4 held_first held_last_multi nc256", rgb=1, tile=1000,
        at=(3, 5)),
    dec("al4_410", 1000, 40, 1, 0, 1, 56, "laps al4 span_store held_first held_last_multi", tile=256, at=(0, 2)),
    # ---- any other width: granules by column phase, row ends in the clean-up pass
    dec("phase_444_rgb", 333, 50, 4, 4, 1, 133, "laps phase span_store", rgb=1, tile=256, at=(5, 3)),
    dec("phase_440", 333, 50, 4, 0, 1, 133, "laps phase held_first", tile=256, at=(9, 1)),
    dec("phase_420", 333, 50, 2, 0, 1, 133, "laps phase held_first held_last_multi", tile=256, at=(1, 0)),
    dec("phase_422", 333, 50, 2, 2, 1, 133, "laps phase", tile=256),
    dec("phase_410_rgb", 1001, 30, 1, 0, 1, 75, "laps phase held_first held_last_multi", rgb=1, tile=256),
    dec("phase_411_96", 1001, 30, 1, 1, 1, 111, "laps phase nc96", tile=384, at=(2, 6)),
    # tiles of ~270 five-pixel rows on 256 consumer threads: the clean-up loop's second stride
    dec("cleanup_5_420", 5, 2150, 2, 0, 1, 953, "laps phase held_first held_last_multi cleanup_strides nc256",
        tile=1344),
    # ---- f = 2 planes (hs 1 and 2, no held lines)
    dec("f2_hs0_wide", 1024, 128, 2, 0, 2, 50, "laps wide nc64", tile=256),
    dec("f2_hs1_wide_rgb", 1024, 128, 1, 0, 2, 69, "laps wide nc64", rgb=1, tile=256),
    dec("f2_hs0_phase", 666, 100, 2, 0, 2, 133, "laps phase", tile=256, at=(7, 0)),
    dec("f2_hs1_al4_rgb", 1000, 100, 1, 1, 2, 90, "laps al4", rgb=1, tile=256),
    # ---- the planner's own tile: a small frame is one tile
    dec("one_tile", 96, 64, 2, 0, 1, 40, "one_tile_frames"),
    # ---- plan_decode declines: rows narrower than a granule; 4:4:4 chroma rows too wide for a stage even after the
    # tile is halved to 256 pixels (the LDG decoder runs)
    dec("declined_narrow", 3, 40, 2, 0, 1, 4, "declined_narrow"),
    dec("declined_smem", 30000, 3, 4, 4, 1, 2, "declined_smem"),
]


# ---- the plan driver and the decoder's per-tile rules ---------------------------------------------------------------
def plan_decoders(driver, limits, cases=DEC_CASES):
    """{case name: the extended D line as a dict, or None where plan_decode declines}."""
    import subprocess
    lines = "".join(f"D {c.W} {c.H} {c.a} {c.b} {c.f} {c.n} {c.rgb} {c.tile} walk\n" for c in cases)
    r = subprocess.run([driver, *map(str, limits)], input=lines, capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stderr
    out = r.stdout.splitlines()
    assert len(out) == len(cases)
    plans = {}
    for c, line in zip(cases, out):
        assert not line.startswith("error"), (c.name, line)
        v = list(map(int, line.split()))
        plans[c.name] = dict(zip(DFIELDS, v)) if v[0] else None
    return plans


def out_wh(c):
    return -(-c.W // c.f), -(-c.H // c.f)


def tile_walk(c, P):
    """Per tile of the launch, what the kernel computes from it (numpy arrays, one entry per tile)."""
    Wo, _ = out_wh(c)
    tpf, T, A, cw, hs, vh, last_c = (P[k] for k in ("tiles_per_frame", "tile_px", "A", "cw", "hs_sh", "vhold", "last_c"))
    # the producer, csrc/csic_decode_kernel.cu:229-232
    t = np.arange(P["n_tiles"], dtype=np.int64)
    k = t // tpf
    p0 = (t - k * tpf) * T
    npx = np.minimum(T, A - p0)
    p1 = p0 + npx - 1
    r0, col0, r1 = p0 // Wo, p0 % Wo, p1 // Wo
    frame = c.at[0] + k * P["frame_bytes"]                # stage slots are 16-byte aligned: only addresses mod 16 matter
    y_al = (frame + p0) & 15                              # d->y_s (:242)
    h0 = (r0 & 1).astype(bool) & bool(vh)
    first = np.where(vh, r0 >> 1, r0) * cw + np.where(h0, last_c, col0 >> hs)           # (:249-250)
    cb_s, cr_s = (((frame + off + first) & 15) - first for off in (P["cb_off"], P["cr_off"]))   # the bias (:255)
    galign = (c.at[1] + (k * A + p0) * 3) & 15            # (:277)
    wide = (Wo % 16 == 0) & ((galign & 12) == 0) & (y_al == 0) & (((cb_s | cr_s) & ((16 >> hs) - 1)) == 0)   # (:281)
    wide_no_phase = (Wo % 16 == 0) & (y_al == 0) & (((cb_s | cr_s) & ((16 >> hs) - 1)) == 0)
    return dict(k=k, p0=p0, npx=npx, r0=r0, r1=r1, galign=galign, wide=wide, wide_no_phase=wide_no_phase)


def dec_regimes(c, P):
    """The labels the plan `P` (None: declined) of decoder case `c` reaches."""
    Wo, _ = out_wh(c)
    if P is None:
        return {"declined_narrow" if Wo < 4 else "declined_smem"}     # csrc/csic_plan.cpp:465, :507
    got = set()
    nc = P["threads"] - 32                                            # consumer threads (:516-517)
    got.add({64: "nc64", 96: "nc96", 256: "nc256"}.get(nc, "nc_mid"))
    if P["n_tiles"] // P["grid"] >= 2 * P["stages"] + 1:              # the CTA with the fewest tiles laps the ring twice
        got.add("laps")
    got.add("one_tile_frames" if P["tiles_per_frame"] == 1 else "many_tile_frames")
    w = tile_walk(c, P)
    wide = w["wide"]
    narrow = ~wide
    if wide.any():
        got.add("wide")
    if narrow.any():
        got.add("al4" if Wo % 4 == 0 else "phase")                   # (:283-284)
        if wide.any():
            got.add("mixed")
    bulk = (w["galign"] & 3) == 0                                     # (:290)
    length = w["npx"] * 3
    head = np.minimum(length, (16 - w["galign"]) & 15)
    tail = length - head - ((length - head) & ~15)                    # (:296)
    if bulk.any():
        got.add("bulk_store")
        if (bulk & ((head > 0) | (tail > 0))).any():
            got.add("head_tail")
    if (~bulk).any():
        got.add("span_store")
    if P["vhold"]:                                                    # (:249-251)
        if (w["r0"] & 1).any():
            got.add("held_first")
        if ((w["r1"] > w["r0"]) & (w["r1"] & 1).astype(bool)).any():
            got.add("held_last_multi")
    if Wo % 4 and (narrow & (w["r1"] - w["r0"] + 1 > nc)).any():      # row ends past NC threads (:200-201)
        got.add("cleanup_strides")
    return got


def check_dec_plans(plans):
    wrong = []
    for c in DEC_CASES:
        lost = c.labels - dec_regimes(c, plans[c.name])
        if lost:
            wrong.append(f"{c.name} no longer reaches {sorted(lost)}: {plans[c.name]}")
    assert not wrong, "\n".join(wrong)


def test_decoder_cases_reach_their_regimes(driver):
    """Every decoder case reaches every regime it claims under the B200 limits."""
    check_dec_plans(plan_decoders(driver, B200))


def test_decoder_table_covers_every_instance_and_regime(driver):
    """The table's coverage, as the decoder's tests need it -- in cases that lap the ring, except the declines and the
    one-tile frames: every csic_decode_kernel<HS, VHOLD, RGB> instance at f = 1 and the f = 2 planes of hs 1 and 2, each
    compute path at each hold width, per-tile switching, both store paths, held first and last lines, the clean-up
    stride, 64 / 96 / 256 consumer threads, and ring laps at depth 2 and 3."""
    plans = plan_decoders(driver, B200)
    lapping = [c for c in DEC_CASES if "laps" in c.labels]
    inst = {(plans[c.name]["hs_sh"], plans[c.name]["vhold"], c.rgb) for c in lapping if c.f == 1}
    assert inst == {(h, v, r) for h in (0, 1, 2) for v in (0, 1) for r in (0, 1)}, inst
    assert {plans[c.name]["hs_sh"] for c in lapping if c.f == 2} >= {0, 1}
    for path in ("wide", "al4", "phase"):
        assert {plans[c.name]["hs_sh"] for c in lapping if path in c.labels} == {0, 1, 2}, path
    need = {"mixed", "span_store", "head_tail", "held_first", "held_last_multi", "cleanup_strides", "nc64", "nc96",
            "nc256"}
    assert need <= set().union(*(c.labels for c in lapping)), need - set().union(*(c.labels for c in lapping))
    assert {plans[c.name]["stages"] for c in lapping} == {2, 3}
    # the planner's own choices of tile and stage depth are covered too, not only CSIC_DEC_TILE's
    assert any(c.tile == 0 for c in DEC_CASES if "one_tile_frames" in c.labels)
    assert {"declined_narrow", "declined_smem"} <= set().union(*(c.labels for c in DEC_CASES))
    # the (galign & 12) term of `wide` decides some tile of a lapping case: word-aligned output off its 16-byte phase
    assert any((w["wide_no_phase"] & ~w["wide"]).any() for w in (tile_walk(c, plans[c.name]) for c in lapping))


# ---- the decoder on the GPU ---------------------------------------------------------------------------------------
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
def live_dec_plans(driver):
    """The plans for this device's limits: the two values csic_create reads."""
    import torch
    prop = torch.cuda.get_device_properties(0)
    plans = plan_decoders(driver, (prop.multi_processor_count, prop.shared_memory_per_block_optin))
    check_dec_plans(plans)
    return plans


def planar_params(csic, W, H, a, b, f):
    return csic.make_params(W, H, a, b, 8, 8, 8, f, CSQ, 0, 0, PLANAR, 0)


@pytest.mark.gpu
@pytest.mark.parametrize("c", DEC_CASES, ids=[c.name for c in DEC_CASES])
def test_decode_walk_on_gpu(csic, gctx, live_dec_plans, c, monkeypatch):
    """Case `c` decoded with its tile: every frame against the replay rule, the canaries around the output, and the whole
    buffer against the LDG decoder.  Which decoder ran is not observable through the C ABI: for the declined cases the
    planner test above pins that plan_decode declines, and this test checks the result only."""
    import torch
    from csic_b200 import _ffi
    from csic_b200.api import check
    from test_gpu_parity import _planar_decode_ref
    monkeypatch.delenv("CSIC_DEC_NO_TMA", raising=False)
    if c.tile:
        monkeypatch.setenv("CSIC_DEC_TILE", str(c.tile))
    else:
        monkeypatch.delenv("CSIC_DEC_TILE", raising=False)
    p = planar_params(csic, c.W, c.H, c.a, c.b, c.f)
    w, h, _, fb = csic.out_shape(p)
    oi, oo = c.at
    rng = np.random.default_rng(sum(map(ord, c.name)))
    planar = rng.integers(0, 256, size=(c.n, fb), dtype=np.uint8)       # different bytes in every frame
    d_in = torch.zeros(oi + c.n * fb + 64, dtype=torch.uint8, device="cuda")
    d_in[oi:oi + c.n * fb] = torch.from_numpy(planar.reshape(-1)).cuda()
    want = _planar_decode_ref(csic, p, planar, c.rgb).reshape(c.n, -1)
    G, size = 4096, c.n * w * h * 3
    S = torch.cuda.current_stream().cuda_stream or 1

    def decode():
        buf = torch.full((G + oo + size + G,), 0xA5, dtype=torch.uint8, device="cuda")
        check(_ffi.lib().csic_expand_planar_device(gctx._h, ctypes.byref(p), d_in.data_ptr() + oi, c.n,
                                                   buf.data_ptr() + G + oo, c.rgb, S))
        torch.cuda.synchronize()
        return buf

    buf = decode()
    got = buf[G + oo:G + oo + size].view(c.n, -1).cpu().numpy()
    bad = [k for k in range(c.n) if not np.array_equal(got[k], want[k])]
    if bad:
        k = bad[0]
        i = int(np.flatnonzero(got[k] != want[k])[0])
        pytest.fail(f"{c.name}: {len(bad)} of {c.n} frames differ from the replay rule; frame {k} first at pixel "
                    f"{i // 3} (row {i // 3 // w}, column {i // 3 % w}), channel {i % 3}")
    assert bool((buf[:G + oo] == 0xA5).all()) and bool((buf[G + oo + size:] == 0xA5).all()), \
        f"{c.name}: a write outside the output"
    monkeypatch.setenv("CSIC_DEC_NO_TMA", "1")
    assert torch.equal(buf, decode()), f"{c.name}: differs from the LDG decoder"


# ---- PLANAR row bands -----------------------------------------------------------------------------------------------
# One band case: W x H of 4:a:b at factor f, n frames, the kernel family option (0 auto, 1 gather, 2 flex), cuts that
# tile every frame into bands, a middle band (r0, r1) that must write exactly its own bytes, the family that band must
# take, and forced options (stages, tile bytes, CTAs per SM) as in test_tile_walks.py.
Band = namedtuple("Band", "name W H a b f n family cuts mid kernel opts")


def band(name, W, H, a, b, f, n, family, cuts, mid, kernel, **opts):
    return Band(name, W, H, a, b, f, n, family, cuts, mid, kernel, opts)


BAND_CASES = [
    # the row kernel: bands that start on a chroma row, Wo a multiple of 16 * hs; the unaligned cuts go to flex
    band("rows_420", 256, 36, 2, 0, 1, 5, 0, ((0, 10, 20, 36), (0, 7, 19, 36)), (10, 22), ROWS),
    band("rows_410", 512, 30, 1, 0, 1, 4, 0, ((0, 12, 30), (0, 5, 17, 30)), (4, 12), ROWS),
    band("rows_422", 256, 20, 2, 2, 1, 4, 0, ((0, 3, 11, 20),), (3, 14), ROWS),
    band("rows_f2_420", 512, 40, 2, 0, 2, 4, 0, ((0, 5, 20),), (5, 14), ROWS),
    # a band of 2-segment rows over 31 frames on one CTA per SM at depth 2: the ring laps (checked by the F line)
    band("rows_band_laps", 1024, 40, 2, 0, 1, 31, 0, ((0, 2, 32, 40),), (2, 32), ROWS, stages=2, tile=1024, ctas=1),
    # the flex kernel: odd band starts under 4:2:0 at f = 1, widths the row kernel declines
    band("flex_420_odd", 1000, 30, 2, 0, 1, 4, 2, ((0, 7, 13, 30), (0, 1, 29, 30)), (7, 20), FLEX),
    band("flex_410_odd", 1000, 22, 1, 0, 1, 3, 2, ((0, 3, 8, 22),), (3, 16), FLEX),
    band("flex_f2_411", 600, 24, 1, 1, 2, 3, 2, ((0, 5, 12),), (1, 10), FLEX),
    band("flex_420_w256", 256, 36, 2, 0, 1, 3, 2, ((0, 9, 36),), (9, 26), FLEX),
    # the gather kernel
    band("gather_420_odd", 333, 25, 2, 0, 1, 3, 1, ((0, 7, 13, 25),), (7, 20), GENERIC),
    band("gather_f2_410", 250, 20, 1, 0, 2, 3, 1, ((0, 3, 10),), (3, 8), GENERIC),
    band("gather_422", 256, 20, 2, 2, 1, 3, 1, ((0, 11, 20),), (5, 16), GENERIC),
]
LAPPING_BAND = "rows_band_laps"


def band_case_for_driver(c):
    """The middle band of `c` as a test_tile_walks case, for the plan driver's F line."""
    return tw.case(c.name, c.W, c.H, c.a, c.b, c.f, c.n, c.kernel, "", fmt=PLANAR, path="band",
                   at=(c.mid[0], c.mid[1] - c.mid[0]), **({"family": c.family} if c.family else {}), **c.opts)


def test_band_cases_plan_their_kernel(driver):
    """Every middle band takes the kernel it names under the B200 limits, and the forced row-kernel band laps its ring."""
    import subprocess
    cases = [band_case_for_driver(c) for c in BAND_CASES]
    r = subprocess.run([driver, *map(str, B200)], input="".join(tw.driver_line(c) + "\n" for c in cases),
                       capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stderr
    for c, t, line in zip(BAND_CASES, cases, r.stdout.splitlines()):
        k = dict(zip(tw.FIELDS, map(int, line.split())))
        assert k["family"] == c.kernel, (c.name, k)
        if c.name == LAPPING_BAND:
            assert {"laps", "segments"} <= tw.regimes(t, k), (c.name, k)
    # every family, 4:2:0 / 4:2:2 / 4:1:0, f = 1 and 2, odd band starts on flex
    assert {c.kernel for c in BAND_CASES} == {ROWS, FLEX, GENERIC}
    assert {(c.a, c.b) for c in BAND_CASES} >= {(2, 0), (2, 2), (1, 0)} and {c.f for c in BAND_CASES} == {1, 2}
    assert any(c.kernel == FLEX and c.f == 1 and c.b == 0 and c.mid[0] % 2 for c in BAND_CASES)


def band_bytes(csic, p, r0, r1):
    """The bytes of one PLANAR frame that output rows [r0, r1) own: their Y rows, and the chroma rows rc with
    r0 <= rc * vs < r1 of each chroma plane."""
    w, h, _, fb = csic.out_shape(p)
    cw, ch, ob, orr = csic.planar_shape(p)
    vs = max(1, (2 if p.chroma_b == 0 else 1) // p.factor)
    m = np.zeros(fb, bool)
    m[r0 * w:r1 * w] = True
    for rc in range(ch):
        if r0 <= rc * vs < r1:
            m[ob + rc * cw:ob + (rc + 1) * cw] = True
            m[orr + rc * cw:orr + (rc + 1) * cw] = True
    return m


def test_band_cuts_own_every_byte_once(csic):
    """The ownership rule partitions a frame: the bands of every cut own each byte of the PLANAR frame exactly once."""
    for c in BAND_CASES:
        p = planar_params(csic, c.W, c.H, c.a, c.b, c.f)
        for cuts in c.cuts:
            owners = sum(band_bytes(csic, p, r0, r1).astype(int) for r0, r1 in zip(cuts[:-1], cuts[1:]))
            assert (owners == 1).all(), (c.name, cuts)


@pytest.mark.gpu
@pytest.mark.parametrize("c", BAND_CASES, ids=[c.name for c in BAND_CASES])
def test_planar_band_on_gpu(csic, gctx, c):
    """Bands that tile every frame rebuild the whole-frame output and the oracle; a middle band writes exactly the bytes
    it owns (every other byte of every frame, and the bytes around the batch, keep their canary)."""
    import torch
    p = planar_params(csic, c.W, c.H, c.a, c.b, c.f)
    po = oracle.make_params(c.W, c.H, c.a, c.b, (8, 8, 8), c.f, "CSQ", 0, 0, PLANAR, 0)
    _, oh, _, fb = csic.out_shape(p)
    rgb = np.random.default_rng(sum(map(ord, c.name))).integers(0, 256, size=(c.n, c.H, c.W, 3), dtype=np.uint8)
    want = oracle.process(po, rgb, threads=8).reshape(c.n, fb)
    d_in = torch.from_numpy(rgb).cuda()
    G, S = 4096, torch.cuda.current_stream().cuda_stream or 1

    def fresh():
        buf = torch.full((G + c.n * fb + G,), 0xA5, dtype=torch.uint8, device="cuda")
        return buf, buf.data_ptr() + G

    def frames(buf):
        assert bool((buf[:G] == 0xA5).all()) and bool((buf[G + c.n * fb:] == 0xA5).all()), f"{c.name}: outside the batch"
        return buf[G:G + c.n * fb].view(c.n, fb).cpu().numpy()

    try:
        ctx = gctx
        ctx.set_option(tw.OPT["family"], c.family)
        for name, v in c.opts.items():
            ctx.set_option(tw.OPT[name], v)
        buf, out = fresh()
        ctx.process_device(p, d_in.data_ptr(), c.n, out, S)
        torch.cuda.synchronize()
        whole = frames(buf)
        assert np.array_equal(whole, want), f"{c.name}: the whole frame differs from the oracle"
        for cuts in c.cuts:
            buf, out = fresh()
            for r0, r1 in zip(cuts[:-1], cuts[1:]):
                ctx.process_band(p, d_in.data_ptr(), c.n, out, r0, r1 - r0, S)
            torch.cuda.synchronize()
            assert np.array_equal(frames(buf), whole), f"{c.name}: bands {cuts} do not rebuild the frame"
        r0, r1 = c.mid
        buf, out = fresh()
        ctx.process_band(p, d_in.data_ptr(), c.n, out, r0, r1 - r0, S)
        torch.cuda.synchronize()
        assert ctx.last_kernel()[0] == c.kernel, (c.name, ctx.last_kernel())
        got = frames(buf)
        own = band_bytes(csic, p, r0, r1)
        assert np.array_equal(got[:, own], want[:, own]), f"{c.name}: band {c.mid} differs from the oracle"
        stray = np.flatnonzero((got[:, ~own] != 0xA5).any(0))
        assert stray.size == 0, f"{c.name}: band {c.mid} wrote byte {np.flatnonzero(~own)[stray[0]]} it does not own"
    finally:
        for name in tw.OPT:
            gctx.set_option(tw.OPT[name], 0)


@pytest.mark.gpu
def test_planar_host_layout_contracts(csic, gctx):
    """What csic_plan.cpp enforces for PLANAR: no host row bands and no pitched output (three planes are not rows), and
    a batch of fewer frames than contexts goes to one context as whole frames instead of row bands."""
    import torch
    W, H, n = 256, 32, 1
    p = planar_params(csic, W, H, 2, 0, 1)
    po = oracle.make_params(W, H, 2, 0, (8, 8, 8), 1, "CSQ", 0, 0, PLANAR, 0)
    _, _, _, fb = csic.out_shape(p)
    rgb = np.random.default_rng(4).integers(0, 256, size=(n, H, W, 3), dtype=np.uint8)
    want = oracle.process(po, rgb)
    out = np.full((n, fb), 0xA5, np.uint8)
    with pytest.raises(csic.IllegalArgumentException) as e:
        gctx.process_host_band(p, rgb, out, 2, 8)
    assert e.value.status == CSIC_EINVAL_MODE and (out == 0xA5).all()
    d_in = torch.from_numpy(rgb).cuda()
    d_out = torch.full((2 * fb + 4096,), 0xA5, dtype=torch.uint8, device="cuda")
    S = torch.cuda.current_stream().cuda_stream or 1
    for out_pitch, out_frame in ((W, 0), (0, 2 * fb), (W + 16, 2 * fb)):
        with pytest.raises(csic.IllegalArgumentException) as e:
            gctx.process_device_pitched(p, d_in.data_ptr(), W * 3, 0, n, d_out.data_ptr(), out_pitch, out_frame, S)
        assert e.value.status == CSIC_EINVAL_MODE, (out_pitch, out_frame)
    torch.cuda.synchronize()
    assert bool((d_out == 0xA5).all())
    with csic.MultiContext([0, 0, 0]) as multi:
        before = multi.host_bytes()
        assert np.array_equal(multi.process_host(p, rgb), want)
        shipped = [a - b for a, b in zip(multi.host_bytes(), before)]
        assert sorted(shipped) == [0, 0, rgb.nbytes], shipped        # one context, the whole frame
