"""Parity tests proper: the CUDA path, called through the C ABI (libcsic.so via ctypes), against the
CPU oracle on the same inputs.  Bit-exact: everything on this path is 8-bit integer work.

Run on the B200 box: python -m pytest tests -m gpu
"""
import itertools
import os

import numpy as np
import pytest

import oracle
from conftest import ALL_AB, ALL_ORDERS, load_png_rgb, manifest, synth_frames

pytestmark = pytest.mark.gpu

ORD = {"S": 1, "Q": 2, "C": 3}


@pytest.fixture(scope="module")
def csic():
    import csic_b200
    return csic_b200


@pytest.fixture(scope="module")
def ctx(csic):
    c = csic.Context(0)
    yield c
    c.close()


def both_params(csic, W, H, a, b, q, f, order, round_mode=0, pool_mode=0, out_format=0, in_format=0):
    ops = tuple(ORD[ch] for ch in order)
    p = csic.make_params(W, H, a, b, q[0], q[1], q[2], f, ops, round_mode, pool_mode, out_format, in_format)
    po = oracle.make_params(W, H, a, b, q, f, order, round_mode, pool_mode, out_format, in_format)
    return p, po


def run_both_kernels(ctx, p, rgb):
    """Every kernel family that can run the parameter set must produce the same bytes: the automatic choice (TMA
    row / pooling kernel when eligible), the generic gather kernel (family option 1), and the any-alignment flex
    kernel (family option 2: no TMA kernels, no re-pitching in the host path -> dense odd rows reach it as they are)."""
    ctx.set_option(0, 0)
    out_auto = ctx.process_host(p, rgb)
    fam_auto = ctx.last_kernel()[0]
    ctx.set_option(0, 1)
    out_gen = ctx.process_host(p, rgb)
    assert ctx.last_kernel()[0] == 1
    ctx.set_option(0, 2)
    out_flex = ctx.process_host(p, rgb)
    fam_flex = ctx.last_kernel()[0]
    ctx.set_option(0, 0)
    assert fam_flex in (1, 4)
    if p.pool_mode == 0 or p.factor == 1:
        case_b = p.factor > 1 and [p.op[0], p.op[1], p.op[2]].index(1) < [p.op[0], p.op[1], p.op[2]].index(3)
        if not case_b or (p.chroma_a == 4 and p.chroma_b == 4):
            assert fam_flex == 4, "every chroma-first DECIMATE pipeline must be eligible for the flex kernel"
    assert np.array_equal(out_auto, out_gen), "automatic kernel and generic kernel disagree"
    assert np.array_equal(out_flex, out_gen), "flex kernel and generic kernel disagree"
    return out_auto, fam_auto


# ---- the reference's committed outputs, through the reference-shaped API --------------------------
@pytest.mark.parametrize("entry", [e for e in manifest()["goldens"] if e["forward"] != "identity"],
                         ids=lambda e: e["file"])
def test_golden_png_gpu(csic, ctx, entry):
    rgb = load_png_rgb(entry["input"])
    want = load_png_rgb(entry["file"])
    H, W = rgb.shape[:2]
    p, _ = both_params(csic, W, H, entry["a"], entry["b"], entry["q"], entry["factor"], entry["order"],
                       round_mode=0 if entry["forward"] == "floor" else 1, out_format=1)
    out, _ = run_both_kernels(ctx, p, rgb)
    assert np.array_equal(out.reshape(want.shape), want)


def test_baseline_config0_via_legacy_enums_and_app(csic, ctx, tmp_path):
    """BASELINE.json configs[0]: in128x128.png, CHROMA_420 + Q_8BIT + sf1 -- through the legacy enum
    constructor and through ImageCompressionApp.processImage."""
    from csic_b200 import app
    from conftest import GOLDEN
    want = load_png_rgb("G_top_legacy_CHROMA_420_Q_8BIT_sf1_128x128.png")
    top = csic.ImageCompressorTop.legacy(128, 128, csic.ChromaSubsamplingMode.CHROMA_420,
                                         csic.QuantizationMode.Q_8BIT, 1, out_format=csic.OutFormat.RGB888, ctx=ctx)
    assert np.array_equal(top.process(load_png_rgb("in128x128.png"))[0], want)
    S = csic.ProcessingStep
    outp = tmp_path / "o.png"
    got = app.processImage(f"{GOLDEN}/in128x128.png", str(outp), 2, 0, 3, 3, 2, 1, S.ChromaSubsampling,
                           S.ColorQuantization, S.SpatialSampling, ctx=ctx)
    assert np.array_equal(got, want)
    assert np.array_equal(csic.ImageProcessorModel.readImage(str(outp)), want)


def test_image_processor_integration(csic, ctx):
    """SpatialDownsamplerSpec.scala:155-230: 16x16, 4:2:0, f=2 through ImageProcessor -> G23."""
    img = csic.ImageProcessorModel.readImage(__import__("conftest").GOLDEN + "/in16x16.png")
    params = csic.ImageProcessorParams(width=16, height=16, factor=2, chromaParamA=2, chromaParamB=0)
    out = csic.ImageProcessor(params, out_format=csic.OutFormat.RGB888, ctx=ctx).process(img)
    assert out.shape == (1, 8, 8, 3)
    assert np.array_equal(out[0], load_png_rgb("G_imageprocessor_420_sf2_16x16.png"))


# ---- exhaustive forward / inverse transform -------------------------------------------------------
@pytest.mark.parametrize("round_mode", [0, 1])
@pytest.mark.parametrize("out_format", [0, 1])
def test_colour_cube_exhaustive(csic, ctx, round_mode, out_format):
    """All 2^24 RGB values as one 4096x4096 frame (row kernel) -- vs the oracle."""
    v = np.arange(1 << 24, dtype=np.uint32)
    rgb = np.stack([(v >> 16) & 255, (v >> 8) & 255, v & 255], -1).astype(np.uint8).reshape(1, 4096, 4096, 3)
    p, po = both_params(csic, 4096, 4096, 4, 4, (8, 8, 8), 1, "CSQ", round_mode, 0, out_format)
    out = ctx.process_host(p, rgb)
    assert ctx.last_kernel()[0] == 2
    assert np.array_equal(out, oracle.process(po, rgb, threads=8))


def test_inverse_on_quantised_pipeline_outputs(csic, ctx):
    """The fused RGB888 reconstruction on what the forward path can produce, with 1-bit..8-bit quantisers (the
    quantiser widens the reachable YCbCr set a little); the full YCbCr cube is the next test."""
    rgb = synth_frames(2, 64, 256, seed=5)
    for q in [(8, 8, 8), (1, 1, 1), (2, 7, 3), (6, 5, 5), (3, 3, 2)]:
        p, po = both_params(csic, 256, 64, 4, 4, q, 1, "CSQ", 0, 0, 1)
        out, _ = run_both_kernels(ctx, p, rgb)
        assert np.array_equal(out, oracle.process(po, rgb))


@pytest.mark.parametrize("W,H", [(4096, 4096), (4092, 4101), (4099, 4094)], ids=["w%16", "w%4", "w odd"])
def test_inverse_exhaustive_ycc_cube(csic, ctx, W, H):
    """YCbCr2RGB.scala:17-26 / RGB2YCbCr.scala:123-132 over ALL 2^24 (Y,Cb,Cr) triples, most of which no RGB input
    reaches through the forward transform (the clamps fire on 42 / 27 / 51 % of the cube for R / G / B): a synthetic
    4:4:4 PLANAR frame whose three planes enumerate the cube is decoded on the GPU by csic_expand_planar_device (the
    same reconstruction arithmetic the fused kernels use) and compared with the oracle's ycbcr2rgb.  Three widths = the
    three paths of the TMA-staged decoder (16 pixels per thread, 4 per thread with a fixed hold pattern, any width)."""
    import torch
    n = W * H
    assert n >= 1 << 24
    v = (np.arange(n, dtype=np.uint32) * np.uint32(2654435761 if W != 4096 else 1)) & 0xFFFFFF   # odd multiplier: a bijection mod 2^24
    assert W == 4096 or len(np.unique(v[:1 << 24])) == 1 << 24
    y, cb, cr = ((v >> 16) & 255).astype(np.uint8), ((v >> 8) & 255).astype(np.uint8), (v & 255).astype(np.uint8)
    p, _ = both_params(csic, W, H, 4, 4, (8, 8, 8), 1, "CSQ", 0, 0, 4)
    planar = np.concatenate([y, cb, cr])
    assert planar.size == csic.out_shape(p)[3]
    want_ycc = np.stack([y, cb, cr], -1)
    want_rgb = oracle.ycbcr2rgb_array(want_ycc)
    # the clamps really fire on this input (and on far more of it than the forward map can reach)
    wide = want_ycc.astype(np.int32)
    r_raw = (298 * wide[:, 0] + 409 * (wide[:, 2] - 128) + 128) >> 8
    assert 0.35 < np.mean((r_raw < 0) | (r_raw > 255)) < 0.5
    d = torch.from_numpy(planar[None]).cuda()
    got_ycc = ctx.expand_planar_torch(p, d, to_rgb=False)
    got_rgb = ctx.expand_planar_torch(p, d, to_rgb=True)
    ctx.synchronize(); torch.cuda.synchronize()
    assert np.array_equal(got_ycc.cpu().numpy().reshape(-1, 3), want_ycc)
    assert np.array_equal(got_rgb.cpu().numpy().reshape(-1, 3), want_rgb)


# ---- every mode x order x factor x format, eligible and non-eligible shapes ------------------------
SHAPES = [(64, 16), (128, 6), (256, 9), (48, 8), (40, 12), (5, 3), (33, 7), (16, 16), (1, 1), (1024, 4)]
FORMATS = [(0, (8, 8, 8)), (0, (4, 4, 4)), (1, (6, 5, 5)), (2, (3, 3, 2)), (3, (6, 5, 5)), (3, (8, 8, 8)), (2, (8, 7, 8))]


@pytest.mark.parametrize("ab", ALL_AB, ids=lambda ab: f"4{ab[0]}{ab[1]}")
@pytest.mark.parametrize("f", [1, 2, 4, 8])
def test_mode_sweep(csic, ctx, ab, f):
    seen_rows_kernel = False
    for (W, H), order, (fmt, q), rm in itertools.product(SHAPES, ALL_ORDERS, FORMATS, (0, 1)):
        if rm == 1 and (order not in ("CSQ", "SQC") or fmt != 0):
            continue
        rgb = synth_frames(3, H, W, seed=W * 7 + H * 3 + f)
        p, po = both_params(csic, W, H, ab[0], ab[1], q, f, order, rm, 0, fmt)
        out, fam = run_both_kernels(ctx, p, rgb)
        seen_rows_kernel |= fam == 2
        want = oracle.process(po, rgb)
        assert np.array_equal(out, want), (W, H, ab, f, order, fmt, q, rm, fam)
    assert seen_rows_kernel


@pytest.mark.parametrize("order", ALL_ORDERS)
def test_average_extension(csic, ctx, order):
    """pool_mode=AVERAGE (extension, parity unpinned): the TMA pooling kernel (aligned shapes; chroma-first orders and
    pooling-first orders, whose held lines replay a block the producer warp pools itself) and the generic kernel both
    equal the oracle; 3- and 4-byte pixels; both roundings; held 4:2:0 lines both inside the tile (whole rows) and
    TMA-fetched (rows split into segments)."""
    fams = set()
    shapes = [(64, 16), (32, 8), (128, 24), (40, 8), (2048, 8), (4096, 16), (344, 16), (1368, 8)]
    for (W, H), ab, f in itertools.product(shapes, ALL_AB, (2, 4, 8)):
        if W >= 2048 and (ab not in ((2, 0), (4, 4)) or order not in ("CSQ", "QCS", "SQC")):
            continue
        if W in (344, 1368) and ab not in ((2, 0), (4, 4), (1, 1)):
            continue
        for fmt, q, inf, rm in ((0, (5, 4, 3), 0, 0), (1, (8, 8, 8), 1, 0), (3, (8, 8, 8), 0, 1), (2, (3, 3, 2), 2, 0)):
            ch = 3 if inf == 0 else 4
            rgb = np.random.default_rng(W + f + inf).integers(0, 256, size=(2, H, W, ch), dtype=np.uint8)
            p, po = both_params(csic, W, H, ab[0], ab[1], q, f, order, rm, 1, fmt, inf)
            out, fam = run_both_kernels(ctx, p, rgb)
            fams.add(fam)
            want = oracle.process(po, rgb, threads=2)
            assert np.array_equal(out, want), (W, H, ab, f, fmt, inf, fam)
            # widths that break the 16-byte rules (Wo = 43, 171, 5, ...): the host path re-pitches them in its staging
            # buffers, so the chroma-first orders still run on the pooling kernel; the same frames dense on the device
            # take the generic gather kernel
            if order.index("C") < order.index("S"):
                assert fam == 3, (W, H, ab, f, fmt, inf, fam)
            if (W // f) % 16 != 0:
                import torch
                got = ctx.process_torch(p, torch.from_numpy(rgb).cuda())
                torch.cuda.synchronize()
                assert ctx.last_kernel()[0] == 1 and np.array_equal(got.cpu().numpy(), want), (W, H, ab, f, fmt, inf)
    assert 3 in fams and fams <= {1, 3}, fams      # aligned / re-pitched shapes take the pooling kernel in every order


# ---- BASELINE.json geometries: oracle on sampled frames + size-independent properties -------------
BASELINE_CFGS = {
    # name: (W, H, a, b, q, f, order, out_format)
    "cfg2_512_422_sf2": (512, 512, 2, 2, (8, 8, 8), 2, "CSQ", 0),
    "cfg3_1080p_420_q444": (1920, 1080, 2, 0, (4, 4, 4), 1, "CSQ", 0),
    "cfg4_4k_420_sf2_bundle128": (3840, 2160, 2, 0, (8, 8, 8), 2, "CSQ", 3),
    "cfg4_4k_420_sf2_bundle128_spatial_first": (3840, 2160, 2, 0, (8, 8, 8), 2, "SQC", 3),
    "cfg5_8k_420_sf4_q16_rgb": (7680, 4320, 2, 0, (6, 5, 5), 4, "CSQ", 1),
    "cfg5_8k_420_sf4_q16_rgb_spatial_first": (7680, 4320, 2, 0, (6, 5, 5), 4, "SCQ", 1),
}


@pytest.mark.parametrize("name", list(BASELINE_CFGS))
def test_baseline_geometry(csic, ctx, name):
    import torch
    W, H, a, b, q, f, order, fmt = BASELINE_CFGS[name]
    n = 3
    g = torch.Generator(device="cuda").manual_seed(1234)
    rgb = torch.randint(0, 256, (n, H, W, 3), dtype=torch.uint8, device="cuda", generator=g)
    p, po = both_params(csic, W, H, a, b, q, f, order, 0, 0, fmt)
    ctx.set_option(0, 0)
    out = ctx.process_torch(p, rgb)
    torch.cuda.synchronize(); ctx.synchronize()
    assert ctx.last_kernel()[0] == 2, "BASELINE geometries must take the TMA row kernel"
    # (1) oracle on the middle frame
    want = oracle.process(po, rgb[1].cpu().numpy(), threads=8)[0]
    assert np.array_equal(out[1].cpu().numpy(), want)
    # (2) the independent generic kernel on all frames
    ctx.set_option(0, 1)
    out_gen = ctx.process_torch(p, rgb)
    ctx.synchronize(); ctx.set_option(0, 0)
    assert torch.equal(out, out_gen)
    ctx.set_option(0, 2)      # ... and the any-alignment flex kernel
    out_flex = ctx.process_torch(p, rgb)
    ctx.synchronize(); assert ctx.last_kernel()[0] == 4
    ctx.set_option(0, 0)
    assert torch.equal(out, out_flex)
    # (3) frames are independent: permuting the batch permutes the output
    perm = torch.tensor([2, 0, 1], device="cuda")
    out_perm = ctx.process_torch(p, rgb[perm].contiguous())
    ctx.synchronize()
    assert torch.equal(out_perm, out[perm])
    # (4) row bands tile the frame: aligned bands written into one buffer == whole-frame call
    bands = csic.band_plan(csic.out_shape(p)[1], 8, f, a, b, order.index("C") < order.index("S"))
    out_b = torch.zeros_like(out)
    for r0, rows in bands:
        ctx.process_torch(p, rgb, out=out_b, out_row0=r0, out_rows=rows)
    ctx.synchronize()
    assert torch.equal(out_b, out)
    # (5) unaligned bands too (the held-chroma row is fetched from above the band)
    out_c = torch.zeros_like(out)
    Ho = csic.out_shape(p)[1]
    cuts = [0, 1, 7, Ho // 3 + 1, Ho - 5, Ho]
    for r0, r1 in zip(cuts[:-1], cuts[1:]):
        ctx.process_torch(p, rgb, out=out_c, out_row0=r0, out_rows=r1 - r0)
    ctx.synchronize()
    assert torch.equal(out_c, out)


def test_bundle_unpacks_to_parity_layout(csic, ctx):
    """unpack(BUNDLE) == YCC888 >> shifts, for every slot width, both word sizes."""
    rgb = synth_frames(2, 32, 96, seed=9)
    for q in [(3, 3, 2), (6, 5, 5), (8, 8, 8), (1, 1, 1), (8, 4, 4), (5, 6, 5)]:
        p0, _ = both_params(csic, 96, 32, 2, 0, q, 2, "CSQ", 0, 0, 0)
        ycc = ctx.process_host(p0, rgb).reshape(2, 16, 48, 3).astype(np.uint32)
        for fmt, word in ((2, 8), (3, 16)):
            p, _ = both_params(csic, 96, 32, 2, 0, q, 2, "CSQ", 0, 0, fmt)
            _, _, rb, fb = csic.out_shape(p)
            raw = ctx.process_host(p, rgb).reshape(2, 16, rb)
            sb = 1 if sum(q) <= 8 else (2 if sum(q) <= 16 else 4)
            assert rb % word == 0
            slots = raw[..., :48 * sb].reshape(2, 16, 48, sb).astype(np.uint32)
            v = sum(slots[..., k] << (8 * k) for k in range(sb))
            y = (v >> (q[1] + q[2])) << (8 - q[0])
            cb = ((v >> q[2]) & ((1 << q[1]) - 1)) << (8 - q[1])
            cr = (v & ((1 << q[2]) - 1)) << (8 - q[2])
            assert np.array_equal(np.stack([y, cb, cr], -1), ycc)
            assert not raw[..., 48 * sb:].any()


def test_host_pipeline_chunking_and_pinned(csic, ctx):
    """csic_process_host with many small chunks (buffer ring reuse) and pinned buffers == one call."""
    W, H, n = 256, 64, 37
    rgb = synth_frames(n, H, W, seed=21)
    p, po = both_params(csic, W, H, 2, 0, (6, 5, 5), 2, "SQC", 0, 0, 3)
    want = oracle.process(po, rgb, threads=4)
    ctx.set_option(1, 3 * W * H * 3)          # 3 frames per chunk -> 13 chunks over 3 buffers
    out_small = ctx.process_host(p, rgb)
    ctx.set_option(1, 0)
    assert np.array_equal(out_small, want)
    pin_in = csic.PinnedBuffer(rgb.nbytes)
    pin_out = csic.PinnedBuffer(want.nbytes)
    pin_in.array[:] = rgb.reshape(-1)
    out = ctx.process_host(p, pin_in.array.reshape(rgb.shape), out=pin_out.array.reshape(want.shape))
    assert np.array_equal(out, want)
    pin_in.free(); pin_out.free()


def test_host_path_ships_only_the_rows_decimate_reads(csic, ctx):
    """With DECIMATE and f>1, csic_process_host copies every f-th input row only (1/f of the H2D bytes);
    results must equal the full-frame copy path and the oracle, for both stage orders and both kernels."""
    W, H, n = 128, 64, 5
    rgb = synth_frames(n, H, W, seed=33)
    for f, order, fmt in itertools.product((2, 4, 8), ("CSQ", "SQC"), (0, 3)):
        p, po = both_params(csic, W, H, 2, 0, (8, 8, 8), f, order, 0, 0, fmt)
        want = oracle.process(po, rgb)
        for family in (0, 1):
            ctx.set_option(0, family)
            b0 = ctx.host_bytes()
            got = ctx.process_host(p, rgb)
            assert ctx.host_bytes() - b0 == n * (H // f) * W * 3
            ctx.set_option(6, 1)
            b0 = ctx.host_bytes()
            full = ctx.process_host(p, rgb)
            assert ctx.host_bytes() - b0 == n * H * W * 3
            ctx.set_option(6, 0)
            assert np.array_equal(got, want) and np.array_equal(full, want), (f, order, fmt, family)
    ctx.set_option(0, 0)


def test_empty_batch_and_errors(csic, ctx):
    p, _ = both_params(csic, 16, 16, 4, 4, (8, 8, 8), 1, "CSQ")
    out = ctx.process_host(p, np.zeros((0, 16, 16, 3), np.uint8))
    assert out.shape == (0, 16 * 16 * 3)
    with pytest.raises(csic.IllegalArgumentException):
        ctx.process_band(p, 1, 1, 1, 10, 10)      # band outside the frame
    with pytest.raises(csic.IllegalArgumentException):
        csic.ImageCompressorTop(4, 4, 4, 4, 8, 8, 8, 3, 1, 2, 3)


def test_randomised_parameter_space(csic, ctx):
    """Property-style sweep: 400 random legal parameter sets (sizes incl. odd / prime / 1-pixel, every
    (a,b), order, factor, format, rounding, bit depth, pooling mode), both kernels vs the oracle."""
    # CSIC_RANDOM_CASES / CSIC_RANDOM_SEED: longer one-off runs with other seeds and any width up to 400 (run under gpurun:
    # 20000 cases x 3 seeds green at the end of round 2)
    cases, seed = int(os.environ.get("CSIC_RANDOM_CASES", "400")), os.environ.get("CSIC_RANDOM_SEED")
    rng = np.random.default_rng(int(seed) if seed else 20261018)
    widths = [1, 2, 3, 5, 16, 17, 31, 32, 48, 64, 96, 100, 128, 160, 256, 272, 320]
    if seed:
        widths = widths + list(range(1, 401))
    seen = {1: 0, 2: 0, 3: 0, 4: 0}
    for it in range(cases):
        f = int(rng.choice([1, 2, 4, 8]))
        pool = int(rng.random() < 0.15)
        W = int(rng.choice(widths)) * (f if (pool or rng.random() < 0.6) else 1)
        H = int(rng.integers(1, 24)) * (f if (pool or rng.random() < 0.6) else 1)
        a, b = ALL_AB[int(rng.integers(0, 6))]
        order = ALL_ORDERS[int(rng.integers(0, 6))]
        q = tuple(int(v) for v in rng.integers(1, 9, size=3))
        fmt = int(rng.integers(0, 4))
        rm = int(rng.random() < 0.3)
        n = int(rng.integers(1, 4))
        rgb = rng.integers(0, 256, size=(n, H, W, 3), dtype=np.uint8)
        p, po = both_params(csic, W, H, a, b, q, f, order, rm, pool, fmt)
        out, fam = run_both_kernels(ctx, p, rgb)
        seen[fam] += 1
        assert np.array_equal(out, oracle.process(po, rgb)), (it, W, H, a, b, order, q, f, fmt, rm, pool, fam)
    assert seen[2] > 50 and seen[1] + seen[4] > 20, seen        # TMA and non-TMA families were exercised


def test_writes_stay_inside_the_output_buffer(csic, ctx):
    """compute-sanitizer is closed on this GPU pool, so bound the writes ourselves: the output lives
    between two canary regions which must survive every format / factor / kernel family, full-frame and
    banded; the input is placed at the very end of its allocation-sized tensor."""
    import torch
    G = 8192
    for (W, H), f, fmt, q, order in itertools.product([(256, 32), (64, 16), (40, 9)], (1, 2, 4, 8),
                                                      (0, 1, 2, 3), [(8, 8, 8), (3, 3, 2)], ("CSQ", "SQC")):
        p, po = both_params(csic, W, H, 2, 0, q, f, order, 0, 0, fmt)
        _, oh, _, fb = csic.out_shape(p)
        n = 3
        rgb = torch.randint(0, 256, (n, H, W, 3), dtype=torch.uint8, device="cuda")
        want = torch.from_numpy(oracle.process(po, rgb.cpu().numpy())).cuda()
        for fam in (0, 1, 2):
            ctx.set_option(0, fam)
            buf = torch.full((G + n * fb + G,), 0xA5, dtype=torch.uint8, device="cuda")
            out = buf[G:G + n * fb].view(n, fb)
            ctx.process_torch(p, rgb, out=out)
            ctx.synchronize(); torch.cuda.synchronize()
            assert torch.equal(out, want)
            assert bool((buf[:G] == 0xA5).all()) and bool((buf[G + n * fb:] == 0xA5).all()), (W, H, f, fmt, fam)
            if oh >= 3:      # a middle band must not touch rows outside itself
                buf.fill_(0xA5)
                ctx.process_torch(p, rgb, out=out, out_row0=1, out_rows=oh - 2)
                ctx.synchronize(); torch.cuda.synchronize()
                rb = fb // oh
                o3 = out.view(n, oh, rb)
                assert torch.equal(o3[:, 1:oh - 1], want.view(n, oh, rb)[:, 1:oh - 1])
                assert bool((o3[:, 0] == 0xA5).all()) and bool((o3[:, oh - 1] == 0xA5).all())
    ctx.set_option(0, 0)


@pytest.mark.parametrize("in_format", [1, 2], ids=["RGBA32", "BGRA32"])
def test_four_byte_input_formats(csic, ctx, in_format):
    """RGBA32 / BGRA32 input (alpha ignored, as pixel.red/green/blue ignores it): equals the oracle, and
    equals the RGB24 path on the same colours, on aligned (row kernel) and odd (generic kernel) shapes."""
    sel = [0, 1, 2] if in_format == 1 else [2, 1, 0]
    seen = set()
    for (W, H), f, ab, order, (fmt, q) in itertools.product(
            [(64, 16), (256, 12), (128, 9), (40, 12), (33, 7)], (1, 2, 4, 8), [(4, 4), (2, 0), (1, 0)],
            ("CSQ", "SQC"), [(0, (8, 8, 8)), (1, (6, 5, 5)), (3, (8, 8, 8)), (2, (3, 3, 2))]):
        rgba = np.random.default_rng(W * 13 + f).integers(0, 256, size=(3, H, W, 4), dtype=np.uint8)
        p4, po4 = both_params(csic, W, H, ab[0], ab[1], q, f, order, 0, 0, fmt, in_format)
        p3, _ = both_params(csic, W, H, ab[0], ab[1], q, f, order, 0, 0, fmt, 0)
        out4, fam = run_both_kernels(ctx, p4, rgba)
        seen.add(fam)
        assert np.array_equal(out4, oracle.process(po4, rgba)), (W, H, f, ab, order, fmt)
        assert np.array_equal(out4, ctx.process_host(p3, np.ascontiguousarray(rgba[..., sel])))
    assert 2 in seen and seen <= {1, 2, 4}


def test_pitched_layout_any_width(csic, ctx):
    """csic_process_device_pitched: with 16-byte-multiple pitches covering the width rounded up to 16 output
    pixels, ANY width runs the TMA row kernel (columns past the frame live in the row padding); result == oracle.
    Also: csic_process_host re-pitches odd widths by itself."""
    import torch
    fams = set()
    for (W, H), f, ab, order, (fmt, q), inf in itertools.product(
            [(1000, 12), (37, 9), (5, 3), (130, 8), (250, 16)], (1, 2, 4), [(4, 4), (2, 0), (1, 1)], ("CSQ", "SQC"),
            [(0, (8, 8, 8)), (1, (6, 5, 5)), (2, (3, 3, 2)), (3, (6, 5, 5)), (3, (8, 8, 8))], (0, 1)):
        ipb = 3 if inf == 0 else 4
        n = 2
        rgb = np.random.default_rng(W * 3 + f).integers(0, 256, size=(n, H, W, ipb), dtype=np.uint8)
        p, po = both_params(csic, W, H, ab[0], ab[1], q, f, order, 0, 0, fmt, inf)
        want = oracle.process(po, rgb)
        ow, oh, orb, ofb = csic.out_shape(p)
        wp = (ow + 15) // 16 * 16
        opx = 3 if fmt < 2 else (1 if sum(q) <= 8 else (2 if sum(q) <= 16 else 4))
        in_pitch = (max(W * ipb, wp * f * ipb) + 15) // 16 * 16 + 32          # extra slack: any 16-multiple works
        out_pitch = (max(orb, wp * opx) + 15) // 16 * 16 + 16
        d_in = torch.full((n, H, in_pitch), 0x5A, dtype=torch.uint8, device="cuda")
        d_in[:, :, :W * ipb] = torch.from_numpy(rgb.reshape(n, H, W * ipb)).cuda()
        d_out = torch.full((n, oh, out_pitch), 0xA5, dtype=torch.uint8, device="cuda")
        ctx.process_device_pitched(p, d_in.data_ptr(), in_pitch, 0, n, d_out.data_ptr(), out_pitch, 0,
                                   torch.cuda.current_stream().cuda_stream or 1)
        torch.cuda.synchronize()
        fams.add(ctx.last_kernel()[0])
        got = d_out[:, :, :orb].contiguous().view(n, ofb).cpu().numpy()
        assert np.array_equal(got, want), (W, H, f, ab, order, fmt, q, inf, ctx.last_kernel()[0])
        # host path: re-pitched staging must give the same bytes
        assert np.array_equal(ctx.process_host(p, rgb), want)
    assert 2 in fams
    # a width no dense layout could serve takes the row kernel through the host path
    p, po = both_params(csic, 1000, 16, 2, 0, (8, 8, 8), 4, "CSQ", 0, 0, 0)
    rgb = synth_frames(2, 16, 1000, seed=4)
    assert np.array_equal(ctx.process_host(p, rgb), oracle.process(po, rgb)) and ctx.last_kernel()[0] == 2


def test_host_band_and_multi_context(csic, ctx):
    """csic_process_host_band moves only a band's rows across PCIe and writes only its output rows;
    csic_multi (one process, several contexts -- here three on the same GPU) splits by frames, or by aligned
    row bands when there are fewer frames than contexts.  All equal the oracle."""
    rng = np.random.default_rng(77)
    multi = csic.MultiContext([0, 0, 0])
    assert len(multi) == 3
    for (W, H), f, ab, order, (fmt, q), pool in itertools.product(
            [(128, 48), (250, 36), (64, 64)], (1, 2, 4), [(2, 0), (4, 4), (1, 0)], ("CSQ", "SQC"),
            [(0, (8, 8, 8)), (3, (6, 5, 5)), (1, (3, 3, 2))], (0, 1)):
        if pool and (W % f or H % f):
            continue
        n = 2
        rgb = rng.integers(0, 256, size=(n, H, W, 3), dtype=np.uint8)
        p, po = both_params(csic, W, H, ab[0], ab[1], q, f, order, 0, pool, fmt)
        want = oracle.process(po, rgb)
        _, oh, _, fb = csic.out_shape(p)
        rb = fb // oh
        # arbitrary (unaligned) bands tile the frame; rows outside a band stay untouched
        out = np.full((n, fb), 0xA5, np.uint8)
        cuts = sorted(set([0, oh] + [int(v) for v in rng.integers(1, oh, size=3)]))
        for r0, r1 in zip(cuts[:-1], cuts[1:]):
            before = out.copy()
            ctx.process_host_band(p, rgb, out, r0, r1 - r0)
            o3, b3 = out.reshape(n, oh, rb), before.reshape(n, oh, rb)
            assert np.array_equal(o3[:, :r0], b3[:, :r0]) and np.array_equal(o3[:, r1:], b3[:, r1:])
        assert np.array_equal(out, want), (W, H, f, ab, order, fmt, pool)
        # fewer frames than contexts -> row bands; more -> frame shards
        assert np.array_equal(multi.process_host(p, rgb), want)
        rgb7 = np.concatenate([rgb] * 4)[:7]
        assert np.array_equal(multi.process_host(p, rgb7), np.concatenate([want] * 4)[:7])
    multi.close()


def _multi_cases(csic):
    rng = np.random.default_rng(99)
    for (W, H), f, ab, order, (fmt, q), n in [((256, 64), 2, (2, 0), "CSQ", (3, (8, 8, 8)), 41), ((250, 36), 1, (2, 0), "CSQ", (0, (6, 5, 5)), 23),
                                             ((128, 48), 4, (2, 2), "SQC", (1, (8, 8, 8)), 17), ((512, 128), 2, (2, 0), "CSQ", (1, (6, 5, 5)), 1)]:
        rgb = rng.integers(0, 256, size=(n, H, W, 3), dtype=np.uint8)
        p, po = both_params(csic, W, H, ab[0], ab[1], q, f, order, 0, 0, fmt)
        yield p, rgb, oracle.process(po, rgb, threads=4)


def test_multi_shared_cursor_divides_the_batch(csic):
    """csic_multi_process_host: every context's chunk pipeline pulls its chunks from one shared cursor (dynamic split by
    link speed).  Small chunks force many pulls per context; the even split (CSIC_OPT_MULTI_STATIC_SPLIT) and pinned /
    pageable buffers give the same bytes; the bytes shipped over all contexts add up to exactly one copy of the rows."""
    with csic.MultiContext([0, 0, 0]) as multi:
        multi.set_option(1, 64 << 10)                      # CSIC_OPT_HOST_CHUNK_BYTES on every context
        for p, rgb, want in _multi_cases(csic):
            before = sum(multi.host_bytes())
            assert np.array_equal(multi.process_host(p, rgb), want)
            shipped = sum(multi.host_bytes()) - before
            rows = p.height if p.factor == 1 else -(-p.height // p.factor)
            if p.height % p.factor == 0:
                assert shipped == rgb.shape[0] * rows * p.width * 3, (shipped, rgb.shape, p.factor)
            multi.set_option(csic.MultiContext.STATIC_SPLIT, 1)
            assert np.array_equal(multi.process_host(p, rgb), want)
            multi.set_option(csic.MultiContext.STATIC_SPLIT, 0)
        # a big pinned batch: > 8 MB so that pageable callers would bounce; here pinned in, pinned out
        p, rgb, want = next(_multi_cases(csic))
        n = 400
        pin_in, pin_out = csic.PinnedBuffer(n * rgb[0].size), csic.PinnedBuffer(n * want.shape[1])
        big = pin_in.array.reshape(n, *rgb.shape[1:])
        big[:] = np.concatenate([rgb] * (n // len(rgb) + 1))[:n]
        out = pin_out.array.reshape(n, want.shape[1])
        multi.process_host(p, big, out=out)
        assert np.array_equal(out, np.concatenate([want] * (n // len(want) + 1))[:n])
        pageable = np.array(big)                           # same batch from pageable memory: bounce pipeline per context
        assert np.array_equal(multi.process_host(p, pageable), out)
        pin_in.free(); pin_out.free()


def test_multi_on_two_different_devices(csic):
    """csic_multi_* on devices [0, 1]: two real GPUs, one host thread and one context each (VERDICT r1, weak #1)."""
    if csic.device_count() < 2:
        pytest.skip("needs two GPUs")
    with csic.MultiContext([0, 1]) as multi, csic.Context(1) as ctx1:
        assert len(multi) == 2
        multi.set_option(1, 256 << 10)
        for p, rgb, want in _multi_cases(csic):
            assert np.array_equal(multi.process_host(p, rgb), want)          # frames pulled from the shared cursor / bands when n == 1
            assert np.array_equal(ctx1.process_host(p, rgb), want)            # a plain context on the second GPU
            before = multi.host_bytes()
            multi.set_option(csic.MultiContext.STATIC_SPLIT, 1)
            assert np.array_equal(multi.process_host(p, rgb), want)
            multi.set_option(csic.MultiContext.STATIC_SPLIT, 0)
            assert all(a > b for a, b in zip(multi.host_bytes(), before)), "the even split must use both GPUs"
    with csic.MultiContext() as every:                                        # devices == NULL -> every visible GPU
        assert len(every) == csic.device_count()
        p, rgb, want = next(_multi_cases(csic))
        assert np.array_equal(every.process_host(p, rgb), want)


def test_pooling_first_many_small_frames(csic, ctx):
    """Regression (found by tools/stress.py): with pooling before the chroma stage, the rows of an odd counter line replay
    the pooled chroma of one block of the line above, which the pooling kernel's producer warp reduces and caches -- the
    cache was keyed by the line only, and a CTA's consecutive tiles are often the same line of DIFFERENT frames (static
    round-robin over a batch of small frames).  More tiles than resident CTAs, every frame different."""
    import torch
    for (W, H, f, ab, order, n) in ((640, 8, 2, (1, 0), "QSC", 150), (2176, 240, 8, (1, 0), "SQC", 5), (256, 16, 4, (2, 0), "SCQ", 300),
                                    (128, 8, 2, (2, 0), "SQC", 1200)):
        p, po = both_params(csic, W, H, ab[0], ab[1], (4, 4, 4), f, order, 0, 1, 1)
        rgb = np.random.default_rng(W + n).integers(0, 256, size=(n, H, W, 3), dtype=np.uint8)
        d = torch.from_numpy(rgb).cuda()
        ctx.set_option(0, 0)
        out = ctx.process_torch(p, d)
        ctx.synchronize()
        assert ctx.last_kernel()[0] == 3, (W, H, f, ab, order)
        ctx.set_option(0, 1)
        ref = ctx.process_torch(p, d)
        ctx.synchronize()
        ctx.set_option(0, 0)
        assert torch.equal(out, ref), (W, H, f, ab, order, n, int((out != ref).flatten().nonzero()[0]))
        pick = [0, n // 2, n - 1]
        assert np.array_equal(out[pick].cpu().numpy(), oracle.process(po, rgb[pick])), (W, H, f, ab, order)


def test_planar_output_and_decoder(csic, ctx):
    """out_format PLANAR (SURVEY 8(f) N3): Y plane + the chroma samples that survive.  Both kernels equal the oracle;
    csic_expand_planar_device replays the planes into exactly the YCC888 / RGB888 stream of the same parameters."""
    import torch
    fams = set()
    for (W, H), f, ab, order, q, inf in itertools.product(
            [(128, 16), (256, 9), (64, 64), (40, 12), (33, 7), (2048, 6)], (1, 2, 4, 8), ALL_AB,
            ("CSQ", "QCS", "SQC"), [(8, 8, 8), (5, 4, 3)], (0, 1)):
        if order == "SQC" and f > 1:
            with pytest.raises(csic.IllegalArgumentException):
                both_params(csic, W, H, ab[0], ab[1], q, f, order, 0, 0, 4, inf)
            continue
        ch = 3 if inf == 0 else 4
        rgb = np.random.default_rng(W + 7 * f).integers(0, 256, size=(3, H, W, ch), dtype=np.uint8)
        p, po = both_params(csic, W, H, ab[0], ab[1], q, f, order, 0, 0, 4, inf)
        out, fam = run_both_kernels(ctx, p, rgb)
        fams.add(fam)
        assert np.array_equal(out, oracle.process(po, rgb)), (W, H, f, ab, order, q, inf, fam)
        for to_rgb in (False, True):
            pe, _ = both_params(csic, W, H, ab[0], ab[1], q, f, order, 0, 0, 1 if to_rgb else 0, inf)
            want = ctx.process_host(pe, rgb)
            got = ctx.expand_planar_torch(p, torch.from_numpy(out).cuda(), to_rgb)
            ctx.synchronize(); torch.cuda.synchronize()
            assert np.array_equal(got.cpu().numpy().reshape(3, -1), want), (W, H, f, ab, order, to_rgb)
    assert 2 in fams and fams <= {1, 2, 4}
    cw, chh, ob, orr = csic.planar_shape(both_params(csic, 1920, 1080, 2, 0, (8, 8, 8), 1, "CSQ", 0, 0, 4)[0])
    assert (cw, chh, ob, orr) == (960, 540, 1920 * 1080, 1920 * 1080 + 960 * 540)


def _planar_decode_ref(csic, p, planar, to_rgb):
    """PLANAR -> interleaved stream, restated in numpy: pixel (r, c) shows chroma sample (r // vs, c // hs); the odd
    lines of a vertically subsampled stream replay the LAST sample of the line above (ChromaSubsampler.scala:52-65)."""
    w, h, _, fb = csic.out_shape(p)
    cw, chh, ob, orr = csic.planar_shape(p)
    f = p.factor
    hf, vf = 4 // p.chroma_a, (2 if p.chroma_b == 0 else 1)
    hs, vs = max(1, hf // f), max(1, vf // f)
    last_c = (((p.width - 1) // hf) * hf // f) // hs
    n = planar.shape[0]
    y = planar[:, :w * h].reshape(n, h, w)
    rows = np.arange(h)
    held = (rows & 1).astype(bool) if vs == 2 else np.zeros(h, bool)
    crow = (rows - held) // vs
    planes = []
    for off in (ob, orr):
        c = planar[:, off:off + cw * chh].reshape(n, chh, cw)
        full = c[:, crow][:, :, np.arange(w) // hs]
        full[:, held, :] = c[:, crow[held], last_c][:, :, None]
        planes.append(full)
    ycc = np.stack([y, planes[0], planes[1]], -1)
    return oracle.ycbcr2rgb_array(ycc) if to_rgb else ycc


@pytest.mark.parametrize("no_tma", [False, True], ids=["tma", "ldg"])
def test_decoder_any_width_and_alignment(csic, ctx, no_tma, monkeypatch):
    """csic_expand_planar_device on random planes: widths that are / are not multiples of 4 and 16, frames of one to many
    tiles (CSIC_DEC_TILE shrinks the tile so that tiles start and end mid-row and on held lines), several frames, every
    (a, b), f = 1 and 2, planar and output base pointers at every offset modulo 16 with canaries on both sides of the
    output.  The TMA-staged decoder and the LDG decoders (CSIC_DEC_NO_TMA) must both equal the numpy restatement."""
    import ctypes
    import torch
    from csic_b200 import _ffi
    from csic_b200.api import check
    if no_tma:
        monkeypatch.setenv("CSIC_DEC_NO_TMA", "1")
    rng = np.random.default_rng(11)
    shapes = [(333, 50), (1366, 25), (1918, 13), (37, 300), (4, 5), (5, 5), (7, 1), (6000, 3), (1920, 20), (31, 31), (64, 64), (9, 2),
              (3, 7), (1, 5), (2, 4)]          # rows narrower than a granule: the TMA-staged kernel declines, the LDG kernel runs
    cases = 0
    for (W, H), ab, f, tile in itertools.product(shapes, ALL_AB, (1, 2), (0, 64, 720)):
        if W % f or H % f or (tile and W * H // (f * f) > 40000) or (no_tma and tile):
            continue
        monkeypatch.setenv("CSIC_DEC_TILE", str(tile)) if tile else monkeypatch.delenv("CSIC_DEC_TILE", raising=False)
        try:
            p, _ = both_params(csic, W, H, ab[0], ab[1], (8, 8, 8), f, "CSQ", 0, 0, 4)
        except csic.IllegalArgumentException:
            continue
        w, h, _, fb = csic.out_shape(p)
        n = 3
        planar = rng.integers(0, 256, size=(n, fb), dtype=np.uint8)
        off_in, off_out = (int(rng.integers(0, 16)), int(rng.integers(0, 16))) if cases % 3 else (0, 0)
        d_in = torch.zeros(n * fb + 64, dtype=torch.uint8, device="cuda")
        d_in[off_in:off_in + n * fb] = torch.from_numpy(planar.reshape(-1)).cuda()
        for to_rgb in (False, True):
            want = _planar_decode_ref(csic, p, planar, to_rgb).reshape(-1)
            d_out = torch.full((n * w * h * 3 + 128,), 0xA5, dtype=torch.uint8, device="cuda")
            stream = torch.cuda.current_stream().cuda_stream or 1
            check(_ffi.lib().csic_expand_planar_device(ctx._h, ctypes.byref(p), d_in.data_ptr() + off_in, n,
                                                            d_out.data_ptr() + 48 + off_out, 1 if to_rgb else 0, stream))
            torch.cuda.synchronize()
            got = d_out.cpu().numpy()
            body = got[48 + off_out:48 + off_out + want.size]
            assert np.array_equal(body, want), (W, H, ab, f, tile, to_rgb, off_in, off_out, int(np.flatnonzero(body != want)[0]))
            assert (got[:48 + off_out] == 0xA5).all() and (got[48 + off_out + want.size:] == 0xA5).all(), (W, H, ab, f, tile)
        cases += 1
    assert cases > (60 if no_tma else 200)


@pytest.mark.parametrize("W,H,ab", [(1920, 1080, (2, 0)), (1918, 1078, (2, 0)), (333, 500, (2, 2)), (1001, 999, (1, 0))],
                         ids=["1080p420", "1918x1078", "333x500", "1001x999"])
def test_decoder_full_size_batches(csic, ctx, W, H, ab):
    """The decoder at bench size with the planner's own tiles (every CTA walks many tiles and the stage ring wraps):
    32 frames of random planes against a torch gather on the device (YCC888, all frames) and the oracle's ycbcr2rgb
    (RGB888, first and last frame).  1920 takes the 16-pixel path, the other widths the column-phase path; no shape here
    takes the AL4 path or mixes paths in one launch -- those, and the other regimes, are tests/test_decode_walks.py's."""
    import torch
    p, _ = both_params(csic, W, H, ab[0], ab[1], (8, 8, 8), 1, "CSQ", 0, 0, 4)
    w, h, _, fb = csic.out_shape(p)
    cw, chh, ob, orr = csic.planar_shape(p)
    hf, vs = 4 // ab[0], (2 if ab[1] == 0 else 1)
    last_c = ((W - 1) // hf * hf) // hf
    n = 32
    g = torch.Generator(device="cuda").manual_seed(W + H)
    planar = torch.randint(0, 256, (n, fb), dtype=torch.uint8, device="cuda", generator=g)
    rows = torch.arange(h, device="cuda")
    held = (rows & 1).bool() if vs == 2 else torch.zeros(h, dtype=torch.bool, device="cuda")
    crow = (rows - held.long()) // vs
    ccol = (torch.arange(w, device="cuda") // hf)[None, :].expand(h, w).clone()
    ccol[held] = last_c
    idx = (crow[:, None] * cw + ccol).reshape(-1)
    want = torch.stack([planar[:, :w * h], planar[:, ob:ob + cw * chh][:, idx], planar[:, orr:orr + cw * chh][:, idx]], -1)
    got = ctx.expand_planar_torch(p, planar, to_rgb=False)
    ctx.synchronize(); torch.cuda.synchronize()
    assert torch.equal(got.reshape(n, -1, 3), want)
    rgb = ctx.expand_planar_torch(p, planar, to_rgb=True)
    ctx.synchronize(); torch.cuda.synchronize()
    for k in (0, n - 1):
        assert np.array_equal(rgb[k].cpu().numpy().reshape(-1, 3), oracle.ycbcr2rgb_array(want[k].cpu().numpy()))


def test_row_segments_and_ring_depths(csic, ctx):
    """Force rows to be split into several tiles (CSIC_OPT_TILE_BYTES small -> nsplit > 1: held chroma comes from
    TMA-fetched aux windows, per-segment stores) under other block sizes and CTAs per SM: results never change.  These
    batches are small: no CTA gets more than one tile, so no stage is reused at the forced depths; ring reuse at every
    depth is tests/test_tile_walks.py's."""
    rng = np.random.default_rng(5)
    try:
        for tile_bytes, stages, threads, ctas in [(1024, 2, 128, 1), (3072, 3, 256, 3), (6144, 4, 64, 2), (16384, 2, 512, 1)]:
            ctx.set_option(4, tile_bytes); ctx.set_option(3, stages); ctx.set_option(5, threads); ctx.set_option(2, ctas)
            for (W, H), f, ab, order, (fmt, q), inf in itertools.product(
                    [(1024, 10), (2048, 7), (512, 33)], (1, 2, 4, 8), [(2, 0), (1, 0), (4, 4)], ("CSQ", "SQC"),
                    [(0, (8, 8, 8)), (1, (6, 5, 5)), (3, (8, 8, 8)), (2, (3, 3, 2)), (4, (7, 6, 5))], (0, 1)):
                if fmt == 4 and order == "SQC" and f > 1:
                    continue
                rgb = rng.integers(0, 256, size=(2, H, W, 3 if inf == 0 else 4), dtype=np.uint8)
                p, po = both_params(csic, W, H, ab[0], ab[1], q, f, order, 0, 0, fmt, inf)
                got = ctx.process_host(p, rgb)
                assert ctx.last_kernel()[0] == 2
                assert np.array_equal(got, oracle.process(po, rgb)), (tile_bytes, stages, threads, W, H, f, ab, order, fmt, inf)
    finally:
        for opt in (2, 3, 4, 5):
            ctx.set_option(opt, 0)


def test_pageable_buffers_use_the_bounce_pipeline(csic, ctx):
    """Pageable host arrays (what a JVM / malloc caller has) go through the pinned bounce buffers with parallel
    host copies; pinned arrays go direct; with the bounce path disabled the driver stages.  Same bytes every way --
    whole frames, compacted rows, re-pitched odd widths, row bands, PLANAR."""
    rng = np.random.default_rng(8)
    ctx.set_option(1, 6 << 20)            # 6 MB chunks -> several chunks, ring reuse, deferred drains
    try:
        for (W, H, n), f, order, fmt in itertools.product([(1024, 512, 9), (1000, 300, 14)], (1, 2, 4), ("CSQ", "SQC"), (0, 3, 4)):
            if fmt == 4 and order == "SQC" and f > 1:
                continue
            rgb = rng.integers(0, 256, size=(n, H, W, 3), dtype=np.uint8)        # pageable
            p, po = both_params(csic, W, H, 2, 0, (8, 8, 8), f, order, 0, 0, fmt)
            want = oracle.process(po, rgb, threads=4)
            assert np.array_equal(ctx.process_host(p, rgb), want), (W, H, f, order, fmt)
            ctx.set_option(7, 1)
            assert np.array_equal(ctx.process_host(p, rgb), want)
            ctx.set_option(7, 0)
            if fmt != 4:
                _, oh, _, fb = csic.out_shape(p)
                out = np.zeros((n, fb), np.uint8)
                for r0, r1 in ((0, oh // 3), (oh // 3, oh)):
                    ctx.process_host_band(p, rgb, out, r0, r1 - r0)
                assert np.array_equal(out, want)
    finally:
        ctx.set_option(1, 0)


def test_flex_kernel_any_alignment_pitch_and_band(csic, ctx):
    """The flex kernel (family 4) is what dense odd-width device buffers get automatically.  It must be exact for any
    base-pointer misalignment of input and output (sub-views of a larger buffer), odd pitches, row bands, every
    format -- and touch nothing outside its output rows (canaries all around, pitch padding included)."""
    import torch
    rng = np.random.default_rng(99)
    S = torch.cuda.current_stream().cuda_stream or 1
    seen_auto = set()
    for (W, H), f, ab, order, (fmt, q), inf in itertools.product(
            [(1000, 12), (37, 9), (5, 3), (1, 4), (130, 20), (2050, 5), (4099, 3), (96, 33)], (1, 2, 4, 8),
            [(4, 4), (2, 0), (1, 0), (2, 2)], ("CSQ", "SQC"),
            [(0, (8, 8, 8)), (1, (6, 5, 5)), (2, (3, 3, 2)), (3, (6, 5, 5)), (3, (8, 8, 8)), (2, (8, 8, 8)), (4, (7, 6, 5))], (0, 2)):
        if fmt == 4 and order == "SQC" and f > 1:
            continue
        ipb = 3 if inf == 0 else 4
        n = 2
        rgb = rng.integers(0, 256, size=(n, H, W, ipb), dtype=np.uint8)
        p, po = both_params(csic, W, H, ab[0], ab[1], q, f, order, 0, 0, fmt, inf)
        want = oracle.process(po, rgb)
        ow, oh, orb, ofb = csic.out_shape(p)
        case_b = order == "SQC" and f > 1 and ab != (4, 4)      # 4:4:4 holds nothing: counter alignment is moot
        eligible = (not case_b) or (W % f == 0 and ow % (4 // ab[0]) == 0)
        # (1) dense buffers at odd byte offsets inside larger allocations
        oi, oo = int(rng.integers(0, 16)), int(rng.integers(0, 16))
        G = 256
        d_in = torch.empty(oi + rgb.size + 64, dtype=torch.uint8, device="cuda")
        d_in[oi:oi + rgb.size] = torch.from_numpy(rgb.reshape(-1)).cuda()
        buf = torch.full((G + oo + n * ofb + G,), 0xA5, dtype=torch.uint8, device="cuda")
        ctx.set_option(0, 0)
        ctx.process_device(p, d_in.data_ptr() + oi, n, buf.data_ptr() + G + oo, S)
        torch.cuda.synchronize()
        fam = ctx.last_kernel()[0]
        seen_auto.add(fam)
        if (oi or oo) and fmt != 4:
            assert fam == (4 if eligible else 1), (W, H, f, ab, order, fmt, inf, fam)
        got = buf[G + oo:G + oo + n * ofb].cpu().numpy().reshape(n, ofb)
        assert np.array_equal(got, want), (W, H, f, ab, order, fmt, q, inf, oi, oo, fam)
        assert bool((buf[:G + oo] == 0xA5).all()) and bool((buf[G + oo + n * ofb:] == 0xA5).all())
        if fmt == 4:
            continue
        # (2) odd pitches + frame strides, flex forced; pitch padding and the bytes between frames stay untouched
        ctx.set_option(0, 2)
        in_pitch, out_pitch = W * ipb + int(rng.integers(0, 40)), orb + int(rng.integers(0, 40))
        in_fs, out_fs = in_pitch * H + int(rng.integers(0, 100)), out_pitch * oh + int(rng.integers(0, 100))
        pin = torch.full((n * in_fs,), 0x5A, dtype=torch.uint8, device="cuda")
        pin_v = pin.view(n, in_fs)[:, :in_pitch * H].view(n, H, in_pitch)
        pin_v[:, :, :W * ipb] = torch.from_numpy(rgb.reshape(n, H, W * ipb)).cuda()
        pout = torch.full((n * out_fs + 64,), 0xA5, dtype=torch.uint8, device="cuda")
        ctx.process_device_pitched(p, pin.data_ptr(), in_pitch, in_fs, n, pout.data_ptr(), out_pitch, out_fs, S)
        torch.cuda.synchronize()
        assert ctx.last_kernel()[0] == (4 if eligible else 1)
        po_v = pout[:n * out_fs].view(n, out_fs)
        rows_v = po_v[:, :out_pitch * oh].view(n, oh, out_pitch)
        assert np.array_equal(rows_v[:, :, :orb].contiguous().view(n, ofb).cpu().numpy(), want), (W, H, f, ab, order, fmt, inf)
        assert bool((rows_v[:, :, orb:] == 0xA5).all()) and bool((po_v[:, out_pitch * oh:] == 0xA5).all())
        assert bool((pout[n * out_fs:] == 0xA5).all())
        # (3) a middle band writes only its rows
        if oh >= 3:
            buf.fill_(0xA5)
            ctx.process_band(p, d_in.data_ptr() + oi, n, buf.data_ptr() + G + oo, 1, oh - 2, S)
            torch.cuda.synchronize()
            o3 = buf[G + oo:G + oo + n * ofb].view(n, oh, orb)
            assert np.array_equal(o3[:, 1:oh - 1].cpu().numpy(), want.reshape(n, oh, orb)[:, 1:oh - 1])
            assert bool((o3[:, 0] == 0xA5).all()) and bool((o3[:, oh - 1] == 0xA5).all())
        ctx.set_option(0, 0)
    assert 4 in seen_auto


def test_bounce_buffers_survive_staging_growth(csic, ctx):
    """Regression: growing the device staging buffers (a larger batch after a smaller one) must not disturb the
    pinned bounce buffers of the pageable path."""
    rng = np.random.default_rng(3)
    ctx.set_option(1, 8 << 20)
    try:
        for n in (6, 3, 24, 12, 40):
            for (W, H, f, fmt) in ((1024, 512, 2, 3), (1024, 512, 1, 0)):
                rgb = rng.integers(0, 256, size=(n, H, W, 3), dtype=np.uint8)
                p, po = both_params(csic, W, H, 2, 0, (8, 8, 8), f, "CSQ", 0, 0, fmt)
                assert np.array_equal(ctx.process_host(p, rgb), oracle.process(po, rgb, threads=4)), (n, W, H, f, fmt)
            ctx.set_option(1, (8 << 20) * (1 + n % 3))
    finally:
        ctx.set_option(1, 0)


def test_full_batch_size_independent_properties(csic, ctx):
    """BASELINE configs[3] at its FULL size (1024 4K frames, 25.5 GB in / 8.5 GB out on the device), checked through
    properties that do not need the oracle to replay 8.5 G pixels: (1) three independent kernels (TMA row kernel,
    flex kernel, generic gather kernel) agree byte for byte on the whole batch; (2) splitting the batch anywhere gives
    the same bytes (frames are independent: ImageCompressorTopApp.scala:53 builds a fresh DUT per image); (3) duplicated
    frames give duplicated outputs; (4) the oracle on two frames picked from the ends."""
    import torch
    free, _ = torch.cuda.mem_get_info()
    W, H, a, b, q, f, order, fmt = BASELINE_CFGS["cfg4_4k_420_sf2_bundle128"]
    n = 1024
    p, po = both_params(csic, W, H, a, b, q, f, order, 0, 0, fmt)
    fb = csic.out_shape(p)[3]
    need = n * (W * H * 3 + 2 * fb) + (2 << 30)
    if free < need:
        n = max(16, int((free - (2 << 30)) // (W * H * 3 + 2 * fb)) // 16 * 16)
    g = torch.Generator(device="cuda").manual_seed(99)
    rgb = torch.empty((n, H, W, 3), dtype=torch.uint8, device="cuda")
    for i in range(0, n, 32):
        rgb[i:i + 32] = torch.randint(0, 256, rgb[i:i + 32].shape, dtype=torch.uint8, device="cuda", generator=g)
    rgb[n - 1] = rgb[0]                                   # (3) a duplicated frame
    ctx.set_option(0, 0)
    out = ctx.process_torch(p, rgb)
    torch.cuda.synchronize(); ctx.synchronize()
    assert ctx.last_kernel()[0] == 2
    other = torch.empty_like(out)
    for fam, want_fam in ((2, 4), (1, 1)):                # (1)
        ctx.set_option(0, fam)
        ctx.process_torch(p, rgb, out=other)
        torch.cuda.synchronize(); ctx.synchronize()
        assert ctx.last_kernel()[0] == want_fam
        assert torch.equal(out, other), f"kernel family {want_fam} disagrees with the row kernel on the full batch"
    ctx.set_option(0, 0)
    cut = n // 3 + 1                                      # (2)
    other.zero_()
    ctx.process_torch(p, rgb[:cut], out=other[:cut])
    ctx.process_torch(p, rgb[cut:], out=other[cut:])
    torch.cuda.synchronize(); ctx.synchronize()
    assert torch.equal(out, other)
    assert torch.equal(out[0], out[n - 1])                # (3)
    for k in (0, n - 2):                                  # (4)
        want = oracle.process(po, rgb[k].cpu().numpy(), threads=8)[0]
        assert np.array_equal(out[k].cpu().numpy(), want)
