"""The AVERAGE pooling kernel (family 3) on every colour.  The consumers do their own colour arithmetic -- in the
complement-domain specialisations the chroma sums are flipped once with 255*F*F - sum, which rests on fwd_nc16 < 65536
for every input -- so one wrong byte for one extreme colour would pass the random-input tests almost surely.

First pass: the 4096 x 4096 colour cube with every colour blown up to a uniform f x f block.  The mean of a uniform
block is its colour, and with the chroma stage first, no vertical hold and hf <= f every held sample is the block's own
colour; so the expected output is the oracle's f = 1, 4:4:4 output on the cube itself (same bit depths, rounding and
output format).  Second pass: blocks drawn from colours whose channels are 0, 1, 254 or 255, mixed at random inside
each block, against the oracle proper: block sums at both ends of their range and around the round-half-up point."""
import itertools

import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu

POOL = 3
YCC888, RGB888, BUNDLE64, BUNDLE128 = 0, 1, 2, 3
ORD = {"S": 1, "Q": 2, "C": 3}
N = 4096                                    # the cube: N x N pixels, colour (r, g, b) = index >> 16, >> 8, & 255
HOLDS = ((4, 4), (2, 2), (1, 1))            # (a, b) = (a, a): hf = 1, 2, 4, no vertical hold
# chroma stage first; quantiser after the pooling (MODE 2) or before it with fewer than 8 bits (MODE 0); TRUNC runs
# its own instance whatever the order
QUANT = (("CSQ", (8, 8, 8)), ("CQS", (5, 6, 4)))


@pytest.fixture(scope="module")
def csic():
    import csic_b200
    return csic_b200


@pytest.fixture(scope="module")
def ctx(csic):
    c = csic.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def expected():
    """(order, q, round_mode, out_format) -> the oracle's f = 1, 4:4:4 output on the cube, on the device."""
    import torch
    v = np.arange(N * N, dtype=np.uint32)
    cube = np.stack([(v >> 16) & 255, (v >> 8) & 255, v & 255], -1).astype(np.uint8).reshape(1, N, N, 3)
    want = {}
    for (order, q), rm, fmt in itertools.product(QUANT, (0, 1), (YCC888, RGB888)):
        po = oracle.make_params(N, N, 4, 4, q, 1, order, rm, 0, fmt, 0)
        want[order, q, rm, fmt] = torch.from_numpy(oracle.process(po, cube, threads=8).reshape(-1)).cuda()
    return want


def cube_frame(f, in_format):
    """The cube with every pixel an f x f block, as one (N f) x (N f) frame of RGB24 / RGBA32 / BGRA32 pixels; the
    fourth byte is noise."""
    import torch
    v = torch.arange(N * N, dtype=torch.int32, device="cuda")
    r, g, b = (v >> 16) & 255, (v >> 8) & 255, v & 255
    ch = [r, g, b] if in_format != 2 else [b, g, r]
    if in_format:
        ch.append(torch.zeros_like(v))
    small = torch.stack(ch, -1).to(torch.uint8).view(N, N, len(ch))
    del v, r, g, b, ch
    frame = small.repeat_interleave(f, dim=0).repeat_interleave(f, dim=1)
    del small
    if in_format:
        gen = torch.Generator(device="cuda").manual_seed(f * 10 + in_format)
        frame[..., 3] = torch.randint(0, 256, (N * f, N * f), dtype=torch.uint8, device="cuda", generator=gen)
    return frame


def run(csic, ctx, p, d_in, n, family):
    """n dense frames of d_in through csic_process_device with kernel family option `family` -> (output, the
    family that ran)."""
    import torch
    out = torch.full((n * csic.out_shape(p)[3],), 0xA5, dtype=torch.uint8, device="cuda")
    try:
        ctx.set_option(0, family)
        ctx.process_device(p, d_in.data_ptr(), n, out.data_ptr(), torch.cuda.current_stream().cuda_stream or 1)
        torch.cuda.synchronize()
        return out, ctx.last_kernel()[0]
    finally:
        ctx.set_option(0, 0)


@pytest.mark.parametrize("f", [2, 4, 8])
def test_every_colour_as_uniform_blocks(csic, ctx, expected, f):
    """All 2^24 colours through the pooling kernel at factor f: every hold width hf <= f, FLOOR and TRUNC, YCC888 and
    the fused RGB888, RGB24 / RGBA32 / BGRA32 input, the quantiser after the pooling and before it.  The frames are
    (4096 f)^2 pixels, so rows run in 2, 8 or 32 segments.  The gather kernel must give the same bytes."""
    import torch
    wrong = []
    for inf in (0, 1, 2):
        d_in = cube_frame(f, inf)
        for (a, b), (order, q), rm, fmt in itertools.product(HOLDS, QUANT, (0, 1), (YCC888, RGB888)):
            if 4 // a > f:
                continue
            ops = tuple(ORD[ch] for ch in order)
            p = csic.make_params(N * f, N * f, a, b, *q, f, ops, rm, 1, fmt, inf)
            want = expected[order, q, rm, fmt]
            for family, expect in ((0, POOL), (1, 1)):
                got, fam = run(csic, ctx, p, d_in, 1, family)
                assert fam == expect, (f, inf, a, order, rm, fmt, fam)
                if not torch.equal(got, want):
                    bad = torch.nonzero(got != want)[:, 0]
                    px = int(bad[0]) // 3
                    wrong.append(f"family {fam}, in {inf}, 4:{a}:{b} {order} q={q} rm={rm} fmt={fmt}: {bad.numel()} "
                                 f"bytes differ, first at colour #{px:06x}")
        del d_in
        torch.cuda.empty_cache()
    assert not wrong, "\n".join(wrong)


# (a, b, order, q, round_mode, out_format): each consumer specialisation -- 4:2:0 chroma first (MODE 1), no vertical
# hold (MODE 2), pooling first (MODE 3), quantiser first with fewer bits (MODE 0), TRUNC -- and a bundle format
EDGE_CONFIGS = [
    (2, 0, "CSQ", (8, 8, 8), 0, YCC888),
    (1, 0, "CSQ", (8, 8, 8), 0, RGB888),
    (4, 4, "CSQ", (8, 8, 8), 0, YCC888),
    (2, 2, "CSQ", (6, 5, 5), 0, RGB888),
    (2, 0, "SQC", (8, 8, 8), 0, YCC888),
    (1, 1, "SCQ", (8, 8, 8), 0, RGB888),
    (2, 0, "QCS", (5, 6, 4), 0, YCC888),
    (2, 0, "CSQ", (8, 8, 8), 1, YCC888),
    (4, 0, "SQC", (8, 8, 8), 1, BUNDLE128),
]


@pytest.mark.parametrize("f", [2, 4, 8])
def test_extreme_channel_blocks(csic, ctx, f):
    """Blocks whose channels take two of 0, 1, 254 and 255, mixed in a per-block proportion, against the oracle at
    factor f in every consumer specialisation; the gather kernel must agree."""
    import torch
    n, H, W = 3, 32 * f, 128 * f
    rng = np.random.default_rng(f)
    levels = np.array([0, 1, 254, 255], dtype=np.uint8)
    blocks = (n, H // f, W // f, 1, 1, 3)
    lo = levels[rng.integers(0, 4, size=blocks)]
    hi = levels[rng.integers(0, 4, size=blocks)]
    share = rng.random(size=blocks)
    pick = rng.random(size=(n, H // f, W // f, f, f, 3)) < share
    rgb = np.where(pick, hi, lo).transpose(0, 1, 3, 2, 4, 5).reshape(n, H, W, 3)
    d_in = torch.from_numpy(np.ascontiguousarray(rgb)).cuda()
    wrong = []
    for a, b, order, q, rm, fmt in EDGE_CONFIGS:
        ops = tuple(ORD[ch] for ch in order)
        p = csic.make_params(W, H, a, b, *q, f, ops, rm, 1, fmt, 0)
        want = oracle.process(oracle.make_params(W, H, a, b, q, f, order, rm, 1, fmt, 0), rgb, threads=8)
        for family, expect in ((0, POOL), (1, 1)):
            out, fam = run(csic, ctx, p, d_in, n, family)
            assert fam == expect, (f, a, b, order, rm, fmt, fam)
            got = out.cpu().numpy().reshape(want.shape)
            if not np.array_equal(got, want):
                wrong.append(f"family {fam}, 4:{a}:{b} {order} q={q} rm={rm} fmt={fmt}: "
                             f"{int((got != want).sum())} bytes differ")
    assert not wrong, "\n".join(wrong)
