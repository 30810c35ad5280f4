"""Ticket dealing in the TMA row kernel (KPlan::ticketed: f >= 2 with direct bundle stores).  A CTA's tiles after its
first come from a counter pair that the launch's last CTA zeroes again; each stream of a context has its own pair, and a
launch captured into a CUDA graph walks round robin instead (csic_last_walk reports which walk ran).  Checked here on
shapes whose tile count is not a multiple of the grid: the output equals the generic gather kernel (the static walk of
an independent kernel) byte for byte and the CPU oracle on its first and last frame, and a counter left behind or
shared -- which would make a launch skip tiles -- shows up as stale bytes: outputs are filled with a sentinel before
every launch, launches of different shapes run back to back without a synchronise, on two streams at once, and next to
concurrent replays of graphs captured on their stream."""
import numpy as np
import pytest

import oracle
import conftest  # noqa: F401  (puts the repository root on sys.path)

GENERIC, ROWS = 1, 2
BUNDLE64, BUNDLE128 = 2, 3
ORD = {"S": 1, "Q": 2, "C": 3}
SENTINEL = 0xA5

# name: (W, H, a, b, q, f, order, out_format, in_format, frames, band) -- band = (row0, rows) or None
SHAPES = {
    "cfg4_x7": (3840, 2160, 2, 0, (8, 8, 8), 2, "CSQ", BUNDLE128, 0, 7, None),        # 3780 tiles
    "cfg4s_x3": (3840, 2160, 2, 0, (8, 8, 8), 2, "SQC", BUNDLE128, 0, 3, None),       # spatial first: held pixels fetched
    "thumb32_f2": (32, 32, 2, 0, (8, 8, 8), 2, "CSQ", BUNDLE128, 0, 4099, None),      # tall batch, tiles across frames
    "cfg5_band_f4": (7680, 4320, 2, 0, (6, 5, 5), 4, "CSQ", BUNDLE64, 0, 2, (64, 333)),  # 16-bit slots, a row band
    "rgba_f8_slot8": (2048, 1024, 4, 4, (3, 3, 2), 8, "CSQ", BUNDLE64, 1, 5, None),   # 8-bit slots, 4-byte pixels
}


@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch


@pytest.fixture(scope="module")
def csic():
    import csic_b200
    return csic_b200


@pytest.fixture(scope="module")
def ctx(csic, torch):
    c = csic.Context(0)
    yield c
    c.close()


class Shape:
    """One shape: its parameters, a seeded input batch on the GPU and the generic kernel's output as the reference."""

    def __init__(self, csic, torch, ctx, name):
        W, H, a, b, q, f, order, fmt, inf, n, band = SHAPES[name]
        self.name, self.band, self.n = name, band, n
        self.p = csic.make_params(W, H, a, b, q[0], q[1], q[2], f, tuple(ORD[c] for c in order), out_format=fmt,
                                  in_format=inf)
        self.op = oracle.make_params(W, H, a, b, q, f, order, out_format=fmt, in_format=inf)
        _, oh, self.row_bytes, fb = csic.out_shape(self.p)
        ipb = 3 if inf == 0 else 4
        gen = torch.Generator(device="cuda").manual_seed(sum(map(ord, name)))
        self.rgb = torch.randint(0, 256, (n, H, W, ipb), dtype=torch.uint8, device="cuda", generator=gen)
        self.out = torch.empty((n, fb), dtype=torch.uint8, device="cuda")
        ctx.set_option(0, GENERIC)
        self.ref = torch.full_like(self.out, SENTINEL)
        self.launch(ctx, self.ref)
        ctx.set_option(0, 0)
        torch.cuda.synchronize()

    def launch(self, ctx, out):
        if self.band is None:
            ctx.process_torch(self.p, self.rgb, out=out)
        else:
            ctx.process_torch(self.p, self.rgb, out=out, out_row0=self.band[0], out_rows=self.band[1])

    def check(self, torch, out=None):
        out = self.out if out is None else out
        assert torch.equal(out, self.ref), f"{self.name}: ticketed row kernel != generic gather kernel"


@pytest.fixture(scope="module")
def shapes(csic, torch, ctx):
    return {name: Shape(csic, torch, ctx, name) for name in SHAPES}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SHAPES))
def test_ticketed_equals_static_walk_and_oracle(torch, ctx, shapes, name):
    s = shapes[name]
    s.out.fill_(SENTINEL)
    s.launch(ctx, s.out)
    assert ctx.last_kernel()[0] == ROWS and ctx.last_walk() == 1
    torch.cuda.synchronize()
    s.check(torch)
    if s.band is None:
        for k in sorted({0, s.n - 1}):
            want = oracle.process(s.op, s.rgb[k].cpu().numpy())
            assert np.array_equal(s.out[k].cpu().numpy(), want[0]), f"{name}: frame {k} != oracle"


@pytest.mark.gpu
def test_counter_resets_across_back_to_back_launches(torch, ctx, shapes):
    order = ["cfg4_x7", "thumb32_f2", "cfg5_band_f4"]
    for names in (order, order[::-1]):
        for n in names:
            shapes[n].out.fill_(SENTINEL)
        for n in names:                          # one stream, no synchronise in between
            shapes[n].launch(ctx, shapes[n].out)
            assert ctx.last_walk() == 1
        torch.cuda.synchronize()
        for n in names:
            shapes[n].check(torch)


@pytest.mark.gpu
def test_each_stream_has_its_own_counter(torch, ctx, shapes):
    a, b = shapes["cfg4_x7"], shapes["cfg4s_x3"]
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for _ in range(3):
        a.out.fill_(SENTINEL)
        b.out.fill_(SENTINEL)
        s1.wait_stream(torch.cuda.current_stream())
        s2.wait_stream(torch.cuda.current_stream())
        for _ in range(2):                       # the two streams' launches may overlap
            with torch.cuda.stream(s1):
                a.launch(ctx, a.out)
                assert ctx.last_walk() == 1
            with torch.cuda.stream(s2):
                b.launch(ctx, b.out)
                assert ctx.last_walk() == 1
        torch.cuda.synchronize()
        a.check(torch)
        b.check(torch)


def capture(torch, ctx, stream, launches):
    """One CUDA graph of `launches` [(shape, out)] captured on `stream` (warmed up there first)."""
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        for sh, out in launches:
            sh.launch(ctx, out)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        for sh, out in launches:
            sh.launch(ctx, out)
            assert ctx.last_kernel()[0] == ROWS and ctx.last_walk() == 0     # captured: round robin, no counter
    torch.cuda.synchronize()
    return g


@pytest.mark.gpu
def test_graph_replays_and_the_capture_streams_own_launches(torch, ctx, shapes):
    names = ["cfg4_x7", "rgba_f8_slot8", "cfg4_x7", "thumb32_f2"]    # K = 4 launches in one graph
    side = torch.cuda.Stream()
    g = capture(torch, ctx, side, [(shapes[n], shapes[n].out) for n in names])
    for _ in range(3):
        for n in set(names):
            shapes[n].out.fill_(SENTINEL)
        g.replay()
        torch.cuda.synchronize()
        for n in set(names):
            shapes[n].check(torch)
    # direct launches on the capture stream are ticketed and find their pair zeroed
    s = shapes["cfg4_x7"]
    for _ in range(2):
        s.out.fill_(SENTINEL)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            s.launch(ctx, s.out)
            assert ctx.last_walk() == 1
        torch.cuda.synchronize()
        s.check(torch)


@pytest.mark.gpu
def test_graphs_of_one_stream_replayed_concurrently(torch, ctx, shapes):
    """Two graphs captured on one stream, replayed at the same time on two other streams while the capture stream runs
    its own ticketed launch: nothing may share a counter."""
    a, b = shapes["cfg4_x7"], shapes["cfg4s_x3"]
    out_a, out_b, out_c = (torch.empty_like(a.out), torch.empty_like(b.out), torch.empty_like(a.out))
    cap = torch.cuda.Stream()
    ga = capture(torch, ctx, cap, [(a, out_a), (a, out_a)])
    gb = capture(torch, ctx, cap, [(b, out_b), (b, out_b)])
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for _ in range(3):
        for o in (out_a, out_b, out_c):
            o.fill_(SENTINEL)
        for s in (s1, s2, cap):
            s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s1):
            ga.replay()
        with torch.cuda.stream(s2):
            gb.replay()
        with torch.cuda.stream(cap):
            a.launch(ctx, out_c)
            assert ctx.last_walk() == 1
            a.launch(ctx, out_c)
        torch.cuda.synchronize()
        a.check(torch, out_a)
        b.check(torch, out_b)
        a.check(torch, out_c)
