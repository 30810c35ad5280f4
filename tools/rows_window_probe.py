"""Drift probe of the TMA row kernel: how wide the window of tiles in flight gets over one launch.

Needs a library built with -DCSIC_PROBE_WINDOW, e.g.

    cd chroma-subsampling-image-compressor_b200/csrc && \
        CSIC_LIB_OUT=/tmp/libcsic_probe.so CSIC_OBJ_DIR=/tmp/obj_probe CSIC_DEFINES=-DCSIC_PROBE_WINDOW bash build.sh
    python tools/rows_window_probe.py --lib /tmp/libcsic_probe.so [--workload cfg4] [--frames N] [--out FILE.json]

In that build the producer warp of csic_rows_kernel writes %globaltimer and its CTA for every tile it takes, and every
CTA its end time (KPlan::probe).  From one launch (after one unprobed warm-up launch) this reports, sampled over time:

* the window: max - min of the tiles the running CTAs are on (a CTA is "on" the last tile its producer took), in tiles,
  in MB of input and in frames; a grid in lockstep keeps it near one grid's worth of tiles;
* the per-CTA finish times, relative to the launch's first tile.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def analyse(rec, frames, in_bytes, samples=400):
    """rec: uint64 array (n, 2) of the probe buffer.  -> dict of the window and finish statistics."""
    import numpy as np
    used = rec[:, 0] != 0
    n_used = int(used.sum())
    end_mask = used & ((rec[:, 1] >> 32) == 1)
    n_tiles = n_used - int(end_mask.sum())
    if not used[:n_tiles].all():
        raise RuntimeError("probe buffer: not every tile was recorded")
    t0 = int(rec[:n_tiles, 0].min())
    start = (rec[:n_tiles, 0].astype(np.int64) - t0)
    cta = rec[:n_tiles, 1].astype(np.int64)
    ends = rec[n_tiles:n_used]
    grid = len(ends)
    cta_end = np.zeros(grid, dtype=np.int64)
    cta_end[(ends[:, 1] & 0xFFFFFFFF).astype(np.int64)] = ends[:, 0].astype(np.int64) - t0
    dur = int(cta_end.max())

    # per CTA: its tiles in the order it took them
    order = np.lexsort((start, cta))
    cs, ts = cta[order], start[order]
    bounds = np.searchsorted(cs, np.arange(grid + 1))
    T = np.linspace(0, dur, samples, endpoint=False)[1:]
    lo = np.full(len(T), np.iinfo(np.int64).max)
    hi = np.full(len(T), -1)
    tiles_of_cta = []
    for c in range(grid):
        a, b = bounds[c], bounds[c + 1]
        tiles_of_cta.append(b - a)
        if b == a:
            continue
        idx = np.searchsorted(ts[a:b], T, side="right") - 1          # last tile taken at or before T
        live = (idx >= 0) & (T < cta_end[c])
        cur = order[a:b][np.clip(idx, 0, None)]                       # tile numbers
        lo = np.where(live, np.minimum(lo, cur), lo)
        hi = np.where(live, np.maximum(hi, cur), hi)
    ok = hi >= 0
    width = (hi - lo)[ok]
    tpf = n_tiles / frames
    mb_per_tile = in_bytes / n_tiles / 1e6

    def stats(v):
        return {"median": float(np.median(v)), "p90": float(np.percentile(v, 90)), "max": float(v.max())}

    w = stats(width)
    series = [{"t_ms": round(float(T[ok][i]) / 1e6, 3), "tiles": int(width[i])}
              for i in np.linspace(0, len(width) - 1, 16).astype(int)]
    fin = np.sort(cta_end)
    per_cta = np.array(tiles_of_cta)
    return {
        "tiles": n_tiles, "grid": grid, "tiles_per_frame": tpf, "input_mb_per_tile": mb_per_tile,
        "launch_ms": dur / 1e6,
        "window_tiles": w,
        "window_mb_input": {k: v * mb_per_tile for k, v in w.items()},
        "window_frames": {k: v / tpf for k, v in w.items()},
        "lockstep_window_tiles": grid,
        "window_over_time": series,
        "cta_finish_ms": {"first": fin[0] / 1e6, "median": float(np.median(fin)) / 1e6, "last": fin[-1] / 1e6,
                          "spread": (fin[-1] - fin[0]) / 1e6},
        "tiles_per_cta": {"min": int(per_cta.min()), "max": int(per_cta.max())},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", required=True, help="libcsic.so built with -DCSIC_PROBE_WINDOW")
    ap.add_argument("--workload", default="cfg4")
    ap.add_argument("--frames", type=int, default=0, help="frames (default: the workload's)")
    ap.add_argument("--out", default="", help="also write the result as JSON here")
    args = ap.parse_args()
    os.environ["CSIC_LIB_PATH"] = os.path.abspath(args.lib)
    sys.path.insert(0, ROOT)
    import ctypes
    import numpy as np
    import torch
    import bench
    import csic_b200 as csic

    W, H, frames, a, b, q, f, order, fmt, _ = bench.WORKLOADS[args.workload]
    frames = args.frames or frames
    lib = csic._ffi.lib()
    if not hasattr(lib, "csic_probe_window"):
        raise SystemExit(f"{args.lib} is not a probe build (-DCSIC_PROBE_WINDOW)")
    lib.csic_probe_window.argtypes = [ctypes.c_void_p]
    ops = tuple(bench.ORD[c] for c in order)
    p = csic.make_params(W, H, a, b, q[0], q[1], q[2], f, ops, pool_mode=1 if args.workload.endswith("avg") else 0,
                         out_format=fmt)
    _, out_h, _, out_fb = csic.out_shape(p)
    rgb = bench.make_inputs(torch, frames, H, W, 3, 0x5EED)
    out = torch.empty((frames, out_fb), dtype=torch.uint8, device="cuda")
    cap = frames * out_h * 4 + 65536                 # records: one per tile (a few per output row at most), then the CTAs
    buf = torch.zeros((cap, 2), dtype=torch.int64, device="cuda")
    with csic.Context(0) as ctx:
        ctx.process_torch(p, rgb, out=out)           # warm-up, unprobed
        lib.csic_probe_window(buf.data_ptr())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ctx.process_torch(p, rgb, out=out)
        e1.record()
        torch.cuda.synchronize()
        lib.csic_probe_window(None)
        if ctx.last_kernel()[0] != 2:
            raise SystemExit("the workload does not run the TMA row kernel")
    rec = buf.cpu().numpy().view(np.uint64)
    in_bytes = frames * out_h * W * 3                # DECIMATE: the kernel reads every f-th input row
    res = {"workload": args.workload, "frames": frames, "lib": os.path.basename(args.lib),
           "gpu": torch.cuda.get_device_name(0), "event_ms": e0.elapsed_time(e1)}
    res.update(analyse(rec, frames, in_bytes))
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
