#!/usr/bin/env python3
"""bench.py -- throughput of the pixel-pipeline hot path on B200, one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg4|cfg3|cfg2|cfg5]
                    [--dump-outputs DIR]

Workload (default): BASELINE.json configs[3], the 4K batch `metric` is quoted on -- 1024 frames of
3840x2160 RGB24 per GPU, 4:2:0 (a=2,b=0) -> spatial f=2 -> 8/8/8 bits, BUNDLE128 output, one fused
kernel launch per step.  A "step" = one pass of the hot path over that batch.

  value          input megapixels / s, whole job, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e            same metric through csic_process_host (the reference-facing C-ABI call) with pinned HOST
                 buffers: H2D + kernel + D2H all inside the timed region
  roofline       algorithmic bytes (SURVEY.md 8(d) D3: DECIMATE needs only every f-th input row) / kernel time,
                 against the measured HBM copy peak of this pool (MEASURED_PEAKS.json)
  cpu_baseline   the oracle (CPU restatement of the reference, all host cores) on a bounded sample
  --impl reference   the reference's CPU path.  The Scala/Chisel reference cannot run here (no JVM), so this
                 arm times the oracle port with all host threads on bounded samples of the same workload.

Under torchrun (N > 1) every rank owns one GPU and its own shard of frames; nothing is exchanged on
the data path (torch.distributed is used for the barrier and the max-over-ranks of the time only).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# name: (W, H, frames_per_gpu, a, b, (y,cb,cr) bits, factor, order, out_format, description)
WORKLOADS = {
    "cfg4": (3840, 2160, 1024, 2, 0, (8, 8, 8), 2, "CSQ", 3,
             "BASELINE configs[3]: 3840x2160 x1024 frames, 4:2:0 + f=2 decimate + BUNDLE128"),
    "cfg4s": (3840, 2160, 1024, 2, 0, (8, 8, 8), 2, "SQC", 3,
              "BASELINE configs[3], spatial before chroma (misaligned chroma counters)"),
    "cfg3": (1920, 1080, 256, 2, 0, (4, 4, 4), 1, "CSQ", 0,
             "BASELINE configs[2]: 1920x1080 x256 frames, 4:2:0 + Y4Cb4Cr4, YCC888"),
    "cfg2": (512, 512, 4096, 2, 2, (8, 8, 8), 2, "CSQ", 0,
             "BASELINE configs[1] batched: 512x512 x4096 frames, 4:2:2 + f=2, YCC888"),
    "cfg2x1": (512, 512, 1, 2, 2, (8, 8, 8), 2, "CSQ", 0,
               "BASELINE configs[1]: ONE 512x512 frame, 4:2:2 + f=2, YCC888 (launch-latency bound)"),
    "cfg3b": (1920, 1080, 256, 2, 0, (4, 4, 4), 1, "CSQ", 3,
              "BASELINE configs[2] with 16-bit bundle slots (Y4Cb4Cr4 -> 2 B/px out, 5 B/px total)"),
    "cfg3p": (1920, 1080, 256, 2, 0, (4, 4, 4), 1, "CSQ", 4,
              "cfg3 geometry with PLANAR 4:2:0 output (Y plane + quarter-size Cb/Cr planes, 1.5 B/px out)"),
    "cfg4avg": (3840, 2160, 1024, 2, 0, (8, 8, 8), 2, "CSQ", 3,
                "AVERAGE-pooling extension on the cfg4 geometry: 4:2:0 + 2x2 mean + BUNDLE128 (reads every row)"),
    "cfg4savg": (3840, 2160, 1024, 2, 0, (8, 8, 8), 2, "SQC", 3,
                 "AVERAGE-pooling extension, pooling BEFORE chroma (the app's default order) on the cfg4 geometry"),
    "cfg5savg": (7680, 4320, 64, 2, 0, (6, 5, 5), 4, "SQC", 1,
                 "AVERAGE-pooling extension, pooling BEFORE chroma on the cfg5 geometry: 4x4 mean + Q_16BIT + RGB888"),
    "cfg5avg": (7680, 4320, 64, 2, 0, (6, 5, 5), 4, "CSQ", 1,
                "AVERAGE-pooling extension on the cfg5 geometry: 4:2:0 + 4x4 mean + Q_16BIT + RGB888"),
    "thumb128": (128, 128, 32768, 2, 0, (8, 8, 8), 1, "CSQ", 0,
                 "small frames: 128x128 x32768, 4:2:0, f=1, YCC888 (many short rows per tile)"),
    "cfg4f8": (3840, 2160, 1024, 4, 4, (8, 8, 8), 8, "SQC", 0,
               "the reference app's defaults (ImageCompressorTopApp.scala:164-173: 4:4:4, 8/8/8, sf=8, spatial -> color -> chroma) on 4K x1024"),
    "cfg4f4": (3840, 2160, 1024, 2, 0, (8, 8, 8), 4, "CSQ", 0,
               "4K x1024, 4:2:0 + f=4, YCC888"),
    "thumb64": (64, 64, 131072, 2, 0, (8, 8, 8), 1, "CSQ", 0,
                "tiny frames: 64x64 x131072, 4:2:0, f=1, YCC888 (a tile never spans two frames)"),
    "thumb32": (32, 32, 524288, 2, 0, (8, 8, 8), 1, "CSQ", 0,
                "tiny frames: 32x32 x524288, 4:2:0, f=1, YCC888"),
    "thumb256": (256, 256, 16384, 2, 0, (8, 8, 8), 2, "CSQ", 3,
                 "small frames: 256x256 x16384, 4:2:0 + f=2 + BUNDLE128"),
    "cfg3odd": (1918, 1078, 256, 2, 0, (4, 4, 4), 1, "CSQ", 0,
                "cfg3 with a width no 16-byte rule fits (1918x1078, dense): the any-alignment flex kernel"),
    "cfg4odd": (3838, 2158, 256, 2, 0, (8, 8, 8), 2, "CSQ", 3,
                "cfg4 with odd dimensions (3838x2158 x256, dense): the any-alignment flex kernel"),
    "hd_rgb": (1920, 1080, 512, 2, 0, (6, 5, 5), 1, "CSQ", 1,
               "1080p x512, 4:2:0, f=1, Q_16BIT, fused RGB888 reconstruction (every byte converted: issue-bound case)"),
    "hd_b128": (1920, 1080, 512, 2, 0, (8, 8, 8), 1, "CSQ", 3,
                "1080p x512, 4:2:0, f=1, 8/8/8, BUNDLE128 (3 B/px in, 4 B/px out)"),
    "hd_f2rgb": (1920, 1080, 512, 2, 0, (6, 5, 5), 2, "CSQ", 1,
                 "1080p x512, 4:2:0 + f=2, Q_16BIT, RGB888"),
    "wxga_rgb": (1366, 768, 1024, 2, 0, (6, 5, 5), 1, "CSQ", 1,
                 "1366x768 x1024 dense (no 16-byte rule fits), 4:2:0, f=1, RGB888: flex kernel"),
    "wxga_f2": (1366, 768, 1024, 2, 0, (8, 8, 8), 2, "CSQ", 0,
                "1366x768 x1024 dense, 4:2:0 + f=2, YCC888: flex kernel"),
    "port_f1": (1080, 1920, 512, 2, 0, (8, 8, 8), 1, "CSQ", 0,
                "1080x1920 portrait x512 dense (3240-byte rows), 4:2:0, f=1, YCC888: flex kernel"),
    "sq200_f4": (200, 200, 32768, 2, 0, (8, 8, 8), 4, "CSQ", 0,
                 "200x200 x32768, 4:2:0 + f=4, YCC888 (tiny odd frames)"),
    "sq96_f8": (96, 96, 131072, 2, 0, (8, 8, 8), 8, "CSQ", 0,
                "96x96 x131072, 4:2:0 + f=8, YCC888 (12x12 outputs)"),
    "oddavg": (1366, 768, 512, 2, 0, (8, 8, 8), 2, "CSQ", 0,
               "AVERAGE extension on 1366x768 (Wo = 683: breaks the pooling kernel's 16-byte rules)"),
    "thumb96rgb": (96, 96, 65536, 2, 0, (6, 5, 5), 1, "CSQ", 1,
                   "96x96 x65536, 4:2:0, f=1, RGB888 (tiny frames, fused reconstruction)"),
    "cfg5": (7680, 4320, 64, 2, 0, (6, 5, 5), 4, "CSQ", 1,
             "BASELINE configs[4]: 7680x4320 x64 frames, 4:2:0 + f=4 + Q_16BIT + RGB888 reconstruct"),
}
ORD = {"S": 1, "Q": 2, "C": 3}


def algorithmic_bytes_per_frame(W, H, f, out_frame_bytes, average=False, ipb=3):
    """SURVEY.md 8(d) D3: in_required + out_bytes; DECIMATE with f>1 needs only every f-th row."""
    rows = H if (f == 1 or average) else -(-H // f)
    return ipb * W * rows + out_frame_bytes


def load_peak():
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(d["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (B200_PROFILING.md "clocks" line).
    NVML in a thread every 5 ms (the timed region is a fraction of a second); nvidia-smi -lms as fallback."""
    NAMES = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
             "hw_power_brake_slowdown": 0x80}

    def __init__(self, gpu_index):
        self.idx, self.sm, self.mask, self.max = gpu_index, [], 0, None
        self._stop = threading.Event()
        self.t = None
        self.how = None

    def _uuid_index(self):
        # CUDA_VISIBLE_DEVICES may renumber devices; NVML does not honour it
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            tok = vis.split(",")[self.idx].strip()
            return tok
        return self.idx

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            ident = self._uuid_index()
            if isinstance(ident, str) and not ident.isdigit():
                h = pynvml.nvmlDeviceGetHandleByUUID(ident.encode() if hasattr(ident, "encode") else ident)
            else:
                h = pynvml.nvmlDeviceGetHandleByIndex(int(ident))
            self.max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

            def loop():
                while not self._stop.is_set():
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        self.mask |= int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                    except Exception:
                        pass
                    time.sleep(0.005)
            self.how = "nvml"
            self.t = threading.Thread(target=loop, daemon=True)
            self.t.start()
        except Exception:
            self.how = None

    def stop(self):
        if self.how != "nvml":
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"]}
        self._stop.set()
        self.t.join(timeout=1)
        reasons = sorted(n for n, bit in self.NAMES.items() if self.mask & bit)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_min_mhz": min(self.sm) if self.sm else None,
                "sm_max_mhz": self.max, "samples": len(self.sm), "reasons": reasons, "how": "NVML, 5 ms period"}


def oracle_throughput(wl, frames, threads, steps, warmup):
    """MP/s of the CPU oracle on `frames` synthetic frames per step (same geometry and parameters)."""
    import numpy as np
    import oracle
    W, H, _, a, b, q, f, order, fmt, _ = wl
    rng = np.random.default_rng(7)
    base = rng.integers(0, 256, size=(min(frames, 4), H, W, 3), dtype=np.uint8)
    rgb = np.concatenate([base] * (-(-frames // len(base))))[:frames]       # CPU speed is not data dependent
    po = oracle.make_params(W, H, a, b, q, f, order, out_format=fmt)
    for _ in range(warmup):
        oracle.process(po, rgb, threads=threads)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        oracle.process(po, rgb, threads=threads)
        times.append(time.perf_counter() - t0)
    total = sum(times)
    return frames * W * H * steps / 1e6 / total, total / steps * 1e3


def run_reference(args, wl, name):
    """The reference arm: the reference's own implementation is Scala + Chisel RTL simulation and cannot
    run in this image (no JVM/sbt); its CPU restatement (oracle/, pinned to the reference's golden PNGs)
    is timed instead, on all host threads, on a bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    W, H, _, a, b, q, f, order, fmt, desc = wl
    cores = os.cpu_count() or 1
    per_thread = max(1, min(4, int(3.0e9 / (W * H * 3 * 4 * cores))))          # bounded sample, <= ~3 GB of staging
    frames = cores * per_thread                                                # whole frames per thread: no imbalance
    mps, ms = oracle_throughput(wl, frames, cores, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": "input megapixels/s", "value": round(mps, 2), "unit": "MP/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": config_dict(name, wl, frames, note="reference arm: CPU oracle port, bounded sample per step"),
        "cpu_baseline": {"value": round(mps, 2), "unit": "MP/s", "cores": cores, "kind": "port",
                         "sample": f"{frames} frames of {W}x{H} per step, {cores} host threads"},
        "e2e": {"value": round(mps, 2), "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def config_dict(name, wl, frames_per_gpu, note=None):
    W, H, _, a, b, q, f, order, fmt, desc = wl
    c = {"workload": f"{name}: {desc}", "width": W, "height": H, "frames_per_gpu": frames_per_gpu,
         "chroma": f"4:{a}:{b}", "quant_bits": list(q), "factor": f, "order": order,
         "out_format": ["YCC888", "RGB888", "BUNDLE64", "BUNDLE128", "PLANAR"][fmt], "round_mode": "FLOOR",
         "pool_mode": "AVERAGE (extension)" if name.endswith("avg") else "DECIMATE", "in_format": "RGB24", "sharding": "frames split across ranks, no collective",
         "l2": "inputs (>=1 GB per step) far larger than the 126 MB L2; no flush needed"}
    if note:
        c["note"] = note
    return c


class Env:
    """Rank bookkeeping + the two process groups: NCCL for the timed barrier / max-over-ranks, gloo for waits
    that must not spin a host core (ranks idling while rank 0 times the CPU baseline)."""

    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            sys.exit("bench.py needs a CUDA device: there is no CPU fallback for the pixel path")
        torch.cuda.set_device(self.local)
        self.dist = None
        self.gloo = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
            self.gloo = dist.new_group(backend="gloo")

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def idle_barrier(self):
        if self.dist is not None:
            self.dist.barrier(group=self.gloo)

    def max_over_ranks(self, x):
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device="cuda")
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather(self, values):
        """[world][len(values)] floats, same on every rank."""
        t = self.torch.tensor([float(v) for v in values], dtype=self.torch.float64, device="cuda")
        if self.dist is None:
            return [t.tolist()]
        outt = self.torch.empty((self.world, t.numel()), dtype=self.torch.float64, device="cuda")
        self.dist.all_gather_into_tensor(outt, t)
        return outt.tolist()


def make_inputs(torch, frames, H, W, ipb, seed):
    """The batch a run times: uniform random bytes generated in HBM from `seed`, the same in every run."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    rgb = torch.empty((frames, H, W, ipb), dtype=torch.uint8, device="cuda")
    step_f = max(1, (1 << 29) // (W * H * ipb))      # chunked: randint materialises int64 temporaries for some dtypes
    for i in range(0, frames, step_f):
        rgb[i:i + step_f] = torch.randint(0, 256, rgb[i:i + step_f].shape, dtype=torch.uint8, device="cuda", generator=gen)
    return rgb


DUMP_SAMPLES = 1 << 22      # 16 MB of float32 values + 32 MB of float64 positions: under 64 MB for any workload


def dump_index(total, n=DUMP_SAMPLES):
    """Flat positions of the output bytes --dump-outputs writes: all of them when there are at most n, else a fixed
    seeded sample of n distinct positions, ascending."""
    import numpy as np
    if total <= n:
        return np.arange(total, dtype=np.int64)
    return np.sort(np.random.default_rng(0xD0).choice(total, size=n, replace=False))


def dump_outputs(dirpath, out):
    """Writes the output of the last timed step (`out`, uint8 [frames, bytes per frame]) as DIR/out.npy (float32 byte
    values) and DIR/out_index.npy (float64 flat positions in `out`: frame * bytes_per_frame + byte)."""
    import numpy as np
    import torch
    idx = dump_index(out.numel())
    vals = out.reshape(-1)[torch.from_numpy(idx).to(out.device)].cpu().numpy()
    os.makedirs(dirpath, exist_ok=True)
    np.save(os.path.join(dirpath, "out.npy"), vals.astype(np.float32))
    np.save(os.path.join(dirpath, "out_index.npy"), idx.astype(np.float64))


def device_run(env, ctx, name, frames, shard, steps, warmup, graph, in_format=0, verify=True, replays=1, one_gpu_too=False):
    """Inputs resident in HBM, one kernel launch per step, CUDA events on the launching stream, max over ranks.
    Every rank does the same untimed work first (parity spot check, full-batch cross-check, W warm-up steps).
    shard == "bands": every rank owns one aligned row band of EVERY frame of one shared batch (strong scaling)."""
    import numpy as np
    import csic_b200 as csic
    import oracle
    torch = env.torch
    wl = WORKLOADS[name]
    W, H, _, a, b, q, f, order, fmt, desc = wl
    ops = tuple(ORD[c] for c in order)
    pool = 1 if name.endswith("avg") else 0
    p = csic.make_params(W, H, a, b, q[0], q[1], q[2], f, ops, pool_mode=pool, out_format=fmt, in_format=in_format)
    ipb = 3 if in_format == 0 else 4
    _, out_h, _, out_fb = csic.out_shape(p)

    rgb = make_inputs(torch, frames, H, W, ipb, 0x5EED + (env.rank if shard == "frames" else 0))
    out = torch.empty((frames, out_fb), dtype=torch.uint8, device="cuda")

    # parity spot check (outside the timed region, on every rank): one frame against the oracle
    nchk = min(2, frames)
    ctx.process_torch(p, rgb[:nchk], out=out[:nchk])
    torch.cuda.synchronize()
    want = oracle.process(oracle.make_params(W, H, a, b, q, f, order, pool_mode=pool, out_format=fmt, in_format=in_format),
                          rgb[nchk - 1].cpu().numpy())
    parity = bool(np.array_equal(out[nchk - 1].cpu().numpy(), want[0]))

    band = None
    if shard == "bands":
        chroma_first = order.index("C") < order.index("S")
        band = csic.band_plan(out_h, env.world, f, a, b, chroma_first)[env.rank]

    def step(bnd=band):
        if bnd is None:
            ctx.process_torch(p, rgb, out=out)      # one kernel launch on torch's current stream
        else:
            ctx.process_torch(p, rgb, out=out, out_row0=bnd[0], out_rows=bnd[1])

    # full-size cross-check (outside the timed region, on every rank so that all ranks enter the timed region equally
    # warm): the whole batch through the independent generic gather kernel must equal the fast kernel's output
    full_check = None
    family_opt = ctx_family(ctx)
    if verify and family_opt != 1:
        try:
            ctx.process_torch(p, rgb, out=out)
            fam_fast = ctx.last_kernel()[0]
            ref = torch.empty_like(out)
            ctx.set_option(0, 1)
            ctx.process_torch(p, rgb, out=ref)
            ctx.set_option(0, family_opt)
            torch.cuda.synchronize()
            full_check = {"frames": frames, "kernels": [fam_fast, 1], "equal": bool(torch.equal(out, ref))}
            del ref
            torch.cuda.empty_cache()
        except torch.cuda.OutOfMemoryError:
            full_check = {"skipped": "not enough device memory for a second output buffer"}
            ctx.set_option(0, family_opt)

    def timed(bnd, sampler):
        """-> (total ms of `steps` launches on this rank, per-step ms list)"""
        for _ in range(warmup):
            step(bnd)
        env.barrier() if bnd is band else torch.cuda.synchronize()
        if sampler is not None:
            sampler.start()
        if graph:
            # launch-bound workloads: the K launches are captured once and replayed as one CUDA graph, so the device
            # time holds no host launch cost; `replays` replays are timed one by one, the median is reported
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            g = torch.cuda.CUDAGraph()
            with torch.cuda.stream(side):
                step(bnd)
                with torch.cuda.graph(g, stream=side):
                    for _ in range(steps):
                        step(bnd)
            torch.cuda.current_stream().wait_stream(side)
            g.replay()
            totals = []
            for _ in range(replays):
                env.barrier() if bnd is band else torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); g.replay(); e1.record()
                env.barrier() if bnd is band else torch.cuda.synchronize()
                totals.append(e0.elapsed_time(e1))
            return totals, [t / steps for t in totals]
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        env.barrier() if bnd is band else torch.cuda.synchronize()
        ev[0].record()
        for i in range(steps):
            step(bnd)
            ev[i + 1].record()
        env.barrier() if bnd is band else torch.cuda.synchronize()
        return [ev[0].elapsed_time(ev[-1])], [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]

    fam0, launches0 = ctx.last_kernel()
    sampler = ClockSampler(env.local)
    totals, step_ms = timed(band, sampler)
    clocks = sampler.stop()
    fam, launches1 = ctx.last_kernel()
    launches_timed = steps * (replays if graph else 1)
    # max over ranks, replay by replay; the median replay is the figure (one "replay" for stream launches)
    totals_max = [env.max_over_ranks(t) for t in totals]
    total_ms_max = statistics.median(totals_max)
    mp_per_step_all = frames * W * H * (env.world if band is None else 1) / 1e6
    value = mp_per_step_all * steps / (total_ms_max / 1e3)

    alg_bytes = algorithmic_bytes_per_frame(W, H, f, out_fb, average=bool(pool), ipb=ipb) * frames          # per launch (one rank)
    if band is not None:
        alg_bytes = alg_bytes * band[1] // out_h
    kernel_ms = statistics.median(step_ms) if graph else statistics.mean(step_ms)                        # one launch per step
    peak, peak_src = load_peak()
    achieved = alg_bytes / (kernel_ms / 1e3) / 1e9
    cap_bits = sum(bit for n_, bit in ClockSampler.NAMES.items() if n_ in (clocks.get("reasons") or []))
    per_rank = env.gather([statistics.median(totals), kernel_ms, min(step_ms), max(step_ms), clocks.get("sm_mhz") or 0, cap_bits])
    slowest = max(range(env.world), key=lambda r: per_rank[r][0])
    res = {
        "workload": name, "value": round(value, 1), "unit": "MP/s", "ms_per_step": round(total_ms_max / steps, 4),
        "steps": steps, "frames_per_gpu": frames, "sharding": shard, "scaling": "weak" if band is None else "strong",
        "timed_as": f"cuda_graph_replay (median of {replays} replays of {steps} launches)" if graph else "stream_launches",
        "per_rank_ms": [round(r[0] / steps, 4) for r in per_rank],
        "per_rank_sm_mhz": [r[4] for r in per_rank],
        "per_rank_reasons": [sorted(n_ for n_, bit in ClockSampler.NAMES.items() if int(r[5]) & bit) for r in per_rank],
        "slowest_rank": slowest,
        "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                     "frac": round(achieved / peak, 4), "traffic": None,
                     "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": round(kernel_ms, 4),
                     "kernel": {2: "csic_rows_kernel", 3: "csic_pool_kernel", 4: "csic_flex_kernel"}.get(fam, "csic_generic_kernel"),
                     "peak_source": peak_src, "rank": 0},
        "clocks": clocks, "gpu_launches": launches_timed * env.world,
        "parity_spot_check": parity, "full_batch_cross_check": full_check,
        "step_ms_min": round(min(step_ms), 4), "step_ms_max": round(max(step_ms), 4),
    }
    if band is not None:
        res["band_rows_rank0"] = list(band)
    if one_gpu_too and band is not None and env.world > 1:
        # strong scaling needs the one-GPU time of the SAME batch on the SAME box: rank 0 runs all rows alone
        # (the other ranks wait on a socket, GPUs idle), timed the same way
        if env.rank == 0:
            t1, _ = timed((0, out_h), None)
            one = statistics.median(t1)
        else:
            one = 0.0
        env.idle_barrier()
        one = env.max_over_ranks(one)
        res["one_gpu_ms_per_step"] = round(one / steps, 4)
        res["speedup_vs_one_gpu"] = round(one / total_ms_max, 3)
    res["_state"] = (p, rgb, out, ipb, out_fb)
    return res


def ctx_family(ctx):
    return getattr(ctx, "_bench_family", 0)


def e2e_run(env, ctx, p, rgb, out, W, H, ipb, out_fb, frames, steps):
    """The same metric through csic_process_host (the reference-facing C-ABI call) with pinned HOST buffers: every
    step copies its inputs host->device and its result device->host inside the timed region (wall clock around the
    synchronous calls, barrier on both sides, max over ranks)."""
    import numpy as np
    import csic_b200 as csic
    torch = env.torch
    hb = min(frames, max(1, int(3.2e9 // (W * H * ipb))))         # frames per pinned host batch (~3.2 GB)
    calls = -(-frames // hb)
    pin_in = csic.PinnedBuffer(hb * H * W * ipb)
    pin_out = csic.PinnedBuffer(hb * out_fb)
    hin = torch.from_numpy(pin_in.array)
    hin.copy_(rgb[:hb].reshape(-1))                               # real pixel data in the pinned buffer
    torch.cuda.synchronize()
    hin_np = pin_in.array.reshape(hb, H, W, ipb)
    hout_np = pin_out.array.reshape(hb, out_fb)
    e2e_steps = max(1, min(steps, 3))

    def e2e_step():
        done = 0
        for _ in range(calls):
            n = min(hb, frames - done)
            ctx.process_host(p, hin_np[:n], out=hout_np[:n])   # H2D + kernel + D2H, synchronous
            done += n

    e2e_step()
    env.barrier()
    hb0 = ctx.host_bytes()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    mine = time.perf_counter() - t0
    env.barrier()
    dt = time.perf_counter() - t0
    dt_max = env.max_over_ranks(dt)
    per_rank = env.gather([mine])
    e2e_ok = bool(np.array_equal(hout_np[hb - 1], out[hb - 1].cpu().numpy()))
    h2d = (ctx.host_bytes() - hb0) // e2e_steps
    d2h = frames * out_fb
    mp_all = frames * W * H * env.world / 1e6
    e2e = {"value": round(mp_all * e2e_steps / dt_max, 1), "unit": "MP/s",
           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "h2d_note": "per rank; DECIMATE f>1 reads every f-th input row only; csic_process_host ships just those rows",
           "steps": e2e_steps, "calls_per_step": calls, "host_batch_frames": hb,
           "api": "csic_process_host (pinned host buffers; chunked H2D/kernel/D2H pipeline)",
           "matches_device_path": e2e_ok,
           "per_rank_s_per_step": [round(r[0] / e2e_steps, 4) for r in per_rank],
           "link_gbs": {"h2d": round(h2d * env.world * e2e_steps / dt_max / 1e9, 2),
                        "d2h": round(d2h * env.world * e2e_steps / dt_max / 1e9, 2)}}
    # the ceiling of this figure, measured live on this box in this run: the SAME bytes between the SAME buffers as raw
    # cudaMemcpy calls (no kernel, no library of ours), all ranks at once
    ceil = link_probe(env, pin_in.array.ctypes.data, pin_out.array.ctypes.data, rgb.data_ptr(), out.data_ptr(),
                      hb, H, W, ipb, p.factor if (p.pool_mode == 0 and p.factor > 1 and H % p.factor == 0) else 1, out_fb, calls)
    if ceil is None:
        ceil = load_link_ceiling(env.world)
    if ceil:
        e2e["link_ceiling_gbs"] = ceil
        e2e["frac_of_ceiling"] = round((e2e["link_gbs"]["h2d"] + e2e["link_gbs"]["d2h"]) / (ceil["h2d_gbs"] + ceil["d2h_gbs"]), 3)
    pin_in.free(); pin_out.free()
    return e2e


def link_probe(env, h_in, h_out, d_in, d_out, frames, H, W, ipb, f, out_fb, calls):
    """Host<->device link ceiling for exactly the traffic of one e2e step: `calls` x (H2D of the rows the pipeline
    reads of `frames` frames || D2H of their results), as raw cudaMemcpy2DAsync / cudaMemcpyAsync between the same
    pinned and device buffers on two streams, every rank at the same time; aggregate GB/s = bytes of all ranks /
    max over ranks of the elapsed time.  cuda-python's runtime bindings issue the copies (plumbing, not product)."""
    try:
        from cuda.bindings import runtime as rt
    except Exception:
        return None

    def ck(res):
        if int(res[0]) != 0:
            raise RuntimeError(f"CUDA error {res[0]} in link_probe")
        return res[1] if len(res) > 1 else None
    try:
        s1 = ck(rt.cudaStreamCreateWithFlags(rt.cudaStreamNonBlocking))
        s2 = ck(rt.cudaStreamCreateWithFlags(rt.cudaStreamNonBlocking))
        H2D, D2H = rt.cudaMemcpyKind.cudaMemcpyHostToDevice, rt.cudaMemcpyKind.cudaMemcpyDeviceToHost
        row = W * ipb
        rows = frames * (H // f)

        def one():
            if f > 1:
                ck(rt.cudaMemcpy2DAsync(d_in, row, h_in, f * row, row, rows, H2D, s1))
            else:
                ck(rt.cudaMemcpyAsync(d_in, h_in, rows * row, H2D, s1))
            ck(rt.cudaMemcpyAsync(h_out, d_out, frames * out_fb, D2H, s2))

        def sync():
            ck(rt.cudaStreamSynchronize(s1)); ck(rt.cudaStreamSynchronize(s2))
        one(); sync()
        best = None
        for _ in range(2):
            env.barrier()
            t0 = time.perf_counter()
            for _ in range(calls):
                one()
            sync()
            env.barrier()
            dt = env.max_over_ranks(time.perf_counter() - t0)
            best = dt if best is None else min(best, dt)
        ck(rt.cudaStreamDestroy(s1)); ck(rt.cudaStreamDestroy(s2))
        up, dn = rows * row * calls * env.world, frames * out_fb * calls * env.world
        return {"h2d_gbs": round(up / best / 1e9, 2), "d2h_gbs": round(dn / best / 1e9, 2),
                "how": f"live: raw cudaMemcpy{'2D' if f > 1 else ''}Async H2D || cudaMemcpyAsync D2H of the same bytes between the same "
                       f"pinned/device buffers, {env.world} GPU(s) at once, best of 2 passes, no kernel",
                "see_also": "profiles/r2/pcie_ceiling.json (every subset of GPUs, every direction)"}
    except Exception as e:  # noqa: BLE001
        print(f"link_probe failed: {e}", file=sys.stderr)
        return None


def cpu_baseline(wl):
    W, H = wl[0], wl[1]
    cores = os.cpu_count() or 1
    fr = cores * max(1, min(4, int(3.0e9 / (W * H * 3 * 4 * cores))))
    mps, _ = oracle_throughput(wl, fr, cores, steps=2, warmup=1)
    mps1, _ = oracle_throughput(wl, 2, 1, steps=1, warmup=0)      # SURVEY D5 (i): one thread, streaming form
    return {"value": round(mps, 2), "unit": "MP/s", "cores": cores, "kind": "port",
            "sample": f"{fr} frames of {W}x{H}, 2 timed passes, {cores} host threads (oracle/csic_oracle.c)",
            "value_1thread": round(mps1, 2), "sample_1thread": f"2 frames of {W}x{H}, 1 thread",
            "note": "scalar three-pass CPU restatement of the Scala/Chisel path (the reference itself needs a JVM); "
                    "other ranks idle on a socket while this runs"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg4", choices=list(WORKLOADS))
    ap.add_argument("--frames", type=int, default=0, help="frames per GPU (default: the workload's)")
    ap.add_argument("--graph", action="store_true",
                    help="capture the K timed launches into one CUDA graph and time its replay (launch-bound workloads)")
    ap.add_argument("--replays", type=int, default=5, help="with --graph: timed replays; the median is reported")
    ap.add_argument("--in-format", type=int, default=0, choices=[0, 1, 2], help="0 RGB24, 1 RGBA32, 2 BGRA32")
    ap.add_argument("--generic", action="store_true", help="force the generic gather kernel (family 1)")
    ap.add_argument("--family", type=int, default=0, choices=[0, 1, 2],
                    help="kernel family option: 0 automatic, 1 generic gather kernel, 2 no TMA kernels (flex kernel)")
    ap.add_argument("--no-verify", action="store_true", help="skip the full-batch cross-check against the generic kernel")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the short extra runs of BASELINE configs[2] and configs[4]")
    ap.add_argument("--ctas-per-sm", type=int, default=0)
    ap.add_argument("--stages", type=int, default=0)
    ap.add_argument("--tile-bytes", type=int, default=0)
    ap.add_argument("--block-threads", type=int, default=0)
    ap.add_argument("--chunk-mb", type=int, default=0, help="csic_process_host chunk size (CSIC_OPT_HOST_CHUNK_BYTES)")
    ap.add_argument("--shard", default="frames", choices=["frames", "bands"],
                    help="frames: every rank owns its own batch (weak scaling).  bands: every rank owns one aligned "
                         "row band of EVERY frame of one shared batch (strong scaling; BASELINE configs[4])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write rank 0's output of the last step to DIR/out.npy with the flat "
                         "positions in DIR/out_index.npy (every byte, or a fixed seeded sample of 4 Mi of them)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl, args.workload)
        return

    import csic_b200 as csic
    env = Env()
    torch = env.torch
    W, H, frames, a, b, q, f, order, fmt, desc = wl
    frames = args.frames or frames
    ctx = csic.Context(env.local)
    if args.generic:
        args.family = 1
    if args.family:
        ctx.set_option(0, args.family)
        ctx._bench_family = args.family
    if args.ctas_per_sm:
        ctx.set_option(2, args.ctas_per_sm)
    if args.stages:
        ctx.set_option(3, args.stages)
    if args.tile_bytes:
        ctx.set_option(4, args.tile_bytes)
    if args.block_threads:
        ctx.set_option(5, args.block_threads)
    if args.chunk_mb:
        ctx.set_option(1, args.chunk_mb << 20)
    default_run = args.workload == "cfg4" and args.shard == "frames" and not args.family
    if args.dump_outputs and args.shard == "bands" and env.world > 1:
        sys.exit("--dump-outputs with --shard bands needs one GPU: rank 0 computes only its own band")

    main_res = device_run(env, ctx, args.workload, frames, args.shard, args.steps, args.warmup, args.graph,
                          in_format=args.in_format, verify=not args.no_verify, replays=args.replays)
    p, rgb, out, ipb, out_fb = main_res.pop("_state")
    if args.dump_outputs and env.rank == 0:
        dump_outputs(args.dump_outputs, out)
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp) and args.shard == "frames":
        try:
            tj = json.load(open(tp)).get(args.workload)
            if tj:      # DRAM bytes of one launch measured by ncu, per frame x the frames of this launch
                main_res["roofline"]["traffic"] = tj["dram_bytes_per_frame"] * frames
                main_res["roofline"]["traffic_source"] = tj.get("source")
        except Exception:
            pass

    e2e = None
    if not args.no_e2e and args.shard == "frames":
        e2e = e2e_run(env, ctx, p, rgb, out, W, H, ipb, out_fb, frames, args.steps)
    del rgb, out
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs, witnessed in the same run (short) -----------------------------
    also = None
    if default_run and not args.no_also:
        also = {}
        r = device_run(env, ctx, "cfg3", WORKLOADS["cfg3"][2], "frames", max(args.steps, 20), args.warmup, False, verify=False)
        r.pop("_state")
        also["configs[2] cfg3"] = slim(r, WORKLOADS["cfg3"][9])
        torch.cuda.empty_cache()
        r = device_run(env, ctx, "cfg5", 256, "bands", 50, args.warmup, True, verify=False, replays=7, one_gpu_too=True)
        r.pop("_state")
        also["configs[4] cfg5 row bands"] = slim(r, "BASELINE configs[4]: 7680x4320 x256 frames (one shared batch), every rank "
                                                 "computes one aligned row band of every frame (zero halo), 4:2:0 + f=4 + Q_16BIT + "
                                                 "RGB888 reconstruct; strong scaling")
        torch.cuda.empty_cache()

    # ---- CPU baseline (rank 0, every N; bounded sample; the other ranks wait without spinning) -----
    cpu = None
    if not args.no_cpu:
        if env.rank == 0:
            cpu = cpu_baseline(wl)
        env.idle_barrier()

    if env.rank == 0:
        band_note = None if args.shard == "frames" else \
            f"row-band sharding: {env.world} aligned bands per frame, zero halo, rank 0 band = rows {main_res.get('band_rows_rank0')}"
        line = {
            "metric": "input megapixels/s", "value": main_res["value"], "unit": "MP/s", "n_gpus": env.world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": main_res["ms_per_step"],
            "higher_is_better": True, "scaling": main_res["scaling"], "vs_baseline": None, "dtype": "u8",
            "data": "synthetic (uniform random bytes, torch.randint, seed 0x5EED+rank, generated in HBM)",
            "config": dict(config_dict(args.workload, wl, frames, note=band_note),
                           in_format=["RGB24", "RGBA32", "BGRA32"][args.in_format]),
            "roofline": main_res["roofline"], "cpu_baseline": cpu, "e2e": e2e, "clocks": main_res["clocks"],
            "gpu_launches": main_res["gpu_launches"], "timed_as": main_res["timed_as"],
            "per_rank_ms": main_res["per_rank_ms"], "per_rank_sm_mhz": main_res["per_rank_sm_mhz"],
            "per_rank_reasons": main_res["per_rank_reasons"], "slowest_rank": main_res["slowest_rank"],
            "parity_spot_check": main_res["parity_spot_check"], "full_batch_cross_check": main_res["full_batch_cross_check"],
            "step_ms_min": main_res["step_ms_min"], "step_ms_max": main_res["step_ms_max"],
            "also": also,
        }
        for k in ("one_gpu_ms_per_step", "speedup_vs_one_gpu"):
            if k in main_res:
                line[k] = main_res[k]
        print(json.dumps(line), flush=True)
    if env.dist is not None:
        env.dist.barrier()
        env.dist.destroy_process_group()
    ctx.close()


def slim(r, desc):
    keep = ("value", "unit", "ms_per_step", "steps", "frames_per_gpu", "sharding", "scaling", "timed_as", "per_rank_ms",
            "slowest_rank", "gpu_launches", "parity_spot_check", "one_gpu_ms_per_step", "speedup_vs_one_gpu", "band_rows_rank0")
    d = {"workload": f"{r['workload']}: {desc}"}
    d.update({k: r[k] for k in keep if k in r})
    d["roofline"] = {k: r["roofline"][k] for k in ("achieved", "peak", "frac", "kernel", "kernel_ms", "algorithmic_bytes_per_launch")}
    return d


if __name__ == "__main__":
    main()
