"""Host-side logic: sharding arithmetic (incl. a world_size-2 gloo run), the app's CLI surface, and the
repository rules the product must obey (no oracle on the product path)."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import csic_b200 as csic
from conftest import ALL_AB, ROOT


def test_frame_shard_partitions_exactly():
    for n in (0, 1, 7, 64, 1024, 1025):
        for world in (1, 2, 3, 4, 8):
            cuts = [csic.frame_shard(n, r, world) for r in range(world)]
            assert cuts[0][0] == 0 and cuts[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(cuts, cuts[1:]))
            sizes = [hi - lo for lo, hi in cuts]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        csic.frame_shard(10, 2, 2)


def test_band_plan_is_aligned_and_covers():
    for (a, b) in ALL_AB:
        for f in (1, 2, 4, 8):
            for chroma_first in (True, False):
                for out_h in (1080, 135, 17, 8):
                    for world in (1, 2, 8):
                        bands = csic.band_plan(out_h, world, f, a, b, chroma_first)
                        assert len(bands) == world and sum(r for _, r in bands) == out_h
                        unit = csic.sharding.band_alignment(f, a, b, chroma_first)
                        pos = 0
                        for r0, rows in bands:
                            assert r0 == pos and (r0 % unit == 0 or rows == 0)
                            pos += rows


def test_aligned_bands_need_no_halo():
    """E2 of SURVEY.md: a band starting on an alignment unit reads no row above its own first row."""
    S = csic.ProcessingStep
    for (a, b) in ALL_AB:
        for f in (1, 2, 4, 8):
            for ops, chroma_first in (((S.ChromaSubsampling, S.SpatialSampling, S.ColorQuantization), True),
                                      ((S.SpatialSampling, S.ColorQuantization, S.ChromaSubsampling), False)):
                p = csic.make_params(256, 256, a, b, factor=f, ops=ops)
                out_h = csic.out_shape(p)[1]
                for r0, rows in csic.band_plan(out_h, 8, f, a, b, chroma_first):
                    if rows:
                        in0, _ = csic.band_input_rows(p, r0, rows)
                        assert in0 == r0 * f, (a, b, f, chroma_first, r0)


GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, sys.argv[1])
import torch, torch.distributed as dist
import csic_b200 as csic
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
n = 1024
lo, hi = csic.frame_shard(n, rank, world)
# every rank marks the frames it owns; the sum over ranks must be exactly one owner per frame
owned = torch.zeros(n, dtype=torch.int32); owned[lo:hi] = 1
dist.all_reduce(owned)
assert bool((owned == 1).all()), "frames not partitioned exactly once"
# max-over-ranks timing reduction as bench.py does it
t = torch.tensor([float(rank + 1)], dtype=torch.float64)
dist.all_reduce(t, op=dist.ReduceOp.MAX)
assert t.item() == world
bands = csic.band_plan(1080, world, 4, 2, 0, True)
mine = torch.zeros(1080, dtype=torch.int32); mine[bands[rank][0]:bands[rank][0] + bands[rank][1]] = 1
dist.all_reduce(mine)
assert bool((mine == 1).all())
dist.barrier()
if rank == 0:
    print("GLOO_OK", world)
dist.destroy_process_group()
"""


def test_sharding_world_size_2_gloo(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(GLOO_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29533", str(script), ROOT],
                       capture_output=True, text=True, timeout=240, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "GLOO_OK 2" in r.stdout


def test_bench_reference_arm_prints_contract_line():
    """bench.py --impl reference runs the CPU oracle on a bounded sample and prints one JSON line."""
    import json
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg2",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["unit"] == "MP/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["e2e"]["h2d_bytes_per_step"] == 0


def test_app_cli_surface(tmp_path, monkeypatch, capsys):
    """Flag names, defaults and output naming of ImageCompressionApp (ImageCompressorTopApp.scala:149-190);
    processImage itself is stubbed (it needs a GPU and is covered by tests/test_gpu_parity.py)."""
    from csic_b200 import app
    calls = []
    monkeypatch.setattr(app, "processImage", lambda *a, **k: calls.append(a))
    img = tmp_path / "pic.png"
    csic.ImageProcessorModel.writeImage(np.zeros((8, 8, 3), np.uint8), str(img))
    rc = app.main(["--input", str(img), "--a", "2", "--b", "0", "--yq", "3", "--cbq", "3", "--crq", "2", "--sf", "1",
                   "--op1", "chroma", "--op2", "COLOR", "--op3", "SpatialSampling", "--outdir", str(tmp_path / "o")])
    assert rc == 0
    S = csic.ProcessingStep
    (inp, outp, a, b, yq, cbq, crq, sf, o1, o2, o3), = calls
    assert (a, b, yq, cbq, crq, sf) == (2, 0, 3, 3, 2, 1)
    assert (o1, o2, o3) == (S.ChromaSubsampling, S.ColorQuantization, S.SpatialSampling)
    assert outp.endswith("o/pic_processed_chroma4-2-0_Y3Cb3Cr2_sf1_order-Ch-Co-Sp.png")
    out = capsys.readouterr().out
    assert "Selected Chroma Subsampling (J:a:b): 4:2:0" in out and "Selected Pipeline Order: ChromaSubsampling -> ColorQuantization -> SpatialSampling" in out
    # defaults (:164-173): a=b=4, 8/8/8, sf=8, spatial -> color -> chroma
    calls.clear()
    monkeypatch.chdir(tmp_path)
    os.makedirs("test_images")
    csic.ImageProcessorModel.writeImage(np.zeros((8, 8, 3), np.uint8), "test_images/in128x128.png")
    assert app.main([]) == 0
    (inp, outp, a, b, yq, cbq, crq, sf, o1, o2, o3), = calls
    assert (inp, a, b, yq, cbq, crq, sf) == ("test_images/in128x128.png", 4, 4, 8, 8, 8, 8)
    assert (o1, o2, o3) == (S.SpatialSampling, S.ColorQuantization, S.ChromaSubsampling)
    assert outp == "APP_OUTPUT/in128x128_processed_chroma4-4-4_Y8Cb8Cr8_sf8_order-Sp-Co-Ch.png"
    assert app.main(["--input", "missing.png"]) == 1
    with pytest.raises(csic.IllegalArgumentException):
        app.main(["--op1", "blur"])


def test_image_model_png_roundtrip(tmp_path):
    """ImageProcessorModel.readImage / writeImage / getImagePixels (ImageProcessorModel.scala:14-52)."""
    from conftest import GOLDEN
    M = csic.ImageProcessorModel
    img = M.readImage(os.path.join(GOLDEN, "in128x128.png"))                  # RGBA source: alpha dropped
    assert img.shape == (128, 128, 3) and img.dtype == np.uint8
    out = tmp_path / "deep" / "dir" / "x.png"
    M.writeImage(img, str(out))                                              # creates parent directories
    assert np.array_equal(M.readImage(str(out)), img)
    px = M.getImagePixels(img[:2, :3])
    assert len(px) == 2 and len(px[0]) == 3 and px[1][2] == [int(v) for v in img[1, 2]]
    p = csic.ImageProcessorParams(3, 2, 1, 4, 4)
    M.writeImage(img[:2, :3].reshape(-1, 3), str(out), p)                    # Array[Pixel] + params overload
    assert M.readImage(str(out)).shape == (2, 3, 3)


def test_product_never_touches_the_oracle():
    """The product path must not import, link or call oracle/ (prompt rule 3): grep the package and the
    library's dynamic symbols."""
    pkg = os.path.join(ROOT, "chroma-subsampling-image-compressor_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cpp", ".h", ".cuh", ".sh")):
                text = open(os.path.join(dp, f), errors="ignore").read()
                assert not re.search(r"^\s*(import oracle|from oracle)|csic_oracle|liboracle|oracle\.lib|_build/", text, flags=re.M), \
                    (f, "references the oracle")
    out = subprocess.run(["nm", "-D", os.path.join(pkg, "libcsic.so")], capture_output=True, text=True).stdout
    assert "oracle" not in out


def test_every_bench_workload_is_a_legal_parameter_set():
    """bench.py's named workloads must pass the reference's constructor predicates (csic_validate) and give the
    algorithmic byte counts DESIGN.md quotes for the BASELINE configurations."""
    import bench
    import csic_b200 as csic
    for name, (W, H, frames, a, b, q, f, order, fmt, desc) in bench.WORKLOADS.items():
        pool = 1 if name.endswith("avg") else 0
        p = csic.make_params(W, H, a, b, q[0], q[1], q[2], f, tuple(bench.ORD[c] for c in order), pool_mode=pool, out_format=fmt)
        ow, oh, _, fb = csic.out_shape(p)
        assert ow == -(-W // f) and oh == -(-H // f) and fb > 0 and frames > 0, name
    W, H, _, a, b, q, f, order, fmt, _ = bench.WORKLOADS["cfg4"]
    fb = csic.out_shape(csic.make_params(W, H, a, b, *q, f, tuple(bench.ORD[c] for c in order), out_format=fmt))[3]
    assert fb == 8_294_400 and bench.algorithmic_bytes_per_frame(W, H, f, fb) == 20_736_000
    W, H, _, a, b, q, f, order, fmt, _ = bench.WORKLOADS["cfg3"]
    fb = csic.out_shape(csic.make_params(W, H, a, b, *q, f, tuple(bench.ORD[c] for c in order), out_format=fmt))[3]
    assert bench.algorithmic_bytes_per_frame(W, H, f, fb) == 12_441_600


def test_rtl_crosscheck_harness_plumbing(tmp_path):
    """tools/rtl_crosscheck/crosscheck.py end to end without a JVM: a stand-in for the reference CLI (answers with the
    oracle, file named the way the reference's own committed APP_OUTPUT file is) must pass, and a stand-in that flips
    one byte must be reported -- so on a machine with sbt the only unknown is the RTL itself (SURVEY 8(f) N4)."""
    import subprocess, sys
    tool = os.path.join(ROOT, "tools", "rtl_crosscheck")
    base = [sys.executable, os.path.join(tool, "crosscheck.py"), "--reference", str(tmp_path), "--cases", "6"]
    fake = f"{sys.executable} {os.path.join(tool, 'fake_reference.py')}"
    r = subprocess.run(base + ["--runner", fake], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.count("-> ok") == 6, r.stdout + r.stderr
    r = subprocess.run(base + ["--runner", fake + " --corrupt"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 1 and "MISMATCH" in r.stdout, r.stdout + r.stderr


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the arm the driver runs beside ours): one JSON line with the contract's keys, the CPU
    restatement on a bounded sample, no GPU involved; ranks other than 0 print nothing."""
    import json, subprocess, sys
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--workload", "cfg2"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "data",
              "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in line, k
    assert line["impl"] == "reference" and line["unit"] == "MP/s" and line["value"] > 0 and line["gpu_launches"] == 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and "workload" in line["config"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_bench_rejects_zero_steps():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr


@pytest.mark.gpu
def test_bench_dump_outputs_are_the_timed_outputs(tmp_path):
    """--dump-outputs: two runs with the same arguments write the same files (float32 values, float64 positions, at most
    64 MB), which equal the oracle on the bench's own inputs at the sampled positions; --steps sets the timed launches."""
    import json
    import torch
    import bench
    import oracle
    name, frames = "cfg2", 32                         # 6.3 MB of output: more than the sample, so the seeded sample is taken
    W, H, _, a, b, q, f, order, fmt, _ = bench.WORKLOADS[name]
    dumps = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", name, "--frames", str(frames),
                            "--steps", "4", "--warmup", "0", "--no-e2e", "--no-cpu", "--no-verify", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 4 and line["gpu_launches"] == 4
        assert sorted(os.listdir(d)) == ["out.npy", "out_index.npy"]
        assert sum(os.path.getsize(d / n) for n in os.listdir(d)) <= 64 << 20
        vals, idx = np.load(d / "out.npy"), np.load(d / "out_index.npy")
        assert vals.dtype == np.float32 and idx.dtype == np.float64
        dumps.append((vals, idx))
    assert np.array_equal(dumps[0][0], dumps[1][0]) and np.array_equal(dumps[0][1], dumps[1][1])
    rgb = bench.make_inputs(torch, frames, H, W, 3, 0x5EED).cpu().numpy()
    want = oracle.process(oracle.make_params(W, H, a, b, q, f, order, out_format=fmt), rgb, threads=4).reshape(-1)
    vals, idx = dumps[0]
    assert want.size > bench.DUMP_SAMPLES and np.array_equal(idx, bench.dump_index(want.size))
    assert np.array_equal(vals, want[idx.astype(np.int64)])
