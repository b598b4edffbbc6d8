"""bench.py contract: the reference arm runs on host cores only and prints the required JSON line;
the GPU arm's line is checked on the GPU box."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, synth_np

REQUIRED = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"]


def _run(args, timeout=600):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                         timeout=timeout, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, "bench.py must print exactly one JSON line"
    return json.loads(lines[0])


def _dumped(dirname):
    out = np.load(os.path.join(dirname, "filtered.npy"))
    idx = np.load(os.path.join(dirname, "filtered_frame_index.npy"))
    assert out.dtype == np.float32 and idx.dtype == np.float64
    assert out.ndim == 3 and out.shape[1:] == (480, 640) and idx.shape == (out.shape[0],)
    assert out.nbytes + idx.nbytes <= 64 * 10 ** 6
    return out, idx.astype(np.int64)


def test_reference_arm_line(tmp_path):
    line = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path)])
    for k in REQUIRED + ["impl", "cpu_baseline"]:
        assert k in line, k
    assert line["impl"] == "reference" and line["unit"] == "Mpixel/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["cpu_baseline"]["kind"] in ("reference", "port")
    assert line["cpu_baseline"]["cores"] >= 1 and line["e2e"]["h2d_bytes_per_step"] == 0
    assert "workload" in line["config"] and "model" not in line["config"]
    # the dump holds what the timed path computed: frame 0 of the seeded stream through pre-smooth + filter
    import oracle
    out, idx = _dumped(tmp_path)
    d, c = synth_np(640, 480, seed=1234, frame=0)
    assert idx.tolist() == [0]
    assert np.array_equal(out[0], oracle.jbf_process(d, c, 15))


def test_steps_must_be_positive():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert res.returncode != 0 and "--steps" in res.stderr and res.stdout == ""


def test_reference_arm_non_zero_rank_is_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_static_roofline_fields_parse_from_committed_profiles():
    """roofline.traffic and roofline.pipes_ncu come from the committed `ncu --set full` summary of the dominant kernel
    (labelled static in the line): the parser must find the newest capture and its counters."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    traffic, src = bench.measured_traffic(64 * 640 * 480)
    assert src and src.startswith("profiles/") and "jbf_fast_r7" in src
    # no wasted re-reads: DRAM traffic of a 64-frame launch within 10 % of the 11 B/pixel algorithmic bytes
    assert 0.9 * 64 * 640 * 480 * 11 < traffic < 1.1 * 64 * 640 * 480 * 12
    pipes = bench.profiled_pipes()
    assert pipes["source"].endswith(src)
    for k in ("xu_pipe_busy_pct", "fma_pipe_busy_pct", "alu_pipe_busy_pct", "issue_slots_busy_pct"):
        assert 0.0 < pipes[k] <= 100.0
    assert pipes["xu_pipe_busy_pct"] > pipes["fma_pipe_busy_pct"]      # the kernel is MUFU-bound, not FP32-bound


@pytest.mark.gpu
def test_gpu_arm_line(tmp_path):
    line = _run(["--frames", "256", "--steps", "2", "--warmup", "3", "--e2e-frames", "128", "--cpu-seconds", "3",
                 "--band-size", "2048", "--dump-outputs", str(tmp_path)], timeout=900)
    for k in REQUIRED + ["roofline", "cpu_baseline", "clocks", "parity", "extra", "e2e_u16"]:
        assert k in line, k
    assert line["steps"] == 2 and line["e2e"]["steps"] == 2 and line["e2e_u16"]["steps"] == 2
    # the dump: a seeded sample of the 256 frames the timed path returned, equal to filtering each frame alone
    # (the stream tiles 64 distinct frames) and, independently of the kernels, within the north_star tolerance
    # of the fp64 oracle
    import oracle
    from kinectdepthmapenhancement_b200 import JointBilateralFilter, synth
    out, idx = _dumped(tmp_path)
    assert len(set(idx.tolist())) == out.shape[0] == 48 and 0 <= idx.min() and idx.max() < 256
    f = JointBilateralFilter(640, 480, window_radius=7)
    for k in (0, out.shape[0] - 1):
        d, c = synth.rgbd_frame(640, 480, seed=1234, frame=int(idx[k]) % 64, device="cuda")
        f.Process(d, c)
        assert np.array_equal(f.getFiltered_Device().cpu().numpy().view(np.uint32), out[k].view(np.uint32))
    d, c = synth_np(640, 480, seed=1234, frame=int(idx[0]) % 64)
    par = oracle.parity_block(out[0], d, oracle.presmooth(c), 15)
    assert par["mask_mismatches"] == 0 and par["nan"] == 0 and par["max_abs_regular_mm"] <= 1e-3, par
    rf = line["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in rf, k
    assert 0.3 < rf["frac"] < 1.2 and rf["hbm"]["frac"] < 0.1      # compute-bound stencil
    assert 0.3 < rf["mufu"]["frac"] < 1.05
    assert line["gpu_launches"] == 2 * 4 * 3                        # 2 steps x (256/64 chunks) x (pre-smooth, filter, refine)
    assert line["e2e"]["h2d_bytes_per_step"] == 128 * 640 * 480 * 7 and line["e2e"]["d2h_bytes_per_step"] == 128 * 640 * 480 * 4
    assert line["e2e_u16"]["h2d_bytes_per_step"] == 128 * 640 * 480 * 5
    assert line["scaling"] == "weak" and line["vs_baseline"] is None and line["dtype"] == "f32"
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    # parity block: the north_star tolerance, flat, on the configs[1] stream and on configs[0]
    par = line["parity"]
    assert par["mask_mismatches"] == 0 and par["presmooth_bit_exact"] is True
    assert par["max_abs_regular_mm"] <= 1e-3 and par["config1"]["max_abs_regular_mm"] <= 1e-3
    assert par["frames_checked"] >= 4 and par["refine_queue_dropped"] == 0
    ex = line["extra"]
    assert ex["bands_nccl"]["seam_rows_bitwise_equal_single_gpu_path"] is True
    assert ex["bands_nccl"]["oracle_seam_check"]["mask_mismatches"] == 0
    assert ex["bands_nccl"]["oracle_seam_check"]["max_abs_regular_mm"] <= 1e-3
    assert ex["single_frame"]["r7_us"] > 0 and ex["upsample"]["ms"] > 0 and len(ex["sweep"]["rows"]) == 13
    assert ex["strong"]["scaling"] == "strong"


@pytest.mark.gpu
def test_config1_dump(tmp_path):
    """--config1 dumps its one GPU frame: the bundled colour frame + seeded surrogate depth, reference defaults."""
    import cv2
    import oracle
    line = _run(["--config1", "--cpu-seconds", "0.5", "--dump-outputs", str(tmp_path)])
    assert line["parity"]["mask_bit_exact"] is True
    out, idx = _dumped(tmp_path)
    assert idx.tolist() == [0] and out.shape[0] == 1
    img = cv2.imread(os.path.join(ROOT, "tests", "golden", "guide_frame_640x480.png"), 1)
    d, _ = synth_np(640, 480, seed=2013, frame=0)
    par = oracle.parity_block(out[0], d, oracle.presmooth(img), 5)
    assert par["mask_mismatches"] == 0 and par["nan"] == 0 and par["max_abs_regular_mm"] <= 1e-3, par
