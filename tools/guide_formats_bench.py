"""Per-guide-format timings: GRAY (1 byte/pixel), BGR (3) and BGRX (4).

    python tools/guide_formats_bench.py [--reps 7] [--out FILE.json]

Every figure is the median over --reps repetitions, the repetitions of the three formats interleaved (so a drift of
the shared host or GPU hits all three alike); min and max are reported beside it as the run-to-run spread.  Device
legs are timed with CUDA events, end-to-end legs with the host clock around synchronous calls.  Inputs are seeded
synthetic Kinect frames (kinectdepthmapenhancement_b200.synth); GRAY is their G channel, BGRX appends a random
4th byte.  The 64-frame pre-smooth working set (20-80 MB in, 79 MB out) fits the 126 MB L2 only partly; it is what
a batch of that size costs in practice, not a DRAM-bound figure.

Legs, per format:
  presmooth_us_64x640x480   the guide pre-smooth (ksize 5, 30/30) of 64 frames of 640x480, one launch
  process_batch_mpix_s      jbf_process_batch, 64 frames of 640x480, r = 7 (pre-smooth + filter + fp64 refinement)
  guided_fill_us_1920x1080  kdme_guided_fill_ex, 1920x1080, window 7 (r = 3), no labels
  upsample_us_512x424_to_1920x1080  jbf_upsample (pre-smooth of the 1920x1080 guide + filter), r = 7
  e2e_host_mpix_s / e2e_host_u16_mpix_s  jbf_process_host / _u16 from pinned host buffers, 128 frames of 640x480,
                            H2D + pre-smooth + filter + D2H, one GPU
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FORMATS = {1: "GRAY", 3: "BGR", 4: "BGRX"}


def _as_format(bgr, c, seed=7):
    import torch
    if c == 1:
        return bgr[..., 1].contiguous()
    if c == 4:
        g = torch.Generator(device="cpu").manual_seed(seed)
        x = torch.randint(0, 256, bgr.shape[:-1] + (1,), generator=g, dtype=torch.uint8).to(bgr.device)
        return torch.cat([bgr, x], dim=-1).contiguous()
    return bgr.contiguous()


def _device_us(fn, iters):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters


def _host_s(fn, iters):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / iters


def _gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        return q
    except Exception as e:   # the figures stand without it, but say so
        return f"nvidia-smi unavailable: {e}"


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    args = ap.parse_args()

    import torch
    from kinectdepthmapenhancement_b200 import JointBilateralFilter, synth
    from kinectdepthmapenhancement_b200.guided import guided_fill
    from kinectdepthmapenhancement_b200.jbf import host_buffer
    if not torch.cuda.is_available():
        raise SystemExit("guide_formats_bench.py needs a CUDA device (B200)")
    torch.cuda.set_device(0)
    W, H, NB, NE = 640, 480, 64, 128

    depth, bgr = synth.rgbd_stream(NB, W, H, seed=1234, device="cuda", distinct=16)
    d_hi, bgr_hi = synth.rgbd_frame(1920, 1080, seed=5, frame=0, device="cuda")
    lo, _ = synth.rgbd_frame(512, 424, seed=5, frame=0, device="cuda", noise_rel=0.01)
    host_depth = host_buffer((NE, H, W), torch.float32)
    host_d16 = host_buffer((NE, H, W), torch.int16)
    host_out = host_buffer((NE, H, W), torch.float32)
    for k in range(0, NE, NB):
        host_depth[k:k + NB].copy_(depth.cpu())
    host_d16.copy_(host_depth.round().clamp_(0, 65535).to(torch.int32).to(torch.int16))

    legs = {c: {} for c in FORMATS}
    st = {}
    for c in FORMATS:   # per-format inputs and handles, warmed up once
        g = _as_format(bgr, c)
        s = {"g": g, "g_hi": _as_format(bgr_hi, c)}
        s["f_ps"] = JointBilateralFilter(W, H, window_radius=7, max_batch=NB)
        s["g4"] = s["f_ps"].presmooth(g)
        s["out"] = torch.empty_like(depth)
        s["f_ps"].process_batch(depth, g, s["out"])
        s["f_up"] = JointBilateralFilter(1920, 1080, window_radius=7)
        s["up_out"] = s["f_up"].Upsampling(lo, s["g_hi"])
        s["gf_out"] = guided_fill(d_hi, s["g_hi"], None, 3)
        hc = host_buffer((NE,) + tuple(g.shape[1:]), torch.uint8, write_combined=True)
        for k in range(0, NE, NB):
            hc[k:k + NB].copy_(g.cpu())
        s["hc"] = hc
        s["f_e2e"] = JointBilateralFilter(W, H, window_radius=7, max_batch=NB)
        s["f_e2e"].process_host(host_depth, hc, host_out)
        s["f_e2e"].process_host(host_d16, hc, host_out)
        st[c] = s
    torch.cuda.synchronize()

    for rep in range(args.reps):
        for c, s in st.items():
            L = legs[c]
            L.setdefault("presmooth_us_64x640x480", []).append(
                _device_us(lambda: s["f_ps"].presmooth(s["g"], s["g4"]), 20))
            L.setdefault("process_batch_mpix_s", []).append(
                NB * W * H / _device_us(lambda: s["f_ps"].process_batch(depth, s["g"], s["out"]), 5))
            L.setdefault("guided_fill_us_1920x1080", []).append(
                _device_us(lambda: guided_fill(d_hi, s["g_hi"], None, 3, out=s["gf_out"]), 10))
            L.setdefault("upsample_us_512x424_to_1920x1080", []).append(
                _device_us(lambda: s["f_up"].Upsampling(lo, s["g_hi"], s["up_out"]), 10))
            L.setdefault("e2e_host_mpix_s", []).append(
                NE * W * H / 1e6 / _host_s(lambda: s["f_e2e"].process_host(host_depth, s["hc"], host_out), 3))
            L.setdefault("e2e_host_u16_mpix_s", []).append(
                NE * W * H / 1e6 / _host_s(lambda: s["f_e2e"].process_host(host_d16, s["hc"], host_out), 3))

    res = {"gpu": _gpu_info(), "gpus_used": 1, "reps": args.reps, "formats": {}}
    for c, name in FORMATS.items():
        res["formats"][name] = {
            k: {"median": statistics.median(v), "min": min(v), "max": max(v)} for k, v in legs[c].items()}
        res["formats"][name]["host_bytes_per_pixel"] = {"e2e_host": 4 + c + 4, "e2e_host_u16": 2 + c + 4}
    res["e2e_n8"] = "not measured (one GPU per run)"
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
