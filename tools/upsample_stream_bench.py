"""Upsampling of ToF depth streams: the per-frame loop against upsample_batch (float32 and uint16 depth).

    python tools/upsample_stream_bench.py [--reps 7] [--frames 64] [--max-batch 8] [--out FILE.json]

Sensor shapes, r = 7, guide 1920x1080:
  kinect_v2     512x424 depth
  azure_nfov    640x576 depth (Azure Kinect NFOV unbinned)

Variants, per shape and guide format (BGR, BGRX):
  loop          Upsampling once per frame (pre-smooth, gather, refinement: three launches per frame)
  batch_f32     upsample_batch, float32 depth, chunks of --max-batch frames alternating over two stream lanes
  batch_u16     the same with uint16 depth read by the kernels directly
  batch_f32_one_lane / batch_u16_one_lane   the same on a handle created with KDME_ONE_LANE=1 (every chunk on the
                caller's stream): the A/B of the two lanes

--frames distinct frames per sequence (64 by default: 64 guides of 1920x1080 are 398 MB in BGR and 531 MB in BGRX,
with 531 MB of output, several times the 126 MB L2).  The depth is integer millimetres, so every variant filters the
same samples.  Each figure is the median over --reps repetitions of one whole sequence, timed with CUDA events; the
variants are interleaved inside every repetition so that a drift of the shared machine hits all of them alike; min
and max are the run-to-run spread.  The same run checks that every batch output equals the loop's output bit for bit
and reads the card's name, power limit and max SM clock.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SHAPES = {"kinect_v2": (512, 424), "azure_nfov": (640, 576)}
WH, HH, RADIUS = 1920, 1080, 7
VARIANTS = ("loop", "batch_f32", "batch_u16", "batch_f32_one_lane", "batch_u16_one_lane")


def _gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                               "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # the figures stand without it, but say so
        return f"nvidia-smi unavailable: {e}"


def _device_us(fn):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--max-batch", type=int, default=8)
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    args = ap.parse_args()

    import torch
    from kinectdepthmapenhancement_b200 import JointBilateralFilter, synth
    if not torch.cuda.is_available():
        raise SystemExit("upsample_stream_bench.py needs a CUDA device (B200)")
    torch.cuda.set_device(0)
    n = args.frames

    _, bgr = synth.rgbd_stream(n, WH, HH, seed=77, device="cuda")
    g = torch.Generator(device="cpu").manual_seed(7)
    x = torch.randint(0, 256, (n, HH, WH, 1), generator=g, dtype=torch.uint8).cuda()
    guides = {"BGR": bgr, "BGRX": torch.cat([bgr, x], dim=-1).contiguous()}
    del x

    def handle(one_lane):
        old = os.environ.pop("KDME_ONE_LANE", None)
        if one_lane:
            os.environ["KDME_ONE_LANE"] = "1"
        try:
            return JointBilateralFilter(WH, HH, window_radius=RADIUS, max_batch=args.max_batch)
        finally:
            os.environ.pop("KDME_ONE_LANE", None)
            if old is not None:
                os.environ["KDME_ONE_LANE"] = old

    f2, f1 = handle(False), handle(True)
    res = {"gpu": _gpu_info(), "gpus_used": 1, "reps": args.reps, "frames": n, "max_batch": args.max_batch,
           "radius": RADIUS, "guide": f"{WH}x{HH}", "unit": "us per frame (median, min, max); Mpixel/s of output",
           "shapes": {}}
    for sname, (wl, hl) in SHAPES.items():
        lo = torch.stack([synth.rgbd_frame(wl, hl, seed=11, frame=k, noise_rel=0.01, device="cuda")[0]
                          for k in range(n)]).round_().clamp_(0, 65535)
        lo16 = lo.to(torch.int32).to(torch.int16)   # the uint16 bit patterns
        for gname, gd in guides.items():
            outs = {v: torch.empty((n, HH, WH), dtype=torch.float32, device="cuda") for v in VARIANTS}

            def loop():
                for k in range(n):
                    f2.Upsampling(lo[k], gd[k], outs["loop"][k])

            run = {"loop": loop,
                   "batch_f32": lambda: f2.upsample_batch(lo, gd, outs["batch_f32"]),
                   "batch_u16": lambda: f2.upsample_batch(lo16, gd, outs["batch_u16"]),
                   "batch_f32_one_lane": lambda: f1.upsample_batch(lo, gd, outs["batch_f32_one_lane"]),
                   "batch_u16_one_lane": lambda: f1.upsample_batch(lo16, gd, outs["batch_u16_one_lane"])}
            for v in VARIANTS:   # warm-up (module load, lattice table, queue and lane allocation)
                run[v]()
            torch.cuda.synchronize()
            ref = outs["loop"].view(torch.int32)
            same = {v: bool(torch.equal(outs[v].view(torch.int32), ref)) for v in VARIANTS if v != "loop"}
            t = {v: [] for v in VARIANTS}
            for _ in range(args.reps):
                for v in VARIANTS:
                    t[v].append(_device_us(run[v]) / n)
            row = {}
            for v in VARIANTS:
                med = statistics.median(t[v])
                row[v] = {"us_per_frame": round(med, 2), "min": round(min(t[v]), 2), "max": round(max(t[v]), 2),
                          "mpix_s": round(WH * HH / med, 1)}
            row["speedup_vs_loop"] = {v: round(row["loop"]["us_per_frame"] / row[v]["us_per_frame"], 3)
                                      for v in VARIANTS if v != "loop"}
            row["bit_identical_to_loop"] = same
            res["shapes"].setdefault(f"{sname}_{wl}x{hl}", {})[gname] = row
            del outs
            torch.cuda.empty_cache()
    res["all_bit_identical"] = all(all(r["bit_identical_to_loop"].values())
                                   for s in res["shapes"].values() for r in s.values())
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    if not res["all_bit_identical"]:
        raise SystemExit("a batch output differs from the per-frame loop")


if __name__ == "__main__":
    main()
