"""Guided fill and label-guided upsampling of depth streams: the per-frame loop against one batched call (float32
and uint16 depth).

    python tools/guided_stream_bench.py [--reps 7] [--frames 64] [--out FILE.json]

Cases (sensor shapes; the reference's sigmas 30 / 50 / 70):
  fill_640x480_r3           guided_fill at 640x480, window radius 3 (the reference's window 7), without labels
  fill_640x480_r3_labels    the same with a per-frame label map
  upsample_512x424_r7       guided_upsample 512x424 (Kinect v2) -> 1920x1080, radius 7, per-frame label map
  upsample_640x576_r7       guided_upsample 640x576 (Azure Kinect NFOV) -> 1920x1080, radius 7, per-frame label map

Variants, per case and guide format (BGR, BGRX):
  loop          guided_fill / guided_upsample once per frame from Python, float32 depth (one call, one launch each)
  batch_f32     one call on the [N, ...] float32 depth
  batch_u16     one call on the same depth as uint16 millimetres, read by the kernels directly

--frames distinct frames per sequence (64 by default: at 640x480 the depth, guides, labels and outputs of the
sequence are 295 MB in BGR, at 1920x1080 64 guides alone are 398 MB in BGR; both several times the 126 MB L2).  The
depth is integer millimetres, so every variant filters the same samples.  Each figure is the median over --reps
repetitions of one whole sequence, timed with CUDA events; the variants are interleaved inside every repetition so
that a drift of the shared machine hits all of them alike; min and max are the run-to-run spread.  The same run
checks that every batch output equals the loop's output bit for bit and reads the card's name, power limit and max
SM clock.
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

HI = (1920, 1080)
# name -> (kind, depth size, output size, radius, labels)
CASES = {"fill_640x480_r3": ("fill", (640, 480), (640, 480), 3, False),
         "fill_640x480_r3_labels": ("fill", (640, 480), (640, 480), 3, True),
         "upsample_512x424_r7": ("upsample", (512, 424), HI, 7, True),
         "upsample_640x576_r7": ("upsample", (640, 576), HI, 7, True)}
VARIANTS = ("loop", "batch_f32", "batch_u16")


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


def _labels(n, w, h, device):
    """Superpixel-like label maps: 24x24 blocks whose grid shifts with the frame."""
    import torch
    ys = torch.arange(h, device=device)[:, None]
    xs = torch.arange(w, device=device)[None, :]
    return torch.stack([(((ys + 3 * k) // 24) * 1000 + (xs + 5 * k) // 24).to(torch.int32) for k in range(n)])


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    args = ap.parse_args()

    import torch
    from kinectdepthmapenhancement_b200 import synth
    from kinectdepthmapenhancement_b200.guided import guided_fill, guided_upsample
    if not torch.cuda.is_available():
        raise SystemExit("guided_stream_bench.py needs a CUDA device (B200)")
    torch.cuda.set_device(0)
    n = args.frames
    res = {"gpu": _gpu_info(), "gpus_used": 1, "reps": args.reps, "frames": n,
           "sigmas": {"spatial": 30.0, "color": 50.0, "depth": 70.0},
           "unit": "us per frame (median, min, max); Mpixel/s of output", "cases": {}}
    for cname, (kind, (dw, dh), (w, h), r, use_labels) in CASES.items():
        depth = torch.stack([synth.rgbd_frame(dw, dh, seed=11, frame=k, noise_rel=0.01, device="cuda")[0]
                             for k in range(n)]).round_().clamp_(0, 65535)
        depth16 = depth.to(torch.int32).to(torch.int16)   # the uint16 bit patterns
        _, bgr = synth.rgbd_stream(n, w, h, seed=77, device="cuda")
        g = torch.Generator(device="cpu").manual_seed(7)
        x = torch.randint(0, 256, (n, h, w, 1), generator=g, dtype=torch.uint8).cuda()
        guides = {"BGR": bgr, "BGRX": torch.cat([bgr, x], dim=-1).contiguous()}
        del x
        labels = _labels(n, w, h, "cuda") if use_labels else None
        op = guided_fill if kind == "fill" else guided_upsample
        for gname, gd in guides.items():
            outs = {v: torch.empty((n, h, w), dtype=torch.float32, device="cuda") for v in VARIANTS}

            def loop():
                for k in range(n):
                    op(depth[k], gd[k], labels[k] if labels is not None else None, r, out=outs["loop"][k])

            run = {"loop": loop,
                   "batch_f32": lambda: op(depth, gd, labels, r, out=outs["batch_f32"]),
                   "batch_u16": lambda: op(depth16, gd, labels, r, out=outs["batch_u16"])}
            for v in VARIANTS:   # warm-up (module load)
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
                          "mpix_s": round(w * h / med, 1)}
            row["speedup_vs_loop"] = {v: round(row["loop"]["us_per_frame"] / row[v]["us_per_frame"], 3)
                                      for v in VARIANTS if v != "loop"}
            row["bit_identical_to_loop"] = same
            res["cases"].setdefault(f"{cname}", {})[gname] = row
            del outs
        del depth, depth16, bgr, guides, labels
        torch.cuda.empty_cache()
    res["all_bit_identical"] = all(all(r["bit_identical_to_loop"].values())
                                   for c in res["cases"].values() for r in c.values())
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    if not res["all_bit_identical"]:
        raise SystemExit("a batch output differs from the per-frame loop")


if __name__ == "__main__":
    main()
