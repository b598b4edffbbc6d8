"""Streams of Kinect frames through the MarkovRandomField filter: a per-frame loop against one batched call, and the
single-frame jbf_mrf against an earlier build of the library.

    python tools/mrf_stream_bench.py [--reps 7] [--frames 64] [--parent-lib LIB.so] [--out FILE]

640x480 frames, radii 2 (the reference's window 5) and 5, BGR and BGRX guides.  Variants, per radius and guide:
  loop          JointBilateralFilter.mrf once per frame, float32 depth (the reference's call pattern)
  batch_f32     JointBilateralFilter.mrf of the [N, H, W] stream, float32 depth (jbf_mrf_batch)
  batch_u16     the same with uint16 depth read by the kernel directly (jbf_mrf_batch_u16)
  single        jbf_mrf once per frame, called through ctypes without the Python checks
  single_parent the same call into --parent-lib, an earlier build of the library, loaded into this process

--frames distinct frames per sequence (64: 79 MB of float32 depth, 59 MB of BGR guides and 79 MB of output, above the
126 MB L2 together).  The depth is integer millimetres, so every variant filters the same samples.  Each figure is the
median over --reps repetitions of one whole sequence, timed with CUDA events; the variants are interleaved inside every
repetition so that a drift of the shared machine hits all of them alike; min and max are the run-to-run spread.  The
same run checks that every output equals the per-frame loop's bit for bit and reads the card's name, power limit and
max SM clock.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W, H = 640, 480
RADII = (2, 5)
GUIDES = {"BGR": 3, "BGRX": 4}
SC, SM = 50.0, 150.0


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


class _Handle:
    """A jbf handle of one build of the library, driven through its C ABI (jbf_mrf only)."""

    def __init__(self, path, channels, stream):
        from kinectdepthmapenhancement_b200 import _lib
        self.L = C.CDLL(path)
        for name in ("jbf_create", "jbf_destroy", "jbf_set_guide_channels", "jbf_mrf", "kdme_last_error"):
            fn = getattr(self.L, name)
            fn.restype, fn.argtypes = _lib.SIGNATURES[name]
        self.h = C.c_void_p()
        self.c = channels
        self._check(self.L.jbf_create(C.byref(self.h), W, H, 70.0, 50.0, 20.0, 2, 1, 0, stream))
        self._check(self.L.jbf_set_guide_channels(self.h, channels))

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError(f"kdme error {rc}: {self.L.kdme_last_error()}")

    def run(self, depth, bgr, out, r):
        """jbf_mrf on every frame of the stream."""
        fn, h, step = self.L.jbf_mrf, self.h, self.c * W
        d0, b0, o0 = depth.data_ptr(), bgr.data_ptr(), out.data_ptr()
        for k in range(depth.shape[0]):
            rc = fn(h, d0 + 4 * W * H * k, b0 + step * H * k, step, o0 + 4 * W * H * k, r, SC, SM)
            if rc != 0:
                self._check(rc)

    def close(self):
        self.L.jbf_destroy(self.h)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--parent-lib", default=None, help="an earlier libkdme_b200.so for the single_parent variant")
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    args = ap.parse_args()

    import torch
    from kinectdepthmapenhancement_b200 import JointBilateralFilter, _lib, synth
    if not torch.cuda.is_available():
        raise SystemExit("mrf_stream_bench.py needs a CUDA device (B200)")
    torch.cuda.set_device(0)
    n = args.frames
    depth, bgr3 = synth.rgbd_stream(n, W, H, seed=23, device="cuda")
    depth = depth.round_().clamp_(0, 65535)
    d16 = depth.to(torch.int32).to(torch.int16)   # the uint16 bit patterns
    g = torch.Generator(device="cuda").manual_seed(5)
    guides = {"BGR": bgr3.contiguous(),
              "BGRX": torch.cat([bgr3, torch.randint(0, 256, (n, H, W, 1), generator=g, device="cuda",
                                                     dtype=torch.uint8)], dim=-1).contiguous()}

    res = {"gpu": _gpu_info(), "gpus_used": 1, "reps": args.reps, "frames": n, "size": f"{W}x{H}",
           "sigmas": {"color": SC, "smooth": SM},
           "unit": "us per frame (median, min, max); Mpixel/s", "cases": {}}
    stream = torch.cuda.current_stream().cuda_stream
    f = JointBilateralFilter(W, H)
    for r in RADII:
        for gname, c in GUIDES.items():
            bgr = guides[gname]
            hosts = {"single": _Handle(_lib.LIB_PATH, c, stream)}
            if args.parent_lib:
                hosts["single_parent"] = _Handle(args.parent_lib, c, stream)
            out = {v: torch.empty((n, H, W), dtype=torch.float32, device="cuda")
                   for v in ("loop", "batch_f32", "batch_u16", *hosts)}

            def loop():
                for k in range(n):
                    f.mrf(depth[k], bgr[k], r, SC, SM, out=out["loop"][k])

            run = {"loop": loop,
                   "batch_f32": lambda: f.mrf(depth, bgr, r, SC, SM, out=out["batch_f32"]),
                   "batch_u16": lambda: f.mrf(d16, bgr, r, SC, SM, out=out["batch_u16"])}
            for v, hh in hosts.items():
                run[v] = (lambda hh=hh, v=v: hh.run(depth, bgr, out[v], r))
            for fn in run.values():   # warm-up (module load)
                fn()
            torch.cuda.synchronize()
            ref = out["loop"].view(torch.int32)
            same = {v: bool(torch.equal(o.view(torch.int32), ref)) for v, o in out.items() if v != "loop"}
            t = {v: [] for v in run}
            for _ in range(args.reps):
                for v, fn in run.items():
                    t[v].append(_device_us(fn) / n)
            row = {}
            for v in run:
                med = statistics.median(t[v])
                row[v] = {"us_per_frame": round(med, 2), "min": round(min(t[v]), 2), "max": round(max(t[v]), 2),
                          "mpix_s": round(W * H / med, 1)}
            row["bit_identical_to_loop"] = same
            res["cases"][f"r{r}_{gname}"] = row
            for hh in hosts.values():
                hh.close()
            del out
    f.close()
    res["all_bit_identical"] = all(all(r["bit_identical_to_loop"].values()) for r in res["cases"].values())
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    if not res["all_bit_identical"]:
        raise SystemExit("an output differs from the per-frame loop")


if __name__ == "__main__":
    main()
