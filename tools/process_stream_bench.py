"""Streams of Kinect frames through the joint bilateral filter: float32 against uint16 depth on the device, and the
ways of getting a cloud per frame.

    python tools/process_stream_bench.py [--reps 7] [--frames 64] [--max-batch 16] [--parent-lib LIB.so] [--out FILE]

640x480 frames, BGR guides, radii 7 and 2.  Variants, per radius:
  batch_f32          process_batch, float32 depth (chunks of --max-batch frames over two stream lanes)
  batch_u16          process_batch, uint16 depth read by the filter directly
  xyz_loop           process_xyz once per frame (the reference's Process + projectiveToReal per frame, fused)
  batch_then_project process_batch, then projective_to_real of the [N, H, W] stream (two passes over the planes)
  batch_xyz          process_batch_xyz, float32 depth (the back-projection fused into the filter's epilogue)
  batch_xyz_u16      the same with uint16 depth
  host_u16           jbf_process_host_u16 (pinned host frames in, pinned host planes out; synchronous)
  host_u16_parent    the same call into --parent-lib, an earlier build of the library, loaded into this process

--frames distinct frames per sequence (64: 59 MB of float32 depth, 59 MB of guides, 79 MB of output and 236 MB of
clouds, above the 126 MB L2 together).  The depth is integer millimetres, so every variant filters the same samples.
Each figure is the median over --reps repetitions of one whole sequence, device variants timed with CUDA events and the
host pipeline with the host clock (it ends in a synchronise); the variants are interleaved inside every repetition so
that a drift of the shared machine hits all of them alike; min and max are the run-to-run spread.  The same run checks
that every output equals the per-frame loop's (and the parent library's) bit for bit and reads the card's name, power
limit and max SM clock.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W, H, FX, FY = 640, 480, 525.0, 525.0
RADII = (7, 2)


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


def _host_us(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e6


class _HostHandle:
    """A jbf handle of one build of the library, driven through its C ABI (jbf_process_host_u16 only)."""

    def __init__(self, path, radius, max_batch, stream):
        from kinectdepthmapenhancement_b200 import _lib
        self.L = C.CDLL(path)
        for name in ("jbf_create", "jbf_destroy", "jbf_process_host_u16", "kdme_last_error"):
            fn = getattr(self.L, name)
            fn.restype, fn.argtypes = _lib.SIGNATURES[name]
        self.h = C.c_void_p()
        self._check(self.L.jbf_create(C.byref(self.h), W, H, 70.0, 50.0, 20.0, radius, max_batch, 0, stream))

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError(f"kdme error {rc}: {self.L.kdme_last_error()}")

    def run(self, d16, bgr, out, n):
        self._check(self.L.jbf_process_host_u16(self.h, d16.data_ptr(), bgr.data_ptr(), 3 * W, out.data_ptr(), n))

    def close(self):
        self.L.jbf_destroy(self.h)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--max-batch", type=int, default=16)
    ap.add_argument("--parent-lib", default=None, help="an earlier libkdme_b200.so for the host_u16_parent variant")
    ap.add_argument("--out", default=None, help="write the JSON here as well as to stdout")
    args = ap.parse_args()

    import torch
    from kinectdepthmapenhancement_b200 import JointBilateralFilter, _lib, projective_to_real, synth
    if not torch.cuda.is_available():
        raise SystemExit("process_stream_bench.py needs a CUDA device (B200)")
    torch.cuda.set_device(0)
    n = args.frames
    depth, bgr = synth.rgbd_stream(n, W, H, seed=21, device="cuda")
    depth = depth.round_().clamp_(0, 65535)
    d16 = depth.to(torch.int32).to(torch.int16)   # the uint16 bit patterns
    d16_host = d16.cpu().pin_memory()
    bgr_host = bgr.cpu().pin_memory()

    res = {"gpu": _gpu_info(), "gpus_used": 1, "reps": args.reps, "frames": n, "max_batch": args.max_batch,
           "size": f"{W}x{H}", "guide": "BGR", "library": _lib.LIB_PATH, "parent_library": args.parent_lib,
           "unit": "us per frame (median, min, max); Mpixel/s", "radii": {}}
    stream = torch.cuda.current_stream().cuda_stream
    for r in RADII:
        f = JointBilateralFilter(W, H, window_radius=r, max_batch=args.max_batch)
        hosts = {"host_u16": _HostHandle(_lib.LIB_PATH, r, args.max_batch, stream)}
        if args.parent_lib:
            hosts["host_u16_parent"] = _HostHandle(args.parent_lib, r, args.max_batch, stream)
        out = {v: torch.empty((n, H, W), dtype=torch.float32, device="cuda")
               for v in ("batch_f32", "batch_u16", "xyz_loop", "batch_then_project", "batch_xyz", "batch_xyz_u16")}
        xyz = {v: torch.empty((n, H, W, 3), dtype=torch.float32, device="cuda")
               for v in ("xyz_loop", "batch_then_project", "batch_xyz", "batch_xyz_u16")}
        host_out = {v: torch.empty((n, H, W), dtype=torch.float32).pin_memory() for v in hosts}

        def xyz_loop():
            for k in range(n):
                f.process_xyz(depth[k], bgr[k], FX, FY, W // 2, H // 2, out=xyz["xyz_loop"][k])
                out["xyz_loop"][k].copy_(f.getFiltered_Device())

        def batch_then_project():
            f.process_batch(depth, bgr, out["batch_then_project"])
            xyz["batch_then_project"].copy_(projective_to_real(out["batch_then_project"], FX, FY, W // 2, H // 2))

        run = {"batch_f32": lambda: f.process_batch(depth, bgr, out["batch_f32"]),
               "batch_u16": lambda: f.process_batch(d16, bgr, out["batch_u16"]),
               "xyz_loop": xyz_loop,
               "batch_then_project": batch_then_project,
               "batch_xyz": lambda: f.process_batch_xyz(depth, bgr, FX, FY, W // 2, H // 2, out["batch_xyz"],
                                                        xyz["batch_xyz"]),
               "batch_xyz_u16": lambda: f.process_batch_xyz(d16, bgr, FX, FY, W // 2, H // 2, out["batch_xyz_u16"],
                                                            xyz["batch_xyz_u16"])}
        for v, hh in hosts.items():
            run[v] = (lambda hh=hh, v=v: hh.run(d16_host, bgr_host, host_out[v], n))
        for fn in run.values():   # warm-up (module load, queues, lanes, host pipeline)
            fn()
        torch.cuda.synchronize()
        ref = out["xyz_loop"].view(torch.int32)
        same = {v: bool(torch.equal(o.view(torch.int32), ref)) for v, o in out.items() if v != "xyz_loop"}
        same.update({f"{v}_xyz": bool(torch.equal(x.view(torch.int32), xyz["xyz_loop"].view(torch.int32)))
                     for v, x in xyz.items() if v != "xyz_loop"})
        same.update({v: bool(torch.equal(o.view(torch.int32), ref.cpu())) for v, o in host_out.items()})
        t = {v: [] for v in run}
        for _ in range(args.reps):
            for v, fn in run.items():
                t[v].append((_host_us(fn) if v.startswith("host") else _device_us(fn)) / n)
        row = {}
        for v in run:
            med = statistics.median(t[v])
            row[v] = {"us_per_frame": round(med, 2), "min": round(min(t[v]), 2), "max": round(max(t[v]), 2),
                      "mpix_s": round(W * H / med, 1)}
        row["bit_identical_to_xyz_loop"] = same
        res["radii"][f"r{r}"] = row
        for hh in hosts.values():
            hh.close()
        f.close()
        del out, xyz, host_out
        torch.cuda.empty_cache()
    res["all_bit_identical"] = all(all(r["bit_identical_to_xyz_loop"].values()) for r in res["radii"].values())
    line = json.dumps(res, indent=1)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    if not res["all_bit_identical"]:
        raise SystemExit("an output differs from the per-frame loop")


if __name__ == "__main__":
    main()
