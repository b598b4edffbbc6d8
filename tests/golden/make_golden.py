#!/usr/bin/env python3
"""Generates tests/golden/*.npz from the REFERENCE'S OWN kernel text.

Run with a checkout of the reference:
    python tests/golden/make_golden.py     # checkout found as oracle/build_ref.py describes
It builds oracle/_ref (the reference kernels compiled for the host, read in place from
that checkout by oracle/build_ref.py) and records their outputs on small seeded inputs.
The reference itself ships no golden vectors (SURVEY.md section 4); these fixtures pin the
committed C restatement (oracle/kdme_oracle.c) to the reference wherever the reference
checkout is absent.

guide_frame_640x480.png holds the decoded pixels (cv2.imread(..., 1); pixel sha256 67e5a97a...1614c) of
the reference's bundled sample frame input/color.jpg, written losslessly by this script; the matching
input/depth.xml is a stripped large blob (.MISSING_LARGE_BLOBS) and is replaced by a seeded surrogate
depth everywhere.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from oracle import build_ref  # noqa: E402
from kinectdepthmapenhancement_b200 import synth  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    assert build_ref.available(), "needs a reference checkout (see oracle/build_ref.py)"
    oracle.build(force=True)
    W, H = 96, 64
    d, c = synth.rgbd_frame(W, H, seed=77, frame=3)
    d, c = d.numpy(), c.numpy()
    g = oracle.presmooth(c)
    out = {"depth": d, "bgr": c, "guide": g}
    for ws in (5, 15):
        out[f"jbf_ws{ws}"] = oracle.jbf(d, g, ws, impl="ref", threads=1)
    # exotic sigmas: colour guard fires (sigma_c=20), tiny spatial sigma (S underflows to 0)
    out["jbf_ws7_sc20"] = oracle.jbf(d, g, 7, 70.0, 20.0, 20.0, impl="ref", threads=1)
    out["jbf_ws7_ss05"] = oracle.jbf(d, g, 7, 0.5, 50.0, 20.0, impl="ref", threads=1)
    labels = ((np.arange(H)[:, None] // 16) * 8 + (np.arange(W)[None, :] // 12)).astype(np.int32)
    out["labels"] = labels
    out["guided_ws7"] = oracle.guided_fill(d, c, labels, impl="ref", threads=1)
    out["guided_ws7_nolabel"] = oracle.guided_fill(d, c, None, impl="ref", threads=1)
    out["mrf_ws5"] = oracle.mrf(d, c, impl="ref", threads=1)
    # Buffer2D: 12 noisy frames through updateData, then the maps
    rng = np.random.default_rng(5)
    frames = np.stack([np.where(d > 50, d + rng.uniform(-6, 6, d.shape).astype(np.float32), d)
                       for _ in range(12)]).astype(np.float32)
    frames[3, 10:20, 10:30] = 0.0
    frames[7, 30:40, 50:70] *= 1.5
    b = oracle.Buffer2D(W, H, impl="ref")
    for f in frames:
        b.update(f)
    out["buf_frames"] = frames
    out["buf_depth"] = b.depth_map()
    out["buf_weight"] = b.weight_map()
    b2 = oracle.Buffer2D(W, H, impl="ref")
    xy = np.stack([d, d * 0.5], axis=-1).astype(np.float32)
    b2.insert_f32x2(xy)
    out["buf_xy_raw"] = b2.raw().copy()
    # f2: Projection_GPU::bilateralfilter on the back-projected cloud
    pts = oracle.projective_to_real(d, 525.0, 525.0, W // 2, H // 2)
    z = np.where(pts[..., 2] > 0, pts[..., 2], 1)
    norm = pts.copy()
    norm[..., 0] /= z
    norm[..., 1] /= z
    out["f2_points"] = pts
    out["f2_normalized"] = norm
    out["f2_out"] = oracle.depth_bilateral_xyz(norm, pts, impl="ref", threads=1)
    import cv2
    src = os.path.join(build_ref.REF, "input", "color.jpg")
    if os.path.isfile(src):
        cv2.imwrite(os.path.join(HERE, "guide_frame_640x480.png"), cv2.imread(src, 1), [cv2.IMWRITE_PNG_COMPRESSION, 9])
    np.savez_compressed(os.path.join(HERE, "ref_golden.npz"), **out)
    print("wrote ref_golden.npz:", {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
