"""GPU parity: Buffer2D (bit-exact: un-fused fp32 with integer gate) and the guided fill."""
import os

import numpy as np
import pytest
import torch

from conftest import synth_np
from test_guided_f64 import check_guided_against_f64

import oracle

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("w,h", [(640, 480), (70, 50), (33, 17), (1, 1), (512, 424)])
def test_buffer2d_bit_exact(w, h):
    from kinectdepthmapenhancement_b200 import Buffer2D
    depth, _ = synth_np(w, h, seed=31, frame=0)
    rng = np.random.default_rng(w)
    frames = np.stack([np.where(depth > 50, depth + rng.uniform(-15, 15, depth.shape), depth)
                       for _ in range(9)]).astype(np.float32)
    frames[2, : h // 2] = 0
    frames[5] = frames[5] * 1.3
    b = Buffer2D(w, h)
    o = oracle.Buffer2D(w, h)
    assert torch.count_nonzero(b.getRawPointer()) == 0
    for f in frames:
        b.updateData(torch.from_numpy(f).cuda())
        o.update(f)
    assert np.array_equal(b.getDepthMap().cpu().numpy().view(np.uint32), o.depth_map().view(np.uint32))
    assert np.array_equal(b.getWeightMap().cpu().numpy(), o.weight_map())
    assert np.array_equal(b.getRawPointer().cpu().numpy().view(np.uint32), o.raw().view(np.uint32))
    # fused multi-frame update == frame by frame
    if (w * h) % 4 == 0:
        b2 = Buffer2D(w, h)
        b2.updateData(torch.from_numpy(frames).cuda())
        assert torch.equal(b2.getRawPointer(), b.getRawPointer())
    # insertData(float*), insertData(float2*) (w = row index quirk), insertData(weighted_d*)
    b.insertData(torch.from_numpy(frames[0]).cuda())
    o.insert(frames[0])
    assert np.array_equal(b.getRawPointer().cpu().numpy(), o.raw())
    xy = np.stack([frames[1], frames[2]], axis=-1).astype(np.float32)
    b.insertData2(torch.from_numpy(xy).cuda())
    o.insert_f32x2(xy)
    assert np.array_equal(b.getRawPointer().cpu().numpy(), o.raw())
    b3 = Buffer2D(w, h)
    b3.insertWeighted(b.getRawPointer().clone())
    assert torch.equal(b3.getRawPointer(), b.getRawPointer())
    b.initDeviceMemoryElements()
    assert torch.count_nonzero(b.getRawPointer()) == 0


def test_buffer2d_u16_host_path_and_golden(golden_dir):
    from kinectdepthmapenhancement_b200 import Buffer2D
    gold = np.load(os.path.join(golden_dir, "ref_golden.npz"))
    b = Buffer2D(96, 64)
    for f in gold["buf_frames"]:
        b.updateData(torch.from_numpy(f).cuda())
    assert np.array_equal(b.getDepthMap().cpu().numpy().view(np.uint32), gold["buf_depth"].view(np.uint32))
    assert np.array_equal(b.getWeightMap().cpu().numpy(), gold["buf_weight"])
    d16 = np.clip(gold["depth"], 0, 65535).astype(np.uint16)
    b = Buffer2D(96, 64)
    b.updateDataU16Host(torch.from_numpy(d16.view(np.int16)))
    o = oracle.Buffer2D(96, 64)
    o.update(d16.astype(np.float32))
    assert np.array_equal(b.getRawPointer().cpu().numpy(), o.raw())


@pytest.mark.parametrize("w,h,radius,use_labels", [(160, 120, 3, True), (160, 120, 3, False), (70, 50, 5, True)])
def test_guided_fill_vs_oracle(w, h, radius, use_labels):
    from kinectdepthmapenhancement_b200 import guided_fill
    depth, bgr = synth_np(w, h, seed=17, frame=radius)
    labels = ((np.arange(h)[:, None] // 16) * 64 + (np.arange(w)[None, :] // 12)).astype(np.int32) if use_labels else None
    got = guided_fill(torch.from_numpy(depth).cuda(), torch.from_numpy(bgr).cuda(),
                      torch.from_numpy(labels).cuda() if use_labels else None, radius).cpu().numpy()
    check_guided_against_f64(got, depth, bgr, labels, 2 * radius + 1, what="guided fill")


def test_guided_fill_golden(golden_dir):
    from kinectdepthmapenhancement_b200 import guided_fill
    gold = np.load(os.path.join(golden_dir, "ref_golden.npz"))
    got = guided_fill(torch.from_numpy(gold["depth"]).cuda(), torch.from_numpy(gold["bgr"]).cuda(),
                      torch.from_numpy(gold["labels"]).cuda(), 3).cpu().numpy()
    want = gold["guided_ws7"]
    assert np.array_equal(got > 0, want > 0)
    assert np.quantile(np.abs(got - want), 0.99) <= 5e-3


def test_jbf_golden(golden_dir):
    """GPU vs the reference kernel text's own fp32 outputs (tests/golden/ref_golden.npz, generated from
    the reference checkout by make_golden.py), including the exotic-sigma cases where fp32 products underflow and
    flip `weight > 0` (colour guard at sigma_c = 20 -> generic kernel; spatial LUT underflowing to 0 at
    sigma_s = 0.5): the valid/hole mask must equal the reference's bit for bit, and every value must be as
    close to the reference's as the reference itself is to the exact (fp64) formula, + 1e-3 mm."""
    from test_gpu_jbf import gpu_filter, parity_figures
    gold = np.load(os.path.join(golden_dir, "ref_golden.npz"))
    depth, guide = gold["depth"], gold["guide"]
    for key, r, ss, sc, sd in (("jbf_ws5", 2, 70.0, 50.0, 20.0), ("jbf_ws15", 7, 70.0, 50.0, 20.0),
                               ("jbf_ws7_sc20", 3, 70.0, 20.0, 20.0), ("jbf_ws7_ss05", 3, 0.5, 50.0, 20.0)):
        ref = gold[key]
        out, variant = gpu_filter(depth, guide, r, ss, sc, sd)
        assert np.array_equal(out > 0, ref > 0), f"{key}: mask differs from the reference text"
        assert np.array_equal(out == 0, ref == 0)
        o64, band, err, act = parity_figures(out, depth, guide, 2 * r + 1, ss, sc, sd)
        o64 = o64.astype(np.float64)
        floor = np.abs(ref.astype(np.float64) - o64)           # the reference's own fp32 noise
        dist = np.abs(out.astype(np.float64) - ref.astype(np.float64))
        print(f"\n{key} variant=0x{variant:x}: |gpu - ref| max {dist.max():.2e} median {np.median(dist):.2e}; "
              f"|ref - f64| max {floor.max():.2e}; |gpu - f64| max {np.abs(out - o64).max():.2e}")
        assert np.all(dist <= floor + 1e-3 + (0.05 + band) * act), f"{key}: farther from the reference than its own round-off"
        assert np.median(dist) <= 1e-3


def test_guided_fill_full_size_properties():
    """1920x1080 (config 3's guide size): holes stay holes only where no sample is in the window; values stay
    inside the range of the window's samples; a constant depth is reproduced."""
    from kinectdepthmapenhancement_b200 import guided_fill, synth
    w, h, r = 1920, 1080, 3
    d, c = synth.rgbd_frame(w, h, seed=6, frame=1, device="cuda")
    out = guided_fill(d, c, None, r)
    assert not torch.isnan(out).any()
    valid = (d > 50).float()[None, None]
    dil = torch.nn.functional.max_pool2d(valid, 2 * r + 1, 1, r)[0, 0] > 0
    assert torch.equal(out > 0, dil)
    big = torch.where(d > 50, d, torch.full_like(d, -1e30))[None, None]
    small = torch.where(d > 50, d, torch.full_like(d, 1e30))[None, None]
    mx = torch.nn.functional.max_pool2d(big, 2 * r + 1, 1, r)[0, 0]
    mn = -torch.nn.functional.max_pool2d(-small, 2 * r + 1, 1, r)[0, 0]
    m = out > 0
    assert torch.all(out[m] <= mx[m] + 2e-3) and torch.all(out[m] >= mn[m] - 2e-3)
    const = torch.where(d > 50, torch.full_like(d, 1500.25), torch.zeros_like(d))
    oc = guided_fill(const, c, None, r)
    assert torch.all((oc[oc > 0] - 1500.25).abs() <= 2.5e-4)


def test_guided_upsample_matches_oracle():
    """Config 3, label-guided variant: scatter fused into staging == oracle fill of the materialised sparse image."""
    from kinectdepthmapenhancement_b200.guided import guided_upsample
    from kinectdepthmapenhancement_b200 import guided_fill, synth
    wl, hl, wh, hh, r = 96, 80, 360, 204, 5
    lo, _ = synth.rgbd_frame(wl, hl, seed=6, frame=2, noise_rel=0.01)
    _, hi = synth.rgbd_frame(wh, hh, seed=6, frame=2)
    labels = ((np.arange(hh)[:, None] // 24) * 64 + (np.arange(wh)[None, :] // 30)).astype(np.int32)
    got = guided_upsample(lo.cuda(), hi.cuda(), torch.from_numpy(labels).cuda(), r).cpu().numpy()
    sparse = oracle.scatter_lowres(lo.numpy(), wh, hh)
    check_guided_against_f64(got, sparse, hi.numpy(), labels, 2 * r + 1, what="guided upsample")
    # identical to the same-resolution fill of the materialised sparse image
    dense = guided_fill(torch.from_numpy(sparse).cuda(), hi.cuda(), torch.from_numpy(labels).cuda(), r).cpu().numpy()
    assert np.array_equal(np.nan_to_num(dense, nan=-1).view(np.uint32), np.nan_to_num(got, nan=-1).view(np.uint32))
