"""GPU parity tests of the joint bilateral filter path (C-ABI -> sm_100a kernels) against the oracle.

Tolerance (north_star): valid/hole mask and output indexing bit-exact; filtered depth within
1e-3 mm of the fp64 evaluation of the reference formula.  Written out (check_against_f64):

    |kernel - oracle_f64| <= 1e-3 mm          on EVERY pixel where the skip-if-zero guard is inactive

flat, no conditioning term.  "Skip guard active" = the window holds a valid tap at or beyond the
fp32 expf() underflow distance (288.4 mm at sigma_d = 20) from the pass-1 mean, where
JointBilateralFilter.cu:67-68 gives the tap FULL weight: the output then mixes surfaces > 288 mm
apart and is a discontinuous function of the pass-1 mean (a tap within round-off of the cut-off
flips between ~0 and full weight).  Guard-active pixels are not absorbed into a looser bound: their
count, worst error and coordinates are printed, every one of them must still lie within 0.05 mm +
the fp64 formula's own sensitivity to +-2 fp32 ulps of its mean, and at most 1e-5 of a frame's pixels
(the cut-off flips) may exceed that.
"""
import os

import numpy as np
import pytest
import torch

from conftest import rule_active_mask, synth_np

import oracle

pytestmark = pytest.mark.gpu

TOL_MM = 1e-3          # north_star tolerance, regular pixels
TOL_ACTIVE_MM = 0.05   # skip-guard-active (ill-conditioned) pixels


def _jbf_cls():
    from kinectdepthmapenhancement_b200 import JointBilateralFilter
    return JointBilateralFilter


def gpu_filter(depth, guide3, radius, ss=70.0, sc=50.0, sd=20.0, env=None):
    """Run the GPU filter stage only, feeding the SAME smoothed guide the oracle gets."""
    h, w = depth.shape
    old = {}
    for k, v in (env or {}).items():
        old[k] = os.environ.get(k)
        os.environ[k] = v
    try:
        f = _jbf_cls()(w, h, ss, sc, sd, radius)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    pitch = (w + 3) & ~3
    g4 = np.zeros((1, h, pitch), np.uint32)
    g4[0, :, :w] = guide3[..., 0].astype(np.uint32) | (guide3[..., 1].astype(np.uint32) << 8) | \
        (guide3[..., 2].astype(np.uint32) << 16)
    d = torch.from_numpy(depth[None].copy()).cuda()
    g = torch.from_numpy(g4.view(np.int32)).cuda()
    out = f.filter_guide4(d, g)
    torch.cuda.synchronize()
    return out[0].cpu().numpy(), f.kernel_variant


def parity_figures(out, depth, guide3, ws, ss, sc, sd):
    """The parity block bench.py and smoke() report (same definitions as the asserts below)."""
    o64, band, m64 = oracle.jbf_envelope(depth, guide3, ws, ss, sc, sd)
    err = np.abs(out.astype(np.float64) - o64.astype(np.float64))
    act = rule_active_mask(depth, m64, ws, sd) if sd > 0 else np.zeros(depth.shape, bool)
    return o64, band, err, act


def check_against_f64(out, depth, guide3, ws, ss, sc, sd, label=""):
    """Mask bit-exact; |out - fp64 oracle| <= 1e-3 mm flat on every guard-inactive pixel; guard-active
    pixels listed and sanity-bounded.  See the module docstring and DESIGN.md."""
    o64, band, err, act = parity_figures(out, depth, guide3, ws, ss, sc, sd)
    o32 = oracle.jbf(depth, guide3, ws, ss, sc, sd, precision="f32")
    assert not np.isnan(out).any()
    assert np.array_equal(out > 0, o64 > 0), "valid/hole mask differs from the oracle"
    assert np.array_equal(out == 0, o64 == 0)
    e32 = np.abs(o32.astype(np.float64) - o64.astype(np.float64))
    reg = np.where(act, 0.0, err)
    yr, xr = np.unravel_index(np.argmax(reg), reg.shape)
    ea = np.where(act, err, 0.0)
    ya, xa = np.unravel_index(np.argmax(ea), ea.shape)
    out_act = act & (err > TOL_MM)
    frac = float((err <= TOL_MM).mean())
    frac32 = float((e32 <= TOL_MM).mean())
    print(f"\n{label} ws={ws}: regular max {reg.max():.2e} mm at (y={yr}, x={xr}); guard-active {int(act.sum())} px "
          f"({act.mean() * 100:.1f}%), of which {int(out_act.sum())} beyond 1e-3 mm, worst {ea.max():.2e} mm at "
          f"(y={ya}, x={xa}); within 1e-3 mm overall: kernel {frac * 100:.4f}% (reference-order fp32 {frac32 * 100:.3f}%)")
    assert reg.max() <= TOL_MM, f"guard-inactive pixel (y={yr}, x={xr}) off by {reg.max():.3e} mm (> 1e-3 mm flat)"
    # sanity bound on the ill-conditioned guard-active pixels (listed above, never hidden)
    viol = act & (err > TOL_MM + band + TOL_ACTIVE_MM)
    allowed = max(2, int(1e-5 * err.size))
    assert viol.sum() <= allowed, f"{int(viol.sum())} guard-active pixels beyond the sanity bound"
    return err, act


@pytest.mark.parametrize("w,h,radius", [(640, 480, 2), (640, 480, 7), (320, 240, 9), (256, 128, 15),
                                        (128, 96, 1), (192, 160, 4)])
def test_filter_matches_f64_oracle_tma_path_both_tile_heights(w, h, radius):
    depth, bgr = synth_np(w, h, seed=1234, frame=radius)
    guide = oracle.presmooth(bgr)
    out, variant = gpu_filter(depth, guide, radius)
    assert variant & 0x100, "expected the TMA-staged fast kernel"
    assert (variant & 1) == 0
    check_against_f64(out, depth, guide, 2 * radius + 1, 70.0, 50.0, 20.0, f"{w}x{h} variant=0x{variant:x}")
    # the other tile shape (64x16 instead of the 64x8 picked for small launches) must pass the same bound
    out_big, vbig = gpu_filter(depth, guide, radius, env={"KDME_TILE_H": "16"})
    assert not (vbig & 0xA00)
    check_against_f64(out_big, depth, guide, 2 * radius + 1, 70.0, 50.0, 20.0, f"{w}x{h} variant=0x{vbig:x}")


@pytest.mark.parametrize("w,h,radius", [(70, 50, 2), (70, 50, 7), (33, 17, 3), (5, 3, 2), (1, 1, 2), (101, 67, 5)])
def test_filter_ragged_sizes_plain_staging(w, h, radius):
    """Sizes that are not multiples of the tile (or of 4: no TMA) -- the reference would drop the
    remainder rows/cols (grid W/32 x H/24); every pixel is computed here."""
    depth, bgr = synth_np(w, h, seed=5, frame=radius)
    guide = oracle.presmooth(bgr)
    out, variant = gpu_filter(depth, guide, radius)
    if w % 4:
        assert not (variant & 0x100)
    check_against_f64(out, depth, guide, 2 * radius + 1, 70.0, 50.0, 20.0)


def test_tma_and_plain_staging_bit_identical():
    depth, bgr = synth_np(320, 240, seed=8, frame=0)
    guide = oracle.presmooth(bgr)
    a, va = gpu_filter(depth, guide, 7)
    b, vb = gpu_filter(depth, guide, 7, env={"KDME_NO_TMA": "1"})
    assert (va & 0x100) and not (vb & 0x100)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.parametrize("seed", list(range(24)))
def test_fuzz_small_frames(seed):
    """Random sizes (incl. smaller than a tile and not multiples of 4), radii 0..15, hole densities and
    sigma sets (fast and generic kernels): mask bit-exact and the float bound, against the fp64 oracle."""
    rng = np.random.default_rng(1000 + seed)
    w, h = int(rng.integers(1, 97)), int(rng.integers(1, 81))
    radius = int(rng.integers(0, 16))
    ss = float(rng.choice([0.5, 3.0, 20.0, 70.0]))
    sc = float(rng.choice([0.0, 10.0, 31.0, 50.0, 200.0]))
    sd = float(rng.choice([0.0, 5.0, 20.0, 100.0]))
    hole = float(rng.choice([0.0, 0.08, 0.5, 0.95]))
    depth, bgr = synth_np(w, h, seed=seed, frame=seed, hole_frac=hole)
    if seed % 5 == 0:
        depth[:] = 0.0          # all holes
    guide = oracle.presmooth(bgr)
    out, variant = gpu_filter(depth, guide, radius, ss, sc, sd)
    check_against_f64(out, depth, guide, 2 * radius + 1, ss, sc, sd,
                      f"fuzz {w}x{h} r={radius} ss={ss} sc={sc} sd={sd} holes={hole} variant=0x{variant:x}")


def test_result_independent_of_tile_height():
    """A pixel's arithmetic depends only on the image around it, not on the tile it falls in: 64x16, 64x8
    and 64x4 tiles give the same bits (this is what makes row bands equal the whole frame)."""
    depth, bgr = synth_np(320, 240, seed=8, frame=1)
    guide = oracle.presmooth(bgr)
    for r in (2, 7, 10):
        a, va = gpu_filter(depth, guide, r, env={"KDME_TILE_H": "16"})
        b, vb = gpu_filter(depth, guide, r, env={"KDME_TILE_H": "8"})
        c, vc = gpu_filter(depth, guide, r, env={"KDME_TILE_H": "4"})
        assert not (va & 0xA00) and (vb & 0x200) and (vc & 0x800)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
        assert np.array_equal(a.view(np.uint32), c.view(np.uint32))


def test_fp64_refinement_of_ill_conditioned_pixels():
    """Pixels between two surfaces (no sample near the pass-1 mean) are re-evaluated in fp64 by the whole
    warp; with the refinement disabled the same frame must differ ONLY there, and the refined values are
    the ones within tolerance."""
    depth, bgr = synth_np(320, 240, seed=8, frame=0)
    guide = oracle.presmooth(bgr)
    a, _ = gpu_filter(depth, guide, 7)
    b, _ = gpu_filter(depth, guide, 7, env={"KDME_NO_REFINE": "1"})
    o64, band, err_a, act = parity_figures(a, depth, guide, 15, 70.0, 50.0, 20.0)
    err_b = np.abs(b.astype(np.float64) - o64)
    diff = a != b
    print(f"\nrefined pixels that changed: {int(diff.sum())}; max regular error with / without refinement: "
          f"{np.where(act, 0, err_a).max():.2e} / {np.where(act, 0, err_b).max():.2e} mm")
    assert 0 < diff.sum() < 0.02 * a.size
    assert np.where(act, 0, err_a).max() <= TOL_MM
    assert err_a[diff].max() <= err_b[diff].max() + 1e-9


@pytest.mark.parametrize("ss,sc,sd,radius", [(70.0, 20.0, 20.0, 3),   # colour guard can fire (sigma_c < 30.6)
                                             (0.5, 50.0, 20.0, 3),    # spatial LUT underflows to 0 -> skipped
                                             (70.0, 0.0, 20.0, 2),    # sigma_c == 0: colour factor skipped
                                             (70.0, 50.0, 0.0, 2),    # sigma_d == 0: depth factor skipped
                                             (3.0, 35.0, 5.0, 6), (70.0, 50.0, 20.0, 0)])
def test_exotic_sigmas(ss, sc, sd, radius):
    depth, bgr = synth_np(160, 120, seed=21, frame=radius)
    guide = oracle.presmooth(bgr)
    out, variant = gpu_filter(depth, guide, radius, ss, sc, sd)
    if sc < 30.7 or sd == 0.0 or radius == 0:
        assert variant & 1, "expected the generic kernel for these parameters"
    check_against_f64(out, depth, guide, 2 * radius + 1, ss, sc, sd, f"exotic ss={ss} sc={sc} sd={sd}")


def test_generic_kernel_matches_fast_kernel():
    depth, bgr = synth_np(200, 150, seed=2, frame=1)
    guide = oracle.presmooth(bgr)
    a, va = gpu_filter(depth, guide, 5)
    b, vb = gpu_filter(depth, guide, 5, env={"KDME_FORCE_GENERIC": "1"})
    assert (va & 1) == 0 and (vb & 1) == 1
    assert np.array_equal(a > 0, b > 0)
    assert np.median(np.abs(a - b)) <= 2.5e-4
    check_against_f64(a, depth, guide, 11, 70.0, 50.0, 20.0, "fast")
    check_against_f64(b, depth, guide, 11, 70.0, 50.0, 20.0, "generic")


def test_holes_threshold_and_all_holes():
    JBF = _jbf_cls()
    w, h = 64, 48
    f = JBF(w, h, window_radius=2)
    color = torch.full((h, w, 3), 100, dtype=torch.uint8, device="cuda")
    depth = torch.full((h, w), 30.0, device="cuda")   # <= 50 mm: all holes
    f.Process(depth, color)
    assert torch.count_nonzero(f.getFiltered_Device()) == 0
    depth[20, 30] = 50.0                               # exactly 50 is still a hole (> 50.0f)
    f.Process(depth, color)
    assert torch.count_nonzero(f.getFiltered_Device()) == 0
    depth[20, 30] = 50.5
    f.Process(depth, color)
    out = f.getFiltered_Device()
    assert torch.count_nonzero(out) == 25 and torch.all(out[18:23, 28:33] == 50.5)
    depth[:] = float("nan")                            # NaN fails '> 50' as in the reference
    f.Process(depth, color)
    assert torch.count_nonzero(f.getFiltered_Device()) == 0 and not torch.isnan(f.getFiltered_Device()).any()


def test_presmooth_bit_exact_vs_oracle(golden_dir):
    import cv2
    img = cv2.imread(os.path.join(golden_dir, "guide_frame_640x480.png"), 1)
    h, w, _ = img.shape
    f = _jbf_cls()(w, h)
    g4 = f.presmooth(torch.from_numpy(img[None]).cuda())[0].cpu().numpy().view(np.uint32)
    want = oracle.presmooth(img)
    got = np.stack([(g4 >> s) & 0xFF for s in (0, 8, 16)], axis=-1).astype(np.uint8)[:, :w]
    assert (g4 >> 24).max() == 0
    assert np.array_equal(got, want)
    for (hh, ww) in [(3, 2), (1, 9), (37, 53)]:
        rng = np.random.default_rng(hh)
        im = rng.integers(0, 256, (hh, ww, 3), dtype=np.uint8)
        ff = _jbf_cls()(ww, hh)
        g = ff.presmooth(torch.from_numpy(im[None]).cuda())[0].cpu().numpy().view(np.uint32)
        got = np.stack([(g >> s) & 0xFF for s in (0, 8, 16)], axis=-1).astype(np.uint8)[:, :ww]
        assert np.array_equal(got, oracle.presmooth(im))


def _presmooth_bytes(f, img):
    g = f.presmooth(torch.from_numpy(np.ascontiguousarray(img)[None]).cuda())[0].cpu().numpy().view(np.uint32)
    g = g[:, :img.shape[1]]                      # the pitch is rounded up to 4 words: the pad columns are not written
    assert (g >> 24).max() == 0
    return np.stack([(g >> s) & 0xFF for s in (0, 8, 16)], axis=-1).astype(np.uint8)


@pytest.mark.parametrize("w,h", [(640, 96), (203, 61), (136, 40), (72, 33), (68, 20)])
def test_presmooth_rounding_ties_and_staging_paths(w, h):
    """The pre-smooth output byte is rint(sum / weight).  The kernel rounds s * rcp(ws) and falls back to the IEEE
    division only next to a half-integer, so images built to produce exact ties (two-valued patterns whose
    weighted means are k + 0.5) and near-ties must still match the oracle bit for bit; widths cover the 12-byte
    vector staging (tiles whose 72 columns lie inside 4-byte aligned rows), the byte-wise staging (row pitch
    3*203 is not a multiple of 4) and tiles that reflect at the border."""
    rng = np.random.default_rng(w * 1000 + h)
    f = _jbf_cls()(w, h)
    yy, xx = np.mgrid[0:h, 0:w]
    images = []
    for (a, b, sx, sy) in [(10, 11, 1, 1), (100, 103, 2, 1), (0, 255, 1, 2), (200, 201, 3, 3), (7, 8, 2, 2)]:
        pat = (((xx // sx) + (yy // sy)) & 1).astype(np.uint8)
        images.append(np.repeat((a + (b - a) * pat)[..., None], 3, axis=-1).astype(np.uint8))
    stripes = np.where((xx % 4) < 2, 50, 51).astype(np.uint8)
    images.append(np.stack([stripes, 255 - stripes, stripes // 2], axis=-1))
    images.append(rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
    images.append((rng.integers(0, 4, (h, w, 3)) + 120).astype(np.uint8))        # low contrast: every weight near 1
    images.append(np.full((h, w, 3), 255, np.uint8))
    for im in images:
        assert np.array_equal(_presmooth_bytes(f, im), oracle.presmooth(im))


def test_process_on_bundled_frame_reference_defaults(golden_dir):
    """Config 1: bundled input/color.jpg with the reference's defaults (window 5, 70/50/20, pre-smooth
    5/30/30).  input/depth.xml is a stripped blob in the reference checkout; a seeded surrogate depth
    is used and reported as such."""
    import cv2
    img = cv2.imread(os.path.join(golden_dir, "guide_frame_640x480.png"), 1)
    depth, _ = synth_np(640, 480, seed=2013, frame=0)
    JBF = _jbf_cls()
    f = JBF(640, 480)
    d = torch.from_numpy(depth).cuda()
    c = torch.from_numpy(img).cuda()
    f.Process(d, c)
    out = f.getFiltered_Device().cpu().numpy()
    host = f.getFiltered_Host().numpy()
    assert np.array_equal(out, host)
    smooth = f.getSmoothImage_Device().cpu().numpy()
    guide = oracle.presmooth(img)
    assert np.array_equal(smooth, guide)
    check_against_f64(out, depth, guide, 5, 70.0, 50.0, 20.0, "config1 color.jpg + surrogate depth")


def test_batch_equals_per_frame_and_output_indexing():
    from kinectdepthmapenhancement_b200 import synth
    n, w, h = 5, 128, 96
    depth, bgr = synth.rgbd_stream(n, w, h, seed=3)
    JBF = _jbf_cls()
    fb = JBF(w, h, window_radius=7, max_batch=2)   # forces internal chunking 2+2+1
    out_b = fb.process_batch(depth.cuda(), bgr.cuda()).cpu().numpy()
    f1 = JBF(w, h, window_radius=7)
    for i in range(n):
        f1.Process(depth[i].cuda(), bgr[i].cuda())
        assert np.array_equal(f1.getFiltered_Device().cpu().numpy().view(np.uint32), out_b[i].view(np.uint32))
    # indexing: a single valid pixel at (y, x) lights exactly its window, at out[y*W+x]
    d = torch.zeros((h, w), device="cuda")
    d[10, 100] = 1234.0
    f1.Process(d, bgr[0].cuda())
    o = f1.getFiltered_Device().cpu().numpy()
    ys, xs = np.nonzero(o)
    assert ys.min() == 3 and ys.max() == 17 and xs.min() == 93 and xs.max() == 107
    assert np.allclose(o[3:18, 93:108], 1234.0, atol=1e-3)


def test_process_host_pipeline_matches_device_path():
    from kinectdepthmapenhancement_b200 import synth
    n, w, h = 7, 160, 120
    depth, bgr = synth.rgbd_stream(n, w, h, seed=4)
    JBF = _jbf_cls()
    f = JBF(w, h, window_radius=3, max_batch=3)
    want = f.process_batch(depth.cuda(), bgr.cuda()).cpu()
    dh, ch = depth.pin_memory(), bgr.pin_memory()
    oh = torch.empty_like(depth).pin_memory()
    f.process_host(dh, ch, oh)
    assert torch.equal(oh, want)


def test_two_lane_chunk_pipeline_bit_identical_and_repeatable(monkeypatch):
    """jbf_process_batch / jbf_process_host alternate their chunks between the caller's stream and an internal lane
    (own guide buffer, refinement queue, TMA descriptors).  The lanes must change nothing: same bits and the same
    refinement counts as the single-lane order (KDME_ONE_LANE=1), call after call."""
    from kinectdepthmapenhancement_b200 import synth
    n, w, h = 11, 320, 240
    depth, bgr = synth.rgbd_stream(n, w, h, seed=8)          # this seed's frames hold ill-conditioned pixels
    JBF = _jbf_cls()
    monkeypatch.setenv("KDME_ONE_LANE", "1")
    f1 = JBF(w, h, window_radius=7, max_batch=2)
    monkeypatch.delenv("KDME_ONE_LANE")
    f2 = JBF(w, h, window_radius=7, max_batch=2)              # 2+2+2+2+2+1: six chunks, three per lane
    d, c = depth.cuda(), bgr.cuda()
    want = f1.process_batch(d, c).cpu()
    stats1 = f1.refine_stats()
    assert stats1[0] > 0 and stats1[1] == 0
    for _ in range(3):
        got = f2.process_batch(d, c).cpu()
        assert torch.equal(got.view(torch.int32), want.view(torch.int32))
        assert f2.refine_stats() == stats1
    # a single-frame call on the same handle right after (caller's lane only) still matches
    f2.Process(d[4], c[4])
    assert torch.equal(f2.getFiltered_Device().cpu().view(torch.int32), want[4].view(torch.int32))
    dh, ch = depth.pin_memory(), bgr.pin_memory()
    oh = torch.empty_like(depth).pin_memory()
    f2.process_host(dh, ch, oh)
    assert torch.equal(oh.view(torch.int32), want.view(torch.int32))


def test_two_lane_caches_follow_changing_calls(monkeypatch):
    """Each lane keeps its own TMA descriptors and refinement queue from call to call.  A sequence whose buffers,
    frame counts and kinds change between calls (so both lanes' cached descriptors go stale, and the host pipeline
    and two upsampling sizes follow) gives the same bits and refinement counts as a single-lane handle."""
    from kinectdepthmapenhancement_b200 import synth
    w, h = 320, 240
    depth, bgr = synth.rgbd_stream(12, w, h, seed=8)
    a_d, a_c = depth[:7].cuda(), bgr[:7].cuda()
    b_d, b_c = depth[7:].cuda(), bgr[7:].cuda()
    dh, ch = depth[2:7].pin_memory(), bgr[2:7].pin_memory()
    ups = []
    for wl, hl in ((160, 120), (107, 80)):
        lo = torch.stack([synth.rgbd_frame(wl, hl, seed=8, frame=k, noise_rel=0.01, hole_frac=0.1)[0]
                          for k in range(5)])
        ups.append((lo.cuda(), bgr[:5].cuda()))
    JBF = _jbf_cls()

    def run(f):
        results = []

        def record(out):
            results.append((out.cpu().view(torch.int32), f.refine_stats()))

        record(f.process_batch(a_d, a_c))
        record(f.process_batch(b_d, b_c))
        record(f.process_batch(a_d, a_c))
        oh = torch.empty_like(dh).pin_memory()
        f.process_host(dh, ch, oh)
        record(oh)
        for lo, hi in ups:
            record(f.upsample_batch(lo, hi))
        return results

    monkeypatch.setenv("KDME_ONE_LANE", "1")
    want = run(JBF(w, h, window_radius=7, max_batch=2))
    monkeypatch.delenv("KDME_ONE_LANE")
    got = run(JBF(w, h, window_radius=7, max_batch=2))
    assert sum(stats[0] for _, stats in want) > 0     # the refinement queues are exercised
    for k, ((g, gs), (e, es)) in enumerate(zip(got, want)):
        assert torch.equal(g, e), k
        assert gs == es, k


def test_pitched_gpumat_step_is_honoured():
    """cv::gpu::GpuMat rows may be padded (step > 3*width); the reference ignores step (it indexes
    (y*W+x)*3, JointBilateralFilter.cu:22-24) and only works for continuous images.  Through the C ABI a
    pitched image gives the same result as its continuous copy."""
    import ctypes as C
    from kinectdepthmapenhancement_b200 import _lib, synth
    w, h, pad = 160, 120, 7
    depth, bgr = synth.rgbd_frame(w, h, seed=9, frame=0, device="cuda")
    pitched = torch.zeros((h, w + pad, 3), dtype=torch.uint8, device="cuda")
    pitched[:, :w] = bgr
    f = _jbf_cls()(w, h, window_radius=3)
    f.Process(depth, bgr)
    want = f.getFiltered_Device().clone()
    _lib.check(_lib.lib().jbf_process(f._h, depth.data_ptr(), pitched.data_ptr(), 3 * (w + pad)))
    assert torch.equal(f.getFiltered_Device(), want)
    rc = _lib.lib().jbf_process(f._h, depth.data_ptr(), pitched.data_ptr(), 3 * w - 1)
    assert rc == _lib.KDME_EINVAL


def test_argument_errors():
    from kinectdepthmapenhancement_b200 import KdmeError
    JBF = _jbf_cls()
    with pytest.raises(KdmeError):
        JBF(0, 10)
    with pytest.raises(KdmeError):
        JBF(64, 48, window_radius=16)
    with pytest.raises(KdmeError):
        JBF(64, 48, color_sigma=-1.0)
    with pytest.raises(KdmeError):
        JBF(64, 48, max_batch=70000)
    f = JBF(64, 48)
    with pytest.raises(TypeError):
        f.Process(torch.zeros(48, 64), torch.zeros(48, 64, 3, dtype=torch.uint8))   # CPU tensors
    with pytest.raises(ValueError):
        f.Process(torch.zeros(48, 32, device="cuda"), torch.zeros(48, 64, 3, dtype=torch.uint8, device="cuda"))


# ------------------------------------------------------------------ full-size properties
def _dilate_gpu(valid, r):
    x = valid.float()[None, None]
    return torch.nn.functional.max_pool2d(x, 2 * r + 1, 1, r)[0, 0] > 0


@pytest.mark.parametrize("w,h,radius", [(3840, 2160, 15), (3840, 2160, 3), (1920, 1080, 7)])
def test_full_size_properties(w, h, radius):
    """At BASELINE.json's full sizes the CPU oracle is too slow; check size-independent properties:
    mask == window dilation of (d > 50); output inside [min, max] of the valid window depths;
    a constant valid depth is reproduced; and sampled rows agree with the fp64 oracle."""
    from kinectdepthmapenhancement_b200 import synth
    depth, bgr = synth.rgbd_frame(w, h, seed=99, frame=radius, device="cuda")
    f = _jbf_cls()(w, h, window_radius=radius)
    f.Process(depth, bgr)
    out = f.getFiltered_Device()
    valid = depth > 50
    assert torch.equal(out > 0, _dilate_gpu(valid, radius))
    big = torch.where(valid, depth, torch.full_like(depth, -1e30))[None, None]
    small = torch.where(valid, depth, torch.full_like(depth, 1e30))[None, None]
    mx = torch.nn.functional.max_pool2d(big, 2 * radius + 1, 1, radius)[0, 0]
    mn = -torch.nn.functional.max_pool2d(-small, 2 * radius + 1, 1, radius)[0, 0]
    m = out > 0
    assert torch.all(out[m] <= mx[m] + 2e-3) and torch.all(out[m] >= mn[m] - 2e-3)
    const = torch.where(valid, torch.full_like(depth, 2345.5), depth.clamp(max=50.0))
    f.Process(const, bgr)
    oc = f.getFiltered_Device()
    assert torch.all((oc[oc > 0] - 2345.5).abs() <= 2.5e-4)
    # a horizontal strip against the fp64 oracle (strip rows need the full vertical halo)
    y0 = h // 2 - 8
    rows = slice(y0 - radius, y0 + 16 + radius)
    f.Process(depth, bgr)
    g3 = f.getSmoothImage_Device()[rows].cpu().numpy()
    dnp = depth[rows].cpu().numpy()
    o64, band, m64 = oracle.jbf_envelope(dnp, g3, 2 * radius + 1)
    got = f.getFiltered_Device()[rows].cpu().numpy()
    inner = slice(radius, radius + 16)
    err = np.abs(got[inner].astype(np.float64) - o64[inner])
    act = rule_active_mask(dnp, m64, 2 * radius + 1, 20.0)[inner]
    assert np.where(act, 0, err).max() <= TOL_MM
    assert (act & (err > TOL_MM + band[inner] + TOL_ACTIVE_MM)).sum() <= 2


def test_upsample_matches_oracle_definition():
    """Config 3 (scaled down for the CPU oracle): ToF depth -> high-res guide, gather-form scatter."""
    from kinectdepthmapenhancement_b200 import synth
    wl, hl, wh, hh = 128, 106, 480, 270
    lo, _ = synth.rgbd_frame(wl, hl, seed=6, frame=0, noise_rel=0.01)
    _, hi = synth.rgbd_frame(wh, hh, seed=6, frame=0)
    f = _jbf_cls()(wh, hh, window_radius=7)
    out = f.Upsampling(lo.cuda(), hi.cuda()).cpu().numpy()
    guide = oracle.presmooth(hi.numpy())
    sparse = oracle.scatter_lowres(lo.numpy(), wh, hh)
    check_against_f64(out, sparse, guide, 15, 70.0, 50.0, 20.0, "upsample 128x106 -> 480x270")


def test_upsample_full_size_properties():
    """Config 3 at full size (512x424 ToF depth -> 1920x1080 guide, r=7): every low-res sample lands on its
    own site, the filled mask is the window dilation of the site mask, values stay inside the window range."""
    from kinectdepthmapenhancement_b200 import synth
    wl, hl, wh, hh, r = 512, 424, 1920, 1080, 7
    lo, _ = synth.rgbd_frame(wl, hl, seed=6, frame=0, noise_rel=0.01, device="cuda", hole_frac=0.02)
    _, hi = synth.rgbd_frame(wh, hh, seed=6, frame=0, device="cuda")
    f = _jbf_cls()(wh, hh, window_radius=r)
    out = f.Upsampling(lo, hi)
    sparse = torch.from_numpy(oracle.scatter_lowres(lo.cpu().numpy(), wh, hh)).cuda()
    valid = sparse > 50
    assert int((sparse != 0).sum()) == int((lo != 0).sum())
    assert torch.equal(out > 0, _dilate_gpu(valid, r))
    big = torch.where(valid, sparse, torch.full_like(sparse, -1e30))[None, None]
    small = torch.where(valid, sparse, torch.full_like(sparse, 1e30))[None, None]
    mx = torch.nn.functional.max_pool2d(big, 2 * r + 1, 1, r)[0, 0]
    mn = -torch.nn.functional.max_pool2d(-small, 2 * r + 1, 1, r)[0, 0]
    m = out > 0
    assert torch.all(out[m] <= mx[m] + 2e-3) and torch.all(out[m] >= mn[m] - 2e-3)
    # and the dense path on the materialised sparse image gives the same result bit for bit
    g4 = f.presmooth(hi[None])
    dense = f.filter_guide4(sparse[None].contiguous(), g4)[0]
    assert torch.equal(dense.view(torch.int32), out.view(torch.int32))


def test_mrf_and_projective_to_real():
    from kinectdepthmapenhancement_b200 import projective_to_real
    depth, bgr = synth_np(160, 120, seed=12, frame=0)
    f = _jbf_cls()(160, 120)
    out = f.mrf(torch.from_numpy(depth).cuda(), torch.from_numpy(bgr).cuda()).cpu().numpy()
    want = oracle.mrf(depth, bgr)
    assert np.abs(out - want).max() <= 2e-3
    xyz = projective_to_real(torch.from_numpy(depth).cuda(), 525.0, 525.0, 80, 60).cpu().numpy()
    assert np.array_equal(xyz.view(np.uint32), oracle.projective_to_real(depth, 525.0, 525.0, 80, 60).view(np.uint32))


def test_process_xyz_equals_projective_to_real_of_filtered():
    """f3 as SURVEY 8(f) asks: back-projection fused into the filter epilogue (main.cpp:179 + :182 as one launch
    pair) is bit-identical to projectiveToReal(filtered) -- also on the pixels re-evaluated in fp64."""
    from kinectdepthmapenhancement_b200 import projective_to_real, synth
    for (w, h, r, sc) in [(640, 480, 7, 50.0), (322, 241, 2, 50.0), (70, 50, 3, 50.0), (96, 64, 3, 20.0)]:   # last: generic kernel
        depth, bgr = synth.rgbd_frame(w, h, seed=8, frame=0, device="cuda")
        f = _jbf_cls()(w, h, 70.0, sc, 20.0, window_radius=r)
        xyz = f.process_xyz(depth, bgr, 525.0, 520.0, w // 2, h // 2)
        filt = f.getFiltered_Device().clone()
        f.Process(depth, bgr)
        assert torch.equal(filt.view(torch.int32), f.getFiltered_Device().view(torch.int32))
        want = projective_to_real(filt, 525.0, 520.0, w // 2, h // 2)
        assert torch.equal(xyz.view(torch.int32), want.view(torch.int32))
        assert np.array_equal(want.cpu().numpy().view(np.uint32),
                              oracle.projective_to_real(filt.cpu().numpy(), 525.0, 520.0, w // 2, h // 2).view(np.uint32))


def test_process_host_u16_and_library_pinned_buffers():
    """Sensor-format depth (uint16 mm) uploaded and converted on the device == the float path on the same
    integers; buffers from kdme_host_alloc (plain and write-combined)."""
    from kinectdepthmapenhancement_b200 import synth
    from kinectdepthmapenhancement_b200.jbf import host_buffer
    n, w, h = 5, 160, 120
    depth, bgr = synth.rgbd_stream(n, w, h, seed=4)
    d_int = depth.round().clamp_(0, 65535)
    f = _jbf_cls()(w, h, window_radius=3, max_batch=2)
    want = f.process_batch(d_int.cuda(), bgr.cuda()).cpu()
    for wc in (False, True):
        dh = host_buffer((n, h, w), torch.int16, write_combined=wc)
        ch = host_buffer((n, h, w, 3), torch.uint8, write_combined=wc)
        oh = host_buffer((n, h, w), torch.float32)
        dh.copy_(d_int.to(torch.int32).to(torch.int16))
        ch.copy_(bgr)
        f.process_host(dh, ch, oh)
        assert torch.equal(oh, want)
    with pytest.raises(ValueError):
        f.process_host(torch.zeros((n, h, w)), torch.zeros((n - 1, h, w, 3), dtype=torch.uint8), torch.zeros((n, h, w)))


def test_refine_stats_and_queue():
    """Ill-conditioned pixels are counted; a frame of one flat surface has none."""
    depth, bgr = synth_np(320, 240, seed=8, frame=0)
    f = _jbf_cls()(320, 240, window_radius=7)
    f.Process(torch.from_numpy(depth).cuda(), torch.from_numpy(bgr).cuda())
    refined, dropped = f.refine_stats()
    assert refined > 0 and dropped == 0
    flat = np.full((240, 320), 1500.0, np.float32)
    f.Process(torch.from_numpy(flat).cuda(), torch.from_numpy(bgr).cuda())
    assert f.refine_stats() == (0, 0)


def test_filter_guide4_rejects_mismatched_tensors():
    f = _jbf_cls()(64, 48, window_radius=2)
    d = torch.zeros((2, 48, 64), device="cuda")
    g = torch.zeros((2, 48, 64), dtype=torch.int32, device="cuda")
    f.filter_guide4(d, g)
    with pytest.raises(ValueError):
        f.filter_guide4(d, g[:1])
    with pytest.raises(ValueError):
        f.filter_guide4(d, torch.zeros((2, 48, 62), dtype=torch.int32, device="cuda"))
    with pytest.raises(ValueError):
        f.filter_guide4(d, g, out=torch.zeros((1, 48, 64), device="cuda"))
    with pytest.raises(ValueError):
        f.filter_guide4(d, g, out=d)
    with pytest.raises(ValueError):
        f.filter_guide4(torch.zeros((2, 48, 32), device="cuda"), g)


@pytest.mark.parametrize("wl,hl,wh,hh,r", [(512, 424, 1920, 1080, 7), (64, 48, 64, 48, 3), (50, 37, 131, 97, 5),
                                         (100, 80, 127, 90, 2), (17, 9, 640, 480, 15), (33, 20, 70, 50, 7)])
def test_upsample_gather_equals_dense_bit_for_bit(wl, hl, wh, hh, r):
    """The gather form (site lattice only) and the dense kernel on the scattered tile are the same arithmetic:
    every scale from 1:1 to 37:1, ragged sizes, radii 2..15, holes in the low-res map."""
    from kinectdepthmapenhancement_b200 import synth
    lo, _ = synth.rgbd_frame(wl, hl, seed=6, frame=r, noise_rel=0.01, device="cuda", hole_frac=0.1)
    _, hi = synth.rgbd_frame(wh, hh, seed=6, frame=r, device="cuda")
    f = _jbf_cls()(wh, hh, window_radius=r)
    a = f.Upsampling(lo, hi).clone()
    va = f.kernel_variant
    os.environ["KDME_UPSAMPLE_DENSE"] = "1"
    try:
        b = f.Upsampling(lo, hi).clone()
    finally:
        os.environ.pop("KDME_UPSAMPLE_DENSE", None)
    vb = f.kernel_variant
    assert (va & 0x1000) and not (vb & 0x1000)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    sparse = oracle.scatter_lowres(lo.cpu().numpy(), wh, hh)
    if wh * hh <= 200 * 200:
        guide = oracle.presmooth(hi.cpu().numpy())
        check_against_f64(a.cpu().numpy(), sparse, guide, 2 * r + 1, 70.0, 50.0, 20.0, f"upsample {wl}x{hl}->{wh}x{hh}")
