"""CPU tests of the oracle: pinned to the reference's own kernel text (live when oracle/_ref
is built, and through committed golden vectors always), plus the properties the domain offers."""
import os

import numpy as np
import pytest

from conftest import synth_np

import oracle


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "ref_golden.npz"))


# ---------------------------------------------------------------- golden vectors (reference text)
def test_golden_inputs_reproducible(gold):
    d, c = synth_np(96, 64, seed=77, frame=3)
    assert np.array_equal(d, gold["depth"]) and np.array_equal(c, gold["bgr"])
    assert np.array_equal(oracle.presmooth(c), gold["guide"])


@pytest.mark.parametrize("key,ws,ss,sc,sd", [("jbf_ws5", 5, 70.0, 50.0, 20.0), ("jbf_ws15", 15, 70.0, 50.0, 20.0),
                                             ("jbf_ws7_sc20", 7, 70.0, 20.0, 20.0),
                                             ("jbf_ws7_ss05", 7, 0.5, 50.0, 20.0)])
def test_jbf_restatement_matches_reference_golden(gold, key, ws, ss, sc, sd):
    out = oracle.jbf(gold["depth"], gold["guide"], ws, ss, sc, sd, precision="f32", threads=2)
    assert np.array_equal(out.view(np.uint32), gold[key].view(np.uint32)), "fp32 restatement != reference text"


def test_guided_fill_matches_reference_golden(gold):
    out = oracle.guided_fill(gold["depth"], gold["bgr"], gold["labels"], threads=2)
    assert np.array_equal(out.view(np.uint32), gold["guided_ws7"].view(np.uint32))
    out = oracle.guided_fill(gold["depth"], gold["bgr"], None, threads=2)
    assert np.array_equal(out.view(np.uint32), gold["guided_ws7_nolabel"].view(np.uint32))


# ---------------------------------------------------------------- guided fill: the fp64 guard (DESIGN.md section 2)
def _guided_guard(d, c, lab=None, ws=7, **kw):
    o, mean, guard = oracle.guided_fill(d, c, lab, ws, precision="f64", return_mean=True, return_guard=True,
                                        threads=2, **kw)
    return o, mean, guard


def test_guided_guard_is_clear_on_a_smooth_frame():
    w, h = 64, 48
    yy, xx = np.mgrid[0:h, 0:w]
    d = (1500.0 + 3.0 * xx + 2.0 * yy).astype(np.float32)
    c = np.stack([(xx * 2) % 256, (yy * 3) % 256, np.full_like(xx, 128)], -1).astype(np.uint8)
    for ws in (3, 7, 15):
        o, _, guard = _guided_guard(d, c, ws=ws)
        assert not np.isnan(o).any() and np.all(o > 0)
        assert not guard.any(), ws


def test_guided_guard_flags_a_depth_tap_at_the_cut():
    """Two surfaces with labels of their own: the near one's sweep-1 mean is exactly 1000, and the far one is moved
    so that e^2 kd of its taps lands on the expf() zero cut of sweep 3."""
    w, h, ws, sd = 16, 9, 7, 70.0
    c = np.full((h, w, 3), 100, np.uint8)
    lab = (np.arange(w)[None, :] >= 8).astype(np.int32) * np.ones((h, 1), np.int32)
    kd = 1.0 / (2.0 * sd * sd)
    y, x = 4, 7                                              # the last column of the near surface
    for far, flagged in ((1000.0 + np.sqrt(103.97207708399179 / kd), True), (1000.0 + 1015.0, False)):
        d = np.where(lab == 0, 1000.0, far).astype(np.float32)
        _, mean, guard = _guided_guard(d, c, lab, ws=ws, sigma_d=sd)
        assert mean[y, x] == 1000.0
        assert bool(guard[y, x] & 1) == flagged, far


def test_guided_guard_flags_a_colour_tap_at_the_cut():
    """Sweep 1 with sigma_c chosen so that cd / (2 sigma_c^2) of one tap is the cut exactly."""
    w, h = 5, 5
    d = np.full((h, w), 1000.0, np.float32)
    c = np.full((h, w, 3), 50, np.uint8)
    c[0, 0] = (60, 50, 50)                                   # cd = 100 for the centre pixel
    sc = np.float32(np.sqrt(100.0 / (2.0 * 103.97207708399179)))
    _, _, guard = _guided_guard(d, c, ws=5, sigma_c=float(sc))
    assert guard[2, 2] & 1
    _, _, guard = _guided_guard(d, c, ws=5, sigma_c=float(sc) * 1.01)
    assert not guard[2, 2] & 1


def test_guided_guard_flags_the_recurrence_test():
    """adaptive = 5 dev / mean^2 within a few ulps of sigma * 0.3f at the first valid tap."""
    w, h, ws = 3, 1, 3
    c = np.full((h, w, 3), 7, np.uint8)
    # three taps of one label, depths m - a, m, m + a: dev = 2a/3, adaptive = 10a / (3 m^2)
    m = np.float32(64.0)
    # sigma_c is set so that sigma_c * 0.3f is about adaptive; scan a until the rounding puts it within the margin
    for a in np.linspace(1.0, 14.0, 2000, dtype=np.float32):
        d = np.array([[m - a, m, m + a]], np.float32)
        if (d > 50).all():
            _, _, g = _guided_guard(d, c, ws=ws, sigma_c=float(np.float32(10.0) * np.float32(a) / (3 * m * m) / 0.3))
            if g[0, 1] & 2:
                break
    else:
        pytest.fail("no recurrence-test case found")


def test_guided_guard_flags_the_underflow_of_2_sigma_squared():
    """sigma = adaptive from the first valid tap (sigma_c * 0.3f is below it), with adaptive = 5 dev / mean^2 so small
    that 2 sigma^2 is a few subnormal ulps or 0: the -0/0 NaN is decided there.  A spread of one fp32 ulp at 1e15-1e16
    gives adaptive from 1.5e-22 (2 sigma^2 = 32 subnormal ulps: clear) down to 2.4e-23 (2 sigma^2 = 0: NaN)."""
    c = np.full((1, 3, 3), 7, np.uint8)
    flags = []
    for base in (1e15, 3e15, 1e16):
        b = np.float32(base)
        d = np.array([[b, np.nextafter(b, np.float32(np.inf)), b]], np.float32)
        o, _, guard = _guided_guard(d, c, ws=3, sigma_c=1e-23)
        flags.append((bool(guard[0, 1] & 4), bool(np.isnan(o[0, 1]))))
    assert flags == [(False, False), (True, False), (True, True)]


def test_mrf_matches_reference_golden(gold):
    out = oracle.mrf(gold["depth"], gold["bgr"], threads=2)
    assert np.array_equal(out.view(np.uint32), gold["mrf_ws5"].view(np.uint32))


def _mrf_f32_vs_f64(depth, bgr, ws, sc, sm):
    """The fp64 MRF keeps the fp32 restatement's mask, and differs from it by no more than the fp32 restatement's
    own worst-case rounding: sequential sums of ws*ws non-negative terms (num, den), expf and the quotient."""
    o32 = oracle.mrf(depth, bgr, ws, sc, sm, threads=2)
    o64 = oracle.mrf(depth, bgr, ws, sc, sm, threads=2, precision="f64")
    assert np.array_equal(o32 > 0, o64 > 0) and np.array_equal(o32 == 0, o64 == 0)
    gamma = (2 * ws * ws + 6) * 2.0 ** -24
    err = np.abs(o32.astype(np.float64) - o64.astype(np.float64))
    assert (err <= gamma * np.abs(o64.astype(np.float64)) + 1e-30).all(), err.max()
    return err


@pytest.mark.parametrize("ws,sc,sm", [(5, 50.0, 150.0), (3, 1e-2, 150.0), (11, 1e-3, 1.0), (1, 1e-4, 150.0),
                                      (5, 0.0, 150.0), (5, 50.0, 0.0)])
def test_mrf_f64_keeps_f32_mask_and_values(gold, ws, sc, sm):
    _mrf_f32_vs_f64(gold["depth"], gold["bgr"], ws, sc, sm)
    for seed in (3, 4):
        d, c = synth_np(70, 50, seed=seed, frame=seed)
        _mrf_f32_vs_f64(d, c, ws, sc, sm)


def test_mrf_f64_subnormal_weights_fill_holes():
    """A hole whose only valid neighbours are at colour distance 2: the fp32 reference weight 150 expf(-100) is
    a subnormal, so the hole's output is a tiny positive number, not 0; past the expf() cut it is 0."""
    d = np.zeros((3, 3), np.float32)
    d[0, :] = 1000.0
    c = np.zeros((3, 3, 3), np.uint8)
    c[0, :, 0] = 1
    c[0, :, 1] = 1
    for sc, filled in ((50.0, True), (52.0, False)):
        o32 = oracle.mrf(d, c, 3, sc, 150.0)
        o64 = oracle.mrf(d, c, 3, sc, 150.0, precision="f64")
        assert (o32[1, 1] > 0) == filled and (o64[1, 1] > 0) == filled
        assert o64[1, 1] < 1e-35 and o64[2, 1] == 0


def test_depth_bilateral_xyz_matches_reference_golden(gold):
    out = oracle.depth_bilateral_xyz(gold["f2_normalized"], gold["f2_points"], threads=2)
    assert np.array_equal(out.view(np.uint32), gold["f2_out"].view(np.uint32))


def test_buffer2d_matches_reference_golden(gold):
    b = oracle.Buffer2D(96, 64)
    for f in gold["buf_frames"]:
        b.update(f)
    assert np.array_equal(b.depth_map().view(np.uint32), gold["buf_depth"].view(np.uint32))
    assert np.array_equal(b.weight_map(), gold["buf_weight"])
    b2 = oracle.Buffer2D(96, 64)
    d = gold["depth"]
    b2.insert_f32x2(np.stack([d, d * 0.5], axis=-1).astype(np.float32))
    assert np.array_equal(b2.raw(), gold["buf_xy_raw"])
    # the documented quirk: w == row index (Buffer2D.cu:137)
    assert np.array_equal(b2.weight_map()[:, 0], np.arange(64, dtype=np.float32))


# ---------------------------------------------------------------- live check against oracle/_ref
needs_ref = pytest.mark.skipif(not oracle.ref_available(),
                               reason="oracle/_ref not built (no reference checkout found)")


@needs_ref
@pytest.mark.parametrize("w,h,ws", [(70, 50, 5), (64, 48, 15), (33, 29, 9), (5, 4, 7)])
def test_live_ref_jbf_bit_exact(w, h, ws):
    d, c = synth_np(w, h, seed=9, frame=ws)
    g = oracle.presmooth(c)
    a = oracle.jbf(d, g, ws, precision="f32", threads=2)
    b = oracle.jbf(d, g, ws, precision="f32", impl="ref", threads=2)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


@needs_ref
def test_live_ref_guided_and_buffer_bit_exact():
    d, c = synth_np(48, 40, seed=4, frame=1)
    lab = ((np.arange(40)[:, None] // 10) * 4 + (np.arange(48)[None, :] // 12)).astype(np.int32)
    a = oracle.guided_fill(d, c, lab, threads=2)
    b = oracle.guided_fill(d, c, lab, impl="ref", threads=2)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32), )
    bo, br = oracle.Buffer2D(48, 40), oracle.Buffer2D(48, 40, impl="ref")
    rng = np.random.default_rng(0)
    for _ in range(6):
        f = np.where(d > 50, d + rng.uniform(-8, 8, d.shape), d).astype(np.float32)
        bo.update(f), br.update(f)
    assert np.array_equal(bo.raw().view(np.uint32), br.raw().view(np.uint32))


# ---------------------------------------------------------------- properties
def _dilate(valid, ws):
    h, w = valid.shape
    r = ws // 2
    p = np.pad(valid, r)
    out = np.zeros_like(valid)
    for i in range(ws):
        for j in range(ws):
            out |= p[i:i + h, j:j + w]
    return out


@pytest.mark.parametrize("ws", [5, 15])
@pytest.mark.parametrize("prec", ["f32", "f64"])
def test_mask_is_window_dilation(ws, prec):
    d, c = synth_np(80, 60, seed=3, frame=2, hole_frac=0.6)
    g = oracle.presmooth(c)
    out = oracle.jbf(d, g, ws, precision=prec, threads=2)
    assert not np.isnan(out).any()
    assert np.array_equal(out > 0, _dilate(d > 50, ws))
    assert np.all(out[~_dilate(d > 50, ws)] == 0)


def test_values_of_30mm_are_holes():
    d = np.full((20, 20), 30.0, np.float32)   # below the 50 mm threshold (JointBilateralFilter.cu:21)
    c = np.zeros((20, 20, 3), np.uint8)
    assert np.all(oracle.jbf(d, c, 5) == 0)
    d[10, 10] = 1000.0
    out = oracle.jbf(d, c, 5)
    assert np.all(out[8:13, 8:13] == 1000.0) and out.sum() == 25 * 1000.0


def test_output_within_window_range_and_f32_close_to_f64():
    d, c = synth_np(96, 72, seed=11, frame=0)
    g = oracle.presmooth(c)
    for ws in (5, 15):
        o64 = oracle.jbf(d, g, ws, precision="f64", threads=2)
        o32 = oracle.jbf(d, g, ws, precision="f32", threads=2)
        r = ws // 2
        big = np.pad(np.where(d > 50, d, -np.inf), r, constant_values=-np.inf)
        small = np.pad(np.where(d > 50, d, np.inf), r, constant_values=np.inf)
        mx = np.full(d.shape, -np.inf)
        mn = np.full(d.shape, np.inf)
        for i in range(ws):
            for j in range(ws):
                mx = np.maximum(mx, big[i:i + 72, j:j + 96])
                mn = np.minimum(mn, small[i:i + 72, j:j + 96])
        m = o64 > 0
        assert np.all(o64[m] <= mx[m] + 1e-3) and np.all(o64[m] >= mn[m] - 1e-3)
        assert np.median(np.abs(o32 - o64)) < 1e-3


def test_skip_if_zero_depth_guard():
    """A tap farther than sqrt(103.97*2*sd^2) = 288.4 mm from the pass-1 mean keeps its FULL weight
    (JointBilateralFilter.cu:67-68): two equal populations 1000 mm apart average to the midpoint."""
    d = np.full((9, 9), 1000.0, np.float32)
    d[:, 5:] = 2000.0
    c = np.full((9, 9, 3), 128, np.uint8)
    lut = oracle.spatial_lut(9, 70.0)
    for prec in ("f32", "f64"):
        out = oracle.jbf(d, c, 9, precision=prec)
        w_left = lut.reshape(9, 9)[:, :5].sum()
        w_right = lut.reshape(9, 9)[:, 5:].sum()
        expect = (1000 * w_left + 2000 * w_right) / (w_left + w_right)
        assert abs(out[4, 4] - expect) < 0.05


def test_presmooth_matches_opencv_definition(golden_dir):
    cv2 = pytest.importorskip("cv2")
    img = cv2.imread(os.path.join(golden_dir, "guide_frame_640x480.png"), 1)
    assert img is not None and img.shape == (480, 640, 3)
    ours = oracle.presmooth(img)
    theirs = cv2.bilateralFilter(img, 5, 30, 30)
    diff = np.abs(ours.astype(np.int32) - theirs.astype(np.int32))
    assert diff.max() <= 1
    assert (diff > 0).mean() < 1e-3
    assert np.abs(ours.astype(np.int32) - img.astype(np.int32)).max() > 5   # the smooth is not a no-op


def test_presmooth_border_and_tiny_images():
    rng = np.random.default_rng(1)
    for (h, w) in [(1, 1), (1, 7), (3, 2), (6, 5)]:
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        out = oracle.presmooth(img)
        assert out.shape == img.shape
    flat = np.full((8, 8, 3), 77, np.uint8)
    assert np.array_equal(oracle.presmooth(flat), flat)


def test_upsample_sites_and_fill():
    wl, hl, wh, hh = 16, 12, 60, 34
    lo = np.arange(wl * hl, dtype=np.float32).reshape(hl, wl) + 1000
    sp = oracle.scatter_lowres(lo, wh, hh)
    assert (sp > 0).sum() == wl * hl            # every sample lands on its own site
    ys, xs = np.nonzero(sp)
    assert ys.max() < hh and xs.max() < wh
    c = np.full((hh, wh, 3), 90, np.uint8)
    up = oracle.upsample(lo, c, radius=4)
    assert np.all(up > 0)                       # radius >= ceil(max scale) fills everything


def test_projective_to_real():
    d = np.full((4, 6), 1000.0, np.float32)
    xyz = oracle.projective_to_real(d, 500.0, 500.0, 3, 2)
    assert xyz[2, 3].tolist() == [0.0, 0.0, 1000.0]
    assert xyz[0, 0].tolist() == [-6.0, 4.0, 1000.0]
