"""The next-row operators against the fp64 oracle (DESIGN.md, "Tolerance"):

    f1  MarkovRandomField          jbf_mrf                    mask bit-exact, |out - f64| <= 1e-3 mm on every pixel
    f2  Projection_GPU::bilateral  kdme_depth_bilateral_xyz   mask bit-exact (bar taps at the expf() cut),
                                                              |z - f64| <= 1e-3 mm, x,y = normalized.x,y * z exactly
    f3  projectiveToReal           kdme_projective_to_real    bit-exact against the fp32 restatement
    f4  mean 3-D error             kdme_mean_3d_error         count exact, mean within 1e-12 of an fp64 sum

at the sizes where the 32x8 stencil tiles and the grid-stride loops have ragged or repeated passes, at every
radius class, and off the default sigmas, where the weights are neither all 0 nor all equal.  Only the argument
checks run without a GPU.
"""
import ctypes

import numpy as np
import pytest

from conftest import synth_np

import oracle

TOL_MM = 1e-3
EXP_ZERO_ARG = 103.97207708399179   # fp32 expf(-a) == 0 for a beyond this
SMALL = [(1, 1), (31, 7), (33, 9), (70, 50), (160, 120)]


def sizes_radii(radii):
    """Every size at every radius, except radius 15 above 160x120 (runtime)."""
    return [(w, h, r) for (w, h) in SMALL + [(640, 480)] for r in radii if r < 15 or w * h <= 160 * 120]


def _torch():
    import torch
    return torch


def _frame(w, h, seed=12, frame=0):
    if w * h <= 4:   # the synthetic scene has no structure at this size: a fixed valid/hole pattern
        d = np.array([900.0, 0.0, 1234.5, 30.0], np.float32)[: w * h].reshape(h, w)
        c = np.array([[10, 20, 30], [11, 20, 30], [200, 0, 5], [10, 22, 30]], np.uint8)[: w * h].reshape(h, w, 3)
        return d, c
    return synth_np(w, h, seed=seed, frame=frame)


# ------------------------------------------------------------------------------------------- f1 MRF
_filters = {}


def gpu_mrf(depth, bgr, radius, sc, sm):
    torch = _torch()
    from kinectdepthmapenhancement_b200 import JointBilateralFilter
    h, w = depth.shape
    if (w, h) not in _filters:
        _filters.clear()
        _filters[(w, h)] = JointBilateralFilter(w, h)
    out = _filters[(w, h)].mrf(torch.from_numpy(depth).cuda(), torch.from_numpy(np.ascontiguousarray(bgr)).cuda(),
                               radius, sc, sm)
    return out.cpu().numpy()


def check_mrf(depth, bgr, radius, sc=oracle.MRF_SIGMA_C, sm=oracle.MRF_SMOOTH, label=""):
    out = gpu_mrf(depth, bgr, radius, sc, sm)
    o64 = oracle.mrf(depth, bgr, 2 * radius + 1, sc, sm, precision="f64")
    err = np.abs(out.astype(np.float64) - o64.astype(np.float64))
    y, x = np.unravel_index(np.argmax(err), err.shape)
    mm = (out > 0) != (o64 > 0)
    print(f"\nmrf {label} r={radius} sc={sc} sm={sm}: max {err.max():.2e} mm at (y={y}, x={x}); "
          f"{int(mm.sum())} mask mismatches at {np.argwhere(mm)[:8].tolist()}")
    assert not np.isnan(out).any()
    assert np.array_equal(out > 0, o64 > 0) and np.array_equal(out == 0, o64 == 0), "mask differs from fp64"
    assert err.max() <= TOL_MM, f"(y={y}, x={x}) off by {err.max():.3e} mm"


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,radius", sizes_radii([0, 1, 2, 5, 15]))
def test_mrf_sizes_and_radii(w, h, radius):
    d, c = _frame(w, h)
    check_mrf(d, c, radius, label=f"{w}x{h}")


@pytest.mark.gpu
def test_mrf_full_hd():
    d, c = _frame(1920, 1080, seed=3)
    check_mrf(d, c, 2, label="1920x1080")


@pytest.mark.gpu
@pytest.mark.parametrize("radius", [1, 5, 15])
@pytest.mark.parametrize("sc", [0.0, 1e-4, 1e-3, 1e-2, 50.0])
@pytest.mark.parametrize("sm", [0.0, 1.0, 150.0])
def test_mrf_sigmas(radius, sc, sm):
    """Off the default sigma_c = 50 the weights are no longer 150 or ~0: the sums carry many equal-sized taps."""
    d, c = _frame(160, 120)
    check_mrf(d, c, radius, sc, sm, label="160x120")


@pytest.mark.gpu
@pytest.mark.parametrize("radius", [1, 2, 5])
def test_mrf_crafted(radius):
    w, h = 40, 24
    # hole centres whose only valid neighbours sit at colour distance 2: the weight 150 expf(-100) is an fp32
    # subnormal, so the reference leaves a tiny positive value, not 0 (sigma_c = 52 puts them past the cut)
    d = np.full((h, w), 1000.0, np.float32)
    c = np.full((h, w, 3), 100, np.uint8)
    d[6:18, 10:30] = 0.0
    c[6:18, 10:30] = (101, 101, 100)
    for sc in (50.0, 52.0):
        check_mrf(d, c, radius, sc, 150.0, label="hole ring cd=2")
    # all holes, and a hole frame with a 30 mm (invalid, non-zero) centre value
    check_mrf(np.zeros((h, w), np.float32), c, radius, label="all holes")
    check_mrf(np.full((h, w), 30.0, np.float32), c, radius, label="all 30 mm")
    # a constant guide: every weight is smooth * 1
    d2, _ = _frame(w, h, seed=5)
    check_mrf(d2, np.full((h, w, 3), 7, np.uint8), radius, label="constant guide")


# ---------------------------------------------------------------------------- f2 cloud bilateral
def cloud(depth, fx=525.0, fy=525.0):
    h, w = depth.shape
    pts = oracle.projective_to_real(depth, fx, fy, w // 2, h // 2)
    z = np.where(pts[..., 2] > 0, pts[..., 2], 1)
    norm = pts.copy()
    norm[..., 0] /= z
    norm[..., 1] /= z
    return norm, pts


def gpu_f2(norm, pts, radius, ss, sd):
    torch = _torch()
    from kinectdepthmapenhancement_b200 import evalio
    out = evalio.depth_bilateral_xyz(torch.from_numpy(norm).cuda(), torch.from_numpy(pts).cuda(), radius, ss, sd)
    return out.cpu().numpy()


def at_cut(z, radius, sd):
    """Pixels with a valid tap whose |dz| lies within 2 fp32 ulps of the expf() cut sqrt(2 kExpZeroArg) sd."""
    h, w = z.shape
    cut = np.sqrt(2.0 * EXP_ZERO_ARG) * sd
    zp = np.pad(z, radius)
    near = np.zeros((h, w), bool)
    for i in range(2 * radius + 1):
        for j in range(2 * radius + 1):
            zq = zp[i:i + h, j:j + w]
            band = 2.0 * np.spacing(np.maximum(np.maximum(np.abs(zq), np.abs(z)), np.float32(cut)).astype(np.float32))
            near |= (zq > 50) & (np.abs(np.abs(zq.astype(np.float64) - z) - cut) <= band)
    return near


def check_f2(norm, pts, radius, ss=oracle.PROJ_SIGMA_S, sd=oracle.PROJ_SIGMA_D, label="", got=None):
    out = gpu_f2(norm, pts, radius, ss, sd) if got is None else got
    o64 = oracle.depth_bilateral_xyz(norm, pts, 2 * radius + 1, ss, sd, precision="f64")
    z, z64 = out[..., 2], o64[..., 2]
    mm = (z > 0) != (z64 > 0)
    near = at_cut(pts[..., 2], radius, sd)
    err = np.where(mm, 0.0, np.abs(z.astype(np.float64) - z64.astype(np.float64)))
    y, x = np.unravel_index(np.argmax(err), err.shape)
    print(f"\nf2 {label} r={radius} ss={ss} sd={sd}: z max {err.max():.2e} mm at (y={y}, x={x}); "
          f"{int(mm.sum())} mask mismatches at {np.argwhere(mm)[:8].tolist()} ({int((mm & near).sum())} at the cut)")
    assert not np.isnan(z).any()
    assert not (mm & ~near).any(), "mask differs from fp64 away from the expf() cut"
    assert mm.sum() <= max(2, int(1e-5 * z.size))
    assert err.max() <= TOL_MM, f"(y={y}, x={x}) off by {err.max():.3e} mm"
    assert np.array_equal(out[..., :2].view(np.uint32), (norm[..., :2] * z[..., None]).view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,radius", sizes_radii([0, 1, 3, 7, 15]))
def test_f2_sizes_and_radii(w, h, radius):
    d, _ = _frame(w, h, seed=8, frame=1)
    check_f2(*cloud(d), radius, label=f"{w}x{h}")


@pytest.mark.gpu
def test_f2_full_hd():
    d, _ = _frame(1920, 1080, seed=3)
    check_f2(*cloud(d), 3, label="1920x1080")


@pytest.mark.gpu
@pytest.mark.parametrize("radius", [1, 7, 15])
@pytest.mark.parametrize("ss", [0.5, 5.0, 20.0, 200.0])
@pytest.mark.parametrize("sd", [20.0, 100.0, 300.0, 1000.0])
def test_f2_sigmas(radius, ss, sd):
    d, _ = _frame(160, 120, seed=8, frame=1)
    check_f2(*cloud(d), radius, ss, sd, label="160x120")


@pytest.mark.gpu
@pytest.mark.parametrize("wall", [1400.0, 1445.0, 1460.0, 1475.0, 1485.0])
@pytest.mark.parametrize("radius", [3, 7])
def test_f2_hole_patch_in_a_wall(wall, radius):
    """A 4x4 hole patch in a flat wall: at the default sigma_d = 100 the wall's taps lie 14.42 sd or more from
    the holes' z = 0 from 1442 mm on, where expf() is 0, so the reference leaves the holes empty."""
    h, w = 24, 40
    d = np.full((h, w), wall, np.float32)
    d[10:14, 18:22] = 0.0
    norm, pts = cloud(d)
    out = gpu_f2(norm, pts, radius, 20.0, 100.0)
    filled = int((out[10:14, 18:22, 2] > 0).sum())
    assert filled == (16 if wall < 1442.0 else 0), filled
    check_f2(norm, pts, radius, label=f"wall {wall}", got=out)


@pytest.mark.gpu
@pytest.mark.parametrize("radius", [1, 3, 7])
def test_f2_invalid_nonzero_centre(radius):
    d, _ = _frame(70, 50, seed=9)
    d = d.copy()
    d[d <= 50] = 30.0
    d[20:24, 30:34] = 30.0
    norm, pts = cloud(d)
    check_f2(norm, pts, radius, label="30 mm holes")
    check_f2(norm, pts, radius, 20.0, 2.0, label="30 mm holes, narrow sd")


@pytest.mark.gpu
def test_f2_alternating_parameters_use_their_own_tables():
    """The log2 spatial table is cached per (device, window, sigma_s): every call must still see its own."""
    d, _ = _frame(160, 120, seed=8, frame=1)
    norm, pts = cloud(d)
    for radius, ss in ((3, 20.0), (3, 5.0), (7, 20.0), (3, 20.0), (7, 5.0), (3, 5.0)):
        check_f2(norm, pts, radius, ss, label="alternating")


# ------------------------------------------------------------------------------ f3 back-projection
def _depth_with_holes(w, h, seed):
    rng = np.random.default_rng(seed)
    d = rng.uniform(300.0, 9000.0, (h, w)).astype(np.float32)
    d[rng.random((h, w)) < 0.1] = 0.0
    d[rng.random((h, w)) < 0.02] = 30.0
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(1, 1), (7, 3), (640, 480), (1920, 1080), (3840, 2160)])
def test_projective_to_real_bit_exact(w, h):
    """Bit-exact with the fp32 restatement; 1920x1080 and 3840x2160 exceed the 148*16 blocks of 256 threads, so
    the grid-stride loop runs more than one pass."""
    torch = _torch()
    from kinectdepthmapenhancement_b200 import projective_to_real
    d = _depth_with_holes(w, h, seed=w + h)
    dt = torch.from_numpy(d).cuda()
    for fx, fy, cx, cy in ((525.0, 525.0, w // 2, h // 2), (517.3, 523.9, -40, -7), (588.1, 561.7, w + 100, h + 50),
                           (0.5, 1e4 / 3, 0, h - 1)):
        got = projective_to_real(dt, fx, fy, cx, cy).cpu().numpy()
        want = oracle.projective_to_real(d, fx, fy, cx, cy)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (fx, fy, cx, cy)


# --------------------------------------------------------------------------------- f4 3-D error
_EDGE_Z = np.array([50.0, 15000.0, np.nextafter(np.float32(50.0), np.float32(1e9)),
                    np.nextafter(np.float32(15000.0), np.float32(0.0)), np.nan, np.inf, -np.inf, -700.0, 0.0],
                   np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 255, 257, 148 * 8 * 256 - 1, 148 * 8 * 256 + 1, 3840 * 2160, 4 * 3840 * 2160])
def test_mean_3d_error(n):
    """Count exact and mean within 1e-12 of the fp64 sum of the kernel's fp32 distances, with z on and just inside
    both bounds, NaN, +-inf and negative z in either cloud; n around and past the 148*8 blocks of 256 threads."""
    torch = _torch()
    from kinectdepthmapenhancement_b200 import evalio
    rng = np.random.default_rng(n)
    truth = np.empty((n, 3), np.float32)
    truth[:, 2] = rng.uniform(400.0, 9000.0, n)
    truth[:, :2] = rng.uniform(-3000.0, 3000.0, (n, 2))
    pts = (truth + rng.normal(0.0, 8.0, (n, 3))).astype(np.float32)
    if n > 1:
        k = len(_EDGE_Z)
        idx = rng.choice(n, size=min(n - 1, 4 * k), replace=False)
        for m, i in enumerate(idx):
            (pts if m % 2 == 0 else truth)[i, 2] = _EDGE_Z[(m // 2) % k]
    want, cnt = oracle.mean_3d_error_f64(pts, truth)
    got, gcnt = evalio.mean_3d_error(torch.from_numpy(pts).cuda(), torch.from_numpy(truth).cuda())
    assert gcnt == cnt and cnt >= 1
    assert abs(got - want) <= 1e-12 * want, (got, want)


# ------------------------------------------------------------------------------------ argument checks
@pytest.mark.parametrize("ss,sd", [(0.0, 100.0), (-1.0, 100.0), (float("nan"), 100.0), (20.0, 0.0), (20.0, -5.0),
                                   (20.0, float("nan"))])
def test_f2_rejects_bad_sigmas(ss, sd):
    """sigma_s = 0 would make the centre's spatial weight NaN.  The check comes before any device access, so
    without a GPU stand-in addresses do; with one the clouds are real device buffers."""
    from kinectdepthmapenhancement_b200 import _lib
    torch = _torch()
    if torch.cuda.is_available():
        bufs = [torch.ones((16, 16, 3), device="cuda") for _ in range(3)]
        p = [ctypes.c_void_p(b.data_ptr()) for b in bufs]
        stream = torch.cuda.current_stream().cuda_stream
    else:
        p, stream = [ctypes.c_void_p(a) for a in (0x1000, 0x2000, 0x3000)], None
    rc = _lib.lib().kdme_depth_bilateral_xyz(*p, 16, 16, 3, ss, sd, stream)
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    assert rc == _lib.KDME_EINVAL and b"sigma" in _lib.lib().kdme_last_error()
