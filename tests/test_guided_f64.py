"""The guided cross-bilateral fill (depthmap_enhancement, EdgeRefinedSuperpixel.cu:104-205) and its label-guided
upsampling held to the fp64 contract of DESIGN.md section 2, pixel by pixel.

check_guided_against_f64 is the one check: the NaN positions and the mask `out > 0` equal those of the fp64 oracle,
and every other pixel is within 1e-3 mm of it, except the guard-active pixels the oracle names (a branch of the fp32
formula decided within a few ulps of its threshold), which must stay inside the range of their window's samples.
Nothing here is derived from the kernel's output.  The cases sweep the shapes (ragged against the 32x8 tile, 1x1 to
1920x1080), both forms of the guided kernel (the compile-time window at r = 1..3, the run-time window at r = 0
and r >= 4), the sigmas, labels, the guide formats, uint16 depth and frames built to hit each branch of the formula.
"""
import numpy as np
import pytest

import oracle

SS, SC, SD = oracle.ERS_SIGMA_S, oracle.ERS_SIGMA_C, oracle.ERS_SIGMA_D   # 30, 50, 70
TOL_MM = 1e-3        # every guard-active-free pixel
SANITY_MM = 0.05     # the JBF's sanity bound for guard-active pixels


# ------------------------------------------------------------------ the contract
def window_range(depth, window):
    """Per pixel, [min, max] of the valid (> 50) samples of its window (+inf/-inf where there is none)."""
    d = np.asarray(depth, np.float64)
    h, w = d.shape
    r = window // 2
    valid = d > 50
    lo = np.pad(np.where(valid, d, np.inf), r, constant_values=np.inf)
    hi = np.pad(np.where(valid, d, -np.inf), r, constant_values=-np.inf)
    mn, mx = np.full((h, w), np.inf), np.full((h, w), -np.inf)
    for i in range(window):
        for j in range(window):
            mn = np.minimum(mn, lo[i:i + h, j:j + w])
            mx = np.maximum(mx, hi[i:i + h, j:j + w])
    return mn, mx


def check_guided_against_f64(got, depth, bgr, labels, window, sigma_s=SS, sigma_c=SC, sigma_d=SD, what=""):
    """`got` (the GPU output) against orc_guided_fill_f64 on the same float depth, BGR guide and labels.
    Returns the oracle's output and guard map, for cases that assert a property of the oracle itself."""
    got = np.asarray(got, np.float32)
    o64, guard = oracle.guided_fill(depth, bgr, labels, window, sigma_s, sigma_c, sigma_d, precision="f64",
                                    return_guard=True)
    assert got.shape == o64.shape
    nan = np.isnan(o64)
    assert np.array_equal(np.isnan(got), nan), f"{what}: NaN positions differ ({np.isnan(got).sum()} vs {nan.sum()})"
    ok = ~nan
    bad_mask = ok & ((got > 0) != (o64 > 0))
    assert not bad_mask.any(), f"{what}: mask out > 0 differs at {np.argwhere(bad_mask)[:8].tolist()}"
    err = np.where(ok, np.abs(got.astype(np.float64) - o64.astype(np.float64)), 0.0)
    act = ok & (guard != 0)
    reg = np.where(act, 0.0, err)
    worst = np.unravel_index(np.argmax(reg), reg.shape)
    print(f"\n{what}: {got.shape[1]}x{got.shape[0]} window {window}: max |err| {reg.max():.3e} mm at {list(worst)}, "
          f"{int((reg > TOL_MM).sum())} regular pixels beyond {TOL_MM}")
    if act.any():
        ea = np.where(act, err, 0.0)
        wa = np.unravel_index(np.argmax(ea), ea.shape)
        print(f"  guard-active: {int(act.sum())} pixels (bits {sorted(set(np.unique(guard[act]).tolist()))}), "
              f"worst {ea.max():.3e} mm at {list(wa)}; first {np.argwhere(act)[:6].tolist()}")
    assert reg.max() <= TOL_MM, (f"{what}: {int((reg > TOL_MM).sum())} pixels beyond {TOL_MM} mm, worst "
                                 f"{reg.max():.3e} at {list(worst)}: got {got[worst]!r}, fp64 {o64[worst]!r}")
    if act.any():
        mn, mx = window_range(depth, window)
        v = act & (got > 0)
        assert np.all(got[v] >= mn[v]) and np.all(got[v] <= mx[v]), f"{what}: guard-active pixel outside its window"
        assert int((act & (err > SANITY_MM)).sum()) <= max(2, int(1e-5 * got.size)), f"{what}: too many beyond 0.05 mm"
    return o64, guard


# ------------------------------------------------------------------ inputs
def frame(w, h, seed, edge_mm=0.0, noise_rel=0.01):
    """A synthetic RGB-D frame (float depth with holes, BGR guide); edge_mm > 0 adds that step to the valid depth
    right of a third of the width, a depth edge running through every row."""
    from kinectdepthmapenhancement_b200 import synth
    d, c = synth.rgbd_frame(w, h, seed=seed, frame=seed % 7, noise_rel=noise_rel, hole_frac=0.1)
    d, c = d.numpy().copy(), c.numpy().copy()
    if edge_mm:
        d[:, w // 3:] = np.where(d[:, w // 3:] > 50, d[:, w // 3:] + np.float32(edge_mm), d[:, w // 3:])
    return d, c


def block_labels(w, h, by=16, bx=12):
    return ((np.arange(h)[:, None] // by) * 1000 + (np.arange(w)[None, :] // bx)).astype(np.int32)


def gpu_fill(depth, guide, labels, r, ss=SS, sc=SC, sd=SD):
    import torch
    from kinectdepthmapenhancement_b200 import guided_fill
    lab = torch.from_numpy(labels).cuda() if labels is not None else None
    return guided_fill(torch.from_numpy(depth).cuda(), torch.from_numpy(guide).cuda(), lab, r, ss, sc, sd).cpu().numpy()


def as_bgr(guide):
    """The BGR image a GRAY / BGRX guide stands for: (g, 0, 0) and (b, g, r)."""
    if guide.ndim == 2:
        return np.stack([guide, np.zeros_like(guide), np.zeros_like(guide)], axis=-1)
    return np.ascontiguousarray(guide[..., :3])


def guide_as(bgr, c):
    if c == 1:
        return np.ascontiguousarray(bgr[..., 1])
    if c == 4:
        return np.ascontiguousarray(np.concatenate([bgr, np.full(bgr.shape[:2] + (1,), 77, np.uint8)], axis=-1))
    return bgr


# ------------------------------------------------------------------ sizes, radii, labels, guide formats
@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(1, 1), (5, 3), (33, 17), (161, 121)])
@pytest.mark.parametrize("r", [0, 1, 2, 3, 4, 5, 7, 10, 15])
@pytest.mark.parametrize("use_labels", [False, True])
def test_fill_shapes_and_radii(w, h, r, use_labels):
    d, c = frame(w, h, seed=w + r, edge_mm=1500.0)
    lab = block_labels(w, h, 9, 13) if use_labels else None
    check_guided_against_f64(gpu_fill(d, c, lab, r), d, c, lab, 2 * r + 1, what=f"r={r} labels={use_labels}")


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,r", [(640, 480, 3), (640, 480, 7), (1920, 1080, 7)])
def test_fill_full_frames_with_labels(w, h, r):
    d, c = frame(w, h, seed=5, edge_mm=2000.0)
    lab = block_labels(w, h, 24, 30)
    check_guided_against_f64(gpu_fill(d, c, lab, r), d, c, lab, 2 * r + 1, what=f"{w}x{h} r={r}")


@pytest.mark.gpu
@pytest.mark.parametrize("r,ch", [(2, 1), (5, 4)])   # one non-BGR format per kernel
def test_fill_guide_formats(r, ch):
    d, c = frame(161, 121, seed=40 + r, edge_mm=900.0)
    lab = block_labels(161, 121)
    g = guide_as(c, ch)
    check_guided_against_f64(gpu_fill(d, g, lab, r), d, as_bgr(g), lab, 2 * r + 1, what=f"C={ch} r={r}")


@pytest.mark.gpu
@pytest.mark.parametrize("edge_mm", [700.0, 1500.0, 3000.0])
@pytest.mark.parametrize("r", [3, 5, 7])
def test_fill_depth_edges(edge_mm, r):
    """Depth edges of 0.7-3 m, where fp32 sweeps centred on an fp32 mean miss the fp64 value by up to 4e-2 mm."""
    d, c = frame(160, 120, seed=int(edge_mm) + r, edge_mm=edge_mm)
    check_guided_against_f64(gpu_fill(d, c, None, r), d, c, None, 2 * r + 1, what=f"edge {edge_mm} r={r}")


# ------------------------------------------------------------------ sigmas on both kernels (sc 30.63: sweep 1's colour cut)
@pytest.mark.gpu
@pytest.mark.parametrize("sc", [0.0, 10.0, 30.6, 30.7, 50.0, 200.0])
@pytest.mark.parametrize("r", [3, 5])
def test_fill_colour_sigmas(sc, r):
    d, c = frame(161, 121, seed=60 + r, edge_mm=1200.0)
    lab = block_labels(161, 121)
    check_guided_against_f64(gpu_fill(d, c, lab, r, sc=sc), d, c, lab, 2 * r + 1, sigma_c=sc, what=f"sc={sc} r={r}")


@pytest.mark.gpu
@pytest.mark.parametrize("sd", [0.0, 5.0, 70.0, 1000.0])
@pytest.mark.parametrize("r", [2, 7])
def test_fill_depth_sigmas(sd, r):
    d, c = frame(161, 121, seed=70 + r, edge_mm=800.0)
    check_guided_against_f64(gpu_fill(d, c, None, r, sd=sd), d, c, None, 2 * r + 1, sigma_d=sd, what=f"sd={sd} r={r}")


@pytest.mark.gpu
@pytest.mark.parametrize("ss", [0.5, 30.0, 200.0])
@pytest.mark.parametrize("r", [1, 4])
def test_fill_spatial_sigmas(ss, r):
    d, c = frame(161, 121, seed=80 + r, edge_mm=1000.0)
    lab = block_labels(161, 121)
    check_guided_against_f64(gpu_fill(d, c, lab, r, ss=ss), d, c, lab, 2 * r + 1, sigma_s=ss, what=f"ss={ss} r={r}")


# ------------------------------------------------------------------ crafted frames
@pytest.mark.gpu
@pytest.mark.parametrize("r", [3, 7])
def test_flat_patch_gives_the_fp64_formulas_nan(r):
    """One depth and one colour: the deviation is 0, sigma decays by 0.3 per valid tap until 2 sigma^2 underflows,
    and the next zero-distance tap makes -0/0 = NaN.  This is the NaN of the formula evaluated with an exact mean; the
    fp32 reference text, whose mean of one depth is rarely that depth, gives it on far fewer pixels (DESIGN.md
    section 2)."""
    w, h = 40, 30
    d = np.full((h, w), 1234.5, np.float32)
    d[::7, ::5] = 0.0
    c = np.full((h, w, 3), (90, 120, 200), np.uint8)
    o64, _ = check_guided_against_f64(gpu_fill(d, c, None, r), d, c, None, 2 * r + 1, what=f"flat r={r}")
    assert np.isnan(o64).sum() > 0


@pytest.mark.gpu
def test_zero_distance_taps_before_the_underflow_keep_the_pixel():
    """The 45 taps of the window's first three rows match the centre's colour and come before 2 sigma^2 underflows
    (about the 47th valid tap); every later tap differs in colour, and sigma is 0 by the centre tap: no NaN."""
    r, n = 7, 15
    d = np.full((n, n), 1500.0, np.float32)
    c = np.full((n, n, 3), (10, 20, 30), np.uint8)
    c[3:] = (11, 20, 30)
    c[r, r] = (10, 20, 30)
    o64, _ = check_guided_against_f64(gpu_fill(d, c, None, r), d, c, None, 2 * r + 1, what="underflow after")
    assert not np.isnan(o64[r, r]) and o64[r, r] > 0


def depth_cut_arguments(depth, mean, window, sigma_d):
    """e^2 kd of every (pixel, valid window tap) pair, with e the tap's depth minus the pixel's fp64 sweep-1 mean as
    the oracle computes it (pixels without a mean are left out)."""
    d = np.asarray(depth, np.float64)
    h, w = d.shape
    r = window // 2
    kd = 1.0 / (2.0 * sigma_d * sigma_d)
    dp = np.pad(np.where(d > 50, d, np.nan), r, constant_values=np.nan)
    has = mean > 0
    out = [((dp[i:i + h, j:j + w] - mean) ** 2 * kd)[has] for i in range(window) for j in range(window)]
    z = np.concatenate(out)
    return z[~np.isnan(z)]


@pytest.mark.gpu
@pytest.mark.parametrize("shift_mm", [-0.5, 0.0, 0.5])
@pytest.mark.parametrize("r", [3, 7])
def test_two_surfaces_at_the_depth_cut(shift_mm, r):
    """Two surfaces with labels of their own, 14.42 sigma_d apart: sweep 1 keeps each pixel's mean on its own surface,
    so in sweep 3 the other surface's taps sit at the expf() zero cut of the depth factor, past which the reference
    gives them full weight.  That taps fall just below and just above the cut is asserted from the oracle's mean."""
    w, h = 64, 40
    cut = 103.97207708399179
    rng = np.random.default_rng(10 * r + int(10 * shift_mm) + 5)
    far = np.float32(1200.0 + np.sqrt(cut * 2.0 * SD * SD) + shift_mm)
    left = np.arange(w)[None, :] < w // 2
    d = np.where(left, 1200.0 + rng.uniform(-0.5, 0.5, (h, w)), far + rng.uniform(-1.0, 1.0, (h, w))).astype(np.float32)
    lab = np.where(left, 0, 1).astype(np.int32) * np.ones((h, 1), np.int32)
    c = rng.integers(100, 110, (h, w, 3), dtype=np.uint8)
    _, mean = oracle.guided_fill(d, c, lab, 2 * r + 1, precision="f64", return_mean=True)
    z = depth_cut_arguments(d, mean, 2 * r + 1, SD)
    assert ((z > cut - 0.1) & (z < cut)).sum() >= 20 and ((z > cut) & (z < cut + 0.1)).sum() >= 20
    check_guided_against_f64(gpu_fill(d, c, lab, r), d, c, lab, 2 * r + 1, what=f"cut {shift_mm:+} mm r={r}")


@pytest.mark.gpu
def test_own_label_without_a_sample_gives_zero():
    """A pixel whose label has no valid sample reads 0 although other labels' samples fill its window."""
    w, h, r = 48, 32, 3
    d, c = frame(w, h, seed=9, noise_rel=0.01)
    d[d <= 50] = 1000.0
    lab = np.zeros((h, w), np.int32)
    ys, xs = np.arange(4, h - 4, 5), np.arange(4, w - 4, 7)
    for k, (y, x) in enumerate((y, x) for y in ys for x in xs):
        lab[y, x] = 100 + k
        d[y, x] = 0.0
    o64, _ = check_guided_against_f64(gpu_fill(d, c, lab, r), d, c, lab, 2 * r + 1, what="own label empty")
    assert np.all(o64[lab >= 100] == 0)


@pytest.mark.gpu
@pytest.mark.parametrize("r", [2, 5])
def test_depths_at_the_hole_threshold(r):
    """50 is a hole, 50.5 a sample, NaN a hole."""
    w, h = 70, 50
    d, c = frame(w, h, seed=11)
    rng = np.random.default_rng(r)
    pick = rng.random(d.shape)
    d[pick < 0.15] = 50.0
    d[(pick >= 0.15) & (pick < 0.3)] = 50.5
    d[(pick >= 0.3) & (pick < 0.4)] = np.nan
    check_guided_against_f64(gpu_fill(d, c, None, r), d, c, None, 2 * r + 1, what=f"threshold r={r}")


@pytest.mark.gpu
@pytest.mark.parametrize("r", [3, 7])
def test_uint16_depth_including_65535(r):
    import torch
    from kinectdepthmapenhancement_b200 import guided_fill
    w, h, n = 97, 61, 2
    frames = [frame(w, h, seed=20 + k, edge_mm=1000.0) for k in range(n)]
    d = np.stack([np.clip(np.round(f[0]), 0, 65535) for f in frames]).astype(np.float32)
    c = np.stack([f[1] for f in frames])
    d[:, 10:20, 30:45] = 65535.0
    d[:, 40, :] = 51.0
    lab = np.stack([block_labels(w, h, 11, 17) for _ in range(n)])
    got = guided_fill(torch.from_numpy(d.astype(np.int32)).to(torch.uint16).cuda(), torch.from_numpy(c).cuda(),
                      torch.from_numpy(lab).cuda(), r).cpu().numpy()
    for k in range(n):
        check_guided_against_f64(got[k], d[k], c[k], lab[k], 2 * r + 1, what=f"uint16 frame {k} r={r}")


# ------------------------------------------------------------------ upsampling
def _lowres(wl, hl, seed, edge_mm=1000.0):
    d, _ = frame(wl, hl, seed=seed, edge_mm=edge_mm)
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("wl,hl,w,h,r,use_labels", [(512, 424, 1920, 1080, 7, True), (17, 9, 640, 480, 7, True),
                                                    (1, 1, 9, 5, 1, False), (33, 17, 33, 17, 3, True),
                                                    (96, 80, 360, 204, 5, False)])
@pytest.mark.parametrize("u16", [False, True])
def test_upsample_matches_the_f64_fill_of_the_sparse_image(wl, hl, w, h, r, use_labels, u16):
    import torch
    from kinectdepthmapenhancement_b200.guided import guided_upsample
    lo = _lowres(wl, hl, seed=wl + r)
    if u16:
        lo = np.clip(np.round(lo), 0, 65535).astype(np.float32)
        lo.reshape(-1)[:: max(1, lo.size // 5)] = 65535.0
    _, hi = frame(w, h, seed=h)
    lab = block_labels(w, h, 24, 30) if use_labels else None
    lt = torch.from_numpy(lo.astype(np.int32)).to(torch.uint16)[None] if u16 else torch.from_numpy(lo)[None]
    got = guided_upsample(lt.cuda(), torch.from_numpy(hi)[None].cuda(),
                          torch.from_numpy(lab)[None].cuda() if use_labels else None, r).cpu().numpy()[0]
    sparse = oracle.scatter_lowres(lo, w, h)
    check_guided_against_f64(got, sparse, hi, lab, 2 * r + 1, what=f"upsample {wl}x{hl}->{w}x{h} r={r} u16={u16}")


@pytest.mark.gpu
def test_last_upsampled_frame_of_a_batch():
    import torch
    from kinectdepthmapenhancement_b200.guided import guided_upsample
    n, wl, hl, w, h, r = 3, 64, 48, 320, 240, 7
    lo = np.stack([_lowres(wl, hl, seed=30 + k) for k in range(n)])
    hi = np.stack([frame(w, h, seed=40 + k)[1] for k in range(n)])
    lab = np.stack([block_labels(w, h, 20 + k, 25) for k in range(n)])
    got = guided_upsample(torch.from_numpy(lo).cuda(), torch.from_numpy(hi).cuda(), torch.from_numpy(lab).cuda(),
                          r).cpu().numpy()
    sparse = oracle.scatter_lowres(lo[n - 1], w, h)
    check_guided_against_f64(got[n - 1], sparse, hi[n - 1], lab[n - 1], 2 * r + 1, what="last upsampled frame")
