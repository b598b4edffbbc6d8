"""Guide formats other than packed BGR: GRAY/IR (1 byte per pixel) and BGRX/BGRA (4 bytes per pixel).

One identity defines them, and every GPU test below checks it bit for bit against the same call made with
the derived BGR image:

    GRAY g            == BGR (g, 0, 0)
    BGRX (b, g, r, x) == BGR (b, g, r)        (the 4th byte never enters a weight)

The CPU tests pin the GRAY pre-smooth definition (OpenCV's 1-channel bilateral: L1 colour distance |dg|)
against cv2 and check the C ABI / C++ surface without a device.
"""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT, synth_np

import oracle


# ------------------------------------------------------------------ CPU: ABI surface
def _declared():
    text = open(os.path.join(ROOT, "include", "kdme_b200.h")).read()
    return set(re.findall(r"\b((?:jbf|kdme)_[a-z0-9_]+)\s*\(", re.sub(r"/\*.*?\*/", "", text, flags=re.S)))


def test_header_declares_and_library_exports_the_guide_format_entry_points():
    from kinectdepthmapenhancement_b200 import _lib
    names = ("jbf_set_guide_channels", "kdme_guided_fill_ex", "kdme_guided_upsample_ex")
    assert set(names) <= _declared()
    text = open(os.path.join(ROOT, "include", "kdme_b200.h")).read()
    for c, v in (("GRAY", 1), ("BGR", 3), ("BGRX", 4)):
        assert re.search(rf"#define KDME_GUIDE_{c} {v}\b", text)
        assert getattr(_lib, f"KDME_GUIDE_{c}") == v
    if not os.path.isfile(_lib.LIB_PATH):
        _lib.build()
    L = C.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(L, n) and n in _lib.SIGNATURES


# ------------------------------------------------------------------ CPU: the GRAY pre-smooth definition
def _gray_presmooth_oracle(g):
    """The GRAY pre-smooth: the BGR oracle on (g, 0, 0), channel 0."""
    g = np.ascontiguousarray(g, np.uint8)
    out = oracle.presmooth(np.stack([g, np.zeros_like(g), np.zeros_like(g)], axis=-1))
    assert not out[..., 1:].any(), "zero channels must stay zero"
    return out[..., 0]


def _gray_images():
    import cv2
    img = cv2.imread(os.path.join(ROOT, "tests", "golden", "guide_frame_640x480.png"), 1)
    yield cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
    rng = np.random.default_rng(2024)
    for h, w in [(1, 1), (1, 7), (5, 3), (2, 2), (17, 33), (40, 40), (61, 203)]:
        yield rng.integers(0, 256, (h, w), dtype=np.uint8)
        yield (rng.integers(0, 6, (h, w)) + 100).astype(np.uint8)       # low contrast: many rounding decisions


def test_gray_presmooth_matches_opencv_one_channel_bilateral_up_to_its_truncation():
    """ours - cv2.bilateralFilter(gray, 5, 30, 30) is 0 or +1 everywhere.

    The GRAY pre-smooth is the BGR oracle on (g, 0, 0): L1 distance |dg|, the reference's weights, and the
    byte rounded to nearest (half to even), as the BGR path and OpenCV 2.4.3's GPU filter round.  OpenCV
    4.x's CPU 1-channel 8-bit path TRUNCATES the weighted mean instead (a float model with floor matches it
    on all but ~0.3 % of the pixels of the bundled frame, the same model with rint differs on ~50 %), so the
    rounded result is the truncated one or one level above it, never anything else."""
    import cv2
    for g in _gray_images():
        ours = _gray_presmooth_oracle(g).astype(np.int16)
        ref = cv2.bilateralFilter(g, 5, 30, 30).astype(np.int16)
        d = ours - ref
        assert set(np.unique(d).tolist()) <= {0, 1}, (g.shape, np.unique(d))


# ------------------------------------------------------------------ CPU: C++ drop-in with 1- and 4-channel mats
SNIPPET = r'''
#include "JointBilateralFilter.h"
#include <cstdio>
int run(float* depth, unsigned char* bgrx, unsigned char* gray, float* xyz, int W, int H) {
    JointBilateralFilter JBF(W, H);
    cv::gpu::GpuMat colour4(H, W, bgrx, 4 * (size_t)W, 4);     // Kinect v2 BGRX / Azure Kinect BGRA32
    cv::gpu::GpuMat ir(H, W, gray, (size_t)W, 1);               // IR amplitude, registered to the depth
    JBF.Process(depth, colour4);
    cv::gpu::GpuMat s4 = JBF.getSmoothImage_Device();
    JBF.ProcessXYZ(depth, ir, xyz, 525.f, 525.f, W / 2, H / 2);
    JBF.Upsampling(depth, W / 2, H / 2, colour4);
    JBF.Process(depth, ir);
    cv::gpu::GpuMat s1 = JBF.getSmoothImage_Device();
    JBF.setGuideChannels(4);
    JBF.ProcessBatch(depth, bgrx, 0, depth, 1);
    cv::gpu::GpuMat legacy(H, W, bgrx, 3 * (size_t)W);          // the 4-argument form: BGR
    return s4.channels() == 4 && s1.channels() == 1 && legacy.channels() == 3;
}
int main() {
    cv::gpu::GpuMat legacy(480, 640, 0, 3 * 640);
    if (legacy.channels() != 3) return 2;
    try { JointBilateralFilter JBF(640, 480); }
    catch (const std::exception& e) { std::printf("expected without a GPU: %s\n", e.what()); return 0; }
    return 0;
}
'''


def test_cpp_guide_formats_compile_and_link():
    from kinectdepthmapenhancement_b200 import _lib
    if not os.path.isfile(_lib.LIB_PATH):
        _lib.build()
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "formats.cpp")
        open(src, "w").write(SNIPPET)
        exe = os.path.join(td, "formats")
        libdir = os.path.dirname(_lib.LIB_PATH)
        subprocess.run(["g++", "-std=c++11", "-Wall", "-DKDME_NO_OPENCV", "-I", os.path.join(ROOT, "include"), src,
                        "-o", exe, "-L", libdir, "-lkdme_b200", "-Wl,-rpath," + libdir], check=True)
        res = subprocess.run([exe], capture_output=True, text=True)
        assert res.returncode == 0, res.stdout + res.stderr


# ================================================================== GPU: bit-identity with the derived BGR image
def _torch():
    import torch
    return torch


def _jbf(*a, **kw):
    from kinectdepthmapenhancement_b200 import JointBilateralFilter
    return JointBilateralFilter(*a, **kw)


def _as_format(bgr, c, rng):
    """A guide of format c built from a BGR image, and the BGR image it must filter as."""
    if c == 1:
        g = np.ascontiguousarray(bgr[..., 1])
        return g, np.stack([g, np.zeros_like(g), np.zeros_like(g)], axis=-1)
    if c == 4:
        x = rng.integers(0, 256, bgr.shape[:-1] + (1,), dtype=np.uint8)
        return np.ascontiguousarray(np.concatenate([bgr, x], axis=-1)), np.ascontiguousarray(bgr)
    return np.ascontiguousarray(bgr), np.ascontiguousarray(bgr)


def _cuda(a):
    return _torch().from_numpy(np.ascontiguousarray(a)).cuda()


def _bits(t):
    return t.detach().cpu().numpy().view(np.uint32)


def _guide4(f):
    from kinectdepthmapenhancement_b200 import _lib
    from kinectdepthmapenhancement_b200.jbf import _tensor_view
    step = C.c_size_t()
    ptr = _lib.lib().jbf_guide4_device(f._h, C.byref(step))
    g = _tensor_view(ptr, (f.height, step.value // 4), _torch().int32, f.device, f)
    return g[:, :f.width].clone()


def _pitched(img, c, pad, off):
    """img copied into device rows of c*W + pad bytes starting `off` bytes into an allocation: (keep, ptr, step)."""
    torch = _torch()
    h, w = img.shape[:2]
    step = c * w + pad
    buf = torch.zeros(h * step + off + 16, dtype=torch.uint8, device="cuda")
    rows = buf[off:off + h * step].view(h, step)
    rows[:, :c * w] = _cuda(img.reshape(h, c * w))
    return buf, rows.data_ptr(), step


SIZES = [(1, 1), (5, 3), (33, 17), (70, 50), (101, 67), (640, 480)]
# (pre-smooth ksize, radius, colour sigma): ksize 5 is the unrolled kernel, 3 / 7 the generic one, 0 the raw guide;
# sigma_c = 2 routes the filter to its generic kernel
CONFIGS = [(5, 2, 50.0), (5, 7, 50.0), (3, 2, 50.0), (7, 7, 50.0), (0, 2, 50.0), (0, 7, 50.0), (5, 2, 2.0)]


def _pair(w, h, ps, r, sc, **kw):
    presmooth = None if ps == 0 else (ps, 30.0, 30.0)
    return (_jbf(w, h, 70.0, sc, 20.0, r, presmooth=presmooth, **kw),
            _jbf(w, h, 70.0, sc, 20.0, r, presmooth=presmooth, **kw))


@pytest.mark.gpu
@pytest.mark.parametrize("c", [1, 4])
@pytest.mark.parametrize("w,h", SIZES)
def test_process_and_xyz_equal_the_derived_bgr_image(c, w, h):
    """Process (filtered plane and internal guide) and process_xyz, every pre-smooth / filter kernel, contiguous
    rows and rows that defeat or allow the wide staging (padded steps, unaligned bases)."""
    from kinectdepthmapenhancement_b200 import _lib
    rng = np.random.default_rng(w * 7 + h + c)
    depth, bgr = synth_np(w, h, seed=21, frame=c)
    img, ref = _as_format(bgr, c, rng)
    d = _cuda(depth)
    for ps, r, sc in CONFIGS:
        fc, fb = _pair(w, h, ps, r, sc)
        fb.Process(d, _cuda(ref))
        want, want_g = _bits(fb.getFiltered_Device()), _bits(_guide4(fb))
        fc.Process(d, _cuda(img))
        assert np.array_equal(_bits(fc.getFiltered_Device()), want), (ps, r, sc)
        assert np.array_equal(_bits(_guide4(fc)), want_g), (ps, r, sc)
        # padded / unaligned rows through the C ABI: pad 16 keeps BGRX rows 16-byte aligned when 4W is,
        # pad 4 (and base offset 4) does not; pad 3 / offset 1 makes GRAY rows unaligned
        for pad, off in ((16, 0), (4, 4), (3, 1)):
            keep, ptr, step = _pitched(img, c, pad, off)
            _lib.check(_lib.lib().jbf_process(fc._h, d.data_ptr(), ptr, step))
            assert np.array_equal(_bits(fc.getFiltered_Device()), want), (ps, r, sc, pad, off)
            assert np.array_equal(_bits(_guide4(fc)), want_g), (ps, r, sc, pad, off)
            del keep
        xb = fb.process_xyz(d, _cuda(ref), 525.0, 520.0, w // 2, h // 2)
        xc = fc.process_xyz(d, _cuda(img), 525.0, 520.0, w // 2, h // 2)
        assert np.array_equal(_bits(xc), _bits(xb))


@pytest.mark.gpu
@pytest.mark.parametrize("c", [1, 4])
def test_process_batch_both_chunk_lanes(c):
    torch = _torch()
    from kinectdepthmapenhancement_b200 import synth
    n, w, h = 5, 128, 96
    depth, bgr = synth.rgbd_stream(n, w, h, seed=3)
    rng = np.random.default_rng(c)
    img, ref = _as_format(bgr.numpy(), c, rng)
    for r in (2, 7):
        fc, fb = _pair(w, h, 5, r, 50.0, max_batch=2)     # 2 + 2 + 1: chunks alternate between the two lanes
        want = fb.process_batch(depth.cuda(), _cuda(ref))
        got = fc.process_batch(depth.cuda(), _cuda(img))
        assert np.array_equal(_bits(got), _bits(want))
        if c == 1:   # [N, H, W, 1] is GRAY too
            got1 = fc.process_batch(depth.cuda(), _cuda(img[..., None]))
            assert torch.equal(got1, got)


@pytest.mark.gpu
@pytest.mark.parametrize("c", [1, 4])
@pytest.mark.parametrize("w,h", SIZES)
def test_presmooth_and_row_band_forms_as_guide_words(c, w, h):
    from kinectdepthmapenhancement_b200 import _lib
    torch = _torch()
    rng = np.random.default_rng(w + 1000 * h + c)
    bgr = np.stack([rng.integers(0, 256, (2, h, w), dtype=np.uint8)] * 3, axis=-1)
    bgr[..., 1] //= 2
    bgr[..., 2] = rng.integers(0, 256, (2, h, w), dtype=np.uint8)
    img, ref = _as_format(bgr, c, rng)
    for ps in (5, 3, 7, 0):
        fc, fb = _pair(w, h, ps, 2, 50.0)
        want = fb.presmooth(_cuda(ref))[..., :w]   # the pitch's pad columns are not written
        got = fc.presmooth(_cuda(img))[..., :w]
        assert torch.equal(got, want), ps
        for pad, off in ((16, 0), (4, 4), (3, 1)):
            keep, ptr, step = _pitched(img[0], c, pad, off)
            for p2p in (False, True):
                g4 = torch.full((h, (w + 3) & ~3), -1, dtype=torch.int32, device="cuda")
                if p2p:
                    _lib.check(_lib.lib().jbf_presmooth_rows_p2p(fc._h, ptr, step, g4.data_ptr(), g4.shape[-1] * 4, h,
                                                                 0, h, None, None))
                else:
                    _lib.check(_lib.lib().jbf_presmooth_rows(fc._h, ptr, step, g4.data_ptr(), g4.shape[-1] * 4, h))
                assert torch.equal(g4[:, :w], want[0]), (ps, pad, off, p2p)
            del keep


def _tie_images(w, h):
    """Two-valued patterns whose weighted means are exact or near ties (k + 0.5), as single-channel images."""
    rng = np.random.default_rng(w * 1000 + h)
    yy, xx = np.mgrid[0:h, 0:w]
    ims = []
    for (a, b, sx, sy) in [(10, 11, 1, 1), (100, 103, 2, 1), (0, 255, 1, 2), (200, 201, 3, 3), (7, 8, 2, 2)]:
        ims.append((a + (b - a) * ((((xx // sx) + (yy // sy)) & 1))).astype(np.uint8))
    ims.append(np.where((xx % 4) < 2, 50, 51).astype(np.uint8))
    ims.append(rng.integers(0, 256, (h, w), dtype=np.uint8))
    ims.append((rng.integers(0, 4, (h, w)) + 120).astype(np.uint8))
    ims.append(np.full((h, w), 255, np.uint8))
    return ims


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(640, 96), (203, 61), (136, 40), (72, 33), (68, 20)])
def test_gray_presmooth_rounding_ties_equal_the_oracle(w, h):
    f = _jbf(w, h)
    for g in _tie_images(w, h):
        words = f.presmooth(_cuda(g[None]))[0].cpu().numpy().view(np.uint32)[:, :w]
        assert (words >> 8).max() == 0
        assert np.array_equal(words.astype(np.uint8), _gray_presmooth_oracle(g))


@pytest.mark.gpu
@pytest.mark.parametrize("c", [1, 4])
def test_upsampling_and_smooth_image(c):
    torch = _torch()
    from kinectdepthmapenhancement_b200 import synth
    for wl, hl, wh, hh, r in [(50, 37, 131, 97, 5), (128, 106, 480, 270, 7)]:
        lo, _ = synth.rgbd_frame(wl, hl, seed=6, frame=0, noise_rel=0.01)
        _, hi = synth.rgbd_frame(wh, hh, seed=6, frame=0)
        img, ref = _as_format(hi.numpy(), c, np.random.default_rng(r))
        fc, fb = _pair(wh, hh, 5, r, 50.0)
        want = fb.Upsampling(lo.cuda(), _cuda(ref))
        got = fc.Upsampling(lo.cuda(), _cuda(img))
        assert np.array_equal(_bits(got), _bits(want))
        sb, sc = fb.getSmoothImage_Device().cpu(), fc.getSmoothImage_Device().cpu()
        if c == 1:
            assert tuple(sc.shape) == (hh, wh) and torch.equal(sc, sb[..., 0])
        else:
            assert tuple(sc.shape) == (hh, wh, 4) and torch.equal(sc[..., :3], sb) and bool((sc[..., 3] == 255).all())


@pytest.mark.gpu
@pytest.mark.parametrize("c", [1, 4])
def test_process_host_f32_and_u16(c):
    torch = _torch()
    from kinectdepthmapenhancement_b200 import synth
    n, w, h = 5, 96, 64
    depth, bgr = synth.rgbd_stream(n, w, h, seed=4)
    d16 = depth.round().clamp_(0, 65535).to(torch.int32).to(torch.int16)
    img, ref = _as_format(bgr.numpy(), c, np.random.default_rng(c))
    fc, fb = _pair(w, h, 5, 3, 50.0, max_batch=2)
    for dh in (depth, d16):
        ob, oc = torch.empty((n, h, w)), torch.empty((n, h, w))
        fb.process_host(dh, torch.from_numpy(ref), ob)
        fc.process_host(dh, torch.from_numpy(img), oc)
        assert np.array_equal(oc.numpy().view(np.uint32), ob.numpy().view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("c", [1, 4])
@pytest.mark.parametrize("w,h", [(33, 17), (101, 67), (640, 480)])
def test_mrf_and_guided_fill_and_upsample(c, w, h):
    from kinectdepthmapenhancement_b200.guided import guided_fill, guided_upsample
    depth, bgr = synth_np(w, h, seed=12, frame=c)
    img, ref = _as_format(bgr, c, np.random.default_rng(w))
    d = _cuda(depth)
    fc, fb = _pair(w, h, 5, 2, 50.0)
    for r in (1, 2, 5):
        assert np.array_equal(_bits(fc.mrf(d, _cuda(img), r)), _bits(fb.mrf(d, _cuda(ref), r)))
    labels = _cuda(((np.arange(h)[:, None] // 9) * 64 + (np.arange(w)[None, :] // 11)).astype(np.int32))
    lo = _cuda(depth[::3, ::3])
    for lab in (None, labels):
        for r in (1, 3, 5):   # 1..3 compile-time window, 5 run-time window
            assert np.array_equal(_bits(guided_fill(d, _cuda(img), lab, r)), _bits(guided_fill(d, _cuda(ref), lab, r)))
            assert np.array_equal(_bits(guided_upsample(lo, _cuda(img), lab, r)),
                                  _bits(guided_upsample(lo, _cuda(ref), lab, r)))
        # exotic colour sigma: the generic kernel at a fast radius
        assert np.array_equal(_bits(guided_fill(d, _cuda(img), lab, 2, color_sigma=5.0)),
                              _bits(guided_fill(d, _cuda(ref), lab, 2, color_sigma=5.0)))


@pytest.mark.gpu
def test_channel_order_does_not_matter():
    w, h = 160, 120
    depth, bgr = synth_np(w, h, seed=5, frame=0)
    d = _cuda(depth)
    f = _jbf(w, h, window_radius=7)
    f.Process(d, _cuda(bgr))
    a = _bits(f.getFiltered_Device())
    f.Process(d, _cuda(bgr[..., ::-1]))   # RGB
    assert np.array_equal(_bits(f.getFiltered_Device()), a)
    x = np.full((h, w, 1), 7, np.uint8)
    f.Process(d, _cuda(np.concatenate([bgr[..., ::-1], x], axis=-1)))   # RGBA
    assert np.array_equal(_bits(f.getFiltered_Device()), a)


@pytest.mark.gpu
def test_one_handle_alternates_formats():
    torch = _torch()
    w, h, n = 101, 67, 3
    from kinectdepthmapenhancement_b200 import synth
    depth, bgr = synth.rgbd_stream(n, w, h, seed=9)
    rng = np.random.default_rng(1)
    f = _jbf(w, h, window_radius=7, max_batch=2)
    for c in (1, 4, 3, 1):
        img, _ = _as_format(bgr.numpy(), c, rng)
        fresh = _jbf(w, h, window_radius=7, max_batch=2)
        fresh.Process(depth[0].cuda(), _cuda(img[0]))
        f.Process(depth[0].cuda(), _cuda(img[0]))
        assert np.array_equal(_bits(f.getFiltered_Device()), _bits(fresh.getFiltered_Device())), c
        assert torch.equal(f.getSmoothImage_Device().cpu(), fresh.getSmoothImage_Device().cpu()), c
        of, oh = torch.empty((n, h, w)), torch.empty((n, h, w))
        fresh.process_host(depth, torch.from_numpy(img), of)
        f.process_host(depth, torch.from_numpy(img), oh)
        assert torch.equal(of, oh), c


@pytest.mark.gpu
def test_bad_formats_and_steps_are_rejected():
    torch = _torch()
    from kinectdepthmapenhancement_b200 import _lib
    from kinectdepthmapenhancement_b200.guided import guided_fill
    w, h = 64, 48
    f = _jbf(w, h)
    L = _lib.lib()
    for bad in (0, 2, 5, -3):
        assert L.jbf_set_guide_channels(f._h, bad) == _lib.KDME_EINVAL
    d = torch.zeros((h, w), device="cuda")
    g = torch.zeros((h, 4 * w), dtype=torch.uint8, device="cuda")
    out = torch.empty_like(d)
    for c in (1, 3, 4):
        assert L.jbf_set_guide_channels(f._h, c) == _lib.KDME_OK
        assert L.jbf_process(f._h, d.data_ptr(), g.data_ptr(), c * w - 1) == _lib.KDME_EINVAL
        assert L.jbf_process(f._h, d.data_ptr(), g.data_ptr(), c * w) == _lib.KDME_OK
        assert L.jbf_process(f._h, d.data_ptr(), g.data_ptr(), 0) == _lib.KDME_OK
        assert L.jbf_mrf(f._h, d.data_ptr(), g.data_ptr(), c * w - 1, out.data_ptr(), 2, 50.0, 150.0) == _lib.KDME_EINVAL
        assert L.kdme_guided_fill_ex(d.data_ptr(), None, g.data_ptr(), c * w - 1, c, out.data_ptr(), w, h, 3, 30.0,
                                     50.0, 70.0, None) == _lib.KDME_EINVAL
    assert L.kdme_guided_fill_ex(d.data_ptr(), None, g.data_ptr(), 0, 2, out.data_ptr(), w, h, 3, 30.0, 50.0, 70.0,
                                 None) == _lib.KDME_EINVAL
    assert L.kdme_guided_upsample_ex(d.data_ptr(), 8, 8, None, g.data_ptr(), 0, 5, out.data_ptr(), w, h, 3, 30.0, 50.0,
                                     70.0, None) == _lib.KDME_EINVAL
    torch.cuda.synchronize()
    f2 = _jbf(w, h)
    for shape in ((h, w, 2), (h, w, 5), (h + 1, w, 3), (h, w, 3, 1), (w,)):
        with pytest.raises(ValueError):
            f2.Process(d, torch.zeros(shape, dtype=torch.uint8, device="cuda"))
    with pytest.raises(ValueError):
        f2.process_batch(d[None], torch.zeros((1, h, w, 2), dtype=torch.uint8, device="cuda"))
    with pytest.raises(ValueError):
        f2.presmooth(torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda"))
    with pytest.raises(ValueError):
        guided_fill(d, torch.zeros((h, w, 2), dtype=torch.uint8, device="cuda"))
