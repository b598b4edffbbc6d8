"""Batched Upsampling (jbf_upsample_batch / jbf_upsample_batch_u16, JointBilateralFilter.upsample_batch).

One identity defines the batch, checked bit for bit on the GPU:

    frame k of upsample_batch(depth_lo, colour)  ==  Upsampling(depth_lo[k], colour[k])

whatever the chunking (max_batch), the lanes, the kernel form (gather, dense, generic) and the depth format:
a uint16 sample s filters exactly as the float (float)s.  The frames are distinct and have holes and depth
edges, so the fp64 refinement of ill-conditioned pixels runs in frames after the first, where a wrong frame
offset in the queue or in the low-res read would show.
"""
import ctypes as C
import os
import re
import subprocess
import tempfile

import pytest

from conftest import ROOT

NAMES = ("jbf_upsample_batch", "jbf_upsample_batch_u16")


# ------------------------------------------------------------------ CPU: ABI surface
def test_header_declares_and_library_exports_the_batch_entry_points():
    from kinectdepthmapenhancement_b200 import _lib
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "kdme_b200.h")).read(), flags=re.S)
    for n in NAMES:
        assert re.search(rf"\b{n}\s*\(", text), n
        assert len(_lib.SIGNATURES[n][1]) == 8
    if not os.path.isfile(_lib.LIB_PATH):
        _lib.build()
    L = C.CDLL(_lib.LIB_PATH)
    for n in NAMES:
        assert hasattr(L, n)


SNIPPET = r'''
#include "JointBilateralFilter.h"
#include <cstdio>
int run(const float* lo, const unsigned short* lo16, const unsigned char* bgrx, float* out, int W, int H, int n) {
    JointBilateralFilter JBF(W, H, 70.0f, 50.0f, 20.0f, 7, 4);
    JBF.setGuideChannels(4);                                    // Azure Kinect BGRA32 colour
    JBF.UpsamplingBatch(lo, 640, 576, bgrx, 4 * (size_t)W, out, n);
    JBF.UpsamplingBatch(lo16, 640, 576, bgrx, 0, out, n);       // sensor uint16 millimetres
    return 0;
}
int main() {
    try { JointBilateralFilter JBF(1920, 1080); }
    catch (const std::exception& e) { std::printf("expected without a GPU: %s\n", e.what()); return 0; }
    return 0;
}
'''


def test_cpp_upsampling_batch_overloads_compile_and_link():
    from kinectdepthmapenhancement_b200 import _lib
    if not os.path.isfile(_lib.LIB_PATH):
        _lib.build()
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "ups_batch.cpp")
        open(src, "w").write(SNIPPET)
        exe = os.path.join(td, "ups_batch")
        libdir = os.path.dirname(_lib.LIB_PATH)
        subprocess.run(["g++", "-std=c++11", "-Wall", "-DKDME_NO_OPENCV", "-I", os.path.join(ROOT, "include"), src,
                        "-o", exe, "-L", libdir, "-lkdme_b200", "-Wl,-rpath," + libdir], check=True)
        res = subprocess.run([exe], capture_output=True, text=True)
        assert res.returncode == 0, res.stdout + res.stderr


def test_null_handle_is_rejected_without_a_device():
    from kinectdepthmapenhancement_b200 import _lib
    L = _lib.lib()
    buf = (C.c_uint8 * 64)()
    p = C.addressof(buf)
    for n in NAMES:
        assert getattr(L, n)(None, p, 4, 4, p, 0, p, 1) == _lib.KDME_EINVAL
        assert b"NULL" in L.kdme_last_error()


# ------------------------------------------------------------------ GPU
def _torch():
    import torch
    return torch


def _jbf(*a, **kw):
    from kinectdepthmapenhancement_b200 import JointBilateralFilter
    return JointBilateralFilter(*a, **kw)


def _bits(t):
    return t.contiguous().view(_torch().int32).cpu()


def _frames(n, wl, hl, wh, hh, seed, integer=False):
    """n distinct low-res depth frames with holes and depth edges, and their high-res BGR guides."""
    torch = _torch()
    from kinectdepthmapenhancement_b200 import synth
    lo = torch.stack([synth.rgbd_frame(wl, hl, seed=seed, frame=k, noise_rel=0.01, hole_frac=0.1)[0]
                      for k in range(n)])
    hi = torch.stack([synth.rgbd_frame(wh, hh, seed=seed, frame=k)[1] for k in range(n)])
    # a 1 m step whose column moves with the frame: every frame has a depth edge of its own
    for k in range(n):
        lo[k, :, (wl * (k + 1)) // (n + 2):] += torch.where(lo[k, :, (wl * (k + 1)) // (n + 2):] > 50, 1000.0, 0.0)
    if integer:
        lo = lo.round().clamp_(0, 65535)
    return lo.cuda(), hi.cuda()


def _per_frame(f, lo, hi):
    """Upsampling frame by frame; the fp64-refined pixel count of every frame."""
    outs, refined = [], []
    f.refine_stats()
    for k in range(lo.shape[0]):
        outs.append(f.Upsampling(lo[k], hi[k]).clone())
        r, d = f.refine_stats()
        assert d == 0
        refined.append(r)
    return _torch().stack(outs), refined


# (wl, hl, wh, hh, r, n, max_batch, refinement expected in frames >= 1)
CASES = [(512, 424, 1920, 1080, 7, 5, 2, True),    # Kinect v2: three chunks over two lanes
         (50, 37, 131, 97, 5, 4, 4, True),
         (17, 9, 640, 480, 15, 3, 2, False),       # a window sees at most one site: nothing ill-conditioned
         (64, 48, 64, 48, 3, 4, 3, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("wl,hl,wh,hh,r,n,mb,refines", CASES)
def test_batch_equals_per_frame_bit_for_bit(wl, hl, wh, hh, r, n, mb, refines):
    lo, hi = _frames(n, wl, hl, wh, hh, seed=31 + r)
    f = _jbf(wh, hh, window_radius=r, max_batch=mb)
    want, refined = _per_frame(f, lo, hi)
    got = f.upsample_batch(lo, hi)
    assert f.kernel_variant & 0x1000, "expected the gather form"
    batch_refined, dropped = f.refine_stats()
    assert dropped == 0
    if refines:
        assert sum(refined[1:]) > 0, refined
    assert batch_refined == sum(refined)
    assert torch_equal_bits(got, want)


def torch_equal_bits(a, b):
    return _torch().equal(_bits(a), _bits(b))


@pytest.mark.gpu
@pytest.mark.parametrize("env", ["KDME_ONE_LANE", "KDME_UPSAMPLE_DENSE", "KDME_GATHER_GENERIC"])
@pytest.mark.parametrize("wl,hl,wh,hh,r,n,mb", [(512, 424, 1920, 1080, 7, 5, 2), (50, 37, 131, 97, 5, 5, 2)])
def test_batch_equals_per_frame_on_every_path(monkeypatch, env, wl, hl, wh, hh, r, n, mb):
    lo, hi = _frames(n, wl, hl, wh, hh, seed=47)
    want, refined = _per_frame(_jbf(wh, hh, window_radius=r, max_batch=mb), lo, hi)
    monkeypatch.setenv(env, "1")   # KDME_ONE_LANE is read when the handle is created, the others per launch
    f = _jbf(wh, hh, window_radius=r, max_batch=mb)
    f.refine_stats()
    got = f.upsample_batch(lo, hi)
    assert bool(f.kernel_variant & 0x1000) == (env != "KDME_UPSAMPLE_DENSE")
    assert f.refine_stats() == (sum(refined), 0)
    assert sum(refined[1:]) > 0
    assert torch_equal_bits(got, want)


@pytest.mark.gpu
def test_batch_on_the_generic_kernel():
    """sigma_c = 20: the colour guard can fire, the generic kernel runs (one lane, no refinement queue)."""
    lo, hi = _frames(3, 50, 37, 131, 97, seed=5)
    f = _jbf(131, 97, 70.0, 20.0, 20.0, window_radius=5, max_batch=2)
    want, _ = _per_frame(f, lo, hi)
    got = f.upsample_batch(lo, hi)
    assert f.kernel_variant & 1
    assert torch_equal_bits(got, want)


def _u16_frames(n, wl, hl, seed):
    """Integer depth frames holding 0, every value 1..50 (holes), 51 (the first valid one) and 65535."""
    torch = _torch()
    lo, _ = _frames(n, wl, hl, 8, 8, seed, integer=True)
    lo = lo.cpu()
    special = torch.tensor([0] + list(range(1, 52)) + [65535, 65535], dtype=torch.float32)
    g = torch.Generator().manual_seed(seed)
    for k in range(n):
        idx = torch.randperm(wl * hl, generator=g)[:special.numel()]
        lo[k].view(-1)[idx] = special
    return lo.cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("wl,hl,wh,hh,r,mb", [(17, 13, 131, 97, 5, 2), (512, 424, 1920, 1080, 7, 2),
                                             (33, 21, 33, 21, 2, 4)])
def test_u16_equals_f32_bit_for_bit(wl, hl, wh, hh, r, mb):
    """wl odd: u16 frames and rows start on 2-byte boundaries only."""
    torch = _torch()
    n = 3
    lo = _u16_frames(n, wl, hl, seed=wl)
    _, hi = _frames(n, 8, 8, wh, hh, seed=wl)
    f = _jbf(wh, hh, window_radius=r, max_batch=mb)
    want = f.upsample_batch(lo, hi).clone()
    ints = lo.cpu().to(torch.int32)
    got = f.upsample_batch(ints.to(torch.uint16).cuda(), hi).clone()
    assert torch_equal_bits(got, want)
    got_i16 = f.upsample_batch(ints.to(torch.int16).cuda(), hi)   # the same bits as int16
    assert torch_equal_bits(got_i16, want)
    # and one frame of the u16 batch against the single-frame float call
    assert torch_equal_bits(got[n - 1], f.Upsampling(lo[n - 1].contiguous(), hi[n - 1]))


@pytest.mark.gpu
@pytest.mark.parametrize("c", [1, 4])
def test_guide_formats_equal_bgr_on_the_derived_image(c):
    """GRAY g == BGR (g, 0, 0); BGRX (b, g, r, x) == BGR (b, g, r)."""
    torch = _torch()
    n, wl, hl, wh, hh = 4, 128, 106, 480, 270
    lo, hi = _frames(n, wl, hl, wh, hh, seed=12)
    gen = torch.Generator().manual_seed(c)
    if c == 1:
        img = hi[..., 1].contiguous()
        ref = torch.zeros_like(hi)
        ref[..., 0] = img
    else:
        x = torch.randint(0, 256, (n, hh, wh, 1), generator=gen, dtype=torch.uint8).cuda()
        img = torch.cat([hi, x], dim=-1).contiguous()
        ref = hi
    f = _jbf(wh, hh, window_radius=7, max_batch=3)
    want = f.upsample_batch(lo, ref).clone()
    got = f.upsample_batch(lo, img)
    assert torch_equal_bits(got, want)
    # through the C ABI with a padded guide row: the step is honoured for every frame
    from kinectdepthmapenhancement_b200 import _lib
    step = c * wh + 12
    padded = torch.zeros((n, hh, step), dtype=torch.uint8, device="cuda")
    padded[:, :, :c * wh] = img.reshape(n, hh, c * wh)
    out = torch.empty_like(want)
    assert _lib.lib().jbf_upsample_batch(f._h, lo.data_ptr(), wl, hl, padded.data_ptr(), step, out.data_ptr(),
                                         n) == _lib.KDME_OK
    assert torch_equal_bits(out, want)


@pytest.mark.gpu
def test_last_frame_of_a_batch_matches_the_f64_oracle():
    """Frame offsets against the fp64 formula, not only against the GPU itself."""
    import oracle
    from test_gpu_jbf import check_against_f64
    n, wl, hl, wh, hh = 3, 128, 106, 480, 270
    lo, hi = _frames(n, wl, hl, wh, hh, seed=6)
    f = _jbf(wh, hh, window_radius=7, max_batch=2)
    out = f.upsample_batch(lo, hi)[n - 1].cpu().numpy()
    guide = oracle.presmooth(hi[n - 1].cpu().numpy())
    sparse = oracle.scatter_lowres(lo[n - 1].cpu().numpy(), wh, hh)
    check_against_f64(out, sparse, guide, 15, 70.0, 50.0, 20.0, "batch frame 2, upsample 128x106 -> 480x270")


@pytest.mark.gpu
@pytest.mark.parametrize("wl,hl,wh,hh,r,n,mb", [(50, 37, 131, 97, 5, 3, 2), (64, 48, 70, 50, 7, 4, 4)])
def test_no_write_beyond_the_last_frame(wl, hl, wh, hh, r, n, mb):
    torch = _torch()
    lo, hi = _frames(n, wl, hl, wh, hh, seed=3)
    f = _jbf(wh, hh, window_radius=r, max_batch=mb)
    canary = torch.full((n + 1, hh, wh), -7.25, dtype=torch.float32, device="cuda")
    f.upsample_batch(lo, hi, out=canary[:n])
    torch.cuda.synchronize()
    assert torch.all(canary[n] == -7.25)
    assert torch_equal_bits(canary[:n], f.upsample_batch(lo, hi))
    lo16 = lo.cpu().round().clamp(0, 65535).to(torch.int32).to(torch.uint16).cuda()
    canary[n].fill_(-7.25)
    f.upsample_batch(lo16, hi, out=canary[:n])
    torch.cuda.synchronize()
    assert torch.all(canary[n] == -7.25)


@pytest.mark.gpu
def test_bad_arguments_are_rejected():
    torch = _torch()
    from kinectdepthmapenhancement_b200 import _lib
    L = _lib.lib()
    w, h, n = 64, 48, 2
    f = _jbf(w, h, window_radius=3)
    lo = torch.zeros((n, 20, 16), device="cuda")
    lo16 = torch.zeros((n, 20, 16), dtype=torch.uint16).cuda()
    g = torch.zeros((n, h, 4 * w), dtype=torch.uint8, device="cuda")
    out = torch.empty((n, h, w), device="cuda")
    for fn, d in ((L.jbf_upsample_batch, lo), (L.jbf_upsample_batch_u16, lo16)):
        ok = (f._h, d.data_ptr(), 16, 20, g.data_ptr(), 3 * w, out.data_ptr(), n)
        assert fn(*ok) == _lib.KDME_OK
        for i, bad in ((7, 0), (7, -1), (2, w + 1), (3, h + 1), (2, 0), (3, 0), (5, 3 * w - 1),
                       (1, None), (4, None), (6, None), (0, None)):
            args = list(ok)
            args[i] = bad
            assert fn(*args) == _lib.KDME_EINVAL, (i, bad)
        assert L.jbf_set_guide_channels(f._h, 4) == _lib.KDME_OK
        assert fn(*ok) == _lib.KDME_EINVAL                 # 3*W is below 4*W
        assert L.jbf_set_guide_channels(f._h, 3) == _lib.KDME_OK
    torch.cuda.synchronize()
    f2 = _jbf(w, h, window_radius=3)
    c = torch.zeros((n, h, w, 3), dtype=torch.uint8, device="cuda")
    f2.upsample_batch(lo, c)
    with pytest.raises(ValueError):
        f2.upsample_batch(lo, c[:1])                          # N differs
    with pytest.raises(ValueError):
        f2.upsample_batch(lo, torch.zeros((n, h, w + 4, 3), dtype=torch.uint8, device="cuda"))   # wrong high-res size
    with pytest.raises(ValueError):
        f2.upsample_batch(lo, torch.zeros((n, h, w, 2), dtype=torch.uint8, device="cuda"))       # no such format
    with pytest.raises(ValueError):
        f2.upsample_batch(torch.zeros((n, h + 1, 16), device="cuda"), c)                        # hl > H
    with pytest.raises(ValueError):
        f2.upsample_batch(lo[0], c[0])                        # not a batch
    with pytest.raises(ValueError):
        f2.upsample_batch(lo, c, out=torch.empty((n + 1, h, w), device="cuda"))
    with pytest.raises(TypeError):
        f2.upsample_batch(lo.to(torch.float64), c)
    with pytest.raises(TypeError):
        f2.upsample_batch(lo.to(torch.int32), c)
    with pytest.raises(TypeError):
        f2.upsample_batch(lo.cpu(), c)
