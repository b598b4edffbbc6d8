"""Streams of frames through the joint bilateral filter: uint16 depth on the device (jbf_process_batch_u16), clouds of
a whole stream (jbf_process_batch_xyz[_u16]) and the batched back-projection (kdme_projective_to_real_batch).

Two identities define them, checked bit for bit on the GPU:

    frame k of process_batch(depth_u16, colour)          ==  Process(float(depth_u16[k]), colour[k])
    frame k of process_batch_xyz(depth, colour, ...)     ==  process_xyz(depth[k], colour[k], ...)  (plane and cloud)

whatever the chunking (max_batch), the lanes, the staging (TMA, plain, half units) and the kernel (fast, generic).
The frames are distinct and hold holes, every value 1..50, 51 and 65535, and 1 m depth edges, so the fp64
refinement of ill-conditioned pixels runs in frames after the first, where a wrong frame offset would show.
"""
import ctypes as C
import os
import re
import subprocess
import tempfile

import pytest

from conftest import ROOT

ARITY = {"jbf_process_batch_u16": 6, "jbf_process_batch_xyz": 11, "jbf_process_batch_xyz_u16": 11,
         "kdme_projective_to_real_batch": 10}
FX, FY = 525.0, 519.5


# ------------------------------------------------------------------ CPU: ABI surface
def test_header_declares_and_library_exports_the_entry_points():
    from kinectdepthmapenhancement_b200 import _lib
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "kdme_b200.h")).read(), flags=re.S)
    for n, arity in ARITY.items():
        m = re.search(rf"\b{n}\s*\(([^;]*)\);", text)
        assert m, n
        assert len(m.group(1).split(",")) == arity == len(_lib.SIGNATURES[n][1]), n
    if not os.path.isfile(_lib.LIB_PATH):
        _lib.build()
    L = C.CDLL(_lib.LIB_PATH)
    for n in ARITY:
        assert hasattr(L, n)


SNIPPET = r'''
#include "JointBilateralFilter.h"
#include <cstdio>
int run(const float* d, const unsigned short* d16, const unsigned char* bgrx, float* out, float* xyz, int W, int H, int n) {
    JointBilateralFilter JBF(W, H, 70.0f, 50.0f, 20.0f, 7, 4);
    JBF.setGuideChannels(4);                                             // Azure Kinect BGRA32 colour
    JBF.ProcessBatch(d16, bgrx, 4 * (size_t)W, out, n);                  // sensor uint16 millimetres on the device
    JBF.ProcessXYZBatch(d, bgrx, 0, out, xyz, n, 525.f, 525.f, W / 2, H / 2);
    JBF.ProcessXYZBatch(d16, bgrx, 0, out, xyz, n, 525.f, 525.f, W / 2, H / 2);
    return 0;
}
int main() {
    try { JointBilateralFilter JBF(640, 576); }
    catch (const std::exception& e) { std::printf("expected without a GPU: %s\n", e.what()); return 0; }
    return 0;
}
'''


def test_cpp_batch_overloads_compile_and_link():
    from kinectdepthmapenhancement_b200 import _lib
    if not os.path.isfile(_lib.LIB_PATH):
        _lib.build()
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "batch_xyz.cpp")
        open(src, "w").write(SNIPPET)
        exe = os.path.join(td, "batch_xyz")
        libdir = os.path.dirname(_lib.LIB_PATH)
        subprocess.run(["g++", "-std=c++11", "-Wall", "-DKDME_NO_OPENCV", "-I", os.path.join(ROOT, "include"), src,
                        "-o", exe, "-L", libdir, "-lkdme_b200", "-Wl,-rpath," + libdir], check=True)
        res = subprocess.run([exe], capture_output=True, text=True)
        assert res.returncode == 0, res.stdout + res.stderr


def test_null_arguments_are_rejected_without_a_device():
    from kinectdepthmapenhancement_b200 import _lib
    L = _lib.lib()
    buf = (C.c_uint8 * 64)()
    p = C.addressof(buf)
    assert L.jbf_process_batch_u16(None, p, p, 0, p, 1) == _lib.KDME_EINVAL
    assert b"NULL" in L.kdme_last_error()
    for n in ("jbf_process_batch_xyz", "jbf_process_batch_xyz_u16"):
        assert getattr(L, n)(None, p, p, 0, p, p, 1, FX, FY, 2, 2) == _lib.KDME_EINVAL
        assert b"NULL" in L.kdme_last_error()
    out = (C.c_float * 48)()
    q = C.addressof(out)
    # checked before any device is touched
    assert L.kdme_projective_to_real_batch(None, q, 4, 4, 1, FX, FY, 2, 2, None) == _lib.KDME_EINVAL
    assert L.kdme_projective_to_real_batch(p, None, 4, 4, 1, FX, FY, 2, 2, None) == _lib.KDME_EINVAL
    assert L.kdme_projective_to_real_batch(p, q, 4, 4, 0, FX, FY, 2, 2, None) == _lib.KDME_EINVAL
    assert L.kdme_projective_to_real_batch(p, q, 0, 4, 1, FX, FY, 2, 2, None) == _lib.KDME_EINVAL
    assert L.kdme_projective_to_real_batch(p, q, 4, 4, 1, 0.0, FY, 2, 2, None) == _lib.KDME_EINVAL
    assert L.kdme_projective_to_real_batch(p, q, 4, 4, 1, FX, 0.0, 2, 2, None) == _lib.KDME_EINVAL
    assert L.kdme_projective_to_real_batch(q, q + 4, 4, 4, 1, FX, FY, 2, 2, None) == _lib.KDME_EINVAL   # overlap


# ------------------------------------------------------------------ GPU
def _torch():
    import torch
    return torch


def _jbf(*a, **kw):
    from kinectdepthmapenhancement_b200 import JointBilateralFilter
    return JointBilateralFilter(*a, **kw)


def _bits(t):
    return t.contiguous().view(_torch().int32).cpu()


def _equal(a, b):
    return _torch().equal(_bits(a), _bits(b))


def _frames(n, w, h, c, seed):
    """n distinct integer depth frames (float32 CUDA) with holes, 0, 1..50, 51, 65535 and a 1 m step whose column moves
    with the frame, and their guides of c channels (c = 1: [N, H, W])."""
    torch = _torch()
    from kinectdepthmapenhancement_b200 import synth
    ds, cs = zip(*(synth.rgbd_frame(w, h, seed=seed, frame=k, noise_rel=0.01, hole_frac=0.1) for k in range(n)))
    d, col = torch.stack(ds), torch.stack(cs)
    for k in range(n):
        x0 = (w * (k + 1)) // (n + 2)
        d[k, :, x0:] += torch.where(d[k, :, x0:] > 50, 1000.0, 0.0)
    d = d.round().clamp_(0, 65535)
    special = torch.tensor([0] + list(range(1, 52)) + [65535, 65535], dtype=torch.float32)
    g = torch.Generator().manual_seed(seed)
    for k in range(n):
        m = min(special.numel(), w * h // 4)
        if m:
            idx = torch.randperm(w * h, generator=g)[:m]
            d[k].view(-1)[idx] = special[torch.randperm(special.numel(), generator=g)[:m]]
    if c == 1:
        col = col[..., 1].contiguous()
    elif c == 4:
        col = torch.cat([col, torch.randint(0, 256, (n, h, w, 1), generator=g, dtype=torch.uint8)], dim=-1)
    return d.cuda(), col.contiguous().cuda()


def _u16(d):
    return d.cpu().to(_torch().int32).to(_torch().uint16).cuda()


def _per_frame(f, d, col, cx, cy):
    """process_xyz frame by frame: the planes, the clouds, the fp64-refined pixel count of every frame."""
    torch = _torch()
    planes, clouds, refined = [], [], []
    f.refine_stats()
    for k in range(d.shape[0]):
        clouds.append(f.process_xyz(d[k], col[k], FX, FY, cx, cy).clone())
        planes.append(f.getFiltered_Device().clone())
        r, dropped = f.refine_stats()
        assert dropped == 0
        refined.append(r)
    return torch.stack(planes), torch.stack(clouds), refined


def _check_stream(f, d, col, refines=True):
    """Every batch form of a stream against the single-frame calls on the same handle."""
    n, h, w = d.shape
    cx, cy = w // 2, h // 3
    want, want_xyz, refined = _per_frame(f, d, col, cx, cy)
    d16 = _u16(d)
    assert _equal(f.process_batch(d, col), want)
    assert _equal(f.process_batch(d16, col), want)
    assert _equal(f.process_batch(d16.view(_torch().int16), col), want)   # the same bits as int16
    assert f.refine_stats() == (3 * sum(refined), 0)
    for dd in (d, d16):
        out, xyz = f.process_batch_xyz(dd, col, FX, FY, cx, cy)
        assert _equal(out, want)
        assert _equal(xyz, want_xyz)
    if refines:
        assert sum(refined[1:]) > 0, refined
    return refined


# (w, h, r, n, max_batch, guide channels): max_batch 1, 3 and n; n in 1, 5, 17; every radius class; plain staging
# (1x1 .. 101x67, uint16 rows not 16-byte multiples) and uint16 TMA (640x480)
CASES = [(640, 480, 7, 5, 3, 3), (640, 480, 2, 17, 17, 1), (640, 480, 15, 5, 5, 4), (640, 480, 1, 17, 3, 3),
         (101, 67, 15, 17, 3, 1), (101, 67, 2, 1, 1, 4), (70, 50, 1, 5, 1, 4), (70, 50, 7, 17, 17, 3),
         (5, 3, 2, 5, 5, 3), (1, 1, 7, 1, 1, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,r,n,mb,c", CASES)
def test_batches_equal_single_frames_bit_for_bit(w, h, r, n, mb, c):
    d, col = _frames(n, w, h, c, seed=11 + r + n)
    f = _jbf(w, h, window_radius=r, max_batch=mb)
    _check_stream(f, d, col, refines=n > 1 and w * h >= 50 * 50)


@pytest.mark.gpu
@pytest.mark.parametrize("env", ["KDME_NO_TMA", "KDME_TILE_H=4", "KDME_TILE_H=8", "KDME_TILE_H=16", "KDME_ONE_LANE",
                                 "KDME_FORCE_GENERIC", "KDME_NO_REFINE"])
@pytest.mark.parametrize("w,h,r,n,mb,c", [(640, 480, 7, 5, 2, 3), (101, 67, 2, 5, 3, 4)])
def test_batches_equal_single_frames_on_every_path(monkeypatch, env, w, h, r, n, mb, c):
    name, _, value = env.partition("=")
    monkeypatch.setenv(name, value or "1")   # read when the handle is created
    d, col = _frames(n, w, h, c, seed=5 + r)
    f = _jbf(w, h, window_radius=r, max_batch=mb)
    assert bool(f.kernel_variant & 1) == (name == "KDME_FORCE_GENERIC")
    refined = _check_stream(f, d, col, refines=name not in ("KDME_FORCE_GENERIC", "KDME_NO_REFINE"))
    if name in ("KDME_FORCE_GENERIC", "KDME_NO_REFINE"):
        assert sum(refined) == 0


@pytest.mark.gpu
def test_generic_handle_back_projects_each_chunk():
    """sigma_c = 20: the colour guard can fire, so the generic kernel filters and each chunk is back-projected."""
    d, col = _frames(5, 70, 50, 3, seed=2)
    f = _jbf(70, 50, 70.0, 20.0, 20.0, window_radius=5, max_batch=2)
    assert f.kernel_variant & 1
    _check_stream(f, d, col, refines=False)


@pytest.mark.gpu
def test_u16_tma_runs_and_falls_back_to_plain_staging():
    torch = _torch()
    n, w, h = 3, 640, 480
    d, col = _frames(n, w, h, 3, seed=9)
    f = _jbf(w, h, window_radius=7, max_batch=n)
    want = f.process_batch(d, col).clone()
    d16 = _u16(d)
    assert _equal(f.process_batch(d16, col), want)
    assert f.kernel_variant & 0x100, "expected the uint16 TMA staging"
    # a base 2 bytes off a 16-byte boundary: the same bits through plain staging
    raw = torch.zeros(n * h * w + 8, dtype=torch.int16, device="cuda")
    mis = raw[1:1 + n * h * w].view(n, h, w)
    mis.copy_(d16.view(torch.int16))
    assert mis.data_ptr() % 16 == 2
    assert _equal(f.process_batch(mis, col), want)
    assert not f.kernel_variant & 0x100
    out, xyz = f.process_batch_xyz(mis, col, FX, FY, w // 2, h // 2)
    assert _equal(out, want)
    assert not f.kernel_variant & 0x100
    # width % 8 != 0: float32 frames stage by TMA, uint16 ones by plain loads
    d2, col2 = _frames(2, 100, 60, 3, seed=4)
    f2 = _jbf(100, 60, window_radius=2, max_batch=2)
    want2 = f2.process_batch(d2, col2).clone()
    assert f2.kernel_variant & 0x100
    assert _equal(f2.process_batch(_u16(d2), col2), want2)
    assert not f2.kernel_variant & 0x100


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,n", [(640, 480, 5), (101, 67, 3), (1, 1, 4), (7, 1, 2)])
def test_projective_to_real_of_a_stream_equals_single_frames(w, h, n):
    torch = _torch()
    from kinectdepthmapenhancement_b200 import projective_to_real
    d, _ = _frames(n, w, h, 3, seed=w)
    d = d + torch.rand(d.shape, device="cuda")   # fractional millimetres too
    got = projective_to_real(d, FX, FY, w // 2, h // 3)
    assert tuple(got.shape) == (n, h, w, 3)
    for k in range(n):
        assert _equal(got[k], projective_to_real(d[k].contiguous(), FX, FY, w // 2, h // 3))


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,r,n,mb", [(640, 480, 7, 5, 3), (101, 67, 2, 3, 2)])
def test_no_write_beyond_the_last_frame(w, h, r, n, mb):
    torch = _torch()
    d, col = _frames(n, w, h, 3, seed=3)
    d16 = _u16(d)
    f = _jbf(w, h, window_radius=r, max_batch=mb)
    want, want_xyz = f.process_batch_xyz(d, col, FX, FY, w // 2, h // 2)
    for dd in (d, d16):
        out = torch.full((n + 1, h, w), -7.25, device="cuda")
        xyz = torch.full((n + 1, h, w, 3), -7.25, device="cuda")
        f.process_batch_xyz(dd, col, FX, FY, w // 2, h // 2, out=out[:n], xyz=xyz[:n])
        torch.cuda.synchronize()
        assert torch.all(out[n] == -7.25) and torch.all(xyz[n] == -7.25)
        assert _equal(out[:n], want) and _equal(xyz[:n], want_xyz)
        out[n].fill_(-7.25)
        f.process_batch(dd, col, out=out[:n])
        torch.cuda.synchronize()
        assert torch.all(out[n] == -7.25)
    from kinectdepthmapenhancement_b200 import projective_to_real
    xyz = torch.full((n + 1, h, w, 3), -7.25, device="cuda")
    from kinectdepthmapenhancement_b200 import _lib
    assert _lib.lib().kdme_projective_to_real_batch(want.data_ptr(), xyz.data_ptr(), w, h, n, FX, FY, w // 2, h // 2,
                                                    torch.cuda.current_stream().cuda_stream) == _lib.KDME_OK
    torch.cuda.synchronize()
    assert torch.all(xyz[n] == -7.25)
    assert _equal(xyz[:n], projective_to_real(want, FX, FY, w // 2, h // 2))


@pytest.mark.gpu
def test_bad_arguments_are_rejected():
    torch = _torch()
    from kinectdepthmapenhancement_b200 import _lib
    L = _lib.lib()
    w, h, n = 64, 48, 2
    f = _jbf(w, h, window_radius=3)
    d = torch.zeros((n, h, w), device="cuda")
    d16 = torch.zeros((n, h, w), dtype=torch.uint16).cuda()
    g = torch.zeros((n, h, 3 * w), dtype=torch.uint8, device="cuda")
    out = torch.empty((n, h, w), device="cuda")
    xyz = torch.empty((n, h, w, 3), device="cuda")
    for fn, dd in ((L.jbf_process_batch_u16, d16), (L.jbf_process_batch_xyz, d), (L.jbf_process_batch_xyz_u16, d16)):
        xyz_form = fn is not L.jbf_process_batch_u16
        ok = [f._h, dd.data_ptr(), g.data_ptr(), 3 * w, out.data_ptr()] + \
             ([xyz.data_ptr(), n, FX, FY, w // 2, h // 2] if xyz_form else [n])
        assert fn(*ok) == _lib.KDME_OK
        nf = 6 if xyz_form else 5
        bad = [(nf, 0), (nf, -1), (3, 3 * w - 1), (0, None), (1, None), (2, None), (4, None),
               (4, dd.data_ptr()),                                   # out overlaps the depth input
               (1, out.data_ptr() + 4 * w)]                          # ... from the other side
        if xyz_form:
            bad += [(5, None), (7, 0.0), (8, 0.0), (5, dd.data_ptr()), (5, out.data_ptr()),
                    (4, xyz.data_ptr() + 4)]                         # out overlaps xyz
        for i, v in bad:
            args = list(ok)
            args[i] = v
            assert fn(*args) == _lib.KDME_EINVAL, (fn, i, v)
        assert L.jbf_set_guide_channels(f._h, 4) == _lib.KDME_OK
        assert fn(*ok) == _lib.KDME_EINVAL                                # 3*W is below 4*W
        assert L.jbf_set_guide_channels(f._h, 3) == _lib.KDME_OK
    s = torch.cuda.current_stream().cuda_stream
    ok = [d.data_ptr(), xyz.data_ptr(), w, h, n, FX, FY, 1, 2, s]
    assert L.kdme_projective_to_real_batch(*ok) == _lib.KDME_OK
    for i, v in ((0, None), (1, None), (2, 0), (3, -1), (4, 0), (5, 0.0), (6, 0.0), (1, d.data_ptr() + 4)):
        args = list(ok)
        args[i] = v
        assert L.kdme_projective_to_real_batch(*args) == _lib.KDME_EINVAL, (i, v)
    torch.cuda.synchronize()
    c = torch.zeros((n, h, w, 3), dtype=torch.uint8, device="cuda")
    f2 = _jbf(w, h, window_radius=3)
    f2.process_batch(d16, c)
    with pytest.raises(TypeError):
        f2.process_batch(d.to(torch.int32), c)
    with pytest.raises(TypeError):
        f2.process_batch_xyz(d.to(torch.float64), c, FX, FY, 1, 1)
    with pytest.raises(TypeError):
        f2.process_batch(d16.cpu(), c)
    with pytest.raises(ValueError):
        f2.process_batch(d16, c[:1])                                       # N differs
    with pytest.raises(ValueError):
        f2.process_batch(d16[0], c[0])                                     # not a batch
    with pytest.raises(ValueError):
        f2.process_batch(d16, c, out=torch.empty((n + 1, h, w), device="cuda"))
    with pytest.raises(ValueError):
        f2.process_batch_xyz(d16, c, FX, FY, 1, 1, xyz=torch.empty((n, h, w), device="cuda"))
    with pytest.raises(_lib.KdmeError):
        f2.process_batch_xyz(d16, c, 0.0, FY, 1, 1)
    from kinectdepthmapenhancement_b200 import projective_to_real
    with pytest.raises(ValueError):
        projective_to_real(d[None], FX, FY, 1, 1)
