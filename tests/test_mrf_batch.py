"""Streams of frames through the MarkovRandomField filter (next row f1): jbf_mrf_batch, jbf_mrf_batch_u16, the
[N, H, W] form of JointBilateralFilter.mrf and the header-only C++ class include/MarkovRandomField.h.

The stream form is defined by two identities, checked bit for bit on the GPU:

    frame k of mrf(depth[N, H, W], colour)      ==  mrf(depth[k], colour[k])
    mrf(uint16 depth)                           ==  mrf(float32 image of the same depth)

and every frame meets the fp64 contract of tests/test_next_rows.py.  The frames are distinct and hold holes, every
value 1..50, 51 and 65535, and 1 m depth edges whose column moves with the frame, so a wrong frame offset shows.
"""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT

ARITY = {"jbf_mrf_batch": 9, "jbf_mrf_batch_u16": 9, "jbf_mrf": 8}
TOL_MM = 1e-3
SC, SM = 50.0, 150.0   # MarkovRandomField.cpp:3-6


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


def test_bad_arguments_are_rejected_without_a_device():
    from kinectdepthmapenhancement_b200 import _lib
    L = _lib.lib()
    buf = (C.c_uint8 * 64)()
    p = C.addressof(buf)
    for fn in (L.jbf_mrf_batch, L.jbf_mrf_batch_u16):
        for args, what in (((None, p, p, 0, p, 0, 2, SC, SM), b"n_frames"),
                           ((None, p, p, 0, p, -1, 2, SC, SM), b"n_frames"),
                           ((None, p, p, 0, p, 1, -1, SC, SM), b"radius"),
                           ((None, p, p, 0, p, 1, 16, SC, SM), b"radius"),
                           ((None, p, p, 0, p, 1, 2, SC, SM), b"NULL"),
                           ((1, None, p, 0, p, 1, 2, SC, SM), b"NULL"),
                           ((1, p, None, 0, p, 1, 2, SC, SM), b"NULL"),
                           ((1, p, p, 0, None, 1, 2, SC, SM), b"NULL")):
            assert fn(*args) == _lib.KDME_EINVAL, (fn, args)
            assert what in L.kdme_last_error(), (args, L.kdme_last_error())
    assert L.jbf_mrf(None, p, p, 0, p, 2, SC, SM) == _lib.KDME_EINVAL
    assert L.jbf_mrf(None, p, p, 0, p, 16, SC, SM) == _lib.KDME_EINVAL
    assert b"radius" in L.kdme_last_error()


SNIPPET = r'''
#include "MarkovRandomField.h"
#include <cstdio>
// the reference's call pattern (main.cpp:185-190), then the stream forms
int run(float* d, cv::gpu::GpuMat colour, const float* df, const unsigned short* d16, const unsigned char* bgrx,
        float* out, int W, int H, int n) {
    MarkovRandomField MRF(W, H);
    MRF.Process(d, colour);
    float* filtered = MRF.getFiltered_Device();
    MRF.setGuideChannels(4);
    MRF.ProcessBatch(df, bgrx, 4 * (size_t)W, out, n);
    MRF.ProcessBatch(d16, bgrx, 0, out, n);
    return filtered != 0;
}
int main() {
    try { MarkovRandomField MRF(640, 480); }
    catch (const std::exception& e) { std::printf("expected without a GPU: %s\n", e.what()); return 0; }
    return 0;
}
'''


def test_cpp_markov_random_field_compiles_and_links():
    from kinectdepthmapenhancement_b200 import _lib
    if not os.path.isfile(_lib.LIB_PATH):
        _lib.build()
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "mrf.cpp")
        open(src, "w").write(SNIPPET)
        exe = os.path.join(td, "mrf")
        libdir = os.path.dirname(_lib.LIB_PATH)
        subprocess.run(["g++", "-std=c++11", "-Wall", "-DKDME_NO_OPENCV", "-I", os.path.join(ROOT, "include"), src,
                        "-o", exe, "-L", libdir, "-lkdme_b200", "-Wl,-rpath," + libdir], check=True)
        res = subprocess.run([exe], capture_output=True, text=True)
        assert res.returncode == 0, res.stdout + res.stderr


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
    with the frame, and their guides of c channels (c = 1: [N, H, W]; c = 4: a random 4th byte)."""
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


def _as_bgr(col):
    """The BGR image a guide filters as: GRAY g is (g, 0, 0), BGRX (b, g, r, x) is (b, g, r)."""
    a = col.cpu().numpy()
    if a.ndim == 2:
        z = np.zeros(a.shape + (3,), np.uint8)
        z[..., 0] = a
        return z
    return np.ascontiguousarray(a[..., :3])


# (w, h, r, n, guide channels): sizes 1x1, 33x17, 101x67, 640x480; r = 0, 1, 2, 5, 15; N = 1, 3, 17; every format
CASES = [(1, 1, 0, 1, 1), (1, 1, 15, 3, 3), (1, 1, 2, 17, 4),
         (33, 17, 1, 17, 4), (33, 17, 15, 3, 1), (33, 17, 2, 1, 3), (33, 17, 0, 3, 4),
         (101, 67, 2, 17, 3), (101, 67, 5, 3, 4), (101, 67, 0, 17, 1), (101, 67, 15, 1, 4), (101, 67, 1, 3, 1),
         (640, 480, 2, 17, 4), (640, 480, 2, 3, 1), (640, 480, 5, 3, 3), (640, 480, 0, 1, 3), (640, 480, 15, 3, 1),
         (640, 480, 1, 17, 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,r,n,c", CASES)
def test_stream_equals_single_frames_bit_for_bit(w, h, r, n, c):
    torch = _torch()
    d, col = _frames(n, w, h, c, seed=7 + r + n + c)
    f = _jbf(w, h)
    want = torch.stack([f.mrf(d[k], col[k], r).clone() for k in range(n)])
    d16 = _u16(d)
    assert _equal(f.mrf(d, col, r), want)
    assert _equal(f.mrf(d16, col, r), want)
    assert _equal(f.mrf(d16.view(torch.int16), col, r), want)   # the same bits as int16
    out = torch.full((n + 1, h, w), -7.25, device="cuda")
    f.mrf(d16, col, r, out=out[:n])
    torch.cuda.synchronize()
    assert _equal(out[:n], want) and torch.all(out[n] == -7.25)   # nothing written past the last frame
    if n > 1 and w * h > 1:   # the frames differ, so a frame read at another frame's offset would show
        assert all(not _equal(want[k], want[k + 1]) for k in range(n - 1))


@pytest.mark.gpu
@pytest.mark.parametrize("sc,sm", [(0.0, 150.0), (1e-3, 1.0), (SC, 0.0)])
def test_stream_equals_single_frames_off_the_default_sigmas(sc, sm):
    torch = _torch()
    d, col = _frames(3, 101, 67, 3, seed=3)
    f = _jbf(101, 67)
    want = torch.stack([f.mrf(d[k], col[k], 5, sc, sm).clone() for k in range(3)])
    assert _equal(f.mrf(d, col, 5, sc, sm), want)
    assert _equal(f.mrf(_u16(d), col, 5, sc, sm), want)


def check_mrf(out, depth, bgr, radius, sc=SC, sm=SM, label=""):
    """tests/test_next_rows.py's criterion: no NaN, the mask out > 0 (and out == 0) of the fp64 oracle, and every
    pixel within 1e-3 mm of it."""
    import oracle
    o64 = oracle.mrf(depth, bgr, 2 * radius + 1, sc, sm, precision="f64")
    err = np.abs(out.astype(np.float64) - o64.astype(np.float64))
    y, x = np.unravel_index(np.argmax(err), err.shape)
    assert not np.isnan(out).any(), label
    assert np.array_equal(out > 0, o64 > 0) and np.array_equal(out == 0, o64 == 0), f"{label}: mask differs from fp64"
    assert err.max() <= TOL_MM, f"{label}: (y={y}, x={x}) off by {err.max():.3e} mm"


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,r,n,c", [(640, 480, 2, 3, 3), (640, 480, 2, 3, 4), (101, 67, 5, 5, 1),
                                       (33, 17, 15, 3, 4), (101, 67, 0, 3, 3), (101, 67, 1, 3, 1)])
def test_every_frame_of_a_stream_meets_the_fp64_contract(w, h, r, n, c):
    d, col = _frames(n, w, h, c, seed=40 + r)
    f = _jbf(w, h)
    for dd in (d, _u16(d)):
        got = f.mrf(dd, col, r).cpu().numpy()
        for k in range(n):
            check_mrf(got[k], d[k].cpu().numpy(), _as_bgr(col[k]), r, label=f"{w}x{h} r={r} frame {k} {dd.dtype}")


@pytest.mark.gpu
def test_mrf_leaves_the_handles_guide_and_filtered_plane():
    """Process(A) -> mrf(B) on one handle: the smoothed guide and the filtered plane are still A's."""
    torch = _torch()
    from kinectdepthmapenhancement_b200 import _lib
    from kinectdepthmapenhancement_b200.jbf import _tensor_view
    w, h = 160, 120
    d, col = _frames(3, w, h, 3, seed=8)
    f = _jbf(w, h)
    f.Process(d[0], col[0])
    step = C.c_size_t()
    g4 = _tensor_view(_lib.lib().jbf_guide4_device(f._h, C.byref(step)), (h, step.value), torch.uint8, f.device, f)
    want_g4, want_smooth = g4.clone(), f.getSmoothImage_Device().clone()
    want_plane = f.getFiltered_Device().clone()
    f.mrf(d[1], col[1])
    f.mrf(d[1:], col[1:], 5)
    f.mrf(_u16(d[1:]), col[1:])
    torch.cuda.synchronize()
    assert torch.equal(g4.cpu(), want_g4.cpu())
    assert torch.equal(f.getSmoothImage_Device().cpu(), want_smooth.cpu())
    assert _equal(f.getFiltered_Device(), want_plane)


@pytest.mark.gpu
def test_overlap_and_bad_arguments_are_rejected():
    torch = _torch()
    from kinectdepthmapenhancement_b200 import _lib
    L = _lib.lib()
    w, h, n = 64, 48, 3
    f = _jbf(w, h)
    d = torch.zeros((n, h, w), device="cuda")
    d16 = torch.zeros((n, h, w), dtype=torch.uint16).cuda()
    g = torch.zeros((n, h, 3 * w), dtype=torch.uint8, device="cuda")
    out = torch.empty((n, h, w), device="cuda")
    for fn, dd in ((L.jbf_mrf_batch, d), (L.jbf_mrf_batch_u16, d16)):
        ok = [f._h, dd.data_ptr(), g.data_ptr(), 3 * w, out.data_ptr(), n, 2, SC, SM]
        assert fn(*ok) == _lib.KDME_OK
        for i, v in ((5, 0), (6, 16), (3, 3 * w - 1), (0, None), (1, None), (2, None), (4, None),
                     (4, dd.data_ptr()),                                      # in place
                     (4, dd.data_ptr() + dd.element_size() * (n * h * w - 1)),  # the last sample
                     (1, out.data_ptr() + 4 * w)):                            # out overlaps from the other side
            args = list(ok)
            args[i] = v
            assert fn(*args) == _lib.KDME_EINVAL, (fn, i, v)
        assert L.jbf_set_guide_channels(f._h, 4) == _lib.KDME_OK
        assert fn(*ok) == _lib.KDME_EINVAL                                    # 3*W is below 4*W
        assert L.jbf_set_guide_channels(f._h, 3) == _lib.KDME_OK
    assert L.jbf_mrf(f._h, d.data_ptr(), g.data_ptr(), 0, d.data_ptr(), 2, SC, SM) == _lib.KDME_EINVAL
    torch.cuda.synchronize()
    c = torch.zeros((n, h, w, 3), dtype=torch.uint8, device="cuda")
    f2 = _jbf(w, h)
    with pytest.raises(_lib.KdmeError):
        f2.mrf(d, c, out=d)
    with pytest.raises(TypeError):
        f2.mrf(d16[0], c[0])                                                  # a single frame stays float32
    with pytest.raises(TypeError):
        f2.mrf(d.to(torch.int32), c)
    with pytest.raises(ValueError):
        f2.mrf(d, c[:1])                                                      # N differs
    with pytest.raises(ValueError):
        f2.mrf(d, c, out=torch.empty((n + 1, h, w), device="cuda"))
    with pytest.raises(ValueError):
        f2.mrf(d[:, :, :-1].contiguous(), c)                                  # not the filter's size


CPP_GPU = r'''
#include "MarkovRandomField.h"
#include <cuda_runtime.h>
#include <cstdio>
#include <vector>
// MarkovRandomField MRF(W, H); MRF.Process(d, colour) on frame 0, then ProcessBatch of all n uint16 frames
int main(int argc, char** argv) {
    const int W = atoi(argv[1]), H = atoi(argv[2]), n = atoi(argv[3]);
    const size_t px = (size_t)W * H;
    std::vector<float> d(px * n), out(px * (n + 1));
    std::vector<unsigned short> d16(px * n);
    std::vector<unsigned char> bgr(px * 3 * n);
    FILE* f = fopen(argv[4], "rb");
    if (fread(d.data(), 4, px * n, f) != px * n || fread(d16.data(), 2, px * n, f) != px * n ||
        fread(bgr.data(), 1, 3 * px * n, f) != 3 * px * n) return 2;
    fclose(f);
    float *dd, *od; unsigned short* dd16; unsigned char* bd;
    cudaMalloc(&dd, 4 * px * n); cudaMalloc(&dd16, 2 * px * n); cudaMalloc(&bd, 3 * px * n); cudaMalloc(&od, 4 * px * n);
    cudaMemcpy(dd, d.data(), 4 * px * n, cudaMemcpyHostToDevice);
    cudaMemcpy(dd16, d16.data(), 2 * px * n, cudaMemcpyHostToDevice);
    cudaMemcpy(bd, bgr.data(), 3 * px * n, cudaMemcpyHostToDevice);
    try {
        MarkovRandomField MRF(W, H);
        cv::gpu::GpuMat colour(H, W, bd, 3 * (size_t)W, 3);
        MRF.Process(dd, colour);
        cudaMemcpy(out.data(), MRF.getFiltered_Device(), 4 * px, cudaMemcpyDeviceToHost);
        MRF.ProcessBatch(dd16, bd, 3 * (size_t)W, od, n);
        cudaMemcpy(out.data() + px, od, 4 * px * n, cudaMemcpyDeviceToHost);
    } catch (const std::exception& e) { std::printf("%s\n", e.what()); return 1; }
    f = fopen(argv[5], "wb");
    fwrite(out.data(), 4, out.size(), f);
    fclose(f);
    return 0;
}
'''


@pytest.mark.gpu
def test_cpp_markov_random_field_on_the_gpu_equals_python():
    torch = _torch()
    from kinectdepthmapenhancement_b200 import _lib
    w, h, n = 101, 67, 3
    d, col = _frames(n, w, h, 3, seed=17)
    want = _jbf(w, h).mrf(d, col).cpu()
    with tempfile.TemporaryDirectory() as td:
        src, exe = os.path.join(td, "mrf_gpu.cpp"), os.path.join(td, "mrf_gpu")
        fin, fout = os.path.join(td, "in.bin"), os.path.join(td, "out.bin")
        open(src, "w").write(CPP_GPU)
        libdir = os.path.dirname(_lib.LIB_PATH)
        subprocess.run(["g++", "-std=c++11", "-Wall", "-DKDME_NO_OPENCV", "-I", os.path.join(ROOT, "include"),
                        "-I", "/usr/local/cuda/include", src, "-o", exe, "-L", libdir, "-lkdme_b200",
                        "-L", "/usr/local/cuda/lib64", "-lcudart", "-Wl,-rpath," + libdir], check=True)
        with open(fin, "wb") as fh:
            fh.write(d.cpu().numpy().tobytes())
            fh.write(_u16(d).cpu().view(torch.int16).numpy().tobytes())
            fh.write(col.cpu().numpy().tobytes())
        res = subprocess.run([exe, str(w), str(h), str(n), fin, fout], capture_output=True, text=True)
        assert res.returncode == 0, res.stdout + res.stderr
        got = torch.from_numpy(np.fromfile(fout, np.float32).reshape(n + 1, h, w))
    assert _equal(got[0], want[0])        # Process(frame 0) with the reference's defaults
    assert _equal(got[1:], want)          # ProcessBatch of the uint16 stream
