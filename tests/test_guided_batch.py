"""Streams of frames through the guided cross-bilateral stage (kdme_guided_fill_batch / _u16,
kdme_guided_upsample_batch / _u16; guided_fill / guided_upsample with [N, ...] depth).

One identity defines the batch, checked bit for bit on the GPU:

    frame k of kdme_guided_*_batch(frames)  ==  kdme_guided_*_ex(frame k)

for the fast kernel (r = 1..3) and the runtime-radius kernel, with and without per-frame labels, every guide format,
float32 and uint16 depth, and batches longer than one launch's 65535 frames.  Every frame is distinct, so a wrong
frame offset of any plane shows.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT

NAMES = ("kdme_guided_fill_batch", "kdme_guided_fill_batch_u16", "kdme_guided_upsample_batch",
         "kdme_guided_upsample_batch_u16")
SS, SC, SD = 30.0, 50.0, 70.0   # EdgeRefinedSuperpixel.cpp:4-7


# ------------------------------------------------------------------ CPU: ABI surface
def test_header_declares_and_library_exports_the_guided_batch_entry_points():
    from kinectdepthmapenhancement_b200 import _lib
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "kdme_b200.h")).read(), flags=re.S)
    for n in NAMES:
        assert re.search(rf"\b{n}\s*\(", text), n
        assert len(_lib.SIGNATURES[n][1]) == (14 if "fill" in n else 16), n
    if not os.path.isfile(_lib.LIB_PATH):
        _lib.build()
    L = C.CDLL(_lib.LIB_PATH)
    for n in NAMES:
        assert hasattr(L, n), n


def test_null_pointers_and_empty_batches_are_rejected_without_a_device():
    from kinectdepthmapenhancement_b200 import _lib
    L = _lib.lib()
    buf = (C.c_uint8 * 64)()
    p = C.addressof(buf)
    for n in ("kdme_guided_fill_batch", "kdme_guided_fill_batch_u16"):
        assert getattr(L, n)(None, None, p, 0, 3, p + 32, 2, 2, 1, 1, SS, SC, SD, None) == _lib.KDME_EINVAL
        assert b"NULL" in L.kdme_last_error()
        assert getattr(L, n)(p, None, p, 0, 3, p + 32, 2, 2, 0, 1, SS, SC, SD, None) == _lib.KDME_EINVAL
        assert b"n_frames" in L.kdme_last_error()
    for n in ("kdme_guided_upsample_batch", "kdme_guided_upsample_batch_u16"):
        assert getattr(L, n)(None, 1, 1, None, p, 0, 3, p + 32, 2, 2, 1, 1, SS, SC, SD, None) == _lib.KDME_EINVAL
        assert b"NULL" in L.kdme_last_error()
        assert getattr(L, n)(p, 1, 1, None, p, 0, 3, p + 32, 2, 2, 0, 1, SS, SC, SD, None) == _lib.KDME_EINVAL
        assert b"n_frames" in L.kdme_last_error()


# ------------------------------------------------------------------ GPU helpers
def _torch():
    import torch
    return torch


def _lib():
    from kinectdepthmapenhancement_b200 import _lib as L
    return L


def _bits(t):
    return t.contiguous().view(_torch().int32).cpu()


def _depth(n, w, h, seed, integer=False):
    """n distinct depth frames with holes and a depth edge of their own."""
    torch = _torch()
    from kinectdepthmapenhancement_b200 import synth
    d = torch.stack([synth.rgbd_frame(w, h, seed=seed, frame=k, noise_rel=0.01, hole_frac=0.1)[0] for k in range(n)])
    for k in range(n):
        c0 = (w * (k + 1)) // (n + 2)
        d[k, :, c0:] += torch.where(d[k, :, c0:] > 50, 1000.0, 0.0)
    if integer:
        d = d.round().clamp_(0, 65535)
    return d.cuda()


def _guides(n, w, h, c, seed):
    """n distinct raw guides of c channels: [n,h,w] (GRAY) or [n,h,w,c]."""
    torch = _torch()
    from kinectdepthmapenhancement_b200 import synth
    bgr = torch.stack([synth.rgbd_frame(w, h, seed=seed + 1, frame=k)[1] for k in range(n)])
    if c == 1:
        return bgr[..., 1].contiguous().cuda()
    if c == 4:
        x = torch.randint(0, 256, (n, h, w, 1), generator=torch.Generator().manual_seed(seed), dtype=torch.uint8)
        bgr = torch.cat([bgr, x], dim=-1)
    return bgr.contiguous().cuda()


def _labels(n, w, h, seed):
    """Per-frame superpixel-like label maps: blocks whose size and numbering change with the frame."""
    torch = _torch()
    ys, xs = torch.arange(h)[:, None], torch.arange(w)[None, :]
    return torch.stack([((ys // (5 + k % 4)) * 97 + (xs // (7 + (k + seed) % 5)) + k).to(torch.int32)
                        for k in range(n)]).cuda()


def _stream():
    return _torch().cuda.current_stream().cuda_stream


def _fill_ex(d, lab, g, c, out, w, h, r):
    L = _lib()
    rc = L.lib().kdme_guided_fill_ex(d.data_ptr(), lab.data_ptr() if lab is not None else None, g.data_ptr(), c * w,
                                     c, out.data_ptr(), w, h, r, SS, SC, SD, _stream())
    L.check(rc)


def _fill_per_frame(d, lab, g, c, r):
    torch = _torch()
    n, h, w = d.shape
    want = torch.empty((n, h, w), dtype=torch.float32, device="cuda")
    for k in range(n):
        _fill_ex(d[k], lab[k] if lab is not None else None, g[k], c, want[k], w, h, r)
    return want


def _fill_batch(d, lab, g, c, r, fn="kdme_guided_fill_batch"):
    torch = _torch()
    n, h, w = d.shape
    out = torch.empty((n, h, w), dtype=torch.float32, device="cuda")
    _lib().check(getattr(_lib().lib(), fn)(d.data_ptr(), lab.data_ptr() if lab is not None else None, g.data_ptr(),
                                           c * w, c, out.data_ptr(), w, h, n, r, SS, SC, SD, _stream()))
    return out


def _upsample_per_frame(lo, lab, g, c, w, h, r):
    torch = _torch()
    L = _lib()
    n, hl, wl = lo.shape
    want = torch.empty((n, h, w), dtype=torch.float32, device="cuda")
    for k in range(n):
        L.check(L.lib().kdme_guided_upsample_ex(lo[k].data_ptr(), wl, hl, lab[k].data_ptr() if lab is not None else None,
                                                g[k].data_ptr(), c * w, c, want[k].data_ptr(), w, h, r, SS, SC, SD,
                                                _stream()))
    return want


def _upsample_batch(lo, lab, g, c, w, h, r, fn="kdme_guided_upsample_batch"):
    torch = _torch()
    n, hl, wl = lo.shape
    out = torch.empty((n, h, w), dtype=torch.float32, device="cuda")
    _lib().check(getattr(_lib().lib(), fn)(lo.data_ptr(), wl, hl, lab.data_ptr() if lab is not None else None,
                                           g.data_ptr(), c * w, c, out.data_ptr(), w, h, n, r, SS, SC, SD, _stream()))
    return out


def _equal(a, b):
    return _torch().equal(_bits(a), _bits(b))


# ------------------------------------------------------------------ GPU: batch == loop
@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(1, 1), (33, 17), (70, 50), (640, 480)])
@pytest.mark.parametrize("c", [1, 3, 4])
@pytest.mark.parametrize("use_labels", [False, True])
@pytest.mark.parametrize("r", [1, 2, 3, 5])
def test_fill_batch_equals_per_frame_bit_for_bit(r, use_labels, c, w, h):
    n = 3
    d = _depth(n, w, h, seed=10 * r + c)
    g = _guides(n, w, h, c, seed=r + w)
    lab = _labels(n, w, h, seed=r) if use_labels else None
    want = _fill_per_frame(d, lab, g, c, r)
    got = _fill_batch(d, lab, g, c, r)
    assert _equal(got, want)
    if w * h > 1:
        assert not _equal(got[0], got[1]), "frames must differ for the offsets to be tested"


@pytest.mark.gpu
@pytest.mark.parametrize("wl,hl,w,h,r,use_labels,c", [(17, 9, 70, 50, 3, True, 3), (33, 17, 33, 17, 2, False, 1),
                                                      (50, 37, 131, 97, 5, True, 4), (1, 1, 9, 5, 1, True, 3),
                                                      (512, 424, 1920, 1080, 7, True, 3)])
def test_upsample_batch_equals_per_frame_bit_for_bit(wl, hl, w, h, r, use_labels, c):
    n = 3
    lo = _depth(n, wl, hl, seed=wl + r)
    g = _guides(n, w, h, c, seed=hl)
    lab = _labels(n, w, h, seed=w) if use_labels else None
    want = _upsample_per_frame(lo, lab, g, c, w, h, r)
    got = _upsample_batch(lo, lab, g, c, w, h, r)
    assert _equal(got, want)
    if wl * hl > 1:
        assert not _equal(got[0], got[1]), "frames must differ for the offsets to be tested"


def _u16_frames(n, w, h, seed):
    """Integer depth frames holding 0, every value 1..50 (holes), 51 (the first valid one) and 65535."""
    torch = _torch()
    d = _depth(n, w, h, seed, integer=True).cpu()
    special = torch.tensor([0] + list(range(1, 52)) + [65535, 65535], dtype=torch.float32)
    gen = torch.Generator().manual_seed(seed)
    for k in range(n):
        idx = torch.randperm(w * h, generator=gen)[:special.numel()]
        d[k].view(-1)[idx] = special[:idx.numel()]
    return d.cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,r,c", [(33, 17, 2, 3), (71, 45, 3, 4), (64, 48, 5, 1), (640, 480, 3, 3)])
def test_fill_u16_equals_f32_bit_for_bit(w, h, r, c):
    """w odd: uint16 frames and rows start on 2-byte boundaries only."""
    torch = _torch()
    n = 3
    d = _u16_frames(n, w, h, seed=w)
    g = _guides(n, w, h, c, seed=h)
    lab = _labels(n, w, h, seed=r)
    want = _fill_batch(d, lab, g, c, r)
    ints = d.cpu().to(torch.int32)
    assert (d.cpu() == 65535).any() and (d.cpu() == 51).any() and (d.cpu() == 50).any() and (d.cpu() == 0).any()
    got = _fill_batch(ints.to(torch.uint16).cuda(), lab, g, c, r, fn="kdme_guided_fill_batch_u16")
    assert _equal(got, want)
    # and one frame of the uint16 batch against the single-frame float call
    one = torch.empty((h, w), dtype=torch.float32, device="cuda")
    _fill_ex(d[n - 1].contiguous(), lab[n - 1], g[n - 1], c, one, w, h, r)
    assert _equal(got[n - 1], one)


@pytest.mark.gpu
@pytest.mark.parametrize("wl,hl,w,h,r", [(17, 13, 131, 97, 5), (33, 21, 33, 21, 2), (512, 424, 1920, 1080, 7)])
def test_upsample_u16_equals_f32_bit_for_bit(wl, hl, w, h, r):
    torch = _torch()
    n = 3
    lo = _u16_frames(n, wl, hl, seed=wl)
    g = _guides(n, w, h, 3, seed=hl)
    lab = _labels(n, w, h, seed=r)
    want = _upsample_batch(lo, lab, g, 3, w, h, r)
    got = _upsample_batch(lo.cpu().to(torch.int32).to(torch.uint16).cuda(), lab, g, 3, w, h, r,
                          fn="kdme_guided_upsample_batch_u16")
    assert _equal(got, want)


@pytest.mark.gpu
def test_python_batch_forms_equal_the_per_frame_calls():
    """guided_fill / guided_upsample with [N, ...] depth: float32, uint16 and its int16 view, GRAY as [N,H,W]."""
    torch = _torch()
    from kinectdepthmapenhancement_b200.guided import guided_fill, guided_upsample
    n, w, h, wl, hl = 4, 96, 64, 40, 30
    d = _depth(n, w, h, seed=3, integer=True)
    for c in (1, 3, 4):
        g = _guides(n, w, h, c, seed=c)
        lab = _labels(n, w, h, seed=c)
        want = torch.stack([guided_fill(d[k], g[k], lab[k], 3) for k in range(n)])
        assert _equal(guided_fill(d, g, lab, 3), want)
        ints = d.cpu().to(torch.int32)
        assert _equal(guided_fill(ints.to(torch.uint16).cuda(), g, lab, 3), want)
        assert _equal(guided_fill(ints.to(torch.int16).cuda(), g, lab, 3), want)
        out = torch.full((n + 1, h, w), -7.25, device="cuda")
        guided_fill(d, g, None, 3, out=out[:n])
        assert torch.all(out[n] == -7.25)
        assert _equal(out[:n], torch.stack([guided_fill(d[k], g[k], None, 3) for k in range(n)]))
    lo = _depth(n, wl, hl, seed=4)
    g = _guides(n, w, h, 3, seed=9)
    lab = _labels(n, w, h, seed=9)
    want = torch.stack([guided_upsample(lo[k], g[k], lab[k], 7) for k in range(n)])
    assert _equal(guided_upsample(lo, g, lab, 7), want)
    lo16 = lo.cpu().round().clamp(0, 65535).to(torch.int32)
    want16 = torch.stack([guided_upsample(lo16[k].float().cuda(), g[k], lab[k], 7) for k in range(n)])
    assert _equal(guided_upsample(lo16.to(torch.uint16).cuda(), g, lab, 7), want16)


@pytest.mark.gpu
def test_python_batch_forms_reject_bad_shapes():
    torch = _torch()
    from kinectdepthmapenhancement_b200.guided import guided_fill, guided_upsample
    n, w, h = 2, 16, 12
    d = torch.zeros((n, h, w), device="cuda")
    g = torch.zeros((n, h, w, 3), dtype=torch.uint8, device="cuda")
    guided_fill(d, g)
    with pytest.raises(ValueError):
        guided_fill(d, g[:1])                                                        # N differs
    with pytest.raises(ValueError):
        guided_fill(d, g[0])                                                         # not a batch of guides
    with pytest.raises(ValueError):
        guided_fill(d, torch.zeros((n, h, w, 2), dtype=torch.uint8, device="cuda"))  # no such format
    with pytest.raises(ValueError):
        guided_fill(d, g, torch.zeros((n, h, w + 1), dtype=torch.int32, device="cuda"))
    with pytest.raises(ValueError):
        guided_fill(d, g, out=torch.empty((n + 1, h, w), device="cuda"))
    with pytest.raises(TypeError):
        guided_fill(d.to(torch.float64), g)
    with pytest.raises(TypeError):
        guided_fill(d.cpu(), g)
    with pytest.raises(ValueError):
        guided_upsample(torch.zeros((n, h + 1, 4), device="cuda"), g)                # hl > H
    with pytest.raises(ValueError):
        guided_upsample(torch.zeros((n, 4, 4), device="cuda"), g[0])                 # not a batch of guides
    with pytest.raises(TypeError):
        guided_upsample(torch.zeros((n, 4, 4), dtype=torch.int32, device="cuda"), g)


# ------------------------------------------------------------------ GPU: oracle sanity
@pytest.mark.gpu
def test_last_batch_frame_matches_the_f64_oracle():
    """Frame offsets against the fp64 formula, not only against the GPU itself."""
    from test_guided_f64 import check_guided_against_f64
    n, w, h, r = 3, 160, 120, 3
    d = _depth(n, w, h, seed=17)
    g = _guides(n, w, h, 3, seed=17)
    lab = _labels(n, w, h, seed=17)
    got = _fill_batch(d, lab, g, 3, r)[n - 1].cpu().numpy()
    check_guided_against_f64(got, d[n - 1].cpu().numpy(), g[n - 1].cpu().numpy(), lab[n - 1].cpu().numpy(), 2 * r + 1,
                             SS, SC, SD, what="last batch frame")


# ------------------------------------------------------------------ GPU: more frames than one launch holds
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["fill", "upsample_u16"])
def test_batches_beyond_the_grid_z_limit_equal_the_per_frame_results(kind):
    """70 000 frames: two launches (65535 + 4465 frames); every frame equals its single-frame call."""
    torch = _torch()
    L = _lib()
    n, w, h = 70000, 4, 4
    gen = torch.Generator().manual_seed(70000)
    d = torch.randint(0, 4000, (n, h, w), generator=gen).float()
    d[torch.rand((n, h, w), generator=gen) < 0.2] = 0
    g = torch.randint(0, 256, (n, h, w, 3), generator=gen, dtype=torch.uint8).cuda()
    lab = torch.randint(0, 3, (n, h, w), generator=gen, dtype=torch.int32).cuda()
    want = torch.empty((n, h, w), dtype=torch.float32, device="cuda")
    s, fn = _stream(), L.lib().kdme_guided_fill_ex
    if kind == "fill":
        d = d.cuda()
        got = _fill_batch(d, lab, g, 3, 1)
        dp, lp, gp, op = d.data_ptr(), lab.data_ptr(), g.data_ptr(), want.data_ptr()
        for k in range(n):
            assert fn(dp + 64 * k, lp + 64 * k, gp + 48 * k, 12, 3, op + 64 * k, w, h, 1, SS, SC, SD, s) == 0
    else:
        lo = d[:, :2, :3].contiguous()   # 3x2 -> 4x4
        got = _upsample_batch(lo.to(torch.int32).to(torch.uint16).cuda(), lab, g, 3, w, h, 5,
                              fn="kdme_guided_upsample_batch_u16")
        lo = lo.cuda()
        fn = L.lib().kdme_guided_upsample_ex
        dp, lp, gp, op = lo.data_ptr(), lab.data_ptr(), g.data_ptr(), want.data_ptr()
        for k in range(n):
            assert fn(dp + 24 * k, 3, 2, lp + 64 * k, gp + 48 * k, 12, 3, op + 64 * k, w, h, 5, SS, SC, SD, s) == 0
    torch.cuda.synchronize()
    assert _equal(got, want)
    assert not _equal(got[65534], got[65535])


# ------------------------------------------------------------------ GPU: argument errors
@pytest.mark.gpu
def test_bad_arguments_are_rejected():
    torch = _torch()
    L = _lib()
    lib = L.lib()
    n, w, h = 3, 16, 12
    d = torch.ones((n, h, w), device="cuda")
    d16 = torch.ones((n, h, w), dtype=torch.int16, device="cuda")
    lab = torch.zeros((n, h, w), dtype=torch.int32, device="cuda")
    g = torch.zeros((n, h, 4 * w), dtype=torch.uint8, device="cuda")
    out = torch.empty((n, h, w), device="cuda")
    s = _stream()
    # (fn, ok arguments, {index: bad values})
    fill_bad = {0: [None], 2: [None], 5: [None], 6: [0, -1], 7: [0, -1], 8: [0, -1], 9: [-1, 16], 4: [0, 2, 5],
                3: [3 * w - 1]}
    for fn, dd in ((lib.kdme_guided_fill_batch, d), (lib.kdme_guided_fill_batch_u16, d16)):
        ok = [dd.data_ptr(), lab.data_ptr(), g.data_ptr(), 3 * w, 3, out.data_ptr(), w, h, n, 3, SS, SC, SD, s]
        assert fn(*ok) == L.KDME_OK
        ok[1] = None
        assert fn(*ok) == L.KDME_OK   # one label
        for i, vals in fill_bad.items():
            for bad in vals:
                args = list(ok)
                args[i] = bad
                assert fn(*args) == L.KDME_EINVAL, (fn.__name__, i, bad)
        args = list(ok)
        args[4] = 4
        assert fn(*args) == L.KDME_EINVAL                       # 3*W is below 4*W
    # overlapping input and output byte ranges (the fill does not run in place)
    buf = torch.zeros((3 * n + 1, h, w), device="cuda")
    base, plane = buf.data_ptr(), 4 * w * h
    for i0, o0 in ((0, 0), (0, plane * n - 4), (plane, 0), (plane * n - 4, 0), (0, 2 * plane)):
        rc = lib.kdme_guided_fill_batch(base + i0, None, g.data_ptr(), 0, 3, base + o0, w, h, n, 3, SS, SC, SD, s)
        assert rc == L.KDME_EINVAL, (i0, o0)
    assert lib.kdme_guided_fill_batch(base, None, g.data_ptr(), 0, 3, base + plane * n, w, h, n, 3, SS, SC, SD,
                                      s) == L.KDME_OK   # adjacent, not overlapping
    b16 = base + plane * n   # n uint16 planes take half the bytes of n float planes
    assert lib.kdme_guided_fill_batch_u16(b16, None, g.data_ptr(), 0, 3, b16 + 2 * w * h * n - 4, w, h, n, 3, SS, SC,
                                          SD, s) == L.KDME_EINVAL
    assert lib.kdme_guided_fill_batch_u16(b16, None, g.data_ptr(), 0, 3, b16 + 2 * w * h * n, w, h, n, 3, SS, SC, SD,
                                          s) == L.KDME_OK
    assert lib.kdme_guided_fill_ex(base, None, g.data_ptr(), 0, 3, base + 4, w, h, 3, SS, SC, SD, s) == L.KDME_EINVAL
    ups_bad = {0: [None], 4: [None], 7: [None], 1: [0, w + 1], 2: [0, h + 1], 8: [0], 9: [0], 10: [0, -1],
               11: [-1, 16], 6: [0, 2, 5], 5: [3 * w - 1]}
    lo = torch.ones((n, 5, 7), device="cuda")
    lo16 = torch.ones((n, 5, 7), dtype=torch.int16, device="cuda")
    for fn, dd in ((lib.kdme_guided_upsample_batch, lo), (lib.kdme_guided_upsample_batch_u16, lo16)):
        ok = [dd.data_ptr(), 7, 5, lab.data_ptr(), g.data_ptr(), 3 * w, 3, out.data_ptr(), w, h, n, 3, SS, SC, SD, s]
        assert fn(*ok) == L.KDME_OK
        for i, vals in ups_bad.items():
            for bad in vals:
                args = list(ok)
                args[i] = bad
                assert fn(*args) == L.KDME_EINVAL, (fn.__name__, i, bad)
    # the upsampling reads depth_lo while it writes out_hi: overlapping byte ranges are rejected the same way
    lo_bytes, lo16_bytes, out_bytes = 4 * 7 * 5 * n, 2 * 7 * 5 * n, 4 * w * h * n
    for fn, nb in ((lib.kdme_guided_upsample_batch, lo_bytes), (lib.kdme_guided_upsample_batch_u16, lo16_bytes)):
        for i0, o0 in ((0, 0), (0, (nb - 1) // 4 * 4), (out_bytes - 4, 0)):
            rc = fn(base + i0, 7, 5, None, g.data_ptr(), 0, 3, base + o0, w, h, n, 3, SS, SC, SD, s)
            assert rc == L.KDME_EINVAL, (fn.__name__, i0, o0)
        after = (nb + 255) // 256 * 256   # the first aligned float past the input
        assert fn(base, 7, 5, None, g.data_ptr(), 0, 3, base + after, w, h, n, 3, SS, SC, SD, s) == L.KDME_OK
        assert fn(base + out_bytes, 7, 5, None, g.data_ptr(), 0, 3, base, w, h, n, 3, SS, SC, SD, s) == L.KDME_OK
    assert lib.kdme_guided_upsample_ex(base, 7, 5, None, g.data_ptr(), 0, 3, base + 4, w, h, 3, SS, SC, SD,
                                       s) == L.KDME_EINVAL
    torch.cuda.synchronize()
