"""ctypes front-end of the CPU oracle (oracle/kdme_oracle.c) and, when built,
of the reference's own kernel text compiled for the host (oracle/_ref).

TEST INFRASTRUCTURE ONLY.  Only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs may import this package.  The product
package (kinectdepthmapenhancement_b200) never does.

Reference defaults (JointBilateralFilter.cpp:3-6, JointBilateralFilter.cu:285,
EdgeRefinedSuperpixel.cpp:4-7) are exported as constants.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libkdme_oracle.so")
_REF_PATH = os.path.join(_HERE, "_ref", "libkdme_ref.so")

# JointBilateralFilter.cpp:3-6
JBF_WINDOW, JBF_SIGMA_S, JBF_SIGMA_C, JBF_SIGMA_D = 5, 70.0, 50.0, 20.0
# JointBilateralFilter.cu:285  (kernel_size, sigma_color, sigma_spatial)
PRESMOOTH_KSIZE, PRESMOOTH_SIGMA_C, PRESMOOTH_SIGMA_S = 5, 30.0, 30.0
# EdgeRefinedSuperpixel.cpp:4-7
ERS_WINDOW, ERS_SIGMA_S, ERS_SIGMA_C, ERS_SIGMA_D = 7, 30.0, 50.0, 70.0
# MarkovRandomField.cpp:3-6
MRF_WINDOW, MRF_SIGMA_C, MRF_SMOOTH = 5, 50.0, 150.0


def build(force: bool = False) -> None:
    """Compile the C restatement (and oracle/_ref where oracle/build_ref.py finds a reference checkout)."""
    src = os.path.join(_HERE, "kdme_oracle.c")
    if force or not os.path.isfile(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.run(
            ["gcc", "-O2", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
             "-fvisibility=hidden", "-std=c11", src, "-o", _LIB_PATH, "-lm"], check=True)
    from . import build_ref
    if build_ref.available():
        shim_m = max(os.path.getmtime(os.path.join(_HERE, f)) for f in
                     ("ref_shim_pre.h", "ref_shim_post.h", "build_ref.py"))
        if force or not os.path.isfile(_REF_PATH) or os.path.getmtime(_REF_PATH) < shim_m:
            build_ref.build(verbose=False)


_lib = None
_ref = None
_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")


def lib():
    global _lib
    if _lib is None:
        if not os.path.isfile(_LIB_PATH):
            build()
        L = C.CDLL(_LIB_PATH)
        L.orc_spatial_lut.argtypes = [_f32p, C.c_int, C.c_float]
        L.orc_presmooth_luts.argtypes = [_f32p, _f32p, C.c_int, C.c_float, C.c_float]
        L.orc_presmooth_bgr.argtypes = [_u8p, C.c_size_t, _u8p, C.c_size_t, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_float, C.c_float]
        L.orc_jbf_f32.argtypes = [C.c_int, C.c_int, _f32p, _u8p, _f32p, _f32p, C.c_int, C.c_float,
                                  C.c_float, C.c_int]
        L.orc_jbf_f64.argtypes = [C.c_int, C.c_int, _f32p, _u8p, _f32p, _f32p, C.c_void_p, C.c_int,
                                  C.c_float, C.c_float, C.c_int, C.c_double]
        L.orc_guided_fill_f32.argtypes = [C.c_int, C.c_int, _f32p, _u8p, C.c_void_p, _f32p, _f32p,
                                          C.c_int, C.c_float, C.c_float, C.c_int]
        L.orc_guided_fill_f64.argtypes = [C.c_int, C.c_int, _f32p, _u8p, C.c_void_p, _f32p, _f32p, C.c_void_p,
                                          C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_int]
        L.orc_scatter_lowres.argtypes = [_f32p, C.c_int, C.c_int, _f32p, C.c_int, C.c_int]
        for name in ("orc_buf_insert_f32", "orc_buf_insert_f32x2", "orc_buf_get_depth",
                     "orc_buf_get_weight", "orc_buf_update"):
            getattr(L, name).argtypes = [_f32p, _f32p, C.c_int, C.c_int]
        L.orc_buf_init.argtypes = [_f32p, C.c_int, C.c_int]
        L.orc_mrf_f32.argtypes = [C.c_int, C.c_int, _f32p, _u8p, _f32p, C.c_int, C.c_float, C.c_float,
                                  C.c_int]
        L.orc_mrf_f64.argtypes = L.orc_mrf_f32.argtypes
        L.orc_projective_to_real.argtypes = [_f32p, _f32p, C.c_int, C.c_int, C.c_float, C.c_float,
                                             C.c_int, C.c_int]
        L.orc_depth_bilateral_xyz.argtypes = [_f32p, _f32p, _f32p, _f32p, C.c_int, C.c_float, C.c_int, C.c_int, C.c_int]
        L.orc_depth_bilateral_xyz_f64.argtypes = L.orc_depth_bilateral_xyz.argtypes
        L.orc_mean_3d_error.argtypes = [_f32p, _f32p, C.c_int, C.POINTER(C.c_int)]
        L.orc_mean_3d_error.restype = C.c_float
        _lib = L
    return _lib


def ref_available() -> bool:
    return os.path.isfile(_REF_PATH)


def ref():
    """The reference's own kernel text compiled for the host (oracle/_ref)."""
    global _ref
    if _ref is None:
        if not ref_available():
            raise FileNotFoundError(_REF_PATH + " (run oracle/build_ref.py with a reference checkout)")
        R = C.CDLL(_REF_PATH)
        R.ref_jbf.argtypes = [C.c_int, C.c_int, _f32p, _u8p, _f32p, _f32p, C.c_int, C.c_float, C.c_float,
                              C.c_int]
        R.ref_guided_fill.argtypes = [C.c_int, C.c_int, _f32p, _u8p, C.c_void_p, _f32p, _f32p, C.c_int,
                                      C.c_float, C.c_float, C.c_int]
        R.ref_mrf.argtypes = [C.c_int, C.c_int, _f32p, _u8p, _f32p, C.c_int, C.c_float, C.c_float, C.c_int]
        for name in ("ref_buf_insert_f32", "ref_buf_insert_f32x2", "ref_buf_get_depth",
                     "ref_buf_get_weight", "ref_buf_update"):
            getattr(R, name).argtypes = [_f32p, _f32p, C.c_int, C.c_int]
        R.ref_buf_init.argtypes = [_f32p, C.c_int, C.c_int]
        R.ref_depth_bilateral_xyz.argtypes = [_f32p, _f32p, _f32p, _f32p, C.c_int, C.c_float, C.c_int, C.c_int, C.c_int]
        _ref = R
    return _ref


def n_cores() -> int:
    return len(os.sched_getaffinity(0))


# --------------------------------------------------------------------------- helpers
def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _bgr(a):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    assert a.ndim == 3 and a.shape[2] == 3, "guide must be HxWx3 packed BGR"
    return a


def spatial_lut(window: int, sigma_s: float) -> np.ndarray:
    lut = np.empty(window * window, np.float32)
    lib().orc_spatial_lut(lut, window, sigma_s)
    return lut


def presmooth(bgr, ksize=PRESMOOTH_KSIZE, sigma_color=PRESMOOTH_SIGMA_C, sigma_spatial=PRESMOOTH_SIGMA_S):
    """cv::gpu::bilateralFilter stand-in (JointBilateralFilter.cu:285).  HxWx3 u8 -> HxWx3 u8."""
    bgr = _bgr(bgr)
    h, w, _ = bgr.shape
    out = np.empty_like(bgr)
    lib().orc_presmooth_bgr(bgr, w * 3, out, w * 3, 3, w, h, ksize, sigma_color, sigma_spatial)
    return out


def jbf(depth, guide, window=JBF_WINDOW, sigma_s=JBF_SIGMA_S, sigma_c=JBF_SIGMA_C, sigma_d=JBF_SIGMA_D,
        precision="f32", threads=0, impl="oracle", return_mean=False, mean_shift_ulps=0.0):
    """Two-pass JBF kernel (JointBilateralFilter.cu:4-83) on an already smoothed guide.

    precision: "f32" (reference order, un-fused) or "f64" (exact-math with the fp32 skip rule).
    impl: "oracle" (C restatement) or "ref" (the reference's kernel text, fp32 only).
    """
    depth = _f32(depth)
    guide = _bgr(guide)
    h, w = depth.shape
    assert guide.shape[:2] == (h, w)
    lut = spatial_lut(window, sigma_s)
    out = np.empty((h, w), np.float32)
    threads = threads or n_cores()
    if impl == "ref":
        assert precision == "f32"
        ref().ref_jbf(w, h, depth, guide, lut, out, window, sigma_c, sigma_d, threads)
        return out
    if precision == "f32":
        lib().orc_jbf_f32(w, h, depth, guide, lut, out, window, sigma_c, sigma_d, threads)
        return out
    mean = np.empty((h, w), np.float64) if return_mean else None
    lib().orc_jbf_f64(w, h, depth, guide, lut, out, mean.ctypes.data if return_mean else None, window,
                      sigma_c, sigma_d, threads, float(mean_shift_ulps))
    return (out, mean) if return_mean else out


def jbf_envelope(depth, guide, window=JBF_WINDOW, sigma_s=JBF_SIGMA_S, sigma_c=JBF_SIGMA_C, sigma_d=JBF_SIGMA_D,
                 ulps=2.0, threads=0):
    """fp64 oracle output plus the per-pixel half-width of the envelope its output spans when the
    pass-1 mean moves by +-`ulps` fp32 ulps (the reference holds that mean in a float)."""
    o, mean = jbf(depth, guide, window, sigma_s, sigma_c, sigma_d, "f64", threads, return_mean=True)
    hi = jbf(depth, guide, window, sigma_s, sigma_c, sigma_d, "f64", threads, mean_shift_ulps=ulps)
    lo = jbf(depth, guide, window, sigma_s, sigma_c, sigma_d, "f64", threads, mean_shift_ulps=-ulps)
    band = np.maximum(np.abs(hi.astype(np.float64) - o), np.abs(lo.astype(np.float64) - o))
    return o, band, mean


def guard_active_mask(depth, mean64, window, sigma_d, margin_mm=1.0):
    """Pixels whose window holds a valid tap at or beyond the fp32 expf() underflow distance from the
    pass-1 mean, where the skip-if-zero guard (JointBilateralFilter.cu:67-68) gives the tap FULL weight.
    There the output is a discontinuous, ill-conditioned function of the pass-1 mean."""
    depth = _f32(depth)
    h, w = depth.shape
    r = window // 2
    thr = np.sqrt(103.97207708399179 * 2.0 * sigma_d * sigma_d)
    dp = np.pad(depth, r)
    act = np.zeros((h, w), bool)
    if not sigma_d > 0:
        return act
    for i in range(window):
        for j in range(window):
            dq = dp[i:i + h, j:j + w]
            act |= (dq > 50) & (np.abs(dq - mean64) > thr - margin_mm)
    return act


def parity_block(out, depth, guide, window=JBF_WINDOW, sigma_s=JBF_SIGMA_S, sigma_c=JBF_SIGMA_C,
                 sigma_d=JBF_SIGMA_D, threads=0):
    """Parity figures of a filtered frame `out` against the fp64 evaluation of the reference formula, as
    reported by bench.py / smoke() and asserted by tests/test_gpu_jbf.py (same definitions): mask
    mismatches, max |err| on guard-inactive ("regular") pixels, max |err| and count on guard-active pixels."""
    o64, mean = jbf(depth, guide, window, sigma_s, sigma_c, sigma_d, "f64", threads, return_mean=True)
    act = guard_active_mask(depth, mean, window, sigma_d)
    err = np.abs(np.asarray(out, np.float64) - o64.astype(np.float64))
    reg = np.where(act, 0.0, err)
    yr, xr = np.unravel_index(np.argmax(reg), reg.shape)
    ea = np.where(act, err, 0.0)
    ya, xa = np.unravel_index(np.argmax(ea), ea.shape)
    return {
        "mask_mismatches": int(np.count_nonzero((np.asarray(out) > 0) != (o64 > 0))),
        "nan": int(np.count_nonzero(np.isnan(out))),
        "max_abs_regular_mm": float(reg.max()), "worst_regular_yx": [int(yr), int(xr)],
        "max_abs_active_mm": float(ea.max()), "worst_active_yx": [int(ya), int(xa)],
        "n_active": int(act.sum()), "n_active_beyond_1e-3": int((act & (err > 1e-3)).sum()),
        "frac_within_1e-3": float((err <= 1e-3).mean()), "pixels": int(err.size),
    }


def jbf_process(depth, bgr, window=JBF_WINDOW, sigma_s=JBF_SIGMA_S, sigma_c=JBF_SIGMA_C,
                sigma_d=JBF_SIGMA_D, precision="f32", threads=0):
    """JointBilateralFilter::Process (JointBilateralFilter.cu:283-290): pre-smooth then filter."""
    return jbf(depth, presmooth(bgr), window, sigma_s, sigma_c, sigma_d, precision, threads)


def guided_fill(depth, guide, labels=None, window=ERS_WINDOW, sigma_s=ERS_SIGMA_S, sigma_c=ERS_SIGMA_C,
                sigma_d=ERS_SIGMA_D, threads=0, impl="oracle", precision="f32", return_mean=False, return_guard=False):
    """depthmap_enhancement (EdgeRefinedSuperpixel.cu:104-205), race-free; raw (un-smoothed) guide.

    precision "f64" only: return_mean adds the double sweep-1 mean, return_guard a uint8 map of the guard-active
    pixels (non-zero: a branch of the fp32 formula is decided within a few ulps of its threshold; the bits are
    those of orc_guided_fill_f64).  The result is out, then the mean and the guard in that order, as asked."""
    depth = _f32(depth)
    guide = _bgr(guide)
    h, w = depth.shape
    lut = spatial_lut(window, sigma_s)
    out = np.empty((h, w), np.float32)
    lab = None
    if labels is not None:
        lab = np.ascontiguousarray(labels, dtype=np.int32)
        assert lab.shape == (h, w)
    threads = threads or n_cores()
    if precision == "f64":
        mean = np.empty((h, w), np.float64) if return_mean else None
        guard = np.empty((h, w), np.uint8) if return_guard else None
        lib().orc_guided_fill_f64(w, h, depth, guide, lab.ctypes.data if lab is not None else None, lut, out,
                                  mean.ctypes.data if return_mean else None, guard.ctypes.data if return_guard else None,
                                  window, sigma_c, sigma_d, threads)
        extra = [a for a in (mean, guard) if a is not None]
        return (out, *extra) if extra else out
    if impl == "ref":
        if lab is None:
            lab = np.zeros((h, w), np.int32)
        ref().ref_guided_fill(w, h, depth, guide, lab.ctypes.data, lut, out, window, sigma_c, sigma_d, threads)
    else:
        lib().orc_guided_fill_f32(w, h, depth, guide, lab.ctypes.data if lab is not None else None, lut,
                                  out, window, sigma_c, sigma_d, threads)
    return out


def scatter_lowres(depth_lo, wh, hh):
    depth_lo = _f32(depth_lo)
    hl, wl = depth_lo.shape
    out = np.empty((hh, wh), np.float32)
    lib().orc_scatter_lowres(depth_lo, wl, hl, out, wh, hh)
    return out


def upsample(depth_lo, bgr_hi, radius=7, sigma_s=JBF_SIGMA_S, sigma_c=JBF_SIGMA_C, sigma_d=JBF_SIGMA_D,
             precision="f32", threads=0, presmoothed=False):
    """Upsampling (declared, never implemented: JointBilateralFilter.h:14); SURVEY.md 8(d) config 3."""
    bgr_hi = _bgr(bgr_hi)
    hh, wh, _ = bgr_hi.shape
    sparse = scatter_lowres(depth_lo, wh, hh)
    guide = bgr_hi if presmoothed else presmooth(bgr_hi)
    return jbf(sparse, guide, 2 * radius + 1, sigma_s, sigma_c, sigma_d, precision, threads)


def mrf(depth, guide, window=MRF_WINDOW, sigma_c=MRF_SIGMA_C, smooth=MRF_SMOOTH, threads=0, impl="oracle",
        precision="f32"):
    """MarkovRandomField.cu:4-40.  precision: "f32" (reference order) or "f64" (exact-math with the fp32
    expf() == 0 rule); impl: "oracle" (C restatement) or "ref" (the reference's kernel text, fp32 only)."""
    depth = _f32(depth)
    guide = _bgr(guide)
    h, w = depth.shape
    out = np.empty((h, w), np.float32)
    threads = threads or n_cores()
    if impl == "ref":
        assert precision == "f32"
        ref().ref_mrf(w, h, depth, guide, out, window, sigma_c, smooth, threads)
    elif precision == "f64":
        lib().orc_mrf_f64(w, h, depth, guide, out, window, sigma_c, smooth, threads)
    else:
        lib().orc_mrf_f32(w, h, depth, guide, out, window, sigma_c, smooth, threads)
    return out


def projective_to_real(depth, fx, fy, cx, cy):
    depth = _f32(depth)
    h, w = depth.shape
    out = np.empty((h, w, 3), np.float32)
    lib().orc_projective_to_real(depth, out.reshape(-1), w, h, fx, fy, int(cx), int(cy))
    return out


# Projection_GPU.cpp:3-5
PROJ_WINDOW, PROJ_SIGMA_S, PROJ_SIGMA_D = 7, 20.0, 100.0


def depth_bilateral_xyz(normalized, points, window=PROJ_WINDOW, sigma_s=PROJ_SIGMA_S, sigma_d=PROJ_SIGMA_D,
                        threads=0, impl="oracle", precision="f32"):
    """Projection_GPU::bilateralfilter (Projection_GPU.cu:213-246), race-free.  [H,W,3] float32 each."""
    normalized, points = _f32(normalized), _f32(points)
    h, w, _ = points.shape
    lut = spatial_lut(window, sigma_s)   # same formula as Projection_GPU.cpp:35-43
    out = np.empty_like(points)
    threads = threads or n_cores()
    fn = ref().ref_depth_bilateral_xyz if impl == "ref" else (
        lib().orc_depth_bilateral_xyz_f64 if precision == "f64" else lib().orc_depth_bilateral_xyz)
    fn(normalized.reshape(-1), points.reshape(-1), out.reshape(-1), lut, window, sigma_d, w, h, threads)
    return out


def mean_3d_error(points, truth):
    """main.cpp:217-308: mean 3-D distance over pixels with both z in (50, 15000).  Returns (mean, count)."""
    points, truth = _f32(points).reshape(-1), _f32(truth).reshape(-1)
    cnt = C.c_int()
    m = lib().orc_mean_3d_error(points, truth, points.size // 3, C.byref(cnt))
    return float(m), cnt.value


def mean_3d_error_f64(points, truth):
    """f4 with an fp64 sum: every distance is the fp32 sqrtf((dz*dz + dy*dy) + dx*dx) (each operation rounded to
    fp32, no contraction), so only the order of the sum differs from a kernel that evaluates them the same way.
    Returns (mean, count)."""
    p, t = _f32(points).reshape(-1, 3), _f32(truth).reshape(-1, 3)
    z, zt = p[:, 2], t[:, 2]
    m = (z > 50.0) & (z < 15000.0) & (zt > 50.0) & (zt < 15000.0)
    d = p[m] - t[m]
    dist = np.sqrt((d[:, 2] * d[:, 2] + d[:, 1] * d[:, 1]) + d[:, 0] * d[:, 0])
    n = int(m.sum())
    return (float(dist.astype(np.float64).sum()) / n if n else 0.0), n


class Buffer2D:
    """Host model of ArrayBuffer/Buffer2D (ArrayBuffer.h:9-45, Buffer2D.cu)."""

    def __init__(self, width, height, impl="oracle"):
        self.w, self.h = width, height
        self.buf = np.empty(width * height * 2, np.float32)
        self._L = ref() if impl == "ref" else lib()
        self._p = "ref_buf_" if impl == "ref" else "orc_buf_"
        getattr(self._L, self._p + "init")(self.buf, width, height)

    def _call(self, name, arr):
        getattr(self._L, self._p + name)(self.buf, arr, self.w, self.h)

    def insert(self, depth):
        self._call("insert_f32", _f32(depth).reshape(-1))

    def insert_f32x2(self, data_xy):
        self._call("insert_f32x2", _f32(data_xy).reshape(-1))

    def update(self, depth):
        self._call("update", _f32(depth).reshape(-1))

    def depth_map(self):
        out = np.empty(self.w * self.h, np.float32)
        self._call("get_depth", out)
        return out.reshape(self.h, self.w)

    def weight_map(self):
        out = np.empty(self.w * self.h, np.float32)
        self._call("get_weight", out)
        return out.reshape(self.h, self.w)

    def raw(self):
        return self.buf.reshape(self.h, self.w, 2)
