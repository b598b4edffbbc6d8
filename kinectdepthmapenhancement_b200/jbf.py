"""Host-side mirror of the reference's JointBilateralFilter class for torch tensors.

Same names, argument meaning and defaults as JointBilateralFilter.h:9-36 /
JointBilateralFilter.cpp:3-20; all compute happens in the sm_100a library behind
include/kdme_b200.h.  torch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib


def _ptr(t: torch.Tensor) -> int:
    return t.data_ptr()


def _check_cuda(t: torch.Tensor, dtype, name: str, device: torch.device):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError(f"{name} must be a CUDA tensor (there is no CPU path)")
    if t.device != device:
        raise ValueError(f"{name} lives on {t.device}, the filter on {device}")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")


def guide_channels(color: torch.Tensor, lead: tuple, name: str = "color") -> int:
    """Guide format of a uint8 image whose leading dimensions are `lead` ([H, W] or [N, H, W]): no channel
    dimension or 1 channel is GRAY (1), 3 channels BGR, 4 channels BGRX/BGRA.  Any other shape is a ValueError."""
    shape, lead = tuple(color.shape), tuple(int(v) for v in lead)
    if shape == lead:
        return 1
    if len(shape) == len(lead) + 1 and shape[:-1] == lead and shape[-1] in (1, 3, 4):
        return shape[-1]
    dims = ", ".join(str(v) for v in lead)
    raise ValueError(f"{name} must be [{dims}] or [{dims}, C] with C in (1, 3, 4) (GRAY, BGR, BGRX), got {list(shape)}")


class JointBilateralFilter:
    """JointBilateralFilter(width, height) -- JointBilateralFilter.h:11.

    The reference's static consts (JointBilateralFilter.cpp:3-6) are constructor
    arguments with the reference's values as defaults: window 5 (radius 2),
    sigma_spatial 70, sigma_color 50, sigma_depth 20; the guide pre-smooth is
    cv::gpu::bilateralFilter(color, smooth, 5, 30, 30) (JointBilateralFilter.cu:285).

    Every colour argument may be a GRAY/IR ([..., H, W] or [..., H, W, 1]), BGR ([..., 3]) or BGRX/BGRA
    ([..., 4]) uint8 image; the format is taken from the tensor's shape.  GRAY g filters exactly as the BGR
    image (g, 0, 0) and BGRX (b, g, r, x) exactly as (b, g, r).
    """

    WindowSize = 5
    SpatialSigma = 70.0
    ColorSigma = 50.0
    DepthSigma = 20.0

    def __init__(self, width: int, height: int, spatial_sigma: float = 70.0, color_sigma: float = 50.0,
                 depth_sigma: float = 20.0, window_radius: int = 2, max_batch: int = 1,
                 device: int | torch.device | None = None, stream: torch.cuda.Stream | None = None,
                 presmooth: tuple[int, float, float] | None = (5, 30.0, 30.0)):
        if not torch.cuda.is_available():
            raise RuntimeError("JointBilateralFilter needs a CUDA device (B200); there is no CPU fallback")
        if device is None:
            device = torch.cuda.current_device()
        self.device = torch.device("cuda", device if isinstance(device, int) else device.index or 0)
        self.width, self.height = int(width), int(height)
        self.radius, self.max_batch = int(window_radius), int(max_batch)
        self._stream = stream
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            sptr = stream.cuda_stream if stream is not None else torch.cuda.current_stream().cuda_stream
            self._sptr = sptr
            _lib.check(_lib.lib().jbf_create(C.byref(self._h), self.width, self.height, spatial_sigma,
                                             color_sigma, depth_sigma, self.radius, self.max_batch,
                                             self.device.index, sptr))
        if presmooth is None:
            _lib.check(_lib.lib().jbf_set_presmooth(self._h, 0, 0.0, 0.0))
        elif tuple(presmooth) != (5, 30.0, 30.0):
            _lib.check(_lib.lib().jbf_set_presmooth(self._h, int(presmooth[0]), float(presmooth[1]),
                                                    float(presmooth[2])))
        self._keep = None
        self._guide_c = 3   # the handle's guide format (jbf_set_guide_channels)

    def _use_guide(self, color: torch.Tensor, lead: tuple, name: str) -> int:
        """Set the handle's guide format from `color`'s shape; returns the row step in bytes."""
        c = guide_channels(color, lead, name)
        if c != self._guide_c:
            _lib.check(_lib.lib().jbf_set_guide_channels(self._h, c))
            self._guide_c = c
        return c * self.width

    # -- lifetime ----------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            _lib.lib().jbf_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- reference surface ---------------------------------------------------
    def Process(self, depth_device: torch.Tensor, color_image: torch.Tensor) -> None:
        """void Process(float* depth_device, cv::gpu::GpuMat color_image) -- JointBilateralFilter.cu:283-290.

        depth_device: [H, W] float32 CUDA; color_image: [H, W, 3] uint8 CUDA (BGR, continuous), or [H, W] /
        [H, W, 1] (GRAY) or [H, W, 4] (BGRX).  Asynchronous; result via getFiltered_Device()."""
        _check_cuda(depth_device, torch.float32, "depth_device", self.device)
        _check_cuda(color_image, torch.uint8, "color_image", self.device)
        if tuple(depth_device.shape) != (self.height, self.width):
            raise ValueError(f"depth must be [{self.height}, {self.width}]")
        step = self._use_guide(color_image, (self.height, self.width), "color image")
        self._keep = (depth_device, color_image)
        _lib.check(_lib.lib().jbf_process(self._h, _ptr(depth_device), _ptr(color_image), step))

    def process_xyz(self, depth_device: torch.Tensor, color_image: torch.Tensor, fx: float, fy: float, cx: int,
                    cy: int, out: torch.Tensor | None = None) -> torch.Tensor:
        """Process + DimensionConvertor::projectiveToReal fused (main.cpp:179 + :182): returns the float3
        cloud [H, W, 3]; the depth plane is in getFiltered_Device() as after Process."""
        _check_cuda(depth_device, torch.float32, "depth_device", self.device)
        _check_cuda(color_image, torch.uint8, "color_image", self.device)
        if tuple(depth_device.shape) != (self.height, self.width):
            raise ValueError(f"depth must be [{self.height}, {self.width}]")
        step = self._use_guide(color_image, (self.height, self.width), "color image")
        if out is None:
            out = torch.empty((self.height, self.width, 3), dtype=torch.float32, device=self.device)
        _check_cuda(out, torch.float32, "out", self.device)
        if tuple(out.shape) != (self.height, self.width, 3):
            raise ValueError(f"out must be [{self.height}, {self.width}, 3]")
        self._keep = (depth_device, color_image)
        _lib.check(_lib.lib().jbf_process_xyz(self._h, _ptr(depth_device), _ptr(color_image), step,
                                              _ptr(out), float(fx), float(fy), int(cx), int(cy)))
        return out

    def refine_stats(self) -> tuple[int, int]:
        """(pixels re-evaluated in fp64, pixels dropped because the queue was full) since the last call."""
        a, b = C.c_ulonglong(), C.c_ulonglong()
        _lib.check(_lib.lib().jbf_refine_stats(self._h, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def getFiltered_Device(self) -> torch.Tensor:
        """float* getFiltered_Device() const -- JointBilateralFilter.cpp:41-43 (borrowed view)."""
        ptr = _lib.lib().jbf_filtered_device(self._h)
        return _tensor_view(ptr, (self.height, self.width), torch.float32, self.device, self)

    def getFiltered_Host(self) -> torch.Tensor:
        """float* getFiltered_Host() const -- JointBilateralFilter.cpp:44-46 (copies D2H, synchronises)."""
        ptr = _lib.lib().jbf_filtered_host(self._h)
        if not ptr:
            _lib.check(_lib.KDME_EINVAL)
        buf = (C.c_float * (self.width * self.height)).from_address(ptr)
        return torch.frombuffer(buf, dtype=torch.float32).view(self.height, self.width).clone()

    def getSmoothImage_Device(self) -> torch.Tensor:
        """cv::gpu::GpuMat getSmoothImage_Device() -- JointBilateralFilter.cpp:47-49 (u8 view in the format of the
        last guide: [H,W] GRAY, [H,W,3] BGR, [H,W,4] BGRX with the 4th byte 255)."""
        step = C.c_size_t()
        ptr = _lib.lib().jbf_smooth_device(self._h, C.byref(step))
        if not ptr:
            _lib.check(_lib.KDME_EINVAL)
        shape = (self.height, self.width) if self._guide_c == 1 else (self.height, self.width, self._guide_c)
        return _tensor_view(ptr, shape, torch.uint8, self.device, self)

    def Upsampling(self, depthlow_device: torch.Tensor, colorhigh_image: torch.Tensor,
                   out: torch.Tensor | None = None) -> torch.Tensor:
        """void Upsampling(float* depthlow_device, cv::gpu::GpuMat colorhigh_image) -- declared only,
        JointBilateralFilter.h:14; semantics per SURVEY.md 8(d) config 3."""
        _check_cuda(depthlow_device, torch.float32, "depthlow_device", self.device)
        _check_cuda(colorhigh_image, torch.uint8, "colorhigh_image", self.device)
        hl, wl = depthlow_device.shape
        step = self._use_guide(colorhigh_image, (self.height, self.width), "colour image")
        if out is None:
            out = torch.empty((self.height, self.width), dtype=torch.float32, device=self.device)
        _check_cuda(out, torch.float32, "out", self.device)
        _lib.check(_lib.lib().jbf_upsample(self._h, _ptr(depthlow_device), wl, hl, _ptr(colorhigh_image),
                                           step, _ptr(out)))
        return out

    def upsample_batch(self, depth_lo: torch.Tensor, color_hi: torch.Tensor,
                       out: torch.Tensor | None = None) -> torch.Tensor:
        """N independent Upsampling calls: depth_lo [N, hl, wl] float32 millimetres or uint16 millimetres (the ToF
        sensor's format, read directly; torch.uint16 or a torch.int16 view of the same bits), color_hi
        [N, H, W, 3] u8 (or [N, H, W] / [N, H, W, 1] GRAY, [N, H, W, 4] BGRX) -> out [N, H, W] float32.  Frame k
        equals Upsampling of frame k alone, bit for bit."""
        if not isinstance(depth_lo, torch.Tensor) or depth_lo.dtype not in (torch.float32, torch.uint16, torch.int16):
            raise TypeError("depth_lo must be a float32 or uint16 tensor")
        _check_cuda(depth_lo, depth_lo.dtype, "depth_lo", self.device)
        _check_cuda(color_hi, torch.uint8, "color_hi", self.device)
        if depth_lo.dim() != 3 or depth_lo.shape[0] < 1:
            raise ValueError(f"depth_lo must be [N, hl, wl] with N >= 1, got {list(depth_lo.shape)}")
        n, hl, wl = (int(v) for v in depth_lo.shape)
        if not (1 <= wl <= self.width and 1 <= hl <= self.height):
            raise ValueError(f"low-res size {wl}x{hl} must be positive and at most {self.width}x{self.height}")
        step = self._use_guide(color_hi, (n, self.height, self.width), "color_hi")
        if out is None:
            out = torch.empty((n, self.height, self.width), dtype=torch.float32, device=self.device)
        _check_cuda(out, torch.float32, "out", self.device)
        if tuple(out.shape) != (n, self.height, self.width):
            raise ValueError(f"out must be [{n}, {self.height}, {self.width}]")
        fn = _lib.lib().jbf_upsample_batch if depth_lo.dtype == torch.float32 else _lib.lib().jbf_upsample_batch_u16
        _lib.check(fn(self._h, _ptr(depth_lo), wl, hl, _ptr(color_hi), step, _ptr(out), n))
        return out

    # -- batched / staged forms (B200-native additions) ----------------------
    def process_batch(self, depth: torch.Tensor, color: torch.Tensor, out: torch.Tensor | None = None):
        """N independent frames: depth [N,H,W] f32, color [N,H,W,3] u8 (or [N,H,W] / [N,H,W,1] GRAY,
        [N,H,W,4] BGRX) -> out [N,H,W] f32."""
        _check_cuda(depth, torch.float32, "depth", self.device)
        _check_cuda(color, torch.uint8, "color", self.device)
        n = depth.shape[0]
        if tuple(depth.shape[1:]) != (self.height, self.width):
            raise ValueError("depth must be [N,H,W] at the filter's size")
        step = self._use_guide(color, (n, self.height, self.width), "color")
        if out is None:
            out = torch.empty_like(depth)
        _check_cuda(out, torch.float32, "out", self.device)
        _lib.check(_lib.lib().jbf_process_batch(self._h, _ptr(depth), _ptr(color), step, _ptr(out), n))
        return out

    def presmooth(self, color: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """Guide pre-smooth only: [N,H,W,3] u8 (or [N,H,W] / [N,H,W,1] GRAY, [N,H,W,4] BGRX) -> internal guide
        [N,H,pitch] int32 words {B,G,R,0} ({g,0,0,0} for GRAY)."""
        _check_cuda(color, torch.uint8, "color", self.device)
        n = color.shape[0] if color.dim() >= 3 else 0
        step = self._use_guide(color, (n, self.height, self.width), "color")
        pitch = (self.width + 3) & ~3
        if out is None:
            g4 = torch.empty((n, self.height, pitch), dtype=torch.int32, device=self.device)
        else:
            _check_cuda(out, torch.int32, "out", self.device)
            if tuple(out.shape) != (n, self.height, pitch):
                raise ValueError(f"out must be [{n}, {self.height}, {pitch}]")
            g4 = out
        _lib.check(_lib.lib().jbf_presmooth(self._h, _ptr(color), step, _ptr(g4), pitch * 4, n))
        return g4

    def filter_guide4(self, depth: torch.Tensor, guide4: torch.Tensor, out: torch.Tensor | None = None):
        """Filter only, on an already smoothed internal guide (see presmooth()): depth [N,H,W] f32,
        guide4 [N,H,pitch] int32 words {B,G,R,0} with pitch >= W and a multiple of 4."""
        _check_cuda(depth, torch.float32, "depth", self.device)
        _check_cuda(guide4, torch.int32, "guide4", self.device)
        if depth.dim() != 3 or tuple(depth.shape[1:]) != (self.height, self.width):
            raise ValueError(f"depth must be [N, {self.height}, {self.width}]")
        n = depth.shape[0]
        if guide4.dim() != 3 or guide4.shape[0] != n or guide4.shape[1] != self.height or \
                guide4.shape[2] < self.width or guide4.shape[2] % 4:
            raise ValueError(f"guide4 must be [{n}, {self.height}, pitch] with pitch >= {self.width} and a multiple of 4")
        if out is None:
            out = torch.empty_like(depth)
        _check_cuda(out, torch.float32, "out", self.device)
        if tuple(out.shape) != tuple(depth.shape):
            raise ValueError("out must have the shape of depth")
        if out.data_ptr() == depth.data_ptr():
            raise ValueError("in-place filtering is not supported")
        _lib.check(_lib.lib().jbf_filter_guide4(self._h, _ptr(depth), _ptr(guide4), guide4.shape[-1] * 4,
                                                _ptr(out), n))
        return out

    def process_host(self, depth_host: torch.Tensor, color_host: torch.Tensor, out_host: torch.Tensor):
        """End-to-end with HOST tensors (ideally pinned, see host_buffer()): upload, Process, download;
        synchronous.  depth_host may be float32 millimetres or uint16 millimetres (the sensor's format,
        converted on the device)."""
        if depth_host.dtype not in (torch.float32, torch.uint16, torch.int16):
            raise TypeError("depth_host must be float32 or uint16")
        for t, dt, nm in ((depth_host, depth_host.dtype, "depth_host"), (color_host, torch.uint8, "color_host"),
                          (out_host, torch.float32, "out_host")):
            if t.is_cuda or t.dtype != dt or not t.is_contiguous():
                raise TypeError(f"{nm} must be a contiguous CPU tensor of {dt}")
        n = depth_host.shape[0]
        if tuple(depth_host.shape) != (n, self.height, self.width):
            raise ValueError(f"depth_host must be [N, {self.height}, {self.width}]")
        if tuple(out_host.shape) != (n, self.height, self.width):
            raise ValueError(f"out_host must be [{n}, {self.height}, {self.width}]")
        step = self._use_guide(color_host, (n, self.height, self.width), "color_host")
        fn = _lib.lib().jbf_process_host if depth_host.dtype == torch.float32 else _lib.lib().jbf_process_host_u16
        _lib.check(fn(self._h, _ptr(depth_host), _ptr(color_host), step, _ptr(out_host), n))
        return out_host

    def mrf(self, depth: torch.Tensor, color: torch.Tensor, window_radius=2, color_sigma=50.0, smooth_sigma=150.0):
        """MarkovRandomField::Process -- MarkovRandomField.cu:4-49 (next row f1)."""
        _check_cuda(depth, torch.float32, "depth", self.device)
        _check_cuda(color, torch.uint8, "color", self.device)
        if tuple(depth.shape) != (self.height, self.width):
            raise ValueError(f"depth must be [{self.height}, {self.width}]")
        step = self._use_guide(color, (self.height, self.width), "color")
        out = torch.empty_like(depth)
        _lib.check(_lib.lib().jbf_mrf(self._h, _ptr(depth), _ptr(color), step, _ptr(out),
                                      window_radius, color_sigma, smooth_sigma))
        return out

    @property
    def kernel_variant(self) -> int:
        return _lib.lib().jbf_kernel_variant(self._h)


class _HostBlock:
    def __init__(self, nbytes: int, write_combined: bool):
        self.ptr = _lib.lib().kdme_host_alloc(nbytes, 1 if write_combined else 0)
        if not self.ptr:
            _lib.check(_lib.KDME_EINVAL)
        self.buf = (C.c_uint8 * nbytes).from_address(self.ptr)

    def __del__(self):
        try:
            _lib.lib().kdme_host_free(self.ptr)
        except Exception:
            pass


def host_buffer(shape, dtype: torch.dtype, write_combined: bool = False) -> torch.Tensor:
    """Page-locked host tensor owned by the library (cudaHostAlloc): the buffers jbf_process_host expects.
    write_combined=True for input buffers the CPU only fills front to back; never for results."""
    n = 1
    for s_ in shape:
        n *= int(s_)
    nbytes = max(1, n * torch.empty((), dtype=dtype).element_size())
    blk = _HostBlock(nbytes, write_combined)
    t = torch.frombuffer(blk.buf, dtype=dtype, count=n).view(*shape)
    t._kdme_block = blk   # keeps the allocation alive as long as the tensor object
    return t


def _tensor_view(ptr: int, shape, dtype, device, owner):
    """Zero-copy torch view of library-owned device memory (borrowed, like the reference's raw pointer)."""
    n = 1
    for s in shape:
        n *= s
    itemsize = torch.empty((), dtype=dtype).element_size()

    class _Holder:
        pass

    hold = _Holder()
    hold.__cuda_array_interface__ = {
        "shape": tuple(shape), "typestr": {torch.float32: "<f4", torch.uint8: "|u1", torch.int32: "<i4"}[dtype],
        "data": (int(ptr), False), "version": 2, "strides": None,
    }
    hold.owner = owner
    with torch.cuda.device(device):
        t = torch.as_tensor(hold, device=device)
    assert t.numel() == n and t.element_size() == itemsize
    return t


def projective_to_real(depth: torch.Tensor, fx: float, fy: float, cx: int, cy: int) -> torch.Tensor:
    """DimensionConvertor::projectiveToReal(float*, float3*) -- DimensionConvertor.cu:3-23 (next row f3)."""
    if not depth.is_cuda or depth.dtype != torch.float32 or not depth.is_contiguous():
        raise TypeError("depth must be a contiguous float32 CUDA tensor")
    h, w = depth.shape
    out = torch.empty((h, w, 3), dtype=torch.float32, device=depth.device)
    with torch.cuda.device(depth.device):
        _lib.check(_lib.lib().kdme_projective_to_real(_ptr(depth), _ptr(out), w, h, fx, fy, int(cx), int(cy),
                                                      torch.cuda.current_stream().cuda_stream))
    return out
