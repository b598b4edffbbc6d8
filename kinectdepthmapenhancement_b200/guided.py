"""Guided cross-bilateral fill: the depthmap_enhancement stage of EdgeRefinedSuperpixel
(EdgeRefinedSuperpixel.cu:104-205), reached from TOFDepthInterpolation.cpp:65."""
from __future__ import annotations

import torch

from . import _lib
from .jbf import _check_cuda, _ptr, guide_channels

# EdgeRefinedSuperpixel.cpp:4-7
WindowSize, SpatialSigma, ColorSigma, DepthSigma = 7, 30.0, 50.0, 70.0


def guided_fill(depth: torch.Tensor, color: torch.Tensor, labels: torch.Tensor | None = None,
                window_radius: int = 3, spatial_sigma: float = SpatialSigma, color_sigma: float = ColorSigma,
                depth_sigma: float = DepthSigma, out: torch.Tensor | None = None) -> torch.Tensor:
    """depth [H,W] f32, color [H,W,3] u8 (RAW guide; [H,W] / [H,W,1] GRAY or [H,W,4] BGRX also), labels [H,W]
    i32 or None -> refined depth [H,W]."""
    dev = depth.device
    _check_cuda(depth, torch.float32, "depth", dev)
    _check_cuda(color, torch.uint8, "color", dev)
    h, w = depth.shape
    c = guide_channels(color, (h, w))
    if labels is not None:
        _check_cuda(labels, torch.int32, "labels", dev)
        if tuple(labels.shape) != (h, w):
            raise ValueError("labels must be [H,W]")
    if out is None:
        out = torch.empty_like(depth)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().kdme_guided_fill_ex(_ptr(depth), _ptr(labels) if labels is not None else None,
                                                  _ptr(color), c * w, c, _ptr(out), w, h, window_radius, spatial_sigma,
                                                  color_sigma, depth_sigma, torch.cuda.current_stream().cuda_stream))
    return out


def guided_upsample(depth_lo: torch.Tensor, color_hi: torch.Tensor, labels_hi: torch.Tensor | None = None,
                    window_radius: int = 7, spatial_sigma: float = SpatialSigma, color_sigma: float = ColorSigma,
                    depth_sigma: float = DepthSigma, out: torch.Tensor | None = None) -> torch.Tensor:
    """Label-guided upsampling (SURVEY.md 8(d) config 3): low-res depth [hl,wl] -> high-res [H,W] using the
    depthmap_enhancement sweeps with the high-res label map (or None) and RAW high-res guide ([H,W,3] BGR,
    [H,W] / [H,W,1] GRAY or [H,W,4] BGRX)."""
    dev = depth_lo.device
    _check_cuda(depth_lo, torch.float32, "depth_lo", dev)
    _check_cuda(color_hi, torch.uint8, "color_hi", dev)
    hl, wl = depth_lo.shape
    if color_hi.dim() not in (2, 3):
        raise ValueError(f"color_hi must be [H,W] or [H,W,C], got {list(color_hi.shape)}")
    h, w = color_hi.shape[:2]
    c = guide_channels(color_hi, (h, w), "color_hi")
    if labels_hi is not None:
        _check_cuda(labels_hi, torch.int32, "labels_hi", dev)
        if tuple(labels_hi.shape) != (h, w):
            raise ValueError("labels must be [H,W] at the high-res size")
    if out is None:
        out = torch.empty((h, w), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().kdme_guided_upsample_ex(_ptr(depth_lo), wl, hl,
                                                      _ptr(labels_hi) if labels_hi is not None else None,
                                                      _ptr(color_hi), c * w, c, _ptr(out), w, h, window_radius,
                                                      spatial_sigma, color_sigma, depth_sigma,
                                                      torch.cuda.current_stream().cuda_stream))
    return out
