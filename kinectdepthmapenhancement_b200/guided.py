"""Guided cross-bilateral fill: the depthmap_enhancement stage of EdgeRefinedSuperpixel
(EdgeRefinedSuperpixel.cu:104-205), reached from TOFDepthInterpolation.cpp:65."""
from __future__ import annotations

import torch

from . import _lib
from .jbf import _check_cuda, _depth_entry, _ptr, guide_channels

# EdgeRefinedSuperpixel.cpp:4-7
WindowSize, SpatialSigma, ColorSigma, DepthSigma = 7, 30.0, 50.0, 70.0


def _one(t):
    """One frame as a batch of one (its [None] view); None stays None."""
    return None if t is None else t[None]


def _batch_depth(depth: torch.Tensor, name: str, entry: str) -> tuple:
    """Checks a [N, rows, cols] float32 or uint16 depth batch (torch.uint16 or an int16 view of the same bits):
    (`entry` for its dtype, its shape)."""
    entry = _depth_entry(depth, name, entry)
    _check_cuda(depth, depth.dtype, name, depth.device)
    if depth.shape[0] < 1:
        raise ValueError(f"{name} must be [N, ...] with N >= 1, got {list(depth.shape)}")
    return entry, tuple(int(v) for v in depth.shape)


def _batch_labels(labels: torch.Tensor | None, lead: tuple, dev, name: str):
    if labels is not None:
        _check_cuda(labels, torch.int32, name, dev)
        if tuple(labels.shape) != lead:
            raise ValueError(f"{name} must be {list(lead)}, got {list(labels.shape)}")
        return _ptr(labels)
    return None


def _batch_out(out: torch.Tensor | None, lead: tuple, dev) -> torch.Tensor:
    if out is None:
        return torch.empty(lead, dtype=torch.float32, device=dev)
    _check_cuda(out, torch.float32, "out", dev)
    if tuple(out.shape) != lead:
        raise ValueError(f"out must be {list(lead)}, got {list(out.shape)}")
    return out


def guided_fill(depth: torch.Tensor, color: torch.Tensor, labels: torch.Tensor | None = None,
                window_radius: int = 3, spatial_sigma: float = SpatialSigma, color_sigma: float = ColorSigma,
                depth_sigma: float = DepthSigma, out: torch.Tensor | None = None) -> torch.Tensor:
    """depth [H,W] f32, color [H,W,3] u8 (RAW guide; [H,W] / [H,W,1] GRAY or [H,W,4] BGRX also), labels [H,W]
    i32 or None -> refined depth [H,W].

    A stream of frames in one call: depth [N,H,W] float32 or uint16 millimetres (torch.uint16 or an int16 view of
    the same bits; values <= 50 are holes), color [N,H,W] / [N,H,W,C], labels [N,H,W] or None -> [N,H,W].  The
    depth's rank decides which form runs; frame k equals the fill of frame k alone, bit for bit."""
    if isinstance(depth, torch.Tensor) and depth.dim() == 3:
        return _guided_fill_batch(depth, color, labels, window_radius, spatial_sigma, color_sigma, depth_sigma, out)
    _check_cuda(depth, torch.float32, "depth", depth.device)
    res = _guided_fill_batch(depth[None], _one(color), _one(labels), window_radius, spatial_sigma, color_sigma,
                             depth_sigma, _one(out))
    return res[0] if out is None else out


def _guided_fill_batch(depth, color, labels, window_radius, spatial_sigma, color_sigma, depth_sigma, out):
    entry, (n, h, w) = _batch_depth(depth, "depth", "kdme_guided_fill_batch")
    dev = depth.device
    _check_cuda(color, torch.uint8, "color", dev)
    c = guide_channels(color, (n, h, w))
    lab = _batch_labels(labels, (n, h, w), dev, "labels")
    out = _batch_out(out, (n, h, w), dev)
    fn = getattr(_lib.lib(), entry)
    with torch.cuda.device(dev):
        _lib.check(fn(_ptr(depth), lab, _ptr(color), c * w, c, _ptr(out), w, h, n, window_radius, spatial_sigma,
                      color_sigma, depth_sigma, torch.cuda.current_stream().cuda_stream))
    return out


def guided_upsample(depth_lo: torch.Tensor, color_hi: torch.Tensor, labels_hi: torch.Tensor | None = None,
                    window_radius: int = 7, spatial_sigma: float = SpatialSigma, color_sigma: float = ColorSigma,
                    depth_sigma: float = DepthSigma, out: torch.Tensor | None = None) -> torch.Tensor:
    """Label-guided upsampling (SURVEY.md 8(d) config 3): low-res depth [hl,wl] -> high-res [H,W] using the
    depthmap_enhancement sweeps with the high-res label map (or None) and RAW high-res guide ([H,W,3] BGR,
    [H,W] / [H,W,1] GRAY or [H,W,4] BGRX).

    A stream of frames in one call: depth_lo [N,hl,wl] float32 or uint16 millimetres, color_hi [N,H,W] /
    [N,H,W,C], labels_hi [N,H,W] or None -> [N,H,W]; frame k equals the upsampling of frame k alone, bit for bit."""
    if isinstance(depth_lo, torch.Tensor) and depth_lo.dim() == 3:
        return _guided_upsample_batch(depth_lo, color_hi, labels_hi, window_radius, spatial_sigma, color_sigma,
                                      depth_sigma, out)
    _check_cuda(depth_lo, torch.float32, "depth_lo", depth_lo.device)
    res = _guided_upsample_batch(depth_lo[None], _one(color_hi), _one(labels_hi), window_radius, spatial_sigma,
                                 color_sigma, depth_sigma, _one(out))
    return res[0] if out is None else out


def _guided_upsample_batch(depth_lo, color_hi, labels_hi, window_radius, spatial_sigma, color_sigma, depth_sigma,
                           out):
    entry, (n, hl, wl) = _batch_depth(depth_lo, "depth_lo", "kdme_guided_upsample_batch")
    dev = depth_lo.device
    _check_cuda(color_hi, torch.uint8, "color_hi", dev)
    if color_hi.dim() not in (3, 4):
        raise ValueError(f"color_hi must be [N,H,W] or [N,H,W,C], got {list(color_hi.shape)}")
    h, w = (int(v) for v in color_hi.shape[1:3])
    c = guide_channels(color_hi, (n, h, w), "color_hi")
    if not (1 <= wl <= w and 1 <= hl <= h):
        raise ValueError(f"low-res size {wl}x{hl} must be positive and at most the high-res {w}x{h}")
    lab = _batch_labels(labels_hi, (n, h, w), dev, "labels_hi")
    out = _batch_out(out, (n, h, w), dev)
    fn = getattr(_lib.lib(), entry)
    with torch.cuda.device(dev):
        _lib.check(fn(_ptr(depth_lo), wl, hl, lab, _ptr(color_hi), c * w, c, _ptr(out), w, h, n, window_radius,
                      spatial_sigma, color_sigma, depth_sigma, torch.cuda.current_stream().cuda_stream))
    return out
