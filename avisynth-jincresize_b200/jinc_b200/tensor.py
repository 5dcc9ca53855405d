"""PyTorch front-end: Jinc resizes of CUDA tensors, differentiable for float16 / float32.

    y = jinc_resize(x, 1920, 1080, tap=3)

`x` is a CUDA tensor (..., H, W); every leading index is one plane, and all planes go out in one launch per kernel
(jinc_resize_planes_device).  The arguments are those of the VapourSynth filter core.jinc.JincResize on a GRAY clip, with
its defaults, so a call on one plane equals that filter on that plane, byte for byte.  The resize is a fixed linear map
out = A * src; for float16 and float32 inputs the op is a torch.autograd.Function whose backward runs the adjoint A^T
(jinc_resize_adjoint_planes_device) in float32 and casts the result to x.dtype.  There is no gradient with respect to the
geometry arguments, and none for integer planes.

Work runs on torch.cuda.current_stream(x.device) with no host synchronisation.  One library context is kept per device and
a small LRU cache of coefficient tables keyed by (device, table parameters); building a table is synchronous, so a cached
table is ready before any launch reads it.
"""
from __future__ import annotations

import threading
from collections import OrderedDict

import numpy as np
import torch

from . import capi

_SAMPLE = {torch.uint8: 1, torch.uint16: 2, torch.float16: capi.SAMPLE_F16, torch.float32: 4}
_TABLE_CACHE_SIZE = 32

_lock = threading.Lock()
_contexts: dict[int, capi.Context] = {}
_tables: OrderedDict = OrderedDict()


def _f32(v) -> float:
    return float(np.float32(v))  # script floats are 32-bit


def _check_args(x, width, height, tap, quant_x, quant_y, bits) -> int:
    """Validates everything that needs no GPU; returns the bits per sample (0 for float planes)."""
    if not isinstance(x, torch.Tensor):
        raise TypeError(f"jinc_resize: expected a torch.Tensor, got {type(x).__name__}")
    if x.dtype not in _SAMPLE:
        raise TypeError(f"jinc_resize: unsupported dtype {x.dtype} (uint8, uint16, float16 or float32)")
    if x.dtype == torch.uint8:
        if bits not in (None, 8):
            raise ValueError(f"jinc_resize: bits must be 8 for uint8 planes, got {bits}")
        bits = 8
    elif x.dtype == torch.uint16:
        bits = 16 if bits is None else bits
        if not (isinstance(bits, int) and 9 <= bits <= 16):
            raise ValueError(f"jinc_resize: bits must be 9..16 for uint16 planes, got {bits}")
    else:
        if bits is not None:
            raise ValueError(f"jinc_resize: bits applies to integer planes only, got bits={bits} for {x.dtype}")
        bits = 0
    if x.device.type != "cuda":
        raise ValueError(f"jinc_resize: x is on {x.device}; the resize has no CPU path, move the tensor to a CUDA device")
    if x.dim() < 2:
        raise ValueError("jinc_resize: x must have shape (..., H, W)")
    if not (1 <= tap <= 16):
        raise ValueError("jinc_resize: tap must be between 1..16.")
    if not (1 <= quant_x <= 256) or not (1 <= quant_y <= 256):
        raise ValueError("jinc_resize: quant_x and quant_y must be between 1..256.")
    if width < 1 or height < 1:
        raise ValueError("jinc_resize: width and height must be positive.")
    return bits


def _table(device: int, key: tuple) -> capi.Table:
    with _lock:
        t = _tables.get((device, key))
        if t is not None:
            _tables.move_to_end((device, key))
            return t
        ctx = _contexts.get(device)
        if ctx is None:
            ctx = _contexts[device] = capi.Context(device)
        qx, qy, sw, sh, dw, dh, radius, blur, cl, ct, cw, ch = key
        t = capi.Table(ctx, quant_x=qx, quant_y=qy, src_w=sw, src_h=sh, dst_w=dw, dst_h=dh, radius=radius, blur=blur,
                       crop_left=cl, crop_top=ct, crop_w=cw, crop_h=ch)
        _tables[(device, key)] = t
        if len(_tables) > _TABLE_CACHE_SIZE:
            # dropped from the cache; an autograd graph that still holds it keeps it alive.  Destroying a table frees device
            # memory, which waits for the kernels still reading it.
            _tables.popitem(last=False)
        return t


def _planes(x: torch.Tensor) -> torch.Tensor:
    """x as (N, H, W) planes that do not overlap: unit column stride, a row pitch of at least W and one plane stride of at
    least H rows.  A view of x when its layout allows (a crop or a slice of a larger tensor), else a contiguous copy (e.g. a
    gradient expanded over some dimensions)."""
    H, W = x.shape[-2:]
    if x.stride(-1) == 1 and x.stride(-2) >= W:
        try:
            v = x.view(-1, H, W)
            if v.shape[0] <= 1 or v.stride(0) >= H * v.stride(1):
                return v
        except RuntimeError:
            pass
    return x.contiguous().view(-1, H, W)


_CUDA_STREAM_LEGACY = 0x1  # cudaStreamLegacy


def _stream(device: torch.device) -> int:
    """Handle of torch's current stream on `device`.  torch reports its default stream as 0, which the C ABI reads as the
    library context's own stream; it is passed as cudaStreamLegacy instead, so the work stays ordered with torch's."""
    return torch.cuda.current_stream(device).cuda_stream or _CUDA_STREAM_LEGACY


def _forward(x: torch.Tensor, table: capi.Table, width: int, height: int, peak: float) -> torch.Tensor:
    src = _planes(x)
    n = src.shape[0]
    isz = x.element_size()
    pitch = (width * isz + 15) // 16 * 16 // isz  # destination rows 16-byte aligned
    # the result is a tensor of its own (not a view), so it can be modified in place: rows `pitch` samples apart, the leading
    # dimensions packed
    shape = (*x.shape[:-2], height, width)
    out = torch.empty_strided(shape, _packed_strides(shape, pitch), dtype=x.dtype, device=x.device)
    if n:
        table.resize_planes_device(_SAMPLE[x.dtype], peak, n, src.data_ptr(), src.stride(1) * isz, src.stride(0) * isz,
                                   out.data_ptr(), pitch * isz, height * pitch * isz, _stream(x.device))
    return out


def _packed_strides(shape, pitch: int) -> tuple:
    """Strides of `shape` (..., h, w) with rows `pitch` elements apart and every leading dimension packed."""
    strides = [pitch, 1]
    step = shape[-2] * pitch
    for d in reversed(shape[:-2]):
        strides.insert(0, step)
        step *= d
    return tuple(strides)


def _adjoint(grad: torch.Tensor, table: capi.Table, H: int, W: int) -> torch.Tensor:
    g = _planes(grad.to(torch.float32))
    n, h, w = g.shape
    out = torch.empty((n, H, W), dtype=torch.float32, device=grad.device)
    if n:
        table.adjoint_planes_device(n, g.data_ptr(), g.stride(1) * 4, g.stride(0) * 4, out.data_ptr(), W * 4, H * W * 4,
                                    _stream(grad.device))
    return out


class _JincResizeFloat(torch.autograd.Function):
    """float16 / float32 planes: forward resize, backward adjoint (float32, cast to x.dtype)."""

    @staticmethod
    def forward(ctx, x, table, width, height):
        ctx.table = table
        ctx.src_shape = x.shape
        ctx.x_dtype = x.dtype
        with torch.cuda.device(x.device):
            return _forward(x, table, width, height, 0.0)

    @staticmethod
    def backward(ctx, grad_out):
        H, W = ctx.src_shape[-2:]
        with torch.cuda.device(grad_out.device):
            g = _adjoint(grad_out, ctx.table, H, W)
        return g.view(ctx.src_shape).to(ctx.x_dtype), None, None, None


def jinc_resize(x: torch.Tensor, width: int, height: int, *, tap: int = 3, src_left: float = 0.0, src_top: float = 0.0,
                src_width: float | None = None, src_height: float | None = None, quant_x: int = 256, quant_y: int = 256,
                blur: float = 0.0, bits: int | None = None) -> torch.Tensor:
    """Jinc (EWA) resize of every (H, W) plane of the CUDA tensor `x` (..., H, W) to (..., height, width).

    dtypes: uint8 (bits 8), uint16 (bits 9..16, default 16; samples are clamped to 2**bits - 1), float16 and float32 (raw
    sums, no clamp).  src_left / src_top / src_width / src_height crop the source as in core.jinc.JincResize (a width or
    height <= 0 counts from the right / bottom edge); floats are rounded to float32 first, as script floats are.  blur 0
    means 1.0.  Chroma siting is not applied: shift chroma planes with src_left / src_top.

    The result's rows are padded to 16 bytes: when width * x.element_size() is not a multiple of 16 it is not contiguous
    (stride(-2) > width, the leading dimensions packed).  It is a tensor of its own, not a view, so it may be modified in
    place before backward.  float16 / float32 inputs are differentiable with
    respect to x (the adjoint of the resize); the geometry arguments are not.
    """
    bits = _check_args(x, width, height, tap, quant_x, quant_y, bits)
    H, W = x.shape[-2:]
    src_left, src_top = _f32(src_left), _f32(src_top)
    crop_w = _f32(src_width) if src_width is not None else float(W)
    crop_h = _f32(src_height) if src_height is not None else float(H)
    if crop_w <= 0.0:
        crop_w = W - src_left + crop_w
    if crop_h <= 0.0:
        crop_h = H - src_top + crop_h
    key = (quant_x, quant_y, W, H, width, height, capi.radius_for_tap(tap), _f32(blur), src_left, src_top, crop_w, crop_h)
    device = x.device.index if x.device.index is not None else torch.cuda.current_device()
    with torch.cuda.device(device):
        table = _table(device, key)
    if bits == 0:
        return _JincResizeFloat.apply(x, table, width, height)
    with torch.cuda.device(device):
        return _forward(x, table, width, height, float((1 << bits) - 1))


__all__ = ["jinc_resize"]
