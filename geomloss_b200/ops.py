"""Torch-facing wrappers of the C-ABI kernels: device buffers in, device buffers out, autograd wired.

Mirrors the reference's operator seam — ``softmin(eps, C_xy, h_y) -> f_x`` with ``C_xy = (x, y)``
(src/geomloss/_legacy/sinkhorn_samples.py:337-346, sinkhorn_divergence.py:291-303) and the kernel
matvecs of ``kernel_loss`` (kernel_samples.py:128-137) — but every call lands in libb200ot.so.
PyTorch is used for memory, streams and autograd bookkeeping only.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib

KERNEL_KINDS = {"gaussian": 0, "laplacian": 1, "energy": 2}
# flags of include/b200ot.h: the pykeops convention for sqrt(|x-y|^2) (no 1e-8 clamp, zero gradient at 0), used by
# the reference's "online" / "multiscale" backends; the plain values are the "tensorized" convention
P_UNCLAMPED = 0x100
KERNEL_UNCLAMPED = 0x100
MAX_D = 8  # dimensions instantiated in this build of libb200ot.so (supported_simt_dim in csrc/host_util.cuh)

# Number of kernels of libb200ot.so enqueued so far by this process (bench.py reports the delta over its
# timed region as `gpu_launches`).  Every one-call entry point is pack + partial reduction + finalize.
_launches = 0


def count_launches(n: int):
    global _launches
    _launches += n


# NVTX ranges around every reduction (SURVEY.md section 5: the reference's only tracing hook is the torch profiler in
# examples/performances/plot_profile.py).  Off by default; B200OT_NVTX=1 brackets each softmin / kernel matvec so that a
# timeline (nsys, or ncu --nvtx --nvtx-include) shows the Sinkhorn loop iteration by iteration.
import os as _os

NVTX = _os.environ.get("B200OT_NVTX", "0") == "1"


class nvtx_range:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if NVTX:
            torch.cuda.nvtx.range_push(self.name)

    def __exit__(self, *exc):
        if NVTX:
            torch.cuda.nvtx.range_pop()


def launches() -> int:
    return _launches


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream(dev):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _f32c(t, name):
    if t is None:
        return None
    if not t.is_cuda:
        raise _lib.B200OTError(f"{name} must live on a CUDA device (geomloss_b200 has no CPU path), got {t.device}")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32 (the engine computes in fp32), got {t.dtype}")
    return t.contiguous()


MAX_D_TC = 64  # softmin (p = 2) and kernel convolutions, forward + row gradients: tensor-core path, 8 < D <= 64


def _check_clouds(x, y, max_d=None):
    max_d = MAX_D if max_d is None else max_d
    if x.dim() != 2 or y.dim() != 2 or x.shape[1] != y.shape[1]:
        raise ValueError(f"expected x:(N,D), y:(M,D); got {tuple(x.shape)}, {tuple(y.shape)}")
    if x.shape[0] == 0 or y.shape[0] == 0:
        raise ValueError("empty point cloud")
    if x.shape[1] > max_d:
        raise NotImplementedError(f"D = {x.shape[1]} > {max_d}: not instantiated in this build (CUDA-core kernels "
                                  f"serve D <= {MAX_D}; the tensor-core kernels serve the p = 2 softmin and the "
                                  f"gaussian / laplacian / energy kernel convolutions, forward and row gradients, "
                                  f"up to D = {MAX_D_TC})")
    if x.device != y.device:
        raise ValueError("x and y must be on the same device")


_scratch_cache: dict = {}


def _scratch(nbytes: int, dev, tag: str):
    """Per-(device, stream, tag) scratch buffer, grown geometrically; stream-ordered reuse is safe because
    every kernel that touches it is enqueued on that same stream."""
    key = (dev, torch.cuda.current_stream(dev).cuda_stream, tag)
    buf = _scratch_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=dev)
        _scratch_cache[key] = buf
    return buf


_extent_scratch: dict = {}


def cloud_extent(x, y=None):
    """(2, D) device tensor [minima; maxima] over the rows of x (and y) in ONE launch (b200ot_cloud_extent), or None
    when the clouds are not float32 CUDA tensors with D <= MAX_D (callers then use torch reductions)."""
    if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and 1 <= x.shape[1] <= MAX_D and x.shape[0] > 0):
        return None
    if y is not None and not (y.is_cuda and y.dtype == torch.float32 and y.dim() == 2 and y.shape[1] == x.shape[1]
                              and y.device == x.device):
        return None
    x = x.detach().contiguous()
    y = None if y is None or y.shape[0] == 0 else y.detach().contiguous()
    dev = x.device
    L = _lib.lib()
    with torch.cuda.device(dev):
        key = (dev, torch.cuda.current_stream(dev).cuda_stream)
        scratch = _extent_scratch.get(key)
        if scratch is None:  # zero once: the kernel's ticket counter returns to zero after every launch
            scratch = _extent_scratch[key] = torch.zeros(L.b200ot_cloud_extent_scratch_bytes(), dtype=torch.uint8,
                                                         device=dev)
        out = torch.empty(2, x.shape[1], dtype=torch.float32, device=dev)
        rc = L.b200ot_cloud_extent(_ptr(x), x.shape[0], _ptr(y), 0 if y is None else y.shape[0], x.shape[1], _ptr(out),
                                   _ptr(scratch), scratch.numel(), _stream(dev))
    _lib.check(rc, "b200ot_cloud_extent")
    count_launches(1)
    return out


def default_center(x, y):
    """Mid-point of the joint bounding box: the origin of the |x|^2 - 2x.y + |y|^2 expansion."""
    lh = cloud_extent(x, y)
    if lh is not None:
        return (0.5 * (lh[0] + lh[1])).contiguous()
    lo = torch.minimum(x.min(0).values, y.min(0).values)
    hi = torch.maximum(x.max(0).values, y.max(0).values)
    return (0.5 * (lo + hi)).float().contiguous()


# ------------------------------------------------------------------------------------------------
# softmin
# ------------------------------------------------------------------------------------------------


def softmin_raw(eps, x, y, h_a, h_b=None, h_scale_b=0.0, *, p=2, center=None, out_old=None, alpha_old=0.0,
                beta=1.0, out=None, want_lse2=False):
    """One fused launch group: ``out <- alpha_old*out_old + beta*softmin(eps, (x, y), h_a + h_scale_b*h_b)``.

    No autograd.  Returns ``(out, lse2 | None)``.
    """
    x, y, h_a, h_b = _f32c(x, "x"), _f32c(y, "y"), _f32c(h_a, "h_a"), _f32c(h_b, "h_b")
    center, out_old = _f32c(center, "center"), _f32c(out_old, "out_old")
    _check_clouds(x, y, MAX_D_TC if (p & 0xFF) == 2 else MAX_D)
    N, D = x.shape
    M = y.shape[0]
    if h_a.numel() != M or (h_b is not None and h_b.numel() != M):
        raise ValueError("h must have one entry per column")
    dev = x.device
    L = _lib.lib()
    with torch.cuda.device(dev), nvtx_range(f"b200ot.softmin N={N} M={M} D={D} eps={float(eps):.3g}"):
        if out is None:
            out = torch.empty(N, dtype=torch.float32, device=dev)
        lse2 = torch.empty(N, dtype=torch.float32, device=dev) if want_lse2 else None
        nbytes = L.b200ot_softmin_scratch_bytes(N, M, D)
        scratch = _scratch(nbytes, dev, "softmin")
        rc = L.b200ot_softmin_fwd(_ptr(x), _ptr(y), _ptr(h_a), _ptr(h_b), float(h_scale_b), _ptr(center),
                                  _ptr(out_old), float(alpha_old), float(beta), _ptr(out), _ptr(lse2), N, M, D,
                                  int(p), float(eps), _ptr(scratch), scratch.numel(), _stream(dev))
    _lib.check(rc, "b200ot_softmin_fwd")
    count_launches(3)
    return out, lse2


def softmin_grad_rows(eps, x, y, h_a, h_b, h_scale_b, lse2, grad_out, *, p=2, center=None):
    """grad_x of <grad_out, softmin(eps, (x, y), h)> with y, h constant (b200ot_softmin_bwd_x)."""
    x, y, h_a, h_b = _f32c(x, "x"), _f32c(y, "y"), _f32c(h_a, "h_a"), _f32c(h_b, "h_b")
    center, lse2, grad_out = _f32c(center, "center"), _f32c(lse2, "lse2"), _f32c(grad_out, "grad_out")
    _check_clouds(x, y, MAX_D_TC if (p & 0xFF) == 2 else MAX_D)
    N, D = x.shape
    M = y.shape[0]
    dev = x.device
    L = _lib.lib()
    with torch.cuda.device(dev):
        gx = torch.empty_like(x)
        nbytes = L.b200ot_softmin_scratch_bytes(N, M, D)
        scratch = _scratch(nbytes, dev, "softmin")
        rc = L.b200ot_softmin_bwd_x(_ptr(x), _ptr(y), _ptr(h_a), _ptr(h_b), float(h_scale_b), _ptr(center),
                                    _ptr(lse2), _ptr(grad_out), _ptr(gx), N, M, D, int(p), float(eps),
                                    _ptr(scratch), scratch.numel(), _stream(dev))
    _lib.check(rc, "b200ot_softmin_bwd_x")
    count_launches(3)
    return gx


class _Softmin(torch.autograd.Function):
    """softmin(eps, (x, y), h) with the reference's autograd contract: the gradient flows to the row
    cloud x only; y and h are treated as constants (they are ``.detach()``-ed at every call site of the
    reference: sinkhorn_samples.py:392-393, sinkhorn_divergence.py:616-623)."""

    @staticmethod
    def forward(ctx, x, y, h_a, h_b, h_scale_b, eps, p, center, scale_out):
        need_grad = ctx.needs_input_grad[0]
        out, lse2 = softmin_raw(eps, x, y, h_a, h_b, h_scale_b, p=p, center=center, beta=scale_out,
                                want_lse2=need_grad)
        if need_grad:
            ctx.save_for_backward(x, y, h_a, h_b if h_b is not None else h_a, center if center is not None else h_a,
                                  lse2)
            ctx.meta = (float(h_scale_b), float(eps), int(p), float(scale_out), h_b is not None, center is not None)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        x, y, h_a, h_b, center, lse2 = ctx.saved_tensors
        h_scale_b, eps, p, scale_out, has_hb, has_center = ctx.meta
        go = (grad_out * scale_out).contiguous()
        gx = softmin_grad_rows(eps, x, y, h_a, h_b if has_hb else None, h_scale_b, lse2, go, p=p,
                               center=center if has_center else None)
        return gx, None, None, None, None, None, None, None, None


def softmin(eps, x, y, h_a, h_b=None, h_scale_b=0.0, *, p=2, center=None, scale_out=1.0):
    """Differentiable (w.r.t. x) ``scale_out * softmin(eps, (x, y.detach()), (h_a + h_scale_b*h_b).detach())``."""
    return _Softmin.apply(x, y.detach(), h_a.detach(), None if h_b is None else h_b.detach(), h_scale_b, eps, p,
                          center, scale_out)


# ------------------------------------------------------------------------------------------------
# kernel convolutions
# ------------------------------------------------------------------------------------------------


def kind_id(kind):
    """Kernel name (tensorized convention) or an integer kind, possibly or-ed with KERNEL_UNCLAMPED."""
    return KERNEL_KINDS[kind] if isinstance(kind, str) else int(kind)


def kernel_conv_raw(kind, x, y, w, blur, *, center=None):
    """out_i = sum_j k(x_i, y_j) w_j, no autograd."""
    x, y, w, center = _f32c(x, "x"), _f32c(y, "y"), _f32c(w, "w"), _f32c(center, "center")
    _check_clouds(x, y, MAX_D_TC)
    N, D = x.shape
    M = y.shape[0]
    if w.numel() != M:
        raise ValueError("w must have one entry per column")
    dev = x.device
    L = _lib.lib()
    with torch.cuda.device(dev), nvtx_range(f"b200ot.kernel_conv kind={kind} N={N} M={M} D={D}"):
        out = torch.empty(N, dtype=torch.float32, device=dev)
        nbytes = L.b200ot_kernel_conv_scratch_bytes(N, M, D)
        scratch = _scratch(nbytes, dev, "conv")
        rc = L.b200ot_kernel_conv_fwd(_ptr(x), _ptr(y), _ptr(w), _ptr(center), _ptr(out), N, M, D,
                                      kind_id(kind), float(blur), _ptr(scratch), scratch.numel(), _stream(dev))
    _lib.check(rc, "b200ot_kernel_conv_fwd")
    count_launches(3)
    return out


def kernel_conv_grad_rows(kind, x, y, w, blur, grad_out, *, center=None):
    x, y, w, center = _f32c(x, "x"), _f32c(y, "y"), _f32c(w, "w"), _f32c(center, "center")
    grad_out = _f32c(grad_out, "grad_out")
    _check_clouds(x, y, MAX_D_TC)
    N, D = x.shape
    M = y.shape[0]
    dev = x.device
    L = _lib.lib()
    with torch.cuda.device(dev):
        gx = torch.empty_like(x)
        nbytes = L.b200ot_kernel_conv_scratch_bytes(N, M, D)
        scratch = _scratch(nbytes, dev, "conv")
        rc = L.b200ot_kernel_conv_bwd_x(_ptr(x), _ptr(y), _ptr(w), _ptr(center), _ptr(grad_out), _ptr(gx), N, M, D,
                                        kind_id(kind), float(blur), _ptr(scratch), scratch.numel(),
                                        _stream(dev))
    _lib.check(rc, "b200ot_kernel_conv_bwd_x")
    count_launches(3)
    return gx


def kernel_conv_value_and_grad_rows(kind, x, y, w, blur, *, center=None):
    """(out, grad_unit) with out_i = sum_j k(x_i, y_j) w_j and grad_unit[i] = sum_j w_j dk(x_i, y_j)/dx_i from ONE
    pass over the pairs (gaussian kernel; b200ot_kernel_conv_fwd_bwd_x).  No autograd."""
    x, y, w, center = _f32c(x, "x"), _f32c(y, "y"), _f32c(w, "w"), _f32c(center, "center")
    if (kind_id(kind) & 0xFF) != 0:
        raise ValueError("the one-pass value + row gradient exists for the gaussian kernel only")
    _check_clouds(x, y, MAX_D_TC)
    N, D = x.shape
    M = y.shape[0]
    if w.numel() != M:
        raise ValueError("w must have one entry per column")
    dev = x.device
    L = _lib.lib()
    with torch.cuda.device(dev), nvtx_range(f"b200ot.kernel_conv value+grad kind={kind} N={N} M={M} D={D}"):
        out = torch.empty(N, dtype=torch.float32, device=dev)
        gunit = torch.empty_like(x)
        nbytes = L.b200ot_kernel_conv_scratch_bytes(N, M, D)
        scratch = _scratch(nbytes, dev, "conv")
        rc = L.b200ot_kernel_conv_fwd_bwd_x(_ptr(x), _ptr(y), _ptr(w), _ptr(center), _ptr(out), _ptr(gunit), N, M, D,
                                            kind_id(kind), float(blur), _ptr(scratch), scratch.numel(), _stream(dev))
    _lib.check(rc, "b200ot_kernel_conv_fwd_bwd_x")
    count_launches(3)
    return out, gunit


# A gaussian matvec whose ROW cloud requires a gradient is evaluated by the row-gradient reduction, which accumulates
# sum_j w_j k_ij next to sum_j w_j k_ij y_j anyway: value and unit gradient come from one pass over the N x M pairs and
# backward() is an N x D elementwise product — 3 reductions instead of 5 for SamplesLoss("gaussian")(x, y) + grad w.r.t.
# x.  Measured on B200 (tools/ab_tc_route.py part D: BASELINE configs[2], N = M = 1e6, D = 64, forward + gradient):
# 2.64 s two-pass -> 1.92 s one-pass (1.72 s with the merged GEMM-2 instruction); N = M = 4e5, D = 3: 90 -> 53 ms per
# (value, gradient) pair of reductions.  The price: a forward whose result is never differentiated although x requires a
# gradient pays the (slower) gradient reduction, and (N, D) floats are kept until backward.
# B200OT_FUSED_CONV_GRAD=0 restores the two-pass evaluation.
FUSED_CONV_GRAD = _os.environ.get("B200OT_FUSED_CONV_GRAD", "1") == "1"


class _KernelConv(torch.autograd.Function):
    """out = K(x, y) @ w, differentiable w.r.t. x, y and w (kernels are symmetric, so the y- and
    w-gradients are the same reduction with the roles of the clouds swapped)."""

    @staticmethod
    def forward(ctx, x, y, w, kind, blur, center, fused):
        if fused:
            out, gunit = kernel_conv_value_and_grad_rows(kind, x, y, w, blur, center=center)
        else:
            out, gunit = kernel_conv_raw(kind, x, y, w, blur, center=center), None
        ctx.save_for_backward(x, y, w, center if center is not None else w, gunit if fused else w)
        ctx.meta = (kind, float(blur), center is not None, fused)
        return out

    @staticmethod
    def backward(ctx, go):
        x, y, w, center, gunit = ctx.saved_tensors
        kind, blur, has_center, fused = ctx.meta
        center = center if has_center else None
        go = go.contiguous()
        gx = gy = gw = None
        if ctx.needs_input_grad[0]:
            if fused:
                gx = go.unsqueeze(1) * gunit
            else:
                gx = kernel_conv_grad_rows(kind, x, y, w, blur, go, center=center)
        if ctx.needs_input_grad[1]:
            # d/dy_j sum_i go_i k(x_i, y_j) w_j = w_j * sum_i go_i dk(y_j, x_i)/dy_j
            gy = kernel_conv_grad_rows(kind, y, x, go, blur, w, center=center)
        if ctx.needs_input_grad[2]:
            gw = kernel_conv_raw(kind, y, x, go, blur, center=center)
        return gx, gy, gw, None, None, None, None


def kernel_conv(kind, x, y, w, blur, *, center=None):
    fused = (FUSED_CONV_GRAD and torch.is_grad_enabled() and x.requires_grad and (kind_id(kind) & 0xFF) == 0)
    return _KernelConv.apply(x, y, w, kind, blur, center, bool(fused))
