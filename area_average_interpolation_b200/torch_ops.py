"""Differentiable resampling of CUDA tensors: the forward of ``aai_run_device_batch`` and its transpose
``aai_run_device_adjoint`` as a ``torch.autograd.Function``.

Tensors stay in device memory and every call is enqueued on ``torch.cuda.current_stream(device)`` without a
synchronisation.  Images are ``[H, W]``, ``[N, H, W]`` or ``[N, H, W, C]`` with C = 1..4 interleaved channels (note: the
numpy operator ``AreaAverageInterpolation`` takes a single ``[h, w, c]`` image instead; here a rank-3 tensor is a stack).
A stack of N images is one kernel launch.  There is no CPU fallback: a CPU tensor raises.
"""
from __future__ import annotations

import torch

from . import (AAI_OK, ARITH_F64, ERR_ARGUMENT, MODE_AREA_AVERAGE, AaiError, Plan, run_device_adjoint,
               run_device_batch, status_string, tensor_image)

_CANVAS_DTYPE = {torch.float64: torch.float64, torch.float32: torch.float32, torch.uint8: torch.float32,
                 torch.uint16: torch.float32}


def _check_plan(plan: Plan, who: str) -> None:
    if not isinstance(plan, Plan):
        raise TypeError(f"{who}: plan must be an area_average_interpolation_b200.Plan (make_plan)")
    if plan.status != AAI_OK:
        raise AaiError(plan.status, f"{who}: the plan is not valid: {status_string(plan.status)}")


def _check_tensor(t, who: str, dtypes) -> None:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{who}: expected a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise RuntimeError(f"{who}: the tensor is on {t.device}; this library runs on CUDA devices only and has no CPU "
                           "fallback")
    if t.dtype not in dtypes:
        raise TypeError(f"{who}: unsupported dtype {t.dtype}; expected one of {', '.join(str(d) for d in dtypes)}")
    if t.dim() not in (2, 3, 4) or (t.dim() == 4 and not 1 <= t.shape[3] <= 4):
        raise ValueError(f"{who}: expected [H, W], [N, H, W] or [N, H, W, C] with C = 1..4, got {tuple(t.shape)}")


def _as_stack(t):
    """[N, H, W, C] view of a [H, W] / [N, H, W] / [N, H, W, C] tensor."""
    if t.dim() == 2:
        return t[None, :, :, None]
    if t.dim() == 3:
        return t[..., None]
    return t


def _dense(t):
    """Dense rows, as the library needs them (uint16 goes through its int16 view: torch has few uint16 CUDA kernels)."""
    if t.is_contiguous():
        return t
    if t.dtype == torch.uint16:
        return t.view(torch.int16).contiguous().view(torch.uint16)
    return t.contiguous()


def _images(stack):
    """One aai_image per image of a dense [N, H, W, C] tensor (a contiguous stack: equally strided)."""
    return [tensor_image(stack[k, :, :, 0] if stack.shape[3] == 1 else stack[k]) for k in range(stack.shape[0])]


def _out_shape(rank: int, n: int, h: int, w: int, c: int):
    return (h, w) if rank == 2 else (n, h, w) if rank == 3 else (n, h, w, c)


def _forward(src, plan: Plan, mode: int, arith: int):
    stack = _as_stack(_dense(src))
    n, h, w, c = stack.shape
    if (w, h) != (plan.src_w, plan.src_h):
        raise AaiError(ERR_ARGUMENT, f"resample: the source is {w}x{h}, the plan expects {plan.src_w}x{plan.src_h}")
    out = torch.empty((n, plan.dst_h, plan.dst_w, c), dtype=_CANVAS_DTYPE[src.dtype], device=src.device)
    if n:
        with torch.cuda.device(src.device):
            run_device_batch(plan, _images(stack), _images(out), mode=mode, arith=arith, device=src.device.index,
                             stream=torch.cuda.current_stream(src.device).cuda_stream)
    return out.view(_out_shape(src.dim(), n, plan.dst_h, plan.dst_w, c))


def _adjoint(canvas, plan: Plan, mode: int):
    stack = _as_stack(_dense(canvas))
    n, h, w, c = stack.shape
    if (w, h) != (plan.dst_w, plan.dst_h):
        raise AaiError(ERR_ARGUMENT, f"resample_adjoint: the canvas is {w}x{h}, the plan gives {plan.dst_w}x{plan.dst_h}")
    out = torch.empty((n, plan.src_h, plan.src_w, c), dtype=canvas.dtype, device=canvas.device)
    if n:
        with torch.cuda.device(canvas.device):
            run_device_adjoint(plan, _images(stack), _images(out), mode=mode, device=canvas.device.index,
                               stream=torch.cuda.current_stream(canvas.device).cuda_stream)
    return out.view(_out_shape(canvas.dim(), n, plan.src_h, plan.src_w, c))


class _Resample(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src, plan, mode, arith):
        ctx.plan, ctx.mode = Plan.from_buffer_copy(plan), mode  # a copy: the caller may reuse its Plan before backward
        return _forward(src, plan, mode, arith)

    @staticmethod
    def backward(ctx, grad):
        return _ResampleAdjoint.apply(grad, ctx.plan, ctx.mode), None, None, None


class _ResampleAdjoint(torch.autograd.Function):
    @staticmethod
    def forward(ctx, canvas, plan, mode):
        ctx.plan, ctx.mode = Plan.from_buffer_copy(plan), mode
        return _adjoint(canvas, plan, mode)

    @staticmethod
    def backward(ctx, grad):
        # the transpose of the adjoint is the forward (FP64 arithmetic: the adjoint's weights)
        return _Resample.apply(grad, ctx.plan, ctx.mode, ARITH_F64), None, None


def resample(src, plan: Plan, mode: int = MODE_AREA_AVERAGE, arith: int = ARITH_F64):
    """Resample CUDA tensor ``src`` with ``plan`` (``make_plan``; its ``src_w`` x ``src_h`` must be the image size).

    ``src``: ``[H, W]``, ``[N, H, W]`` or ``[N, H, W, C]`` (C = 1..4 interleaved channels; the numpy operator's
    ``[h, w, c]`` is a single image, here rank 3 is a stack).  float64 gives a float64 canvas; float32, uint8 and uint16
    give a float32 canvas.  The result has the rank of ``src`` and lives on its device; the call is enqueued on the
    current stream of that device and does not synchronise.

    Differentiable with respect to float32 / float64 ``src``: the backward is ``resample_adjoint`` in the same mode,
    itself differentiable (its derivative is this forward), so higher derivatives work.  The adjoint uses the FP64
    forward's weights: under ``ARITH_F32`` the forward differs from them by its FP32 tolerance, so its gradient is exact
    only to that tolerance.  uint8 / uint16 sources are forward only.  There are no gradients with respect to the plan
    (angle, resolution, isocentre): the reference's shape quirk makes the weights discontinuous in them.
    """
    _check_tensor(src, "resample", tuple(_CANVAS_DTYPE))
    _check_plan(plan, "resample")
    if src.dtype in (torch.float32, torch.float64):
        return _Resample.apply(src, plan, int(mode), int(arith))
    return _forward(src, plan, int(mode), int(arith))


def resample_adjoint(canvas, plan: Plan, mode: int = MODE_AREA_AVERAGE):
    """Transpose of ``resample`` (FP64 weights): spreads each canvas value over the source pixels its footprint covers,
    with the operator's own weights divided by the footprint's total weight -- the back-projection of a canvas-grid
    result onto the source grid.  ``resample_adjoint(ones)`` is the coverage of each source pixel.

    ``canvas``: float32 / float64 CUDA tensor ``[dst_h, dst_w]``, ``[N, dst_h, dst_w]`` or ``[N, dst_h, dst_w, C]``;
    the result has the same rank, dtype and device, with the source size of ``plan``.  Enqueued on the current stream,
    no synchronisation; differentiable (its derivative is the FP64 forward)."""
    _check_tensor(canvas, "resample_adjoint", (torch.float32, torch.float64))
    _check_plan(plan, "resample_adjoint")
    return _ResampleAdjoint.apply(canvas, plan, int(mode))


__all__ = ["resample", "resample_adjoint"]
