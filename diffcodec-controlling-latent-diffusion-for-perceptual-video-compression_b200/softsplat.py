"""Drop-in replacement for the reference's ``controlnet/softsplat.py``.

Same public surface -- ``softsplat(tenIn, tenFlow, tenMetric, strMode)`` (reference
``controlnet/softsplat.py:232-274``) and ``softsplat_func.apply(tenIn, tenFlow)``
(``:277-528``) -- same asserts, same autograd and AMP behaviour, output NCHW-contiguous in the
dtype of the (cast) input. What is different is everything underneath: no CuPy, no NVRTC, no
per-shape recompilation, no eager pre/post ops. One call is one pass through the precompiled
sm_100a library behind ``include/diffcodec_b200.h``:

    forward  = dcb_splat_fwd   (scatter with in-register pre-op + fused normalise epilogue)
    backward = dcb_splat_bwd   (one gather pass -> gradIn, gradFlow, gradMetric)

There is no CPU path (the reference has none either, ``softsplat.py:347-348``) and no fallback.

Extensions over the reference (all opt-in, defaults reproduce the reference):
  * bfloat16 tensors (the reference asserts on them, ``softsplat.py:105-107``): inputs bf16,
    positions / weights / accumulation fp32, one rounding at the output;
  * float16 tensors (the reference's kernel names ``half`` but cannot compile it): the same rule
    as bf16 -- loads widened to fp32, fp32 arithmetic, one ``__float2half_rn`` at each store; a
    value beyond the fp16 range becomes +-inf, as a torch fp16 op gives;
  * ``deterministic(True)``: bit-reproducible sort-then-reduce forward.
"""
from __future__ import annotations

import contextlib
import os
import threading

import torch

from . import _lib

__all__ = ["softsplat", "softsplat_func", "deterministic", "is_deterministic"]

_MODES = {"sum": _lib.MODE_SUM, "avg": _lib.MODE_AVG, "linear": _lib.MODE_LINEAR, "soft": _lib.MODE_SOFT}
_EPS = {"addeps": _lib.EPS_ADD, "zeroeps": _lib.EPS_ZERO, "clipeps": _lib.EPS_CLIP}

_state = threading.local()
_ws_sizes: dict = {}
_lib._option_hooks.append(_ws_sizes.clear)


def is_deterministic() -> bool:
    return getattr(_state, "det", os.environ.get("DCB_DETERMINISTIC", "0") == "1")


@contextlib.contextmanager
def deterministic(enabled: bool = True):
    """Within the block, forward splats use the bit-exact sort-then-reduce kernels: ``softsplat``, ``compute_mask``, the
    warpers, and the conditioning pyramids (``bidirectional_pyramid``, ``pyramid_conditioning``, ``bidirectional_block``, the
    fp32 extractors) and, in fp32, the conditioning recipes (``residual_conditioning``, ``residual_conditioning_bidir``), which
    keep their single library call in its deterministic form. The backward kernels use no atomics."""
    prev = is_deterministic()
    _state.det = bool(enabled)
    try:
        yield
    finally:
        _state.det = prev


def _acc_dtype(dtype: torch.dtype) -> torch.dtype:
    return torch.float64 if dtype == torch.float64 else torch.float32


def _check_inputs(tenIn, tenFlow):
    assert tenIn.dim() == 4 and tenFlow.dim() == 4, "softsplat expects NCHW tensors"
    assert tenFlow.shape[1] == 2, "tenFlow must have two channels"                      # softsplat.py:296
    assert tenFlow.shape[0] == tenIn.shape[0] and tenFlow.shape[2:] == tenIn.shape[2:], "tenFlow/tenIn shapes differ"
    assert tenIn.is_cuda and tenFlow.is_cuda, "softsplat has no CPU path (reference: softsplat.py:347-348)"


def _match_flow(tenIn, tenFlow):
    # the reference compiles ONE element type into the kernel; a bf16 / fp16 tensor may keep an fp32 flow
    if tenFlow.dtype == tenIn.dtype or (tenIn.dtype in (torch.bfloat16, torch.float16) and tenFlow.dtype == torch.float32):
        return tenFlow
    return tenFlow.to(tenIn.dtype)


def _forward(tenIn, tenFlow, tenMetric, mask, mode: int, eps: int, det: bool, want_norm: bool):
    lib = _lib.lib()
    n, c, h, w = tenIn.shape
    dev = tenIn.device
    out = torch.empty((n, c, h, w), dtype=tenIn.dtype, device=dev)
    norm = None
    if want_norm and mode != _lib.MODE_SUM:
        norm = torch.empty((n, 1, h, w), dtype=_acc_dtype(tenIn.dtype), device=dev)
    flags = _lib.FLAG_DETERMINISTIC if det else 0
    dt = _lib._DTYPES.get(tenIn.dtype)
    if dt is None:
        raise ValueError(f"softsplat: unsupported dtype {tenIn.dtype} (float32, bfloat16, float16, float64)")
    key = (n, c, h, w, dt, mode, flags)
    need = _ws_sizes.get(key)
    if need is None:
        need = _ws_sizes[key] = lib.dcb_splat_fwd_workspace_bytes(n, c, h, w, dt, mode, flags)
    stream = _lib.stream_ptr(dev)
    ws, ws_ptr = None, None
    if need > 0:
        if det or _lib.fwd_is_scratch(n, c, h, w, dt, mode, flags):
            ws = _lib.workspace(dev, need, "scratch", stream)
        else:
            ws = _lib.workspace(dev, need, "acc", stream)
            flags |= _lib.FLAG_WS_CLEAN
        ws_ptr = ws.data_ptr()
    with _lib.on_device(dev):
        rc = lib.dcb_splat_fwd(_lib.desc(tenIn), _lib.desc(tenFlow), _lib.desc(tenMetric), _lib.desc(out),
                               _lib.desc(norm), _lib.desc(mask), ws_ptr, ws.numel() if ws is not None else 0,
                               mode, eps, flags, stream)
    if rc != 0:
        _lib.invalidate_acc(dev)
    _lib.check(rc, "dcb_splat_fwd")
    return out, norm


def _backward(gout, tenIn, tenFlow, tenMetric, out, norm, mask, mode: int, eps: int, need):
    lib = _lib.lib()
    n, c, h, w = tenIn.shape
    dev = tenIn.device
    gin = torch.empty_like(tenIn, memory_format=torch.contiguous_format) if need[0] else None
    gflow = torch.empty((n, 2, h, w), dtype=tenFlow.dtype, device=dev) if need[1] else None
    gmetric = torch.empty((n, 1, h, w), dtype=tenIn.dtype, device=dev) if (need[2] and tenMetric is not None) else None
    nbytes = lib.dcb_splat_bwd_workspace_bytes(n, c, h, w, _lib._DTYPES[tenIn.dtype], mode, 0)
    ws = _lib.workspace(dev, nbytes, "scratch") if (mode != _lib.MODE_SUM and nbytes > 0) else None
    with _lib.on_device(dev):
        rc = lib.dcb_splat_bwd(_lib.desc(gout), _lib.desc(tenIn), _lib.desc(tenFlow), _lib.desc(tenMetric),
                               _lib.desc(out), _lib.desc(norm), _lib.desc(mask), _lib.desc(gin), _lib.desc(gflow),
                               _lib.desc(gmetric), ws.data_ptr() if ws is not None else None,
                               ws.numel() if ws is not None else 0, mode, eps, 0, _lib.stream_ptr(dev))
    _lib.check(rc, "dcb_splat_bwd")
    return gin, gflow, gmetric


class softsplat_func(torch.autograd.Function):
    """``softsplat_func.apply(tenIn, tenFlow)``: plain summation splat (reference ``softsplat.py:277-528``)."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)      # softsplat.py:279
    def forward(ctx, tenIn, tenFlow):
        _check_inputs(tenIn, tenFlow)
        tenFlow = _match_flow(tenIn, tenFlow)
        out, _ = _forward(tenIn, tenFlow, None, None, _lib.MODE_SUM, _lib.EPS_ADD, is_deterministic(), False)
        ctx.save_for_backward(tenIn, tenFlow)                                  # softsplat.py:352
        return out

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")                                  # softsplat.py:358
    def backward(ctx, tenOutgrad):
        tenIn, tenFlow = ctx.saved_tensors
        assert tenOutgrad.is_cuda                                              # softsplat.py:362
        gin, gflow, _ = _backward(tenOutgrad, tenIn, tenFlow, None, None, None, None, _lib.MODE_SUM, _lib.EPS_ADD,
                                  (ctx.needs_input_grad[0], ctx.needs_input_grad[1], False))
        return gin, gflow


class _splat_mode_func(torch.autograd.Function):
    """avg / linear / soft with the pre/post ops fused into the kernels (and their closed-form backward)."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, tenIn, tenFlow, tenMetric, mask, mode, eps):
        _check_inputs(tenIn, tenFlow)
        tenFlow = _match_flow(tenIn, tenFlow)
        if tenMetric is not None:
            assert tenMetric.shape == (tenIn.shape[0], 1, tenIn.shape[2], tenIn.shape[3]), "tenMetric must be [N,1,H,W]"
            if tenMetric.dtype != tenIn.dtype:
                tenMetric = tenMetric.to(tenIn.dtype)
        if mask is not None and mask.dtype != tenIn.dtype:
            mask = mask.to(tenIn.dtype)
        needs_grad = any(ctx.needs_input_grad[:3])
        out, norm = _forward(tenIn, tenFlow, tenMetric, mask, mode, eps, is_deterministic(), needs_grad)
        ctx.mode, ctx.eps = mode, eps
        ctx.has_metric, ctx.has_mask = tenMetric is not None, mask is not None
        if needs_grad:
            saved = [tenIn, tenFlow, out, norm]
            if tenMetric is not None:
                saved.append(tenMetric)
            if mask is not None:
                saved.append(mask)
            ctx.save_for_backward(*saved)
        return out

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, tenOutgrad):
        saved = list(ctx.saved_tensors)
        tenIn, tenFlow, out, norm = saved[:4]
        rest = saved[4:]
        tenMetric = rest.pop(0) if ctx.has_metric else None
        mask = rest.pop(0) if ctx.has_mask else None
        gin, gflow, gmetric = _backward(tenOutgrad, tenIn, tenFlow, tenMetric, out, norm, mask, ctx.mode, ctx.eps,
                                        ctx.needs_input_grad[:3])
        return gin, gflow, gmetric, None, None, None


def _needs_autograd(*tensors) -> bool:
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


def _splat_normalised(tenIn, tenFlow, tenMetric, mode: int, eps: int, mask=None):
    if _needs_autograd(tenIn, tenFlow, tenMetric) or torch.is_autocast_enabled("cuda"):
        return _splat_mode_func.apply(tenIn, tenFlow, tenMetric, mask, mode, eps)
    # inference fast path: same kernels, no autograd.Function / custom_fwd bookkeeping (~15 us per call)
    _check_inputs(tenIn, tenFlow)
    tenFlow = _match_flow(tenIn, tenFlow)
    if tenMetric is not None:
        assert tenMetric.shape == (tenIn.shape[0], 1, tenIn.shape[2], tenIn.shape[3]), "tenMetric must be [N,1,H,W]"
        if tenMetric.dtype != tenIn.dtype:
            tenMetric = tenMetric.to(tenIn.dtype)
    if mask is not None and mask.dtype != tenIn.dtype:
        mask = mask.to(tenIn.dtype)
    return _forward(tenIn, tenFlow, tenMetric, mask, mode, eps, is_deterministic(), False)[0]


def softsplat(tenIn: torch.Tensor, tenFlow: torch.Tensor, tenMetric: torch.Tensor, strMode: str):
    """Forward-splat ``tenIn`` along ``tenFlow`` (reference ``controlnet/softsplat.py:232-274``).

    strMode: ``sum`` | ``avg`` | ``linear[-addeps|-zeroeps|-clipeps]`` | ``soft[-...]``.
    """
    parts = strMode.split("-")
    assert parts[0] in ["sum", "avg", "linear", "soft"]                        # softsplat.py:233
    if strMode == "sum": assert tenMetric is None                              # softsplat.py:235
    if strMode == "avg": assert tenMetric is None                              # softsplat.py:236
    if parts[0] == "linear": assert tenMetric is not None                      # softsplat.py:237
    if parts[0] == "soft": assert tenMetric is not None                        # softsplat.py:238

    if strMode == "sum":
        if _needs_autograd(tenIn, tenFlow) or torch.is_autocast_enabled("cuda"):
            return softsplat_func.apply(tenIn, tenFlow)
        _check_inputs(tenIn, tenFlow)
        return _forward(tenIn, _match_flow(tenIn, tenFlow), None, None, _lib.MODE_SUM, _lib.EPS_ADD, is_deterministic(), False)[0]

    if parts[0] in ("sum", "avg") and strMode != parts[0]:
        # Reference quirk kept on purpose: 'avg-<eps>' / 'sum-<eps>' fail the exact-match tests of
        # softsplat.py:240, so nothing is appended, and ('avg-*' only, :253) the LAST input channel
        # is used as the normaliser. Composed from the sum splat so that values and gradients are
        # what the reference yields.
        tenOut = softsplat_func.apply(tenIn, tenFlow)
        if parts[0] == "sum":
            return tenOut
        tenNormalize = tenOut[:, -1:, :, :]
        if len(parts) == 1 or parts[1] == "addeps":
            tenNormalize = tenNormalize + 0.0000001
        elif parts[1] == "zeroeps":
            tenNormalize = torch.where(tenNormalize == 0.0, torch.ones_like(tenNormalize), tenNormalize)
        elif parts[1] == "clipeps":
            tenNormalize = tenNormalize.clip(0.0000001, None)
        return tenOut[:, :-1, :, :] / tenNormalize

    # eps rule: no suffix behaves as addeps; an unknown suffix leaves the normaliser untouched in the
    # reference (softsplat.py:256-268 has no else branch) -- we refuse it instead of dividing by 0
    eps = _EPS.get(parts[1]) if len(parts) > 1 else _lib.EPS_ADD
    assert eps is not None, f"unknown normaliser rule in strMode={strMode!r}"
    return _splat_normalised(tenIn, tenFlow, tenMetric, _MODES[parts[0]], eps)
