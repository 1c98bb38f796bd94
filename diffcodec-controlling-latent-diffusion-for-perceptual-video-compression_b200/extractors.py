"""The motion-compensation part of a bi-directional conditioning block (SURVEY.md section 8 f-1).

The reference's ``Bi_Dir_FeatureExtractor.forward`` (``controlnet/extractors.py:280-314``) does, per
pyramid scale: two occlusion masks, two soft splats with ``(1 - mask)``, a confidence fusion
(cat / clamp / sum / divide / two products / add) and a double-hole fill guarded by
``holes.any()`` -- a device->host sync four times per ControlNet forward. Its conv stacks are
cuDNN business and stay where they are; this module provides the rest as three fused calls with
no host sync:

    occ_fwd, occ_bwd = compute_mask(...)                (dcb_occlusion_mask, x2)
    warped, conf     = warper(feat, flow, mask=occ)     (dcb_splat_fwd with mask, x2)
    fused            = bidir_fuse(...)                  (dcb_bidir_fuse_fwd / _bwd)
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from .control_utils import FeatureWarperSoftsplat, compute_mask, resize_and_normalize_flow_batched, zero_module
from .softsplat import is_deterministic

__all__ = ["bidir_fuse", "bidirectional_warp_fuse", "bidirectional_block", "Bi_Dir_FeatureExtractor", "Bi_Dir_ResidueExtractor",
           "WarpExtractor", "ConvBlock"]


def _fuse_forward(A, B, conf_a, conf_b, occ_a, occ_b):
    assert A.is_cuda and A.dim() == 4 and A.shape == B.shape, "bidir_fuse expects two [N,C,H,W] CUDA tensors"
    dt = A.dtype
    if B.dtype != dt: B = B.to(dt)
    if conf_a.dtype != dt: conf_a = conf_a.to(dt)
    if conf_b.dtype != dt: conf_b = conf_b.to(dt)
    if occ_a is not None and (occ_a.dtype != dt or occ_b.dtype != dt):
        occ_a, occ_b = occ_a.to(dt), occ_b.to(dt)
    lib = _lib.lib()
    dev = A.device
    fused = torch.empty(A.shape, dtype=dt, device=dev)
    with _lib.on_device(dev):
        rc = lib.dcb_bidir_fuse_fwd(_lib.desc(A), _lib.desc(B), _lib.desc(conf_a), _lib.desc(conf_b),
                                    _lib.desc(occ_a), _lib.desc(occ_b), _lib.desc(fused), _lib.stream_ptr(dev))
    _lib.check(rc, "dcb_bidir_fuse_fwd")
    return fused, (A, B, conf_a, conf_b, occ_a, occ_b)


class _bidir_fuse_func(torch.autograd.Function):
    @staticmethod
    def forward(ctx, A, B, conf_a, conf_b, occ_a, occ_b):
        fused, (A, B, conf_a, conf_b, occ_a, occ_b) = _fuse_forward(A, B, conf_a, conf_b, occ_a, occ_b)
        ctx.has_occ = occ_a is not None
        ctx.save_for_backward(*([A, B, conf_a, conf_b] + ([occ_a, occ_b] if occ_a is not None else [])))
        return fused

    @staticmethod
    def backward(ctx, g):
        saved = ctx.saved_tensors
        A, B, conf_a, conf_b = saved[:4]
        occ_a, occ_b = (saved[4], saved[5]) if ctx.has_occ else (None, None)
        need = ctx.needs_input_grad
        lib = _lib.lib()
        dev = A.device
        gA = torch.empty_like(A, memory_format=torch.contiguous_format) if need[0] else None
        gB = torch.empty_like(A, memory_format=torch.contiguous_format) if need[1] else None
        gca = torch.empty(conf_a.shape, dtype=A.dtype, device=dev) if need[2] else None
        gcb = torch.empty(conf_a.shape, dtype=A.dtype, device=dev) if need[3] else None
        with _lib.on_device(dev):
            rc = lib.dcb_bidir_fuse_bwd(_lib.desc(g.to(A.dtype)), _lib.desc(A), _lib.desc(B), _lib.desc(conf_a),
                                        _lib.desc(conf_b), _lib.desc(occ_a), _lib.desc(occ_b), _lib.desc(gA),
                                        _lib.desc(gB), _lib.desc(gca), _lib.desc(gcb), _lib.stream_ptr(dev))
        _lib.check(rc, "dcb_bidir_fuse_bwd")
        return gA, gB, gca, gcb, None, None


def bidir_fuse(warped_a, warped_b, conf_a, conf_b, occ_a=None, occ_b=None):
    """``w = clamp(conf, 0) / (sum + 1e-6); fused = w0*A + w1*B``; where both are occluded
    (``occ_a + occ_b > 1.5``) ``0.5*(A + B)`` -- reference ``extractors.py:298-310`` -- in one kernel,
    differentiable w.r.t. both maps and both confidences, without the ``holes.any()`` host sync."""
    assert (occ_a is None) == (occ_b is None)
    if torch.is_grad_enabled() and any(t.requires_grad for t in (warped_a, warped_b, conf_a, conf_b)):
        return _bidir_fuse_func.apply(warped_a, warped_b, conf_a, conf_b, occ_a, occ_b)
    return _fuse_forward(warped_a, warped_b, conf_a, conf_b, occ_a, occ_b)[0]     # inference: no autograd.Function bookkeeping


def _block_sizes(n, c, h, w, dt):
    key = (n, c, h, w, dt)
    v = _block_ws.get(key)
    if v is None:
        lib = _lib.lib()
        v = _block_ws[key] = tuple(int(lib.dcb_bidir_block_workspace_bytes(n, c, h, w, dt, k)) for k in (0, 1, 2))
    return v


_block_ws: dict = {}
_lib._option_hooks.append(_block_ws.clear)


class _bidir_block_func(torch.autograd.Function):
    """The whole block -- both occlusion masks, both masked soft splats, confidence fusion, double-hole fill -- as ONE
    autograd node and ONE library call each way (dcb_bidir_block_fwd / the one-level dcb_bidir_pyramid_bwd), with the
    learned metric of the live consumer (gradients reach the features, the flows and, through the splat weights AND the
    fusion weights, the metric)."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)       # the splats run in fp32 (control_utils.py:61)
    def forward(ctx, first, last, flow_f, flow_b, metric_f, metric_b, holes):
        lib = _lib.lib()
        n, c, h, w = first.shape
        dev, dt = first.device, first.dtype
        need = any(ctx.needs_input_grad[:6])
        fused = torch.empty((n, c, h, w), dtype=dt, device=dev)
        saved = None
        if need:
            warped = torch.empty((2, n, c, h, w), dtype=dt, device=dev)
            planes = torch.empty((2, n, 1, h, w), dtype=torch.float32, device=dev)
            occ = torch.empty((2, n, 1, h, w), dtype=dt, device=dev)
            saved = (warped[0], warped[1], planes[0], planes[1], occ[0], occ[1])
        acc_b, scr_b, _ = _block_sizes(n, c, h, w, _lib._DTYPES[dt])
        stream = _lib.stream_ptr(dev)
        ws_acc = _lib.workspace(dev, acc_b, "acc", stream)
        ws_scr = None if need else _lib.workspace(dev, scr_b, "scratch", stream)
        D = _lib.desc
        with _lib.on_device(dev):
            rc = lib.dcb_bidir_block_fwd(D(first), D(last), D(flow_f), D(flow_b), D(metric_f), D(metric_b), D(fused),
                                         *([D(t) for t in saved] if need else [None] * 6),
                                         ws_acc.data_ptr(), ws_acc.numel(), None if need else ws_scr.data_ptr(), 0 if need else ws_scr.numel(),
                                         _lib.FLAG_WS_CLEAN, stream)
        if rc != 0:
            _lib.invalidate_acc(dev)
        _lib.check(rc, "dcb_bidir_block_fwd")
        ctx.holes = holes
        if need:
            ctx.save_for_backward(first, last, flow_f, flow_b, metric_f, metric_b, *saved)
        return fused

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, g):
        t = ctx.saved_tensors
        return tuple(_pyramid_backward([t[:6]], [t[6:]], [g], [ctx.needs_input_grad[:6]], 0)[0]) + (None,)


def _block_forward_nograd(first, last, flow_f, flow_b, metric_f, metric_b):
    """Inference path of the fused block: no autograd node, nothing saved, intermediate maps in library scratch."""
    lib = _lib.lib()
    n, c, h, w = first.shape
    dev, dt = first.device, first.dtype
    fused = torch.empty((n, c, h, w), dtype=dt, device=dev)
    acc_b, scr_b, _ = _block_sizes(n, c, h, w, _lib._DTYPES[dt])
    stream = _lib.stream_ptr(dev)
    ws_acc = _lib.workspace(dev, acc_b, "acc", stream)
    ws_scr = _lib.workspace(dev, scr_b, "scratch", stream)
    D = _lib.desc
    with _lib.on_device(dev):
        rc = lib.dcb_bidir_block_fwd(D(first), D(last), D(flow_f), D(flow_b), D(metric_f), D(metric_b), D(fused), None, None, None, None,
                                     None, None, ws_acc.data_ptr(), ws_acc.numel(), ws_scr.data_ptr(), ws_scr.numel(), _lib.FLAG_WS_CLEAN, stream)
    if rc != 0:
        _lib.invalidate_acc(dev)
    _lib.check(rc, "dcb_bidir_block_fwd")
    return fused


def bidirectional_block(first_features, last_features, flow_f, flow_b, metric_f=None, metric_b=None):
    """masks + both masked soft splats + confidence fusion + double-hole fill of ONE pyramid scale
    (``extractors.py:289-310``), given the two metric maps (``metric_net`` outputs, or None for a warper without one).
    One library call forward, one backward (two launches); no host sync. Gradients reach the features, the flows and the
    metrics; the occlusion masks carry none (``compute_mask`` thresholds, as in the reference)."""
    dt = first_features.dtype
    if metric_f is None:
        metric_f = torch.ones_like(flow_f[:, :1], dtype=dt)
    if metric_b is None:
        metric_b = torch.ones_like(flow_b[:, :1], dtype=dt)
    if is_deterministic():                                     # the deterministic form of the block is the one-level pyramid
        return bidirectional_pyramid([(first_features, last_features, flow_f, flow_b, metric_f, metric_b)])[0]
    needs_grad = torch.is_grad_enabled() and any(t.requires_grad for t in (first_features, last_features, flow_f, flow_b, metric_f, metric_b))
    if (not needs_grad and not torch.is_autocast_enabled("cuda") and dt in (torch.float32, torch.bfloat16, torch.float16)
            and last_features.dtype == dt and flow_f.dtype == dt and flow_b.dtype == dt and metric_f.dtype == dt and metric_b.dtype == dt):
        return _block_forward_nograd(first_features, last_features, flow_f, flow_b, metric_f, metric_b)
    cast = lambda t: t if t.dtype == dt else t.to(dt)
    return _bidir_block_func.apply(first_features, cast(last_features), cast(flow_f), cast(flow_b), cast(metric_f), cast(metric_b), True)


# -------------------------------------------------------------------------------------------------
# whole pyramids: every scale of one forward in one library call (csrc/pyramid.cu)
# -------------------------------------------------------------------------------------------------
def resample_batch(jobs):
    """Bilinear resampling of several tensors to several sizes in ONE launch (``dcb_resample_batch``).
    jobs: (src [N,C,H,W], (th, tw), align_corners, op, factor0, factor1[, dtype]) with op one of ``_lib.RESAMPLE_*``;
    returns the list of resampled tensors. No autograd (the pyramids resample inputs, not activations)."""
    packed, outs = [], []
    for job in jobs:
        src, (th, tw), align, op, f0, f1 = job[:6]
        dt = job[6] if len(job) > 6 else src.dtype
        dst = torch.empty((src.shape[0], src.shape[1], th, tw), dtype=dt, device=src.device)
        packed.append((src, dst, align, op, f0, f1)); outs.append(dst)
    if packed:
        dev = packed[0][0].device
        with _lib.on_device(dev):
            _lib.check(_lib.lib().dcb_resample_batch(_lib.pack_resample(packed), len(packed), _lib.stream_ptr(dev)), "dcb_resample_batch")
    return outs


_pyr_ws: dict = {}
_lib._option_hooks.append(_pyr_ws.clear)


def _pyramid_forward(levels, flags, want_saved, want_warped=False):
    """levels: per scale (first, last, flow_f, flow_b, metric_f | None, metric_b | None), one dtype. One dcb_bidir_pyramid_fwd
    call: two kernel launches for the whole pyramid, or under ``deterministic()`` the bit-reproducible sort-then-reduce form
    (11 launches). Returns (fused list, per-scale saved tensors or None)."""
    det = is_deterministic()
    lib = _lib.lib()
    dev, dt = levels[0][0].device, levels[0][0].dtype
    outs, fused, saved = [], [], []
    for first, *_ in levels:
        n, c, h, w = first.shape
        f = torch.empty((n, c, h, w), dtype=dt, device=dev)
        fused.append(f)
        if want_saved:
            warped = torch.empty((2, n, c, h, w), dtype=dt, device=dev)
            planes = torch.empty((2, n, 1, h, w), dtype=torch.float32, device=dev)
            occ = torch.empty((2, n, 1, h, w), dtype=dt, device=dev)
            sv = (warped[0], warped[1], planes[0], planes[1], occ[0], occ[1])
        elif want_warped:
            warped = torch.empty((2, n, c, h, w), dtype=dt, device=dev)
            sv = (warped[0], warped[1], None, None, None, None)
        else:
            sv = (None,) * 6
        saved.append(sv)
        outs.append((f,) + sv)
    stream = _lib.stream_ptr(dev)
    with _lib.on_device(dev):
        arr = _lib.pack_pyramid(levels, outs)
        key = (tuple(tuple(lv[0].shape) for lv in levels), dt, det)
        need = _pyr_ws.get(key)
        if need is None:
            query = lib.dcb_bidir_pyramid_det_workspace_bytes if det else lib.dcb_bidir_pyramid_workspace_bytes
            need = _pyr_ws[key] = int(query(arr, len(levels)))
        if det:
            ws = _lib.workspace(dev, need, "scratch", stream)
            flags |= _lib.FLAG_DETERMINISTIC
        else:
            ws = _lib.workspace(dev, need, "acc", stream)
            flags |= _lib.FLAG_WS_CLEAN
        rc = lib.dcb_bidir_pyramid_fwd(arr, len(levels), ws.data_ptr(), ws.numel(), flags, stream)
    if rc != 0 and not det:
        _lib.invalidate_acc(dev)
    _lib.check(rc, "dcb_bidir_pyramid_fwd")
    return fused, saved


def _pyramid_backward(levels, saved, grads, needs, flags):
    """ONE dcb_bidir_pyramid_bwd call (two kernel launches) for every scale that wants a gradient. levels: per scale (first,
    last, flow_f, flow_b, metric_f | None, metric_b | None); saved: per scale the six forward outputs; grads: grad_fused per
    scale; needs: per scale six flags in the order of `levels`. Returns per scale the six gradients (None where not wanted)."""
    res, ins, svs, outs = [], [], [], []
    for lv, sv, g, need in zip(levels, saved, grads, needs):
        if g is None or not any(need):
            res.append((None,) * 6)
            continue
        first = lv[0]
        n, c, h, w = first.shape
        gr = tuple(torch.empty((n, ch, h, w), dtype=first.dtype, device=first.device) if want else None
                   for ch, want in zip((c, c, 2, 2, 1, 1), need))
        ins.append((g.to(first.dtype),) + tuple(lv)); svs.append(sv); outs.append(gr); res.append(gr)
    if not ins:
        return res
    lib = _lib.lib()
    dev = ins[0][1].device
    stream = _lib.stream_ptr(dev)
    with _lib.on_device(dev):
        arr = _lib.pack_pyramid_bwd(ins, svs, outs)
        ws = _lib.workspace(dev, int(lib.dcb_bidir_pyramid_bwd_workspace_bytes(arr, len(ins))), "scratch", stream)
        rc = lib.dcb_bidir_pyramid_bwd(arr, len(ins), ws.data_ptr(), ws.numel(), flags, stream)
    _lib.check(rc, "dcb_bidir_pyramid_bwd")
    return res


class _bidir_pyramid_func(torch.autograd.Function):
    """All scales of a bi-directional conditioning pyramid as ONE autograd node: one library call forward, one backward (two
    launches each). Inputs: the holes flag, then per scale first, last, flow_f, flow_b, metric_f | None, metric_b | None."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)       # the splats run in fp32 (control_utils.py:61)
    def forward(ctx, holes, *tensors):
        levels = [tuple(tensors[i:i + 6]) for i in range(0, len(tensors), 6)]
        need = any(ctx.needs_input_grad[1:])
        ctx.flags = 0 if holes else _lib.PYRAMID_NO_HOLES
        fused, saved = _pyramid_forward(levels, ctx.flags, need)
        ctx.n_levels = len(levels)
        if need:
            flat = []
            for lv, sv in zip(levels, saved):
                flat += list(lv) + list(sv)
            ctx.save_for_backward(*flat)
        return tuple(fused)

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, *grads):
        t, L = ctx.saved_tensors, ctx.n_levels
        need = ctx.needs_input_grad[1:]
        res = _pyramid_backward([t[12 * l:12 * l + 6] for l in range(L)], [t[12 * l + 6:12 * l + 12] for l in range(L)], grads,
                                [need[6 * l:6 * l + 6] for l in range(L)], ctx.flags)
        return (None,) + tuple(x for r in res for x in r)


_PYRAMID_MAX_LEVELS = 4


def bidirectional_pyramid(levels, holes=True):
    """Every scale of ``Bi_Dir_FeatureExtractor.forward`` between the conv stacks (``extractors.py:282-310``) in one call:
    levels = [(first, last, flow_f, flow_b, metric_f | None, metric_b | None), ...] -> [fused, ...]. Two kernel launches
    for the whole pyramid each way, no host sync; gradients reach the features, the flows and the metrics (the occlusion
    masks carry none, as in the reference). ``holes=False``: the fusion without the double-hole fill, as
    ``Bi_Dir_ResidueExtractor`` (``extractors.py:193-199``). Under ``deterministic()`` the forward is bit-reproducible (in
    fp32 bit-identical to the composition of the deterministic single ops); the backward has no atomics either way."""
    levels = [tuple(lv) for lv in levels]
    if len(levels) > _PYRAMID_MAX_LEVELS:
        return bidirectional_pyramid(levels[:_PYRAMID_MAX_LEVELS], holes) + bidirectional_pyramid(levels[_PYRAMID_MAX_LEVELS:], holes)
    dt = levels[0][0].dtype
    grad = torch.is_grad_enabled() and any(t is not None and t.requires_grad for lv in levels for t in lv)
    plain = (not grad and not torch.is_autocast_enabled("cuda") and dt in (torch.float32, torch.bfloat16, torch.float16)
             and all(t is None or t.dtype == dt for lv in levels for t in lv))
    if plain:
        return _pyramid_forward(levels, 0 if holes else _lib.PYRAMID_NO_HOLES, False)[0]
    flat = []
    for first, last, ff, fb, mf, mb in levels:
        d = first.dtype
        cast = lambda t: t if t is None or t.dtype == d else t.to(d)
        flat += [first, cast(last), cast(ff), cast(fb), cast(mf), cast(mb)]
    return list(_bidir_pyramid_func.apply(holes, *flat))


def pyramid_conditioning(img1, img2, flow1, flow2, sizes=(128, 64, 32)):
    """The multi-scale conditioning loop of ``improv_experiments.ipynb`` cell 5 (SURVEY.md section 8, row f-4): per size,
    both frames resized (bilinear, align_corners=False), both flows resized and scaled by size / W, each frame soft-splatted
    by its flow with an all-ones metric, the two warps fused by ``soft_fuse`` with identity masks (cell 3). The reference runs
    ~30 eager kernels and 2 NVRTC lookups per size; here: one resampling launch for all 4 x len(sizes) resizes, then ONE
    pyramid call (two launches). Returns [(warped1, warped2, fused), ...] per size."""
    assert img1.is_cuda and img1.shape == img2.shape and flow1.shape == flow2.shape
    dt = img1.dtype
    out = []
    for s0 in range(0, len(sizes), _PYRAMID_MAX_LEVELS):
        chunk = sizes[s0:s0 + _PYRAMID_MAX_LEVELS]
        jobs = []
        for size in chunk:
            scale = float(size) / float(flow1.shape[-1])
            jobs += [(img1, (size, size), False, _lib.RESAMPLE_NONE, 1.0, 1.0), (img2, (size, size), False, _lib.RESAMPLE_NONE, 1.0, 1.0),
                     (flow1, (size, size), False, _lib.RESAMPLE_MUL, scale, scale, dt), (flow2, (size, size), False, _lib.RESAMPLE_MUL, scale, scale, dt)]
        r = resample_batch(jobs)
        levels = [(r[4 * i], r[4 * i + 1], r[4 * i + 2], r[4 * i + 3], None, None) for i in range(len(chunk))]
        fused, saved = _pyramid_forward(levels, _lib.PYRAMID_NO_MASKS, False, want_warped=True)
        out += [(sv[0], sv[1], f) for f, sv in zip(fused, saved)]
    return out


def _block_fusable(first, last, flow_f, flow_b):
    return first.is_cuda and first.shape == last.shape and first.dtype in (torch.float32, torch.bfloat16, torch.float16) and not is_deterministic()


def bidirectional_warp_fuse(first_features, last_features, flow_f, flow_b, warper):
    """The per-scale block of ``Bi_Dir_FeatureExtractor.forward`` between the conv stacks
    (``extractors.py:289-310``): masks, both warps, fusion. ``warper`` is a ``FeatureWarperSoftsplat``."""
    if _block_fusable(first_features, last_features, flow_f, flow_b):
        learn = getattr(warper, "with_learnable_metric", False)
        mf = warper.metric_net(first_features) if learn else None
        mb = warper.metric_net(last_features) if learn else None
        with torch.autocast(device_type="cuda", enabled=False):
            return bidirectional_block(first_features, last_features, flow_f, flow_b, mf, mb)
    occ_fwd = compute_mask(flow_f, flow_b)
    occ_bwd = compute_mask(flow_b, flow_f)
    warped_first, conf_fwd = warper(first_features, flow_f, mask=occ_fwd)
    warped_last, conf_bwd = warper(last_features, flow_b, mask=occ_bwd)
    return bidir_fuse(warped_first, warped_last, conf_fwd, conf_bwd, occ_fwd, occ_bwd)


# -------------------------------------------------------------------------------------------------
# Drop-in modules for ``controlnet/extractors.py``: same class names, constructor arguments, parameter names (checkpoints
# load with ``load_state_dict``) and forward signatures. The conv stacks are plain cuDNN modules and are only declared
# here so that the state_dict keys match; what changes is the motion-compensation part of ``forward``.
# -------------------------------------------------------------------------------------------------
def _silu_convs(*spec):
    """nn.Sequential of (Conv2d 3x3 pad 1, SiLU) pairs; spec entries are (c_in, c_out, stride)."""
    layers = []
    for cin, cout, stride in spec:
        layers += [nn.Conv2d(cin, cout, 3, padding=1, stride=stride), nn.SiLU()]
    return nn.Sequential(*layers)


class ConvBlock(nn.Module):                                   # extractors.py:14-24
    def __init__(self, in_ch, out_ch, stride=1):
        super().__init__()
        self.block = _silu_convs((in_ch, out_ch, stride), (out_ch, out_ch, 1))

    def forward(self, x):
        return self.block(x)


class WarpExtractor(nn.Module):                               # extractors.py:26-65 (no motion compensation inside)
    def __init__(self, inject_channels=[320, 320, 640, 1280]):
        super().__init__()
        self.inject_channels = inject_channels
        widths = (64, 320, 320, 640, 1280)
        for i, (cin, cout, stride) in enumerate(zip((3,) + widths[:-1], widths, (4, 2, 2, 2, 2)), start=1):
            setattr(self, f"enc{i}", ConvBlock(cin, cout, stride=stride))
        self.zero_convs = nn.ModuleList([zero_module(nn.Conv2d(c, inject_channels[i], 3, padding=1)) for i, c in enumerate(widths[1:])])

    def forward(self, x):
        feats = []
        for i in range(1, 6):
            x = getattr(self, f"enc{i}")(x)
            feats.append(x)
        return [zc(f) for zc, f in zip(self.zero_convs, feats[1:])]


class Bi_Dir_FeatureExtractor(nn.Module):
    """``controlnet/extractors.py:209-316``. Everything between the stride-2 convs and the zero convs of all four scales is
    ONE fused call each way (``bidirectional_pyramid``, two launches forward and two backward): no ``holes.any()`` host
    sync. Flows that carry a gradient receive it through the same call."""

    def __init__(self, inject_channels):
        super().__init__()
        self.inject = inject_channels
        self.split_res = [int(i / 2) for i in self.inject]
        pre = ((3, 16, 1), (16, 32, 2), (32, 32, 1), (32, 64, 2), (64, 64, 1))
        self.first_pre_extractor = _silu_convs(*pre)
        self.last_pre_extractor = _silu_convs(*pre)
        self.wrapper = nn.ModuleList([FeatureWarperSoftsplat(with_learnable_metric=True, in_channels=c) for c in self.split_res])
        chain = [64] + self.split_res
        self.extractors_first = nn.ModuleList([_silu_convs((chain[i], chain[i + 1], 2)) for i in range(4)])
        self.extractors_last = nn.ModuleList([_silu_convs((chain[i], chain[i + 1], 2)) for i in range(4)])
        self.zero_convs = nn.ModuleList([zero_module(nn.Conv2d(c // 2, c, 3, padding=1)) for c in inject_channels])

    def forward(self, local_conditions, flow):
        first_features = self.first_pre_extractor(local_conditions[:, 3:])      # extractors.py:266-272
        last_features = self.last_pre_extractor(local_conditions[:, :3])
        flow_fwd, flow_bwd = flow[:, :2], flow[:, 2:]
        flow_res = (64, 32, 16, 8)                                               # extractors.py:278
        # Under deterministic() only fp32 takes the pyramid: the 16-bit composition thresholds masks computed from 16-bit warps,
        # and the deterministic bits it gives today are kept.
        fp32 = flow.dtype == torch.float32 and first_features.dtype == torch.float32
        whole = first_features.is_cuda and flow.dtype in (torch.float32, torch.bfloat16, torch.float16) and (fp32 or not is_deterministic())
        if not whole:                                                            # what the pyramid does not take: scale by scale
            outs = []
            for idx, res in enumerate(flow_res):
                first_features = self.extractors_first[idx](first_features)
                last_features = self.extractors_last[idx](last_features)
                flow_f = resize_and_normalize_flow_batched(flow_fwd, res, res)
                flow_b = resize_and_normalize_flow_batched(flow_bwd, res, res)
                fused = bidirectional_warp_fuse(first_features, last_features, flow_f, flow_b, self.wrapper[idx])
                outs.append(self.zero_convs[idx](fused))
            return outs
        # The conv chains of the two frames do not depend on the fused maps, so they run first; then all eight flow resizes are
        # one launch (resize_and_normalize_flow_batched, control_utils.py:74-97: divide by ((w - 1) / 2, (h - 1) / 2)) and the
        # motion compensation of all four scales is one call (two launches) instead of 16 splats + 4 host syncs.
        feats = []
        for idx in range(len(flow_res)):
            first_features = self.extractors_first[idx](first_features)
            last_features = self.extractors_last[idx](last_features)
            feats.append((first_features, last_features))
        if torch.is_grad_enabled() and flow.requires_grad:                      # differentiable resizes (dcb_resample_batch has no backward)
            flows = [resize_and_normalize_flow_batched(fl, res, res) for res in flow_res for fl in (flow_fwd, flow_bwd)]
        else:
            with torch.no_grad():
                jobs = []
                for (f, _), res in zip(feats, flow_res):
                    dt = torch.float32 if (torch.is_autocast_enabled("cuda") or f.dtype not in (torch.float32, torch.bfloat16, torch.float16)) else f.dtype
                    for fl in (flow_fwd, flow_bwd):
                        jobs.append((fl, (res, res), False, _lib.RESAMPLE_DIV, (res - 1) / 2.0, (res - 1) / 2.0, dt))
                flows = resample_batch(jobs)
        levels = []
        for idx, (f, l) in enumerate(feats):
            learn = getattr(self.wrapper[idx], "with_learnable_metric", False)
            mf = self.wrapper[idx].metric_net(f) if learn else None
            mb = self.wrapper[idx].metric_net(l) if learn else None
            levels.append((f, l, flows[2 * idx], flows[2 * idx + 1], mf, mb))
        with torch.autocast(device_type="cuda", enabled=False):
            fused = bidirectional_pyramid(levels)
        return [zc(x) for zc, x in zip(self.zero_convs, fused)]


class Bi_Dir_ResidueExtractor(nn.Module):
    """``controlnet/extractors.py:67-205``. The flows pass through learned refiners here and carry a gradient; the motion
    compensation of all four scales (masks, both splats, fusion without the hole branch, :193-199) is ONE
    ``bidirectional_pyramid(..., holes=False)`` call each way, whose backward reaches the refiners through the flows."""

    def __init__(self, inject_channels):
        super().__init__()
        self.inject = inject_channels
        self.split_res = [int(i // 2) for i in inject_channels]
        c = self.split_res
        pre = ((3, 32, 1), (32, 64, 2), (64, 64, 2))
        self.prev_pre = _silu_convs(*pre)
        self.next_pre = _silu_convs(*pre)
        chain = [64] + c
        self.prev_pyramids = nn.ModuleList([_silu_convs((chain[i], chain[i + 1], 2)) for i in range(4)])
        self.next_pyramids = nn.ModuleList([_silu_convs((chain[i], chain[i + 1], 2)) for i in range(4)])
        self.flow_refiners = nn.ModuleList([nn.Conv2d(2, 2, kernel_size=3, padding=1, groups=2) for _ in range(4)])
        self.flow_feature_encoders = nn.ModuleList([nn.Conv2d(2, w, 3, padding=1) for w in (16, 16, 32, 32)])
        self.warpers = nn.ModuleList([FeatureWarperSoftsplat(with_learnable_metric=True, in_channels=ci) for ci in c])
        self.zero_convs = nn.ModuleList([zero_module(nn.Conv2d(ci, inject_channels[i], kernel_size=3, padding=1)) for i, ci in enumerate(c)])
        self.resolutions = [64, 32, 16, 8]

    def forward(self, prev_frame, next_frame, flow_fwd, flow_bwd, masks=None):
        B, _, H, W = prev_frame.shape
        assert H == 512 and W == 512, "expects 512x512 inputs"                   # extractors.py:157
        x_prev, x_next = self.prev_pre(prev_frame), self.next_pre(next_frame)
        prev_feats, next_feats = [], []
        for enc_prev, enc_next in zip(self.prev_pyramids, self.next_pyramids):
            x_prev, x_next = enc_prev(x_prev), enc_next(x_next)
            prev_feats.append(x_prev); next_feats.append(x_next)
        flows = []
        for i, res in enumerate(self.resolutions):
            factor = H // res                                                    # extractors.py:181-183: resize, then divide by the scale factor
            flow_f = self.flow_refiners[i](F.interpolate(flow_fwd, size=(res, res), mode="bilinear", align_corners=False) / factor)
            flow_b = self.flow_refiners[i](F.interpolate(flow_bwd, size=(res, res), mode="bilinear", align_corners=False) / factor)
            flows.append((flow_f, flow_b))
        fp32 = flows[0][0].dtype == torch.float32 and prev_feats[0].dtype == torch.float32     # deterministic(): as Bi_Dir_FeatureExtractor
        if not (prev_frame.is_cuda and flow_fwd.dtype in (torch.float32, torch.bfloat16, torch.float16) and (fp32 or not is_deterministic())):
            outs = []                                                            # what the pyramid does not take: scale by scale
            for i, (flow_f, flow_b) in enumerate(flows):
                occ_f, occ_b = compute_mask(flow_f, flow_b), compute_mask(flow_b, flow_f)
                warped_prev, conf_prev = self.warpers[i](prev_feats[i], flow_f, mask=occ_f)
                warped_next, conf_next = self.warpers[i](next_feats[i], flow_b, mask=occ_b)
                outs.append(self.zero_convs[i](bidir_fuse(warped_prev, warped_next, conf_prev, conf_next)))
            return outs
        # no refined flow or metric depends on a splat: all of them first, then the four scales in one call
        levels = [(prev_feats[i], next_feats[i], flow_f, flow_b, self.warpers[i].metric_net(prev_feats[i]), self.warpers[i].metric_net(next_feats[i]))
                  for i, (flow_f, flow_b) in enumerate(flows)]
        with torch.autocast(device_type="cuda", enabled=False):
            fused = bidirectional_pyramid(levels, holes=False)
        return [zc(x) for zc, x in zip(self.zero_convs, fused)]
