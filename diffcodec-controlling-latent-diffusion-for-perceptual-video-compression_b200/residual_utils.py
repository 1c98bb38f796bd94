"""Conditioning builders: the arithmetic of the reference's ``ResidueDataset.__getitem__``
(``controlnet/dataset.py:214-276``) and ``WarpingDatasetWrapper.__getitem__``
(``controlnet/residual_utils.py:141-211``), batched and fused.

Per sample the reference issues 4 ``softsplat`` calls (two of them identical, SURVEY.md App. B-6),
two norms / compares, a cat / clamp / sum / div fusion and a subtraction: ~45 launches for a
batch of ONE frame. ``residual_conditioning`` does the same arithmetic for N frames in two
pipeline passes (dcb_residual_fused: four launches per frame group).

``residual_conditioning_bidir`` builds the residual the datasets intended (SURVEY.md App. B-6): BOTH decoded
I-frames warped by their own flows, fused by occlusion, subtracted -- also two pipeline passes (dcb_residual_bidir).

Under ``deterministic()`` both builders keep one library call per frame group in fp32 (DCB_FLAG_DETERMINISTIC: emit, one
radix sort, reduce, fuse -- 11 launches), bit for bit the composition of deterministic single ops that bf16, fp64 and
``C > 3`` still run.
"""
from __future__ import annotations

import torch
from torch.utils.data import Dataset

from . import _lib
from .control_utils import compute_mask
from .extractors import bidir_fuse
from .softsplat import softsplat, is_deterministic

__all__ = ["residual_conditioning", "residual_conditioning_bidir", "ResidueDataset", "WarpingDatasetWrapper"]

_VARIANTS = {"dataset": _lib.RECIPE_DATASET, "wrapper": _lib.RECIPE_WRAPPER}

# Deterministic mode: the workspace of one frame group stays under this many bytes (a group holds one frame at least; a
# 1080p RGB frame needs about 0.55 GB); its 8 sort keys per pixel stay below the ABI's 2^31.
DET_GROUP_BYTES = 2 << 30
_det_groups: dict = {}


def _det_group(n, c, h, w):
    """(frames per group, workspace bytes of one group) of the deterministic recipe for a batch of n frames."""
    key = (n, c, h, w, DET_GROUP_BYTES)
    v = _det_groups.get(key)
    if v is None:
        need = _lib.lib().dcb_residual_det_workspace_bytes
        lo, hi = 1, max(1, min(n, ((1 << 31) - 1) // (8 * h * w)))   # the largest group within the cap: need() grows with it
        while lo < hi:
            mid = (lo + hi + 1) // 2
            if need(mid, c, h, w) <= DET_GROUP_BYTES:
                lo = mid
            else:
                hi = mid - 1
        v = _det_groups[key] = (lo, need(lo, c, h, w))
    return v


def _deterministic_recipe(image1, image2, flow1, flow2, gt, variant):
    """fp32, 1 <= C <= 3, under deterministic(): dcb_residual_fused (image2 None) or dcb_residual_bidir with
    DCB_FLAG_DETERMINISTIC, one call per frame group. Frames are independent, so the bits do not depend on the grouping."""
    lib = _lib.lib()
    n, c, h, w = image1.shape
    dev = image1.device
    fused = torch.empty((n, c, h, w), dtype=torch.float32, device=dev)
    residual = torch.empty_like(fused)
    occ_fwd = torch.empty((n, 1, h, w), dtype=torch.float32, device=dev)
    occ_bwd = torch.empty_like(occ_fwd)
    g, need = _det_group(n, c, h, w)
    stream = _lib.stream_ptr(dev)
    ws = _lib.workspace(dev, need, "scratch", stream)
    d = _lib.desc
    with _lib.on_device(dev):
        for i in range(0, n, g):
            s = slice(i, i + g)
            outs = (d(fused[s]), d(residual[s]), d(occ_fwd[s]), d(occ_bwd[s]))
            if image2 is None:
                rc = lib.dcb_residual_fused(d(image1[s]), d(flow1[s]), d(flow2[s]), d(gt[s]), *outs, ws.data_ptr(), ws.numel(),
                                            _VARIANTS[variant], _lib.FLAG_DETERMINISTIC, stream)
            else:
                rc = lib.dcb_residual_bidir(d(image1[s]), d(image2[s]), d(flow1[s]), d(flow2[s]), d(gt[s]), *outs, ws.data_ptr(),
                                            ws.numel(), _lib.FLAG_DETERMINISTIC, stream)
            _lib.check(rc, "dcb_residual_bidir" if image2 is not None else "dcb_residual_fused")
    return fused, residual, occ_fwd, occ_bwd


def _deterministic_fp32(image1, gt):
    n, c, h, w = image1.shape
    return (is_deterministic() and image1.dtype == torch.float32 and gt.dtype == torch.float32 and 1 <= c <= 3
            and n * h * w > 0)


def _composed(image1, flow1, flow2, gt, variant):
    """General path (any channel count / fp64 / bf16 deterministic): same ops, built from the single-op kernels."""
    metric = torch.ones_like(flow1[:, :1])
    warped1 = softsplat(tenIn=image1, tenFlow=flow1, tenMetric=metric, strMode="soft")
    warped2 = warped1                                          # the reference recomputes the identical splat
    occ_fwd = compute_mask(flow1, flow2).to(image1.dtype)
    occ_bwd = compute_mask(flow2, flow1).to(image1.dtype)
    if variant == "dataset":
        conf = torch.clamp(torch.cat([occ_fwd, occ_bwd], dim=1), min=0)
    else:
        conf = torch.clamp(torch.cat([metric, metric], dim=1), min=0)
    w_norm = conf / (conf.sum(dim=1, keepdim=True) + 1e-6)
    fused = w_norm[:, :1] * warped1 + w_norm[:, 1:] * warped2
    if variant == "wrapper":
        holes = (occ_fwd + occ_bwd) > 1.5
        fused = torch.where(holes.expand_as(fused), 0.5 * (warped1 + warped2), fused)   # no .any() host sync
    return fused, gt - fused, occ_fwd, occ_bwd


@torch.no_grad()
def residual_conditioning(image1, flow1, flow2, gt, variant: str = "dataset", return_masks: bool = False):
    """Warped frame + residual for a batch of frames.

    image1, gt: [N,C,H,W]; flow1 (forward, moves image1), flow2 (backward): [N,2,H,W].
    variant "dataset" -> ``controlnet/dataset.py:233-265``; "wrapper" -> ``controlnet/residual_utils.py:159-199``.
    Returns (fused, residual) or (fused, residual, occ_fwd, occ_bwd).
    """
    assert variant in _VARIANTS
    assert image1.dim() == 4 and image1.shape == gt.shape and flow1.shape == flow2.shape
    assert image1.is_cuda, "residual_conditioning has no CPU path"
    n, c, h, w = image1.shape
    fusable = (c <= 3 and image1.dtype in (torch.float32, torch.bfloat16) and flow1.dtype == image1.dtype
               and flow2.dtype == image1.dtype and gt.dtype == image1.dtype and not is_deterministic())
    if _deterministic_fp32(image1, gt):
        fused, residual, occ_fwd, occ_bwd = _deterministic_recipe(image1, None, flow1.to(image1.dtype), flow2.to(image1.dtype),
                                                                  gt, variant)
    elif not fusable:
        fused, residual, occ_fwd, occ_bwd = _composed(image1, flow1.to(image1.dtype), flow2.to(image1.dtype), gt, variant)
    else:
        lib = _lib.lib()
        dev = image1.device
        fused = torch.empty((n, c, h, w), dtype=image1.dtype, device=dev)
        residual = torch.empty_like(fused)
        # always hand the masks their own storage: the library's in-workspace mask scratch would
        # dirty the shared, kept-zero accumulator buffer
        occ_fwd = torch.empty((n, 1, h, w), dtype=image1.dtype, device=dev)
        occ_bwd = torch.empty_like(occ_fwd)
        need = lib.dcb_residual_workspace_bytes(n, c, h, w)
        dt = _lib._DTYPES[image1.dtype]
        scratch = _lib.fwd_is_scratch(n, c, h, w, dt, _lib.MODE_SOFT) and _lib.fwd_is_scratch(n, 2, h, w, dt, _lib.MODE_SOFT)
        ws = _lib.workspace(dev, need, "scratch" if scratch else "acc")
        with _lib.on_device(dev):
            rc = lib.dcb_residual_fused(_lib.desc(image1), _lib.desc(flow1), _lib.desc(flow2), _lib.desc(gt),
                                        _lib.desc(fused), _lib.desc(residual), _lib.desc(occ_fwd), _lib.desc(occ_bwd),
                                        ws.data_ptr(), ws.numel(), _VARIANTS[variant], 0 if scratch else _lib.FLAG_WS_CLEAN,
                                        _lib.stream_ptr(dev))
        if rc != 0:
            _lib.invalidate_acc(dev)
        _lib.check(rc, "dcb_residual_fused")
    if return_masks:
        return fused, residual, occ_fwd, occ_bwd
    return fused, residual


def _composed_bidir(image1, image2, flow1, flow2, gt):
    """General path of the two-reference builder (any channel count / fp64 / bf16 deterministic): the single-op kernels."""
    ones = torch.ones_like(flow1[:, :1])
    warped1 = softsplat(tenIn=image1, tenFlow=flow1, tenMetric=ones, strMode="soft")
    warped2 = softsplat(tenIn=image2, tenFlow=flow2, tenMetric=ones, strMode="soft")
    occ_fwd = compute_mask(flow1, flow2).to(image1.dtype)
    occ_bwd = compute_mask(flow2, flow1).to(image1.dtype)
    if image1.dtype == torch.float64:
        # the fusion kernel is F32/BF16/F16 only: the fp64 composition fuses as _composed does (soft_fuse, improv_experiments.ipynb
        # cell 3, on the valid masks; no .any() host sync)
        conf = torch.cat([1 - occ_fwd, 1 - occ_bwd], dim=1)
        w = conf / (conf.sum(dim=1, keepdim=True) + 1e-6)
        fused = w[:, :1] * warped1 + w[:, 1:] * warped2
        holes = (occ_fwd + occ_bwd) > 1.5
        fused = torch.where(holes.expand_as(fused), 0.5 * (warped1 + warped2), fused)
    else:
        # soft_fuse on the valid masks 1 - occ == bidir_fuse with the occlusion masks as the hole test (binary masks)
        fused = bidir_fuse(warped1, warped2, 1 - occ_fwd, 1 - occ_bwd, occ_fwd, occ_bwd)
    return fused, gt - fused, occ_fwd, occ_bwd


@torch.no_grad()
def residual_conditioning_bidir(image1, image2, flow1, flow2, gt, return_masks: bool = False):
    """Two-reference fused frame + residual for a batch of inter frames.

    image1, image2, gt: [N,C,H,W]; flow1 moves image1, flow2 moves image2: [N,2,H,W]. The caller states the pairing (the
    reference's dataset and extractor pair the frames of ``local_conditions`` with the flows in opposite ways). Computes
    ``soft_fuse(softsplat(image1, flow1), softsplat(image2, flow2), 1 - compute_mask(flow1, flow2),
    1 - compute_mask(flow2, flow1))`` (improv_experiments.ipynb cell 3, mask pairing of ``extractors.py:290-295``) and
    ``gt - fused``. Inputs may be strided views; an I-frame shared by several inter frames can be an ``expand``ed batch.
    Returns (fused, residual) or (fused, residual, occ_fwd, occ_bwd).
    """
    assert image1.dim() == 4 and image1.shape == image2.shape == gt.shape and flow1.shape == flow2.shape
    assert flow1.shape[0] == image1.shape[0] and flow1.shape[1] == 2 and flow1.shape[2:] == image1.shape[2:]
    assert image1.is_cuda, "residual_conditioning_bidir has no CPU path"
    n, c, h, w = image1.shape
    dt_ = image1.dtype
    fusable = (c <= 3 and dt_ in (torch.float32, torch.bfloat16) and all(t.dtype == dt_ for t in (image2, flow1, flow2, gt))
               and not is_deterministic())
    if _deterministic_fp32(image1, image1):                     # gt is cast to image1's dtype, as the composition casts it
        fused, residual, occ_fwd, occ_bwd = _deterministic_recipe(image1, image2.to(dt_), flow1.to(dt_), flow2.to(dt_), gt.to(dt_),
                                                                  "bidir")
    elif not fusable:
        fused, residual, occ_fwd, occ_bwd = _composed_bidir(image1, image2.to(dt_), flow1.to(dt_), flow2.to(dt_), gt.to(dt_))
    else:
        lib = _lib.lib()
        dev = image1.device
        fused = torch.empty((n, c, h, w), dtype=dt_, device=dev)
        residual = torch.empty_like(fused)
        # the masks get their own storage, as in residual_conditioning: the in-workspace planes would dirty the kept-zero buffer
        occ_fwd = torch.empty((n, 1, h, w), dtype=dt_, device=dev)
        occ_bwd = torch.empty_like(occ_fwd)
        need = lib.dcb_residual_workspace_bytes(n, c, h, w)        # the same requirement as dcb_residual_fused
        dt = _lib._DTYPES[dt_]
        scratch = _lib.fwd_is_scratch(n, c, h, w, dt, _lib.MODE_SOFT) and _lib.fwd_is_scratch(n, 2, h, w, dt, _lib.MODE_SOFT)
        ws = _lib.workspace(dev, need, "scratch" if scratch else "acc")
        with _lib.on_device(dev):
            rc = lib.dcb_residual_bidir(_lib.desc(image1), _lib.desc(image2), _lib.desc(flow1), _lib.desc(flow2), _lib.desc(gt),
                                        _lib.desc(fused), _lib.desc(residual), _lib.desc(occ_fwd), _lib.desc(occ_bwd),
                                        ws.data_ptr(), ws.numel(), 0 if scratch else _lib.FLAG_WS_CLEAN, _lib.stream_ptr(dev))
        if rc != 0:
            _lib.invalidate_acc(dev)
        _lib.check(rc, "dcb_residual_bidir")
    if return_masks:
        return fused, residual, occ_fwd, occ_bwd
    return fused, residual


def _sample_to_tensors(sample, device):
    """The reference's host->device step (``dataset.py:224-230``): HWC numpy -> [1,C,W,H] via permute(2,1,0)."""
    local_conditions, flow_conditions, ground_truth = sample["local_conditions"], sample["flow"], sample["jpg"]
    image1 = torch.from_numpy(local_conditions[:, :, :3]).permute(2, 1, 0).unsqueeze(0).to(device)
    flow1 = torch.from_numpy(flow_conditions[:2]).unsqueeze(0).to(device)
    flow2 = torch.from_numpy(flow_conditions[2:]).unsqueeze(0).to(device)
    gt = torch.from_numpy(ground_truth).permute(2, 1, 0).unsqueeze(0).to(device)
    return image1, flow1, flow2, gt


class ResidueDataset(Dataset):
    """Same constructor, ``__len__`` and ``__getitem__`` keys as the reference class (``dataset.py:193-276``)."""

    def __init__(self, original_dataset: Dataset, device: str = "cuda"):
        self.original_dataset = original_dataset
        self.device = device

    def __len__(self):
        return len(self.original_dataset)

    def __getitem__(self, idx):
        sample = self.original_dataset[idx]
        image1, flow1, flow2, gt = _sample_to_tensors(sample, self.device)
        fused, residual = residual_conditioning(image1, flow1, flow2, gt, "dataset")
        return {
            "warped_image": fused.squeeze(0),
            "flow": sample["flow"],
            "txt": sample["txt"],
            "local_conditions": sample["local_conditions"],
            "residual": residual.squeeze(0),
        }


class WarpingDatasetWrapper(Dataset):
    """Same as the reference class (``residual_utils.py:120-211``), minus its last-line crash: the
    reference calls ``.permute()`` on a NumPy array at ``residual_utils.py:207`` and raises
    AttributeError; here ``local_conditions`` is passed through unchanged."""

    def __init__(self, original_dataset: Dataset, device: str = "cuda"):
        self.original_dataset = original_dataset
        self.device = device

    def __len__(self):
        return len(self.original_dataset)

    def __getitem__(self, idx):
        sample = self.original_dataset[idx]
        image1, flow1, flow2, gt = _sample_to_tensors(sample, self.device)
        fused, residual = residual_conditioning(image1, flow1, flow2, gt, "wrapper")
        return {
            "warped_image": fused,
            "flow": sample["flow"],
            "ground_truth": gt,
            "residual": residual.squeeze(0),
            "local_conditions": sample["local_conditions"],
            "txt": sample["txt"],
        }
