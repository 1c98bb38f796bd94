"""Tile utilities of the reference's ``patch_utils.py`` for 1080p inference in 512^2 tiles.

``merge_latent_tiles_from_pixel_coords`` (patch_utils.py:83-174) keeps its name, arguments and
quirks -- the coordinate tuple is read as ``(x1, x2, y1, y2)`` although ``crop_into_tiles`` returns
``(y1, y2, x1, x2)``; canvas pixels whose total Hann weight is below ``eps`` come out as 0 -- but
runs as ONE gather kernel (``dcb_tile_merge``) instead of 6-8 eager kernels and three temporaries
per tile. ``crop_into_tiles`` (patch_utils.py:189-209) is pure indexing and stays on the host side
of the boundary: it returns views, for numpy arrays and torch tensors alike.
"""
from __future__ import annotations

import struct

import torch

from . import _lib

__all__ = ["merge_latent_tiles_from_pixel_coords", "crop_into_tiles"]


def crop_into_tiles(img, tile_size, overlap=0, order="hwc"):
    """Crop image into overlapping tiles of size tile_size; coords are (y, y2, x, x2)."""
    if order == "hwc":
        h, w, c = img.shape
    else:  # chw
        c, h, w = img.shape
    stride_y = tile_size[0] - overlap
    stride_x = tile_size[1] - overlap
    tiles, coords = [], []
    for y in range(0, h, stride_y):
        for x in range(0, w, stride_x):
            y2, x2 = min(y + tile_size[0], h), min(x + tile_size[1], w)
            tiles.append(img[y:y2, x:x2, :] if order == "hwc" else img[:, y:y2, x:x2])
            coords.append((y, y2, x, x2))
    return tiles, coords, (h, w)


def merge_latent_tiles_from_pixel_coords(latents, pixel_coords, full_latent_shape, original_image_size, eps: float = 1e-8):
    """latents: list of (1, C, th, tw) CUDA tensors (one dtype: float32, bfloat16 or float16; the 16-bit merges
    accumulate in fp32 and round once); pixel_coords:
    list of 4-tuples in original pixel space; returns the merged (1, C, H_lat, W_lat) tensor.
    Inference utility: no autograd (the reference's in-place accumulation has none worth keeping)."""
    assert len(latents) == len(pixel_coords), "latents and coords length mismatch"
    assert len(latents) > 0, "no tiles"
    dev, dtype = latents[0].device, latents[0].dtype
    assert dev.type == "cuda", "merge_latent_tiles_from_pixel_coords runs on CUDA tensors"
    n, c, h_lat, w_lat = (int(v) for v in full_latent_shape)
    h_px, w_px = (int(v) for v in original_image_size)
    if dtype not in _lib._DTYPES:
        raise ValueError(f"unsupported dtype {dtype}: float32, bfloat16 and float16 are implemented")
    dt = _lib._DTYPES[dtype]
    lib = _lib.lib()
    out = torch.empty((n, c, h_lat, w_lat), dtype=dtype, device=dev)
    # one packed array of DcbTensor descriptors: this loop is the whole host cost of a merge
    descs = bytearray(80 * len(latents))
    pack = _lib._pack_desc_into
    for i, t in enumerate(latents):
        shape = t.shape
        assert len(shape) == 4 and shape[0] == 1, "expected tile shape (1,C,H,W)"               # patch_utils.py:155
        assert t.dtype is dtype and t.device == dev, "latents must be torch tensors on same device & dtype"
        pack(descs, 80 * i, t.data_ptr(), dt, 0, *shape, *t.stride())
    descs = bytes(descs)
    coords = struct.pack(f"{4 * len(latents)}q", *(int(v) for tup in pixel_coords for v in tup))
    stream = _lib.stream_ptr(dev)
    need = lib.dcb_tile_merge_workspace_bytes(c, h_lat, w_lat, len(latents))
    ws = _lib.workspace(dev, need, "scratch", stream) if need > 0 else None
    with _lib.on_device(dev):
        rc = lib.dcb_tile_merge(descs, coords, len(latents), _lib.desc(out), h_px, w_px, float(eps),
                                ws.data_ptr() if ws is not None else None, ws.numel() if ws is not None else 0, stream)
    _lib.check(rc, "dcb_tile_merge")
    return out
