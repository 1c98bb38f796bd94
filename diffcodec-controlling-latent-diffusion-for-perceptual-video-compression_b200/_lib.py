"""ctypes binding of libdiffcodec_b200.so (the C ABI in include/diffcodec_b200.h).

PyTorch is used here only for device memory, streams and autograd plumbing: every
arithmetic operation of the hot path happens inside the shared library. There is
no fallback: if the library is missing or a call fails, we raise.
"""
from __future__ import annotations

import ctypes
import os
import struct
import subprocess
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DCB_LIB_PATH") or os.path.join(_HERE, "libdiffcodec_b200.so")   # override: A/B builds only

DCB_F32, DCB_BF16, DCB_F64 = 0, 1, 2
DCB_U8, DCB_F16 = 3, 4          # U8: a storage type of dcb_convert only; F16: a tensor dtype wherever BF16 is one
MODE_SUM, MODE_AVG, MODE_LINEAR, MODE_SOFT = 0, 1, 2, 3
EPS_ADD, EPS_ZERO, EPS_CLIP = 0, 1, 2
FLAG_DETERMINISTIC, FLAG_WS_CLEAN = 1, 2
RECIPE_DATASET, RECIPE_WRAPPER = 0, 1
FLOW_BILINEAR_RESCALE, FLOW_ADAPTIVE_AVG, FLOW_BILINEAR_NORMALIZE = 0, 1, 2
PYRAMID_NO_MASKS, PYRAMID_NO_HOLES = 4, 8
RESAMPLE_NONE, RESAMPLE_MUL, RESAMPLE_DIV = 0, 1, 2

E_NULL, E_SHAPE, E_DTYPE, E_MODE, E_WORKSPACE, E_LIMIT, E_ALIGN = -1, -2, -3, -4, -5, -6, -7

_DTYPES = {torch.float32: DCB_F32, torch.bfloat16: DCB_BF16, torch.float16: DCB_F16, torch.float64: DCB_F64}


class DcbTensor(ctypes.Structure):
    _fields_ = [
        ("ptr", ctypes.c_void_p),
        ("dtype", ctypes.c_int32),
        ("reserved", ctypes.c_int32),
        ("size", ctypes.c_int64 * 4),
        ("stride", ctypes.c_int64 * 4),
    ]


# Descriptors are passed as packed bytes with the exact layout of `struct DcbTensor` (80 bytes): building a
# ctypes.Structure costs ~6.5 us per tensor, struct.pack ~1.5 us -- it matters for latent-sized calls.
_P = ctypes.c_void_p
_I64x4 = ctypes.c_int64 * 4
_DESC_STRUCT = struct.Struct("Pii4q4q")
_pack_desc = _DESC_STRUCT.pack
_pack_desc_into = _DESC_STRUCT.pack_into
assert struct.calcsize("Pii4q4q") == ctypes.sizeof(DcbTensor)
_lib = None
_lock = threading.Lock()

# name -> (restype, argtypes); exactly the symbols include/diffcodec_b200.h declares
SYMBOLS = {
    "dcb_version": (ctypes.c_int, []),
    "dcb_last_error": (ctypes.c_char_p, []),
    "dcb_build_info": (ctypes.c_char_p, []),
    "dcb_launch_count": (ctypes.c_int64, []),
    "dcb_splat_workspace_bytes": (ctypes.c_int64, [ctypes.c_int64] * 4 + [ctypes.c_int32] * 3),
    "dcb_splat_fwd_workspace_bytes": (ctypes.c_int64, [ctypes.c_int64] * 4 + [ctypes.c_int32] * 3),
    "dcb_splat_bwd_workspace_bytes": (ctypes.c_int64, [ctypes.c_int64] * 4 + [ctypes.c_int32] * 3),
    "dcb_splat_fwd_workspace_is_scratch": (ctypes.c_int32, [ctypes.c_int64] * 4 + [ctypes.c_int32] * 3),
    "dcb_set_option": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_int64]),
    "dcb_splat_fwd": (ctypes.c_int, [_P] * 6 + [ctypes.c_void_p, ctypes.c_int64] + [ctypes.c_int32] * 3 + [ctypes.c_void_p]),
    "dcb_splat_bwd": (ctypes.c_int, [_P] * 10 + [ctypes.c_void_p, ctypes.c_int64] + [ctypes.c_int32] * 3 + [ctypes.c_void_p]),
    "dcb_backwarp_fwd": (ctypes.c_int, [_P] * 5 + [ctypes.c_int32, ctypes.c_void_p]),
    "dcb_backwarp_bwd_workspace_bytes": (ctypes.c_int64, [ctypes.c_int64] * 4 + [ctypes.c_int32]),
    "dcb_backwarp_bwd": (ctypes.c_int, [_P] * 5 + [ctypes.c_int32, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]),
    "dcb_occlusion_mask_workspace_bytes": (ctypes.c_int64, [ctypes.c_int64] * 3),
    "dcb_occlusion_mask": (ctypes.c_int, [_P] * 3 + [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_void_p]),
    "dcb_residual_workspace_bytes": (ctypes.c_int64, [ctypes.c_int64] * 4),
    "dcb_bidir_fuse_fwd": (ctypes.c_int, [_P] * 7 + [ctypes.c_void_p]),
    "dcb_bidir_fuse_bwd": (ctypes.c_int, [_P] * 11 + [ctypes.c_void_p]),
    "dcb_tile_merge_workspace_bytes": (ctypes.c_int64, [ctypes.c_int64] * 3 + [ctypes.c_int32]),
    "dcb_tile_merge": (ctypes.c_int, [_P, ctypes.c_void_p, ctypes.c_int32, _P, ctypes.c_int64, ctypes.c_int64, ctypes.c_double,
                                      ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]),
    "dcb_bidir_block_workspace_bytes": (ctypes.c_int64, [ctypes.c_int64] * 4 + [ctypes.c_int32] * 2),
    "dcb_bidir_block_fwd": (ctypes.c_int, [_P] * 13 + [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_void_p]),
    "dcb_bidir_block_bwd": (ctypes.c_int, [_P] * 17 + [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]),
    "dcb_flow_resize": (ctypes.c_int, [_P, _P, ctypes.c_int32, ctypes.c_void_p]),
    "dcb_bidir_pyramid_workspace_bytes": (ctypes.c_int64, [ctypes.c_void_p, ctypes.c_int32]),
    "dcb_bidir_pyramid_det_workspace_bytes": (ctypes.c_int64, [ctypes.c_void_p, ctypes.c_int32]),
    "dcb_bidir_pyramid_fwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_void_p]),
    "dcb_bidir_pyramid_bwd_workspace_bytes": (ctypes.c_int64, [ctypes.c_void_p, ctypes.c_int32]),
    "dcb_bidir_pyramid_bwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_void_p]),
    "dcb_resample_batch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p]),
    "dcb_convert": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p]),
    "dcb_residual_fused": (ctypes.c_int, [_P] * 8 + [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p]),
    "dcb_residual_bidir": (ctypes.c_int, [_P] * 9 + [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_void_p]),
}


def build(verbose: bool = False) -> str:
    """Compile the library in-tree for sm_100a with the committed Makefile (nvcc cross-compiles without a GPU)."""
    out = subprocess.run(["make", "-C", os.path.join(_HERE, "csrc"), "-j8"], capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("building libdiffcodec_b200.so failed:\n" + out.stdout[-4000:] + out.stderr[-4000:])
    if verbose:
        print(out.stdout[-2000:])
    return LIB_PATH


def lib() -> ctypes.CDLL:
    """Load the library (once). Raises if it is absent -- there is no other implementation."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(or `make -C <package>/csrc`). diffcodec_b200 has no CPU or PyTorch fallback.")
                handle = ctypes.CDLL(LIB_PATH)
                for name, (res, args) in SYMBOLS.items():
                    fn = getattr(handle, name)
                    fn.restype, fn.argtypes = res, args
                _lib = handle
                for opt in ("fwd_path", "owner_group_bytes", "pipe_group_bytes", "pipe_ring_slots", "bwd_group_bytes", "pipe_tail_percent", "lists_nhwc", "planar_one_launch", "bwd_flat"):      # A/B knobs: DCB_FWD_PATH=1 python ...
                    v = os.environ.get("DCB_" + opt.upper())
                    if v:
                        handle.dcb_set_option(opt.encode(), int(v))
    return _lib


def set_option(name: str, value: int) -> None:
    """Process-wide tuning / test knob of the native library (``dcb_set_option`` in the header)."""
    check(lib().dcb_set_option(name.encode(), int(value)), "dcb_set_option")
    _scratch_cache.clear()
    for hook in _option_hooks:
        hook()


_option_hooks: list = []          # callables that drop size caches derived from the library's dispatch


_scratch_cache: dict = {}


def fwd_is_scratch(n, c, h, w, dt, mode, flags=0) -> bool:
    """True when the forward of these sizes keeps no accumulators in its workspace (plain scratch, no clean protocol)."""
    key = (n, c, h, w, dt, mode, flags)
    v = _scratch_cache.get(key)
    if v is None:
        v = _scratch_cache[key] = bool(lib().dcb_splat_fwd_workspace_is_scratch(n, c, h, w, dt, mode, flags))
    return v


_CONVERT_DTYPES = {torch.uint8: DCB_U8, torch.float16: DCB_F16, torch.bfloat16: DCB_BF16, torch.float32: DCB_F32}


def convert(src: torch.Tensor, dst: torch.Tensor, scale: float = 1.0) -> torch.Tensor:
    """dst = scale * src with a change of element type, on the device, in the native library (dcb_convert)."""
    assert src.is_cuda and dst.is_cuda and src.is_contiguous() and dst.is_contiguous() and src.numel() == dst.numel()
    with on_device(src.device):
        check(lib().dcb_convert(src.data_ptr(), _CONVERT_DTYPES[src.dtype], dst.data_ptr(), _CONVERT_DTYPES[dst.dtype],
                                src.numel(), float(scale), stream_ptr(src.device)), "dcb_convert")
    return dst


class DcbError(RuntimeError):
    pass


def check(rc: int, what: str) -> None:
    """Map ABI return codes to the exceptions the reference would raise."""
    if rc == 0:
        return
    msg = lib().dcb_last_error().decode("utf-8", "replace")
    if rc in (E_SHAPE, E_MODE, E_NULL):
        raise AssertionError(f"{what}: {msg}")          # the reference uses assert for these
    if rc in (E_DTYPE, E_LIMIT, E_ALIGN, E_WORKSPACE):
        raise ValueError(f"{what}: {msg}")
    raise DcbError(f"{what}: CUDA error {rc}: {msg}")


def desc(t: torch.Tensor | None):
    """`const DcbTensor*` argument for a 4-d CUDA tensor (packed bytes), or None for NULL."""
    if t is None:
        return None
    if not t.is_cuda:
        raise AssertionError("diffcodec_b200 runs on CUDA tensors only (the reference asserts the same, softsplat.py:347-348)")
    if t.dim() != 4:
        raise AssertionError(f"expected a 4-d NCHW tensor, got {tuple(t.shape)}")
    if t.dtype not in _DTYPES:
        raise ValueError(f"unsupported dtype {t.dtype}: float32, bfloat16, float16 and float64 are implemented")
    return _pack_desc(t.data_ptr(), _DTYPES[t.dtype], 0, *t.shape, *t.stride())


# -------------------------------------------------------------------------------------------------
# array arguments (DcbPyramidLevel[], DcbResampleJob[]): descriptors and the arrays that point at them live in one
# per-thread ctypes buffer, so a whole pyramid costs one pack per tensor and no ctypes.Structure objects
# -------------------------------------------------------------------------------------------------
_tls = threading.local()
_DESC_BYTES = _DESC_STRUCT.size            # 80
_LEVEL_STRUCT = struct.Struct("13P")       # DcbPyramidLevel: 6 descriptor pointers + 7 raw output pointers
_BWD_LEVEL_STRUCT = struct.Struct("19P")   # DcbPyramidBwdLevel: 7 descriptor pointers + 6 saved + 6 gradient raw pointers
_JOB_STRUCT = struct.Struct("PPiiff")      # DcbResampleJob
_ARENA_BYTES = 1 << 14


def _arena():
    a = getattr(_tls, "arena", None)
    if a is None:
        buf = ctypes.create_string_buffer(_ARENA_BYTES)
        a = _tls.arena = (buf, ctypes.addressof(buf))
    return a


def _tensor_fields(t: torch.Tensor):
    if not t.is_cuda:
        raise AssertionError("diffcodec_b200 runs on CUDA tensors only (the reference asserts the same, softsplat.py:347-348)")
    if t.dim() != 4:
        raise AssertionError(f"expected a 4-d NCHW tensor, got {tuple(t.shape)}")
    if t.dtype not in _DTYPES:
        raise ValueError(f"unsupported dtype {t.dtype}: float32, bfloat16, float16 and float64 are implemented")
    return (t.data_ptr(), _DTYPES[t.dtype], 0, *t.shape, *t.stride())


def pack_pyramid(levels, outputs):
    """levels: per scale (first, last, flow_f, flow_b, metric_f | None, metric_b | None); outputs: per scale 7 tensors or None
    (fused, warped_f, warped_b, norm_f, norm_b, occ_f, occ_b). Returns the address of a DcbPyramidLevel[len(levels)] that
    stays valid until the next pack_* call of this thread."""
    buf, base = _arena()
    n = len(levels)
    off = n * _LEVEL_STRUCT.size
    assert off + n * 6 * _DESC_BYTES <= _ARENA_BYTES
    for l, (ins, outs) in enumerate(zip(levels, outputs)):
        ptrs = []
        for t in ins:
            if t is None:
                ptrs.append(0)
            else:
                _pack_desc_into(buf, off, *_tensor_fields(t))
                ptrs.append(base + off)
                off += _DESC_BYTES
        ptrs += [0 if o is None else o.data_ptr() for o in outs]
        _LEVEL_STRUCT.pack_into(buf, l * _LEVEL_STRUCT.size, *ptrs)
    return base


def pack_pyramid_bwd(levels, saved, grads):
    """levels: per scale (grad_fused, first, last, flow_f, flow_b, metric_f | None, metric_b | None); saved: per scale the six
    forward outputs (warped_f, warped_b, norm_f, norm_b, occ_f, occ_b); grads: per scale six tensors or None (grad_first,
    grad_last, grad_flow_f, grad_flow_b, grad_metric_f, grad_metric_b). Returns the address of a DcbPyramidBwdLevel[len(levels)]
    that stays valid until the next pack_* call of this thread."""
    buf, base = _arena()
    n = len(levels)
    off = n * _BWD_LEVEL_STRUCT.size
    assert off + n * 7 * _DESC_BYTES <= _ARENA_BYTES
    for l, (ins, sv, gr) in enumerate(zip(levels, saved, grads)):
        ptrs = []
        for t in ins:
            if t is None:
                ptrs.append(0)
            else:
                _pack_desc_into(buf, off, *_tensor_fields(t))
                ptrs.append(base + off)
                off += _DESC_BYTES
        ptrs += [0 if o is None else o.data_ptr() for o in tuple(sv) + tuple(gr)]
        _BWD_LEVEL_STRUCT.pack_into(buf, l * _BWD_LEVEL_STRUCT.size, *ptrs)
    return base


def pack_resample(jobs):
    """jobs: (src, dst, align_corners, op, factor0, factor1). Returns the address of a DcbResampleJob[len(jobs)]."""
    buf, base = _arena()
    n = len(jobs)
    off = (n * _JOB_STRUCT.size + 15) // 16 * 16
    assert off + n * 2 * _DESC_BYTES <= _ARENA_BYTES
    for j, (src, dst, align, op, f0, f1) in enumerate(jobs):
        _pack_desc_into(buf, off, *_tensor_fields(src))
        _pack_desc_into(buf, off + _DESC_BYTES, *_tensor_fields(dst))
        _JOB_STRUCT.pack_into(buf, j * _JOB_STRUCT.size, base + off, base + off + _DESC_BYTES, int(bool(align)), int(op), float(f0), float(f1))
        off += 2 * _DESC_BYTES
    return base


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_ptr(device) -> int:
    """cudaStream_t of torch's current stream on `device` (the raw getter costs 0.3 us, the
    Stream object of torch.cuda.current_stream() 5 us -- a quarter of a latent-sized call)."""
    if _raw_stream is not None:
        idx = device.index
        return _raw_stream(torch.cuda.current_device() if idx is None else idx)
    return torch.cuda.current_stream(device).cuda_stream


class on_device:
    """`with on_device(dev):` -- torch.cuda.device(dev) only when dev is not already current (the
    context manager costs ~5 us, more than the kernels of a latent-sized call)."""
    __slots__ = ("ctx",)

    def __init__(self, dev):
        self.ctx = None if torch.cuda.current_device() == dev.index else torch.cuda.device(dev)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)
        return False


# -------------------------------------------------------------------------------------------------
# per-(device, stream) workspace caches. Two kinds:
#   "acc"     accumulators; kept all-zero BETWEEN calls (the epilogue kernels re-zero what they
#             read), so DCB_FLAG_WS_CLEAN can be passed and no memset is launched;
#   "scratch" anything else (backward scalars, deterministic-mode keys); contents arbitrary.
# A workspace is only ever used on the stream it was created for.
# -------------------------------------------------------------------------------------------------
_workspaces: dict = {}


def workspace(device: torch.device, nbytes: int, kind: str, stream: int | None = None) -> torch.Tensor:
    key = (kind, device.index, stream if stream is not None else stream_ptr(device))
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.zeros(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = buf
    return buf


def invalidate_acc(device: torch.device) -> None:
    """Forget the clean accumulator buffer (after a failed call it may hold partial sums)."""
    _workspaces.pop(("acc", device.index, stream_ptr(device)), None)


def release_workspaces() -> None:
    _workspaces.clear()
