"""diffcodec_b200 -- B200-native motion compensation for DiffCodec.

One hot path, rebuilt from scratch for sm_100a behind the reference's Python API:
forward splatting by optical flow (sum / avg / linear / soft) with its backward, the bilinear
backward warp, and the occlusion-mask / fusion / residual arithmetic that builds the ControlNet
conditioning. All arithmetic runs in ``libdiffcodec_b200.so`` (C ABI: ``include/diffcodec_b200.h``);
there is no CPU or PyTorch fallback.

The directory name is the (hyphenated) project name; import it through the ``diffcodec_b200``
alias module at the repository root.
"""
from . import _lib
from .softsplat import softsplat, softsplat_func, deterministic, is_deterministic
from .control_utils import compute_mask, FeatureWarperSoftsplat, resize_and_normalize_flow_batched, FDN, zero_module
from .warp import WarpingLayerBWFlow, backwarp, backwarp_residual
from .extractors import (bidir_fuse, bidirectional_warp_fuse, bidirectional_block, bidirectional_pyramid, pyramid_conditioning, resample_batch,
                         Bi_Dir_FeatureExtractor, Bi_Dir_ResidueExtractor, WarpExtractor, ConvBlock)
from .residual_utils import residual_conditioning, residual_conditioning_bidir, ResidueDataset, WarpingDatasetWrapper
from .sharding import UVG_SEQUENCES, GopUnit, enumerate_gops, shard_units, gather_checksums, gather_outputs, checksum
from .host import softsplat_host, bind_to_gpu_numa
from .patch_utils import merge_latent_tiles_from_pixel_coords, crop_into_tiles
from . import flow_io
from .dropin import install

__version__ = "0.1.0"


def launch_count() -> int:
    """Kernels launched by the native library in this process (bench.py's gpu_launches)."""
    return int(_lib.lib().dcb_launch_count())


def build_info() -> str:
    return _lib.lib().dcb_build_info().decode()
