/*
 * diffcodec_b200.h -- C ABI of the B200-native motion-compensation library
 * (libdiffcodec_b200.so, hand-written sm_100a CUDA).
 *
 * This is the drop-in boundary for ONE path of the reference
 * (Maryamsana-1998/DiffCodec-...): forward splatting by optical flow in the
 * sum / avg / linear / soft modes with its backward, the bilinear backward warp,
 * and the residual / occlusion-mask / fusion arithmetic that builds the
 * ControlNet conditioning. The reference has no C FFI of its own: its de-facto
 * native boundary is the CuPy launch of three JIT-compiled kernels with raw
 * data_ptr()s (controlnet/softsplat.py:285-290, 340-345, 369-376, 430-435,
 * 440-447, 519-524). Each entry point below cites the reference interface it
 * replaces (paths relative to the reference repository root).
 *
 * Contract (all entry points):
 *   - plain pointers and sizes only; no torch types;
 *   - every pointer is DEVICE memory of the current CUDA device, owned by the
 *     caller; the library never allocates, never synchronises, never creates a
 *     stream, and does not retain pointers after returning (CUDA-graph safe);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*);
 *   - returns 0 on success, a negative DCB_E_* for argument errors, a positive
 *     cudaError_t for launch errors; text via dcb_last_error() (thread-local);
 *   - there is no CPU fallback of any kind.
 */
#ifndef DIFFCODEC_B200_H
#define DIFFCODEC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DCB_VERSION 100 /* 0.1.0 */

/* element types */
enum { DCB_F32 = 0, DCB_BF16 = 1, DCB_F64 = 2,
       DCB_U8 = 3 /* storage type of dcb_convert only (host-buffer path) */,
       DCB_F16 = 4 /* IEEE binary16: a tensor dtype wherever BF16 is one (same kernel family, group size and workspace;
                      loads widened to fp32, each store rounded once). Refused (DCB_E_DTYPE) by dcb_backwarp_*,
                      dcb_occlusion_mask, dcb_residual_fused, dcb_residual_bidir and dcb_flow_resize */ };

/* splat modes: controlnet/softsplat.py:232-274 (strMode.split('-')[0]) */
enum { DCB_MODE_SUM = 0, DCB_MODE_AVG = 1, DCB_MODE_LINEAR = 2, DCB_MODE_SOFT = 3 };

/* normaliser variants: controlnet/softsplat.py:256-266 (strMode.split('-')[1]) */
enum { DCB_EPS_ADD = 0, DCB_EPS_ZERO = 1, DCB_EPS_CLIP = 2 };

/* flags */
enum {
    DCB_FLAG_DETERMINISTIC = 1, /* sort-then-reduce: bit-identical run to run and to the sequential oracle */
    DCB_FLAG_WS_CLEAN = 2       /* caller guarantees the accumulator part of the workspace is all-zero on entry;
                                   the library leaves it all-zero on exit (saves the memset) */
};

/* residual recipe variants */
enum {
    DCB_RECIPE_DATASET = 0, /* controlnet/dataset.py:233-265  (occlusion masks are the fusion weights) */
    DCB_RECIPE_WRAPPER = 1  /* controlnet/residual_utils.py:159-199 (ones metrics + double-hole fill) */
};

/* flow resampling conventions of dcb_flow_resize */
enum {
    DCB_FLOW_BILINEAR_RESCALE = 0,   /* controlnet/utils.py:21-28: bilinear, align_corners=True, u *= tw/W, v *= th/H */
    DCB_FLOW_ADAPTIVE_AVG = 1,       /* controlnet/dataset.py:43-50: adaptive average pooling, vectors not rescaled */
    DCB_FLOW_BILINEAR_NORMALIZE = 2  /* controlnet/control_utils.py:74-97: bilinear, align_corners=False, u /= (tw-1)/2, v /= (th-1)/2 */
};

/* error codes */
enum {
    DCB_OK = 0,
    DCB_E_NULL = -1,      /* required pointer missing */
    DCB_E_SHAPE = -2,     /* shapes disagree (the reference would assert / index out of range) */
    DCB_E_DTYPE = -3,     /* unsupported or mixed element types */
    DCB_E_MODE = -4,      /* unknown mode / eps / variant / flag combination */
    DCB_E_WORKSPACE = -5, /* workspace missing, too small or misaligned (256 B) */
    DCB_E_LIMIT = -6,     /* a size exceeds what the kernels index (H*W < 2^31, C <= 65535 ...) */
    DCB_E_ALIGN = -7      /* pointer not aligned to its element size */
};

/* 4-d NCHW-indexed view with arbitrary element strides. */
typedef struct DcbTensor {
    void* ptr;
    int32_t dtype;     /* DCB_F32 / DCB_BF16 / DCB_F16 / DCB_F64 */
    int32_t reserved;
    int64_t size[4];   /* N, C, H, W */
    int64_t stride[4]; /* in elements */
} DcbTensor;

int dcb_version(void);
const char* dcb_last_error(void);
/* static description of the build: arch, kernels, compile flags */
const char* dcb_build_info(void);
/* number of kernels this library has launched in the calling process (all threads); for bench.py's gpu_launches */
int64_t dcb_launch_count(void);

/*
 * Workspace size (bytes) for dcb_splat_fwd / dcb_splat_bwd with these sizes. 0 is a valid answer.
 * `elem_dtype` is the dtype of tenIn.
 */
int64_t dcb_splat_workspace_bytes(int64_t N, int64_t C, int64_t H, int64_t W, int32_t elem_dtype,
                                  int32_t mode, int32_t flags);
/* the two halves of the above (it returns their maximum), for callers that keep separate buffers */
int64_t dcb_splat_fwd_workspace_bytes(int64_t N, int64_t C, int64_t H, int64_t W, int32_t elem_dtype,
                                      int32_t mode, int32_t flags);
int64_t dcb_splat_bwd_workspace_bytes(int64_t N, int64_t C, int64_t H, int64_t W, int32_t elem_dtype,
                                      int32_t mode, int32_t flags);

/*
 * 1 when the forward splat of these sizes keeps NO accumulators in its workspace (target-tile-owner kernels:
 * the workspace only holds small per-strip landing boxes; many channels on large tensors: per-target lists that
 * every call rebuilds): the workspace is then plain scratch, DCB_FLAG_WS_CLEAN buys nothing (if it is passed
 * anyway the library zeroes what it wrote, to honour the flag's exit guarantee -- 40 bytes per pixel for the lists).
 * 0 when the workspace holds accumulators and the all-zero protocol of DCB_FLAG_WS_CLEAN saves a memset.
 */
int32_t dcb_splat_fwd_workspace_is_scratch(int64_t N, int64_t C, int64_t H, int64_t W, int32_t elem_dtype,
                                           int32_t mode, int32_t flags);

/*
 * Tuning / test knobs (process-wide, not thread-safe against concurrent calls; defaults are what ships):
 *   "fwd_path"          0 automatic | 1 round-1 accumulator pipeline (red.global into L2-resident cells)
 *                       | 2 target-tile owner kernels wherever they apply (F32 / BF16 only: F16 stays on the pipelines)
 *   "pipe_group_bytes"  accumulator bytes per ring slot of the accumulator pipelines (tests shrink it so that
 *                       small tensors run through many ring groups); 0 restores the default
 *   "pipe_ring_slots"   1 (default) one accumulator slot, scatter and normalise of a frame group in alternating
 *                       launches | 2 round 1's two-slot ring (normalise of group k-1 inside the launch that scatters group k)
 *   "owner_group_bytes" flow bytes per (pre-pass, owner) launch pair; 0 restores the default
 *   "pipe_tail_percent" share of a frame's rows (at the bottom) cut into single-pass 32 x 4 strips instead of 32 x 8
 *   "bwd_group_bytes"   packed-cell bytes per frame group of the packed backward; 0 = one group
 *   "planar_one_launch" 0 (default) two chained launches | 1 a many-channel call whose frames fit one group and whose warps
 *                       are all resident at once (latents, small feature maps) runs as ONE launch with a grid barrier
 *                       (measured slower on B200: 20.6-22.2 us against 16.4 us for C2 under graph replay); F32 / BF16 only
 *   "bwd_flat"          1 (default) contiguous frames take the compile-time (C, mode) form of the packed backward | 0 never
 *   "lists_nhwc"        1 (default) channels-last many-channel tensors take the channel-quad gather | 0 the NCHW gather
 * Returns DCB_OK, or DCB_E_MODE for an unknown name. There is no equivalent in the reference (its kernels are
 * re-specialised per shape by string templating, controlnet/softsplat.py:27-216).
 */
int dcb_set_option(const char* name, int64_t value);

/*
 * Forward splat. Replaces, in one call, the eager pre-ops, `new_zeros`, the `softsplat_out`
 * kernel and the eager post-ops of softsplat() -- controlnet/softsplat.py:232-274 and
 * softsplat_func.forward :277-355. With mode = DCB_MODE_SUM it is exactly
 * softsplat_func.apply(tenIn, tenFlow).
 *
 *   in      [N,C,H,W]  any strides
 *   flow    [N,2,H,W]  any strides; same dtype as `in`, or F32 when `in` is BF16 or F16
 *   metric  [N,1,H,W]  required for LINEAR/SOFT, must be NULL for SUM/AVG (softsplat.py:235-238)
 *   out     [N,C,H,W]  contiguous NCHW, same dtype as `in` (softsplat.py:281)
 *   norm    [N,1,H,W]  optional (may be NULL): receives the normaliser AFTER the eps rule, in the
 *                      accumulator type (F32 for F32/BF16/F16 input, F64 for F64); dcb_splat_bwd needs it
 *   mask    [N,1,H,W]  optional: out is multiplied by (1 - mask) -- controlnet/control_utils.py:69-70
 */
int dcb_splat_fwd(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric,
                  const DcbTensor* out, const DcbTensor* norm, const DcbTensor* mask,
                  void* workspace, int64_t workspace_bytes,
                  int32_t mode, int32_t eps, int32_t flags, void* stream);

/*
 * Backward of dcb_splat_fwd. Replaces softsplat_func.backward (kernels `softsplat_ingrad`,
 * `softsplat_flowgrad`, controlnet/softsplat.py:357-528) fused with the autograd of the eager
 * pre/post ops (exp, mul, cat, slice, add-eps, div; softsplat.py:240-270) and of the (1 - mask)
 * product. Any of grad_in / grad_flow / grad_metric may be NULL (needs_input_grad gating,
 * softsplat.py:364-365). With mode = DCB_MODE_SUM it is exactly softsplat_func.backward.
 *
 *   grad_out [N,C,H,W] any strides (F16: at most 2^30 elements per plane, else DCB_E_LIMIT);  in/flow/metric/mask as
 *   given to the forward
 *   out, norm: what the forward produced (ignored for SUM)
 *   grad_in [N,C,H,W], grad_flow [N,2,H,W], grad_metric [N,1,H,W]: contiguous, fully overwritten
 */
int dcb_splat_bwd(const DcbTensor* grad_out, const DcbTensor* in, const DcbTensor* flow,
                  const DcbTensor* metric, const DcbTensor* out, const DcbTensor* norm,
                  const DcbTensor* mask,
                  const DcbTensor* grad_in, const DcbTensor* grad_flow, const DcbTensor* grad_metric,
                  void* workspace, int64_t workspace_bytes,
                  int32_t mode, int32_t eps, int32_t flags, void* stream);

/*
 * Bilinear backward warp (+ optional fused residual). Replaces WarpingLayerBWFlow.forward,
 * cmp/models/modules/warp.py:9-25 (flow normalisation, linspace grid, grid_sample with zeros
 * padding). align_corners = 0 reproduces the layer as executed by current torch (grid_sample
 * default), 1 the convention its normalisation was written for.
 *
 *   image [N,C,H,W], flow [N,2,H,W] any strides; warped [N,C,H,W] contiguous
 *   gt / residual: both NULL, or both given: residual = gt - warped (controlnet/residual_utils.py:199)
 */
int dcb_backwarp_fwd(const DcbTensor* image, const DcbTensor* flow, const DcbTensor* gt,
                     const DcbTensor* warped, const DcbTensor* residual,
                     int32_t align_corners, void* stream);

/*
 * Backward of dcb_backwarp_fwd w.r.t. image and flow (what autograd derives through
 * grid_sample in cmp/models/modules/warp.py:25). grad_image is fully overwritten (zeroed, then
 * scatter-added); either output may be NULL. A workspace is needed only for BF16 grad_image
 * (fp32 accumulation, rounded once).
 */
int64_t dcb_backwarp_bwd_workspace_bytes(int64_t N, int64_t C, int64_t H, int64_t W, int32_t elem_dtype);
int dcb_backwarp_bwd(const DcbTensor* grad_warped, const DcbTensor* image, const DcbTensor* flow,
                     const DcbTensor* grad_image, const DcbTensor* grad_flow,
                     int32_t align_corners, void* workspace, int64_t workspace_bytes, void* stream);

/*
 * Occlusion mask. Replaces compute_mask(), controlnet/control_utils.py:11-17:
 *   warp = softsplat(flow_a, flow_b, ones, 'soft');  mask = (||flow_b + warp||_2 > 0.3).float()
 * flow_a, flow_b [N,2,H,W]; mask [N,1,H,W] contiguous, same dtype.
 */
int64_t dcb_occlusion_mask_workspace_bytes(int64_t N, int64_t H, int64_t W);
int dcb_occlusion_mask(const DcbTensor* flow_a, const DcbTensor* flow_b, const DcbTensor* mask,
                       void* workspace, int64_t workspace_bytes, int32_t flags, void* stream);

/*
 * Conditioning builder: warped frame, two occlusion masks, confidence fusion, residual, in two
 * pipeline passes (four launches per frame group: flow1 splatted by flow2 + occlusion epilogue; image1 and
 * flow2 splatted together by flow1 + one epilogue that normalises, tests occlusion, fuses and subtracts).
 * Replaces the arithmetic of ResidueDataset.__getitem__ (controlnet/dataset.py:233-265,
 * variant DCB_RECIPE_DATASET) and WarpingDatasetWrapper.__getitem__
 * (controlnet/residual_utils.py:159-199, variant DCB_RECIPE_WRAPPER), batched over N.
 *
 *   image1, gt [N,C,H,W] (1 <= C <= 3; one dtype, F32 or BF16, for every tensor); flow1, flow2 [N,2,H,W]
 *   fused, residual [N,C,H,W] contiguous; occ_fwd / occ_bwd [N,1,H,W] optional outputs
 *   flags: DCB_FLAG_WS_CLEAN as dcb_splat_fwd; other bits are ignored, except DCB_FLAG_DETERMINISTIC (see below), which
 *   earlier versions ignored too
 *
 * DCB_FLAG_DETERMINISTIC (this entry and dcb_residual_bidir; F32 only, else DCB_E_DTYPE): bit-reproducible, and bit-identical
 * to the composition of deterministic single ops (dcb_splat_fwd's deterministic mode for the warps and for the flows behind
 * the masks, the occlusion test, the fusion, the subtraction). The image splat and one mask splat share the footprints of
 * flow1, the other mask splat (and image2's splat) those of flow2: one key set per flow, 8 x N*H*W keys in all (2^31 or more:
 * DCB_E_LIMIT), ONE radix sort, one reduce, one epilogue -- 11 launches. The workspace is plain scratch of
 * dcb_residual_det_workspace_bytes() bytes (DCB_FLAG_WS_CLEAN with it: DCB_E_MODE).
 */
int64_t dcb_residual_workspace_bytes(int64_t N, int64_t C, int64_t H, int64_t W);
/* workspace of dcb_residual_fused and dcb_residual_bidir with DCB_FLAG_DETERMINISTIC (one size serves both): keys, sorted
 * keys, the sort's temporary storage, the cells of both flows' splats */
int64_t dcb_residual_det_workspace_bytes(int64_t N, int64_t C, int64_t H, int64_t W);
int dcb_residual_fused(const DcbTensor* image1, const DcbTensor* flow1, const DcbTensor* flow2,
                       const DcbTensor* gt, const DcbTensor* fused, const DcbTensor* residual,
                       const DcbTensor* occ_fwd, const DcbTensor* occ_bwd,
                       void* workspace, int64_t workspace_bytes,
                       int32_t variant, int32_t flags, void* stream);

/*
 * Two-reference conditioning builder: the bidirectional blend the reference's datasets intended (SURVEY.md App. B-6) with the
 * mask <-> warp pairing of Bi_Dir_FeatureExtractor (controlnet/extractors.py:290-295), built from reference functions only:
 *   ones = all-ones metric
 *   warped1 = softsplat(image1, flow1, ones, 'soft');  warped2 = softsplat(image2, flow2, ones, 'soft')   (softsplat.py:232-274)
 *   occ_fwd = compute_mask(flow1, flow2);  occ_bwd = compute_mask(flow2, flow1)                          (control_utils.py:11-17)
 *   fused = soft_fuse(warped1, warped2, 1 - occ_fwd, 1 - occ_bwd)     (improv_experiments.ipynb cell 3: where both references
 *                                                                      are occluded, 0.5 * (warped1 + warped2))
 *   residual = gt - fused
 * image_k is moved by flow_k: the caller states the pairing (the reference's dataset and extractor pair the channels of
 * local_conditions with the flows in opposite ways). Rounding follows the composition: warps rounded to the tensor dtype,
 * fused stored, residual of the stored value. Two pipeline passes, four launches per frame group (image2 + flow1 splatted by
 * flow2 with the warp / occ_fwd epilogue; image1 + flow2 splatted by flow1 with the fuse / residual epilogue).
 *
 *   image1, image2, gt [N,C,H,W] (1 <= C <= 3; one dtype, F32 or BF16, for every tensor); flow1, flow2 [N,2,H,W];
 *   inputs may have any strides, a stride-0 batch included (one I-frame serving several inter frames)
 *   fused, residual [N,C,H,W] contiguous; occ_fwd / occ_bwd [N,1,H,W] optional outputs
 *   workspace: dcb_residual_workspace_bytes(N, C, H, W) -- the requirement is the same as dcb_residual_fused's;
 *   DCB_FLAG_WS_CLEAN protocol as dcb_residual_fused; DCB_FLAG_DETERMINISTIC as dcb_residual_fused (same workspace query)
 */
int dcb_residual_bidir(const DcbTensor* image1, const DcbTensor* image2, const DcbTensor* flow1, const DcbTensor* flow2,
                       const DcbTensor* gt, const DcbTensor* fused, const DcbTensor* residual,
                       const DcbTensor* occ_fwd, const DcbTensor* occ_bwd,
                       void* workspace, int64_t workspace_bytes, int32_t flags, void* stream);

/*
 * Confidence fusion of the two warped maps of a bi-directional block, without the host sync.
 * Replaces controlnet/extractors.py:298-310 (also :193-205 and controlnet/residual_utils.py:181-193):
 *   conf = clamp(cat(conf_a, conf_b), min=0); w = conf / (conf.sum(1) + 1e-6);
 *   fused = w0 * A + w1 * B;  where (occ_a + occ_b) > 1.5: fused = 0.5 * (A + B)
 * A, B [N,C,H,W]; conf_a, conf_b, occ_a, occ_b [N,1,H,W] (occ_* both NULL = no hole branch);
 * fused [N,C,H,W] contiguous. The backward fills grad_A, grad_B, grad_conf_a, grad_conf_b (any NULL).
 */
int dcb_bidir_fuse_fwd(const DcbTensor* A, const DcbTensor* B, const DcbTensor* conf_a, const DcbTensor* conf_b,
                       const DcbTensor* occ_a, const DcbTensor* occ_b, const DcbTensor* fused, void* stream);
int dcb_bidir_fuse_bwd(const DcbTensor* grad_fused, const DcbTensor* A, const DcbTensor* B,
                       const DcbTensor* conf_a, const DcbTensor* conf_b, const DcbTensor* occ_a, const DcbTensor* occ_b,
                       const DcbTensor* grad_A, const DcbTensor* grad_B, const DcbTensor* grad_conf_a,
                       const DcbTensor* grad_conf_b, void* stream);

/*
 * One bi-directional conditioning block (one pyramid scale) in ONE call: both occlusion masks, both soft splats with
 * their (1 - mask) product, the confidence fusion and the double-hole fill. Replaces, per scale, the body of
 * Bi_Dir_FeatureExtractor.forward between the conv stacks -- controlnet/extractors.py:289-310 (also :181-205 of
 * Bi_Dir_ResidueExtractor): compute_mask x2 (control_utils.py:11-17), FeatureWarperSoftsplat.forward x2
 * (control_utils.py:49-72, the metric_net conv excluded: pass its output as metric_*), the fusion and the
 * `holes.any()` host sync (extractors.py:298-310).
 *
 *   first, last   [N,C,H,W] feature maps;  flow_f, flow_b [N,2,H,W];  metric_f, metric_b [N,1,H,W] (the warper's
 *                 metric = the fusion confidence; pass ones for a warper without metric_net)
 *   fused         [N,C,H,W] contiguous: the block's result
 *   warped_*, norm_* (F32), occ_*: optional outputs (NULL = kept in scratch / not produced); the backward needs all six
 *   ws_acc        accumulator workspace (dcb_bidir_block_workspace_bytes(.., 0)); DCB_FLAG_WS_CLEAN protocol as dcb_splat_fwd
 *   ws_scratch    plain scratch (.., 1) for the optional outputs the caller left NULL
 * Backward: gradients w.r.t. both feature maps and both metrics (splat path + fusion path summed); it is the one-level
 * dcb_bidir_pyramid_bwd (two launches). ws: plain scratch (dcb_bidir_block_workspace_bytes(.., 2)).
 */
int64_t dcb_bidir_block_workspace_bytes(int64_t N, int64_t C, int64_t H, int64_t W, int32_t elem_dtype, int32_t which);
int dcb_bidir_block_fwd(const DcbTensor* first, const DcbTensor* last, const DcbTensor* flow_f, const DcbTensor* flow_b,
                        const DcbTensor* metric_f, const DcbTensor* metric_b, const DcbTensor* fused,
                        const DcbTensor* warped_f, const DcbTensor* warped_b, const DcbTensor* norm_f, const DcbTensor* norm_b,
                        const DcbTensor* occ_f, const DcbTensor* occ_b,
                        void* ws_acc, int64_t ws_acc_bytes, void* ws_scratch, int64_t ws_scratch_bytes, int32_t flags, void* stream);
int dcb_bidir_block_bwd(const DcbTensor* grad_fused, const DcbTensor* first, const DcbTensor* last,
                        const DcbTensor* flow_f, const DcbTensor* flow_b, const DcbTensor* metric_f, const DcbTensor* metric_b,
                        const DcbTensor* warped_f, const DcbTensor* warped_b, const DcbTensor* norm_f, const DcbTensor* norm_b,
                        const DcbTensor* occ_f, const DcbTensor* occ_b,
                        const DcbTensor* grad_first, const DcbTensor* grad_last, const DcbTensor* grad_metric_f,
                        const DcbTensor* grad_metric_b, void* workspace, int64_t workspace_bytes, void* stream);

/*
 * The motion compensation of a WHOLE conditioning pyramid -- every scale of one forward -- in ONE call and TWO kernel
 * launches (all scatter jobs of all scales; then masks + normalisation + (1 - mask) + confidence fusion + hole fill of all
 * scales), plus one memset. Per scale the arithmetic is that of dcb_bidir_block_fwd. Replaces, for the four scales of
 * Bi_Dir_FeatureExtractor.forward, controlnet/extractors.py:282-310 (16 softsplat() calls, 4 host syncs), and with
 * DCB_PYRAMID_NO_MASKS the multi-scale loop of improv_experiments.ipynb cell 5 (soft splat of both frames per scale +
 * soft_fuse with identity masks, cell 3: no occlusion test, no (1 - mask), no holes).
 *
 *   levels[l].first, last [N,C,H,W]; flow_f, flow_b [N,2,H,W] at the level's resolution; metric_f, metric_b [N,1,H,W]
 *   or NULL = all-ones (never materialised); one dtype (F32, BF16 or F16) for all tensors of all levels
 *   outputs are raw device pointers to NCHW-contiguous buffers of the level's shape and dtype (norm_*: F32):
 *   fused (required); warped_*, norm_*, occ_* optional (NULL = never stored; dcb_bidir_pyramid_bwd needs all six)
 *   n_levels <= 4;  workspace: dcb_bidir_pyramid_workspace_bytes(), DCB_FLAG_WS_CLEAN protocol as dcb_splat_fwd
 *   flags: DCB_PYRAMID_NO_MASKS, or DCB_PYRAMID_NO_HOLES: masks and (1 - mask) as usual, the fusion without the double-hole
 *   fill (Bi_Dir_ResidueExtractor, controlnet/extractors.py:193-199); NO_MASKS | NO_HOLES equals NO_MASKS
 *   DCB_FLAG_DETERMINISTIC (with or without NO_MASKS / NO_HOLES): bit-reproducible. Every splat of every level is one
 *   sort-then-reduce (emit, one radix sort, reduce; about 11 launches whatever the number of levels), in the order and with
 *   the arithmetic of dcb_splat_fwd's deterministic mode; in F32 the outputs equal, bit for bit, the composition of the
 *   deterministic single ops (soft splats of the flows for the masks, masked soft splats, dcb_bidir_fuse_fwd). The workspace is
 *   plain scratch of dcb_bidir_pyramid_det_workspace_bytes() bytes (DCB_FLAG_WS_CLEAN with it: DCB_E_MODE); 4 x N*H*W summed
 *   over levels and both directions must stay below 2^31 (else DCB_E_LIMIT). dcb_bidir_pyramid_bwd takes its saved outputs.
 */
typedef struct DcbPyramidLevel {
    const DcbTensor *first, *last, *flow_f, *flow_b, *metric_f, *metric_b;
    void *fused, *warped_f, *warped_b, *norm_f, *norm_b, *occ_f, *occ_b;
} DcbPyramidLevel;
enum { DCB_PYRAMID_NO_MASKS = 4, DCB_PYRAMID_NO_HOLES = 8 /* flags of dcb_bidir_pyramid_fwd (NO_HOLES: also of _bwd) */ };
int64_t dcb_bidir_pyramid_workspace_bytes(const DcbPyramidLevel* levels, int32_t n_levels);
/* workspace of dcb_bidir_pyramid_fwd with DCB_FLAG_DETERMINISTIC: keys, sorted keys, the sort's temporary storage, the cells */
int64_t dcb_bidir_pyramid_det_workspace_bytes(const DcbPyramidLevel* levels, int32_t n_levels);
int dcb_bidir_pyramid_fwd(const DcbPyramidLevel* levels, int32_t n_levels, void* workspace, int64_t workspace_bytes,
                          int32_t flags, void* stream);

/*
 * Backward of dcb_bidir_pyramid_fwd (with masks; with or without holes) for ALL levels in ONE call and TWO kernel launches
 * (every target pixel of every level; then one source-side gather per level and direction). Gradients w.r.t. both feature
 * maps, both flows (the splat weights' dependence on the flow, as dcb_splat_bwd) and both metrics (splat weights + fusion
 * confidences). The occlusion masks carry no gradient (compute_mask thresholds). No atomics: bit-identical run to run.
 *
 *   grad_fused [N,C,H,W] any strides; first, last, flow_f, flow_b, metric_f, metric_b as given to the forward (a NULL metric
 *   is the all-ones metric); one dtype (F32, BF16 or F16) for all tensors of all levels
 *   warped_*, norm_* (F32), occ_*: what the forward stored for the level (raw pointers, NCHW-contiguous), all six required
 *   grad_*: raw pointers to NCHW-contiguous buffers of the level's dtype, or NULL (not computed); fully overwritten.
 *   grad_metric_* must be NULL where the metric is NULL.
 *   1 <= n_levels <= 4;  flags: 0 or DCB_PYRAMID_NO_HOLES (as passed to the forward); workspace: plain scratch of
 *   dcb_bidir_pyramid_bwd_workspace_bytes() bytes (24 per pixel and level), 256-byte aligned
 */
typedef struct DcbPyramidBwdLevel {
    const DcbTensor *grad_fused, *first, *last, *flow_f, *flow_b, *metric_f, *metric_b;
    const void *warped_f, *warped_b, *norm_f, *norm_b, *occ_f, *occ_b;
    void *grad_first, *grad_last, *grad_flow_f, *grad_flow_b, *grad_metric_f, *grad_metric_b;
} DcbPyramidBwdLevel;
int64_t dcb_bidir_pyramid_bwd_workspace_bytes(const DcbPyramidBwdLevel* levels, int32_t n_levels);
int dcb_bidir_pyramid_bwd(const DcbPyramidBwdLevel* levels, int32_t n_levels, void* workspace, int64_t workspace_bytes,
                          int32_t flags, void* stream);

/*
 * Batched bilinear resampling: every (tensor, scale) pair of a pyramid in ONE launch. dst[j] [N,C,th,tw] (contiguous, F32,
 * BF16 or F16; src and dst in any mix) = bilinear(src[j] [N,C,H,W], any strides), then channel 0 (op) factor0 and every other channel (op) factor1.
 * The index and weight arithmetic is torch's upsample_bilinear2d (fp32, same operation order). Replaces the
 * F.interpolate calls in front of the splats: resize_and_normalize_flow_batched (controlnet/control_utils.py:74-97:
 * align_corners = 0, DIV by ((tw - 1) / 2, (th - 1) / 2)), extractors.py:182-183 (align_corners = 0, DIV by H // res),
 * improv_experiments.ipynb cell 5 (frames: NONE; flows: MUL by size / W), controlnet/utils.py:21-28 (align_corners = 1,
 * MUL by (tw / W, th / H)).
 */
enum { DCB_RESAMPLE_NONE = 0, DCB_RESAMPLE_MUL = 1, DCB_RESAMPLE_DIV = 2 };
typedef struct DcbResampleJob {
    const DcbTensor *src, *dst;
    int32_t align_corners, op;
    float factor0, factor1;
} DcbResampleJob;
int dcb_resample_batch(const DcbResampleJob* jobs, int32_t n_jobs, void* stream);

/*
 * Hann-window merge of overlapping latent tiles into one canvas, in one gather kernel.
 * Replaces merge_latent_tiles_from_pixel_coords(), patch_utils.py:83-174:
 *   per tile (list order): pixel rectangle -> latent rectangle (int(round()), clamped; the 4-tuple is
 *   read as (x1, x2, y1, y2), i.e. entries 2,3 scale with H / H_px and entries 0,1 with W / W_px, as the
 *   reference executes it); bilinear resize (align_corners = 0) if the stored tile size differs;
 *   mask = hann(h) x hann(w) / (max + 1e-12); out[rect] += tile * mask; weight[rect] += mask;
 *   merged = out / max(weight, eps).
 * tiles: array of n_tiles descriptors, each [1,C,th,tw] (any strides, dtype of `out`);
 * pixel_coords: n_tiles * 4 int64; out [N,C,H,W] contiguous (N > 1 receives N copies, like the
 * reference's broadcast); F32, BF16 or F16. Tiles whose rectangle is empty are skipped. Lists longer than
 * 48 tiles need a workspace (dcb_tile_merge_workspace_bytes), shorter ones none.
 */
int64_t dcb_tile_merge_workspace_bytes(int64_t C, int64_t H, int64_t W, int32_t n_tiles);
int dcb_tile_merge(const DcbTensor* tiles, const int64_t* pixel_coords, int32_t n_tiles, const DcbTensor* out,
                   int64_t H_px, int64_t W_px, double eps, void* workspace, int64_t workspace_bytes, void* stream);

/*
 * Flow ingest on the device: resample a flow field [N,2,H,W] (ANY strides -- a raw Middlebury .flo payload uploaded as it is
 * is the view with strides (2HW, 1, 2W, 2); the dataset reader's planar mis-reshape, controlnet/dataset.py:15-24, is the
 * view (2HW, HW, W, 1) of the same bytes) to out [N,2,th,tw] (contiguous, F32 or BF16) with one of the three conventions
 * the reference uses (DCB_FLOW_*). Replaces read_flo + resize_flow_to (controlnet/utils.py:10-28), load_flo_file +
 * fast_downsample_flow (controlnet/dataset.py:15-50) and resize_and_normalize_flow_batched (controlnet/control_utils.py:74-97).
 */
int dcb_flow_resize(const DcbTensor* flow, const DcbTensor* out, int32_t convention, void* stream);

/*
 * Element-type conversion on the device: dst[i] = (dst type)(scale * (float)src[i]) over n contiguous elements.
 * src: DCB_U8 | DCB_F16 | DCB_BF16 | DCB_F32; dst: DCB_F32 | DCB_BF16 | DCB_F16. The host-buffer entry point uploads
 * 8-bit frames and half-precision flows / metrics (9 instead of 24 bytes per pixel over PCIe) and downloads a bf16
 * result; the splat itself runs in fp32. Replaces the host-side `.astype(np.float32) / 255.0` of the reference's
 * dataset code (controlnet/dataset.py:224-230 feeds float arrays prepared on the CPU).
 */
int dcb_convert(const void* src, int32_t src_dtype, void* dst, int32_t dst_dtype, int64_t n, float scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DIFFCODEC_B200_H */
