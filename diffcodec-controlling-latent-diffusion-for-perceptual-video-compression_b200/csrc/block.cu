// block.cu -- the motion-compensation part of one bi-directional conditioning block as ONE C call per pyramid scale
// (SURVEY.md section 8, row f-1), sm_100a.
//
// Replaces, per scale, controlnet/extractors.py:289-310 (and :181-205): two compute_mask() calls
// (control_utils.py:11-17), two FeatureWarperSoftsplat splats with (1 - mask) (control_utils.py:61-72), the confidence
// fusion and the double-hole fill with its `holes.any()` host sync (extractors.py:298-310) -- in the reference ~45 eager
// kernels, 4 NVRTC cache lookups and one device->host stall per scale; in round 1 five library calls from Python. Here
// the host enters the library once. Scales whose accumulators fit the L2 (every pyramid level of the live consumer) run
// as TWO launches (pyramid.cu: all four scatter jobs, then masks + normalisation + fusion); bigger tensors run the
// kernels of recipe.cu / splat_*.cu / fuse.cu back to back on the caller's stream. The backward of every size is the
// one-level pyramid backward (pyramid_bwd.cu, two launches).
#include "dcb_common.cuh"

namespace dcb {

long long mask_workspace(long long N, long long H, long long W);
long long splat_fwd_workspace(long long N, long long C, long long H, long long W, int dtype, int mode);
int occlusion_mask_impl(const DcbTensor*, const DcbTensor*, const DcbTensor*, void*, long long, int, cudaStream_t);
int splat_fwd_impl(const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, void*,
                   long long, int, int, int, cudaStream_t);
int bidir_fuse_fwd_impl(const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*,
                        const DcbTensor*, cudaStream_t);

// pyramid.cu: the two-launch form (every scatter job in one launch, everything else in a second)
long long pyramid_workspace(const DcbPyramidLevel* lv, int n);
int bidir_pyramid_fwd_impl(const DcbPyramidLevel* lv, int n, void* ws, int flags, cudaStream_t st);
long long pyramid_bwd_workspace(const DcbPyramidBwdLevel* lv, int n);
int bidir_pyramid_bwd_impl(const DcbPyramidBwdLevel* lv, int n, void* ws, bool holes, cudaStream_t st);

// One scale goes through the two-launch pyramid kernels when the accumulators of BOTH directions fit the L2 together
// (every pyramid level of the live consumer does); bigger tensors keep the launch sequence below (frame-group pipeline
// or per-target lists per splat).
constexpr long long kFusedLevelBytes = 48ll << 20;
static long long fused_level_bytes(long long N, long long C, long long H, long long W, int dtype) {
    DcbTensor t = {};
    t.dtype = dtype; t.size[0] = N; t.size[1] = C; t.size[2] = H; t.size[3] = W;
    DcbPyramidLevel lv = {};
    lv.first = &t;
    return pyramid_workspace(&lv, 1);
}
static bool block_is_fused(long long N, long long C, long long H, long long W, int dtype) {
    return (dtype == DCB_F32 || is_half_storage(dtype)) && fused_level_bytes(N, C, H, W, dtype) <= kFusedLevelBytes;
}

static DcbTensor contiguous_like(const DcbTensor* t, long long C, int dtype, void* ptr) {
    DcbTensor r = *t;
    r.ptr = ptr; r.dtype = dtype;
    r.size[1] = C;
    r.stride[3] = 1; r.stride[2] = t->size[3]; r.stride[1] = t->size[2] * t->size[3]; r.stride[0] = C * r.stride[1];
    return r;
}

long long block_fwd_acc_bytes(long long N, long long C, long long H, long long W, int dtype) {
    const long long a = mask_workspace(N, H, W), b = splat_fwd_workspace(N, C, H, W, dtype, DCB_MODE_SOFT);
    const long long c = block_is_fused(N, C, H, W, dtype) ? fused_level_bytes(N, C, H, W, dtype) : 0;
    return a > b ? (a > c ? a : c) : (b > c ? b : c);
}

// scratch of the forward: whatever of {warped_f, warped_b, occ_f, occ_b} the caller does not want back
long long block_fwd_scratch_bytes(long long N, long long C, long long H, long long W, int dtype) {
    const long long s = elem_size(dtype);
    return 2 * align_up(N * C * H * W * s, 256) + 2 * align_up(N * H * W * s, 256);
}

// scratch of the backward: that of the one-level pyramid backward (both directions' target scalars, both confidence gradients)
long long block_bwd_scratch_bytes(long long N, long long C, long long H, long long W, int dtype) {
    DcbTensor t = {};
    t.dtype = dtype; t.size[0] = N; t.size[1] = C; t.size[2] = H; t.size[3] = W;
    DcbPyramidBwdLevel lv = {};
    lv.first = &t;
    return pyramid_bwd_workspace(&lv, 1);
}

int bidir_block_fwd_impl(const DcbTensor* first, const DcbTensor* last, const DcbTensor* flow_f, const DcbTensor* flow_b,
                         const DcbTensor* metric_f, const DcbTensor* metric_b, const DcbTensor* fused, const DcbTensor* warped_f,
                         const DcbTensor* warped_b, const DcbTensor* norm_f, const DcbTensor* norm_b, const DcbTensor* occ_f,
                         const DcbTensor* occ_b, void* ws_acc, long long acc_bytes, void* ws_scratch, long long scratch_bytes, int flags,
                         cudaStream_t st) {
    const long long N = first->size[0], C = first->size[1], H = first->size[2], W = first->size[3];
    if (N * C * H * W == 0) return DCB_OK;
    const int dt = first->dtype;
    if (block_is_fused(N, C, H, W, dt)) {
        // two launches for the scale (SURVEY.md section 8, row f-1): outputs the caller does not ask for are never stored
        const long long need = block_fwd_acc_bytes(N, C, H, W, dt);
        if (!ws_acc || acc_bytes < need || ((uintptr_t)ws_acc & 255))
            return set_error(DCB_E_WORKSPACE, "bidir_block_fwd: accumulator workspace of %lld bytes (256 B aligned) required, got %lld", need, acc_bytes);
        DcbPyramidLevel lv = {};
        lv.first = first; lv.last = last; lv.flow_f = flow_f; lv.flow_b = flow_b; lv.metric_f = metric_f; lv.metric_b = metric_b;
        lv.fused = fused->ptr;
        lv.warped_f = warped_f ? warped_f->ptr : nullptr; lv.warped_b = warped_b ? warped_b->ptr : nullptr;
        lv.norm_f = norm_f ? norm_f->ptr : nullptr; lv.norm_b = norm_b ? norm_b->ptr : nullptr;
        lv.occ_f = occ_f ? occ_f->ptr : nullptr; lv.occ_b = occ_b ? occ_b->ptr : nullptr;
        return bidir_pyramid_fwd_impl(&lv, 1, ws_acc, flags & DCB_FLAG_WS_CLEAN, st);
    }
    const long long s = elem_size(dt), big = align_up(N * C * H * W * s, 256), plane = align_up(N * H * W * s, 256);
    char* sc = (char*)ws_scratch;
    long long used = 0;
    DcbTensor t_wf, t_wb, t_of, t_ob;
    auto take = [&](const DcbTensor* given, DcbTensor& slot, long long Cx, long long bytes) -> const DcbTensor* {
        if (given) return given;
        slot = contiguous_like(first, Cx, dt, sc + used);
        used += bytes;
        return &slot;
    };
    const DcbTensor* wf = take(warped_f, t_wf, C, big);
    const DcbTensor* wb = take(warped_b, t_wb, C, big);
    const DcbTensor* of = take(occ_f, t_of, 1, plane);
    const DcbTensor* ob = take(occ_b, t_ob, 1, plane);
    if (used > 0 && (!ws_scratch || scratch_bytes < used || ((uintptr_t)ws_scratch & 255)))
        return set_error(DCB_E_WORKSPACE, "bidir_block_fwd: scratch of %lld bytes (256 B aligned) required, got %lld", used, scratch_bytes);
    const long long need = block_fwd_acc_bytes(N, C, H, W, dt);
    if (need > 0 && (!ws_acc || acc_bytes < need || ((uintptr_t)ws_acc & 255)))
        return set_error(DCB_E_WORKSPACE, "bidir_block_fwd: accumulator workspace of %lld bytes (256 B aligned) required, got %lld", need, acc_bytes);
    const int clean = flags & DCB_FLAG_WS_CLEAN;
    // occ_fwd = compute_mask(flow_f, flow_b), occ_bwd = compute_mask(flow_b, flow_f)      extractors.py:290-291
    int rc = occlusion_mask_impl(flow_f, flow_b, of, ws_acc, acc_bytes, clean, st);
    if (rc != DCB_OK) return rc;
    rc = occlusion_mask_impl(flow_b, flow_f, ob, ws_acc, acc_bytes, DCB_FLAG_WS_CLEAN, st);
    if (rc != DCB_OK) return rc;
    // warped = softsplat(feat, flow, metric, 'soft') * (1 - mask)                          control_utils.py:62-70
    rc = splat_fwd_impl(first, flow_f, metric_f, wf, norm_f, of, ws_acc, acc_bytes, DCB_MODE_SOFT, DCB_EPS_ADD, DCB_FLAG_WS_CLEAN, st);
    if (rc != DCB_OK) return rc;
    rc = splat_fwd_impl(last, flow_b, metric_b, wb, norm_b, ob, ws_acc, acc_bytes, DCB_MODE_SOFT, DCB_EPS_ADD, DCB_FLAG_WS_CLEAN, st);
    if (rc != DCB_OK) return rc;
    // confidence fusion + double-hole fill, no host sync                                   extractors.py:298-310
    return bidir_fuse_fwd_impl(wf, wb, metric_f, metric_b, of, ob, fused, st);
}

// the one-level pyramid backward (pyramid_bwd.cu): two launches whatever the size, with the double-hole fill of the forward
int bidir_block_bwd_impl(const DcbTensor* g, const DcbTensor* first, const DcbTensor* last, const DcbTensor* flow_f,
                         const DcbTensor* flow_b, const DcbTensor* metric_f, const DcbTensor* metric_b, const DcbTensor* warped_f,
                         const DcbTensor* warped_b, const DcbTensor* norm_f, const DcbTensor* norm_b, const DcbTensor* occ_f,
                         const DcbTensor* occ_b, const DcbTensor* g_first, const DcbTensor* g_last, const DcbTensor* g_metric_f,
                         const DcbTensor* g_metric_b, void* ws, long long ws_bytes, cudaStream_t st) {
    const long long N = first->size[0], C = first->size[1], H = first->size[2], W = first->size[3];
    if (N * C * H * W == 0) return DCB_OK;
    const long long need = block_bwd_scratch_bytes(N, C, H, W, first->dtype);
    if (!ws || ws_bytes < need || ((uintptr_t)ws & 255))
        return set_error(DCB_E_WORKSPACE, "bidir_block_bwd: scratch of %lld bytes (256 B aligned) required, got %lld", need, ws_bytes);
    auto ptr = [](const DcbTensor* t) -> void* { return t ? t->ptr : nullptr; };
    DcbPyramidBwdLevel lv = {};
    lv.grad_fused = g; lv.first = first; lv.last = last; lv.flow_f = flow_f; lv.flow_b = flow_b; lv.metric_f = metric_f; lv.metric_b = metric_b;
    lv.warped_f = warped_f->ptr; lv.warped_b = warped_b->ptr; lv.norm_f = norm_f->ptr; lv.norm_b = norm_b->ptr;
    lv.occ_f = occ_f->ptr; lv.occ_b = occ_b->ptr;
    lv.grad_first = ptr(g_first); lv.grad_last = ptr(g_last); lv.grad_metric_f = ptr(g_metric_f); lv.grad_metric_b = ptr(g_metric_b);
    return bidir_pyramid_bwd_impl(&lv, 1, ws, true, st);
}

}  // namespace dcb
