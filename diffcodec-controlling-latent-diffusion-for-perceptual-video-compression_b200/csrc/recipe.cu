// recipe.cu -- occlusion mask and the conditioning builder (K5) for sm_100a.
//
// dcb_occlusion_mask replaces compute_mask(), controlnet/control_utils.py:11-17.
// dcb_residual_fused replaces the arithmetic of ResidueDataset.__getitem__
// (controlnet/dataset.py:233-265) and WarpingDatasetWrapper.__getitem__
// (controlnet/residual_utils.py:159-199): in the reference that is 4 softsplat() calls (each
// cat + memset + scatter + 3 post-ops), 2 norms, 2 compares and ~10 more eager kernels per frame,
// for a batch of ONE frame. Here, for a whole batch:
//
//   pass A  soft splat of flow1 by flow2 with the occlusion epilogue                         -> occ_fwd
//   pass B  soft splat of image1 AND of flow2 by flow1 in ONE scatter (same footprints, same all-ones metric, one shared
//           weight channel: float4 + float2 cells per pixel), and one epilogue per target pixel: normalise, occlusion
//           test (occ_bwd), fusion weights, optional double-hole fill, fused + residual stored once
//
// Both passes are the step pipeline of splat_pipe.cu (L2-resident accumulators, no memset, two launches per frame group).
// Round 1 ran three pipeline passes and an elementwise kernel (flow1 read twice, the warped image written, re-read and
// re-written); a first version that scattered all three splats from one kernel into 40 B/px of accumulators was 7x
// slower on 64 x 1080p because those accumulators (5.3 GB) lived in HBM (profiles/r01/NOTES.md).
// The three-pass composition remains for the forwards the recipe pass does not cover (owner kernels, small frames).
//
// dcb_residual_bidir (residual_bidir_impl) is the two-reference recipe (SURVEY.md App. B-6): image2 splatted by flow2 and
// image1 by flow1, masks with the pairing of extractors.py:290-295, soft_fuse, residual -- two rider passes of splat_pipe.cu
// (bidir_pipe_impl), or four single splats and k_recipe_fuse<T, true> for the forwards the pipeline does not cover.
//
// DCB_FLAG_DETERMINISTIC (both entries, F32): the recipe is one level of the deterministic pyramid's splats (pyramid_det_splats:
// emit, one radix sort, reduce) and one epilogue, k_recipe_det_fuse -- 11 launches per frame group, bit-identical to the
// composition of deterministic single ops (softsplat, compute_mask, the fusion ops, the subtraction).
#include "dcb_common.cuh"

namespace dcb {

// implemented in splat_pipe.cu
long long pipe_workspace(long long N, long long H, long long W);
int splat_pipe_impl(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const DcbTensor* out,
                    const DcbTensor* norm, const DcbTensor* mask, void* ws, int mode, int eps, bool ws_clean,
                    cudaStream_t st, bool ones_metric, const DcbTensor* mask_out);

long long recipe_pipe_workspace(long long N, long long H, long long W);
int recipe_pipe_impl(const DcbTensor* image1, const DcbTensor* flow1, const DcbTensor* flow2, const DcbTensor* gt,
                     const DcbTensor* fused, const DcbTensor* residual, const DcbTensor* occ_fwd, const DcbTensor* occ_bwd,
                     void* ws, int variant, cudaStream_t st);
int bidir_pipe_impl(const DcbTensor* image1, const DcbTensor* image2, const DcbTensor* flow1, const DcbTensor* flow2,
                    const DcbTensor* gt, const DcbTensor* fused, const DcbTensor* residual, const DcbTensor* occ_fwd,
                    const DcbTensor* occ_bwd, void* ws, cudaStream_t st);

// implemented in splat_owner.cu / splat_fwd.cu
long long owner_workspace(long long N, long long H, long long W);
bool use_owner(int dtype, int mode, long long C, long long H, long long W);
bool pipe_supported(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric);
int splat_owner_impl(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const DcbTensor* out,
                     const DcbTensor* norm, const DcbTensor* mask, void* ws, int mode, int eps, cudaStream_t st,
                     bool ones_metric, const DcbTensor* mask_out);

// implemented in splat_small.cu / splat_fwd.cu: small frames take one launch, one thread-block cluster per frame
bool small_frames(int dtype, int mode, long long N, long long C, long long H, long long W);
long long cluster_workspace(long long N, long long C, long long H, long long W, int mode);
int splat_cluster_impl(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const DcbTensor* out,
                       const DcbTensor* norm, const DcbTensor* mask, void* ws, int mode, int eps, bool ws_clean,
                       cudaStream_t st, bool ones_metric, const DcbTensor* mask_out);

// one soft splat with an all-ones metric through whichever forward applies (owner kernels, the cluster kernel for small
// frames, or the accumulator pipeline)
static int ones_splat(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* out, const DcbTensor* mask_out, void* ws,
                      bool owner, bool ws_clean, cudaStream_t st) {
    if (!pipe_supported(in, flow, nullptr))
        return set_error(DCB_E_LIMIT, "conditioning: tensor spans beyond 2^31 elements are not supported (32-bit in-frame offsets)");
    if (owner) return splat_owner_impl(in, flow, nullptr, out, nullptr, nullptr, ws, DCB_MODE_SOFT, DCB_EPS_ADD, st, true, mask_out);
    if (small_frames(in->dtype, DCB_MODE_SOFT, in->size[0], in->size[1], in->size[2], in->size[3]))
        return splat_cluster_impl(in, flow, nullptr, out, nullptr, nullptr, ws, DCB_MODE_SOFT, DCB_EPS_ADD, ws_clean, st, true, mask_out);
    return splat_pipe_impl(in, flow, nullptr, out, nullptr, nullptr, ws, DCB_MODE_SOFT, DCB_EPS_ADD, ws_clean, st, true, mask_out);
}

struct FuseArgs {
    View gt;
    void* fused;           // in: warped (two-reference form: warped2), out: fused   [N,C,H,W]
    void* residual;        // [N,C,H,W] (two-reference form: in warped1, out residual)
    const void* occ_fwd;   // [N,1,H,W]
    const void* occ_bwd;
    unsigned total, HW;
    int C, W;
    int variant;
};

// the fusion weights of the one-reference recipe: the torch ops of residual_utils._composed
__device__ __forceinline__ void recipe_weights(int variant, float of, float ob, float& w0, float& w1) {
    if (variant == DCB_RECIPE_DATASET) {          // dataset.py:255-259: masks are the confidences
        const float ws = add_rn(add_rn(of, ob), 0.000001f);
        w0 = of / ws; w1 = ob / ws;
    } else {                                      // residual_utils.py:181-185: ones are the confidences
        const float ws = add_rn(2.f, 0.000001f);
        w0 = 1.f / ws; w1 = w0;
    }
}

// BIDIR: the two-reference recipe (dcb_residual_bidir); warped1 arrives in `residual`, warped2 in `fused`, and the fusion is
// soft_fuse on the valid masks 1 - occ (bidir_soft_fuse); `variant` is not read
template <class T, bool BIDIR = false>
__global__ void __launch_bounds__(256) k_recipe_fuse(const FuseArgs a) {
    const unsigned p = blockIdx.x * 256 + threadIdx.x;
    if (p >= a.total) return;
    const unsigned n = p / a.HW, r = p - n * a.HW;
    const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
    const float of = ld_stream((const T*)a.occ_fwd + p), ob = ld_stream((const T*)a.occ_bwd + p);
    const T* gp = (const T*)a.gt.p + n * a.gt.sN + (long long)y * a.gt.sH + (long long)x * a.gt.sW;
    T* fo = (T*)a.fused + (long long)n * a.C * a.HW + r;
    T* ro = (T*)a.residual + (long long)n * a.C * a.HW + r;
    if (BIDIR) {
        for (int c = 0; c < a.C; ++c) {
            const float w1 = ld_stream(ro + (long long)c * a.HW), w2 = ld_stream(fo + (long long)c * a.HW);
            const float f = bidir_soft_fuse(w1, w2, of, ob);
            st_stream(fo + (long long)c * a.HW, f);
            st_stream(ro + (long long)c * a.HW, sub_rn(ld_stream(gp + (long long)c * a.gt.sC), round_as<T>(f)));   // residual of the stored value
        }
        return;
    }
    float w0, w1;
    recipe_weights(a.variant, of, ob, w0, w1);
    const bool hole = a.variant == DCB_RECIPE_WRAPPER && add_rn(of, ob) > 1.5f;   // residual_utils.py:190-193
    constexpr int U = 4;                                         // channels in flight: 2 * U loads per thread
    for (int c0 = 0; c0 < a.C; c0 += U) {
        float wv[U], gv[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const bool in = c0 + j < a.C;
            wv[j] = in ? ld_stream(fo + (long long)(c0 + j) * a.HW) : 0.f;                 // warped1 == warped2 (SURVEY.md B-6)
            gv[j] = in ? ld_stream(gp + (long long)(c0 + j) * a.gt.sC) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            if (c0 + j < a.C) {
                float fused = add_rn(mul_rn(w0, wv[j]), mul_rn(w1, wv[j]));
                if (hole) fused = mul_rn(0.5f, add_rn(wv[j], wv[j]));
                st_stream(fo + (long long)(c0 + j) * a.HW, fused);
                st_stream(ro + (long long)(c0 + j) * a.HW, sub_rn(gv[j], round_as<T>(fused)));   // residual of the stored (rounded) value
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
static long long splat_part(long long N, long long C, long long H, long long W) {
    if (use_owner(DCB_F32, DCB_MODE_SOFT, C, H, W)) return owner_workspace(N, H, W);
    if (small_frames(DCB_F32, DCB_MODE_SOFT, N, C, H, W)) return cluster_workspace(N, C, H, W, DCB_MODE_SOFT);
    return pipe_workspace(N, H, W);
}

long long mask_workspace(long long N, long long H, long long W) { return splat_part(N, 2, H, W); }

// the two-pass recipe runs when both forwards would take the accumulator pipeline
static bool recipe_two_pass(int dtype, long long N, long long C, long long H, long long W) {
    return !use_owner(dtype, DCB_MODE_SOFT, C, H, W) && !use_owner(dtype, DCB_MODE_SOFT, 2, H, W) &&
           !small_frames(dtype, DCB_MODE_SOFT, N, C, H, W) && !small_frames(dtype, DCB_MODE_SOFT, N, 2, H, W);
}

long long recipe_workspace(long long N, long long C, long long H, long long W) {
    // splat workspace (landing boxes, or pipeline accumulators) + two mask planes (sized for fp32) when the caller does not want them
    long long a = splat_part(N, C, H, W);
    const long long b = splat_part(N, 2, H, W), c = recipe_pipe_workspace(N, H, W);
    a = a > b ? a : b;
    return (a > c ? a : c) + 2 * align_up(N * H * W * 4, 256);
}

int occlusion_mask_impl(const DcbTensor* flow_a, const DcbTensor* flow_b, const DcbTensor* mask, void* ws,
                        long long ws_bytes, int flags, cudaStream_t st) {
    const long long N = flow_a->size[0], H = flow_a->size[2], W = flow_a->size[3];
    if (N * H * W == 0) return DCB_OK;
    const long long need = mask_workspace(N, H, W);
    if (need > 0 && (!ws || ws_bytes < need || ((uintptr_t)ws & 255)))
        return set_error(DCB_E_WORKSPACE, "occlusion_mask: workspace of %lld bytes required, got %lld", need, ws_bytes);
    // F16 comes only from the bi-directional block's launch sequence (dcb_bidir_block_fwd); dcb_occlusion_mask refuses it
    if (flow_a->dtype != DCB_F32 && !is_half_storage(flow_a->dtype))
        return set_error(DCB_E_DTYPE, "occlusion_mask: F32, BF16 or F16 only, got %d", flow_a->dtype);
    const bool owner = use_owner(flow_a->dtype, DCB_MODE_SOFT, 2, H, W), clean = (flags & DCB_FLAG_WS_CLEAN) != 0;
    const int rc = ones_splat(flow_a, flow_b, nullptr, mask, ws, owner, clean, st);
    if (rc == DCB_OK && owner && clean && need > 0) DCB_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)need, st));
    return rc;
}

template <class T, bool BIDIR = false> static int launch_fuse(const FuseArgs& a, cudaStream_t st) {
    k_recipe_fuse<T, BIDIR><<<(a.total + 255) / 256, 256, 0, st>>>(a);
    DCB_CHECK_LAUNCH("k_recipe_fuse");
    return DCB_OK;
}

int residual_fused_impl(const DcbTensor* image1, const DcbTensor* flow1, const DcbTensor* flow2, const DcbTensor* gt,
                        const DcbTensor* fused, const DcbTensor* residual, const DcbTensor* occ_fwd,
                        const DcbTensor* occ_bwd, void* ws, long long ws_bytes, int variant, int flags,
                        cudaStream_t st) {
    const long long N = image1->size[0], C = image1->size[1], H = image1->size[2], W = image1->size[3];
    if (N * H * W == 0) return DCB_OK;
    const long long need = recipe_workspace(N, C, H, W);
    if (!ws || ws_bytes < need || ((uintptr_t)ws & 255))
        return set_error(DCB_E_WORKSPACE, "residual_fused: workspace of %lld bytes required, got %lld", need, ws_bytes);
    if (image1->dtype != DCB_F32 && image1->dtype != DCB_BF16)
        return set_error(DCB_E_DTYPE, "residual_fused: F32 or BF16 only, got %d", image1->dtype);
    const bool clean = (flags & DCB_FLAG_WS_CLEAN) != 0;
    const long long plane = align_up(N * H * W * 4, 256), pipe_bytes = need - 2 * plane;
    const bool own_img = use_owner(image1->dtype, DCB_MODE_SOFT, C, H, W), own_flow = use_owner(image1->dtype, DCB_MODE_SOFT, 2, H, W);
    // the mask planes live behind the accumulators; they are scratch (not part of the clean region)
    DcbTensor m1 = *flow1, m2 = *flow1;
    m1.size[1] = m2.size[1] = 1;
    m1.stride[0] = m2.stride[0] = H * W; m1.stride[1] = m2.stride[1] = H * W; m1.stride[2] = m2.stride[2] = W; m1.stride[3] = m2.stride[3] = 1;
    m1.ptr = (char*)ws + pipe_bytes;
    m2.ptr = (char*)ws + pipe_bytes + plane;
    const DcbTensor* pf = occ_fwd ? occ_fwd : &m1;
    const DcbTensor* pb = occ_bwd ? occ_bwd : &m2;

    if (recipe_two_pass(image1->dtype, N, C, H, W)) {
        if (!pipe_supported(image1, flow1, nullptr) || !pipe_supported(flow2, flow1, nullptr) || !pipe_supported(gt, flow2, nullptr))
            return set_error(DCB_E_LIMIT, "conditioning: tensor spans beyond 2^31 elements are not supported (32-bit in-frame offsets)");
        if (!clean) DCB_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)pipe_bytes, st));
        // pass A: compute_mask(flow1, flow2) = flow1 splatted by flow2
        int rc = splat_pipe_impl(flow1, flow2, nullptr, nullptr, nullptr, nullptr, ws, DCB_MODE_SOFT, DCB_EPS_ADD, true, st, true, pf);
        if (rc != DCB_OK) return rc;
        // pass B: image1 and flow2 ride on flow1; compute_mask(flow2, flow1), fusion and residual in its epilogue
        return recipe_pipe_impl(image1, flow1, flow2, gt, fused, residual, pf, occ_bwd, ws, variant, st);
    }

    // a pipeline pass after an owner pass would find landing boxes where it expects all-zero accumulators
    const bool mixed = own_img != own_flow;
    int rc = ones_splat(image1, flow1, fused, nullptr, ws, own_img, clean, st);
    if (rc != DCB_OK) return rc;
    if (mixed && own_img) DCB_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)pipe_bytes, st));
    // compute_mask(flow1, flow2): flow1 splatted by flow2; compute_mask(flow2, flow1): the other way round
    rc = ones_splat(flow1, flow2, nullptr, pf, ws, own_flow, !own_img || mixed, st);
    if (rc != DCB_OK) return rc;
    rc = ones_splat(flow2, flow1, nullptr, pb, ws, own_flow, true, st);
    if (rc != DCB_OK) return rc;
    if (clean && own_flow && pipe_bytes > 0) DCB_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)pipe_bytes, st));

    FuseArgs a;
    a.gt = make_view(gt);
    a.fused = fused->ptr; a.residual = residual->ptr;
    a.occ_fwd = pf->ptr; a.occ_bwd = pb->ptr;
    a.HW = (unsigned)(H * W); a.total = (unsigned)(N * H * W);
    a.C = (int)C; a.W = (int)W; a.variant = variant;
    if (image1->dtype == DCB_F32) return launch_fuse<float>(a, st);
    return launch_fuse<__nv_bfloat16>(a, st);
}

// Two references (dcb_residual_bidir): image_k moved by flow_k, fused by occlusion (extractors.py:290-295 pairing), subtracted.
// The workspace requirement is recipe_workspace(): the same splat parts (C-channel images, 2-channel flows), the same rider
// pipeline slot and the same two mask planes.
int residual_bidir_impl(const DcbTensor* image1, const DcbTensor* image2, const DcbTensor* flow1, const DcbTensor* flow2,
                        const DcbTensor* gt, const DcbTensor* fused, const DcbTensor* residual, const DcbTensor* occ_fwd,
                        const DcbTensor* occ_bwd, void* ws, long long ws_bytes, int flags, cudaStream_t st) {
    const long long N = image1->size[0], C = image1->size[1], H = image1->size[2], W = image1->size[3];
    if (N * H * W == 0) return DCB_OK;
    const long long need = recipe_workspace(N, C, H, W);
    if (!ws || ws_bytes < need || ((uintptr_t)ws & 255))
        return set_error(DCB_E_WORKSPACE, "residual_bidir: workspace of %lld bytes required, got %lld", need, ws_bytes);
    if (image1->dtype != DCB_F32 && image1->dtype != DCB_BF16)
        return set_error(DCB_E_DTYPE, "residual_bidir: F32 or BF16 only, got %d", image1->dtype);
    const bool clean = (flags & DCB_FLAG_WS_CLEAN) != 0;
    const long long plane = align_up(N * H * W * 4, 256), pipe_bytes = need - 2 * plane;
    const bool own_img = use_owner(image1->dtype, DCB_MODE_SOFT, C, H, W), own_flow = use_owner(image1->dtype, DCB_MODE_SOFT, 2, H, W);
    // the mask planes live behind the accumulators; they are scratch (not part of the clean region)
    DcbTensor m1 = *flow1, m2 = *flow1;
    m1.size[1] = m2.size[1] = 1;
    m1.stride[0] = m2.stride[0] = H * W; m1.stride[1] = m2.stride[1] = H * W; m1.stride[2] = m2.stride[2] = W; m1.stride[3] = m2.stride[3] = 1;
    m1.ptr = (char*)ws + pipe_bytes;
    m2.ptr = (char*)ws + pipe_bytes + plane;
    const DcbTensor* pf = occ_fwd ? occ_fwd : &m1;
    const DcbTensor* pb = occ_bwd ? occ_bwd : &m2;

    if (recipe_two_pass(image1->dtype, N, C, H, W)) {
        if (!pipe_supported(image1, flow1, nullptr) || !pipe_supported(image2, flow2, nullptr) || !pipe_supported(flow1, flow2, nullptr) ||
            !pipe_supported(gt, flow2, nullptr))
            return set_error(DCB_E_LIMIT, "conditioning: tensor spans beyond 2^31 elements are not supported (32-bit in-frame offsets)");
        if (!clean) DCB_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)pipe_bytes, st));
        return bidir_pipe_impl(image1, image2, flow1, flow2, gt, fused, residual, pf, occ_bwd, ws, st);
    }

    // warped1 in `residual`, warped2 in `fused` (temporaries the fusion kernel reads and overwrites); memsets as in
    // residual_fused_impl: a pipeline pass after an owner pass would find landing boxes where it expects all-zero accumulators
    const bool mixed = own_img != own_flow;
    int rc = ones_splat(image1, flow1, residual, nullptr, ws, own_img, clean, st);
    if (rc != DCB_OK) return rc;
    rc = ones_splat(image2, flow2, fused, nullptr, ws, own_img, !own_img, st);
    if (rc != DCB_OK) return rc;
    if (mixed && own_img) DCB_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)pipe_bytes, st));
    // compute_mask(flow1, flow2): flow1 splatted by flow2; compute_mask(flow2, flow1): the other way round
    rc = ones_splat(flow1, flow2, nullptr, pf, ws, own_flow, !own_img || mixed, st);
    if (rc != DCB_OK) return rc;
    rc = ones_splat(flow2, flow1, nullptr, pb, ws, own_flow, true, st);
    if (rc != DCB_OK) return rc;
    if (clean && own_flow && pipe_bytes > 0) DCB_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)pipe_bytes, st));

    FuseArgs a;
    a.gt = make_view(gt);
    a.fused = fused->ptr; a.residual = residual->ptr;
    a.occ_fwd = pf->ptr; a.occ_bwd = pb->ptr;
    a.HW = (unsigned)(H * W); a.total = (unsigned)(N * H * W);
    a.C = (int)C; a.W = (int)W; a.variant = 0;
    if (image1->dtype == DCB_F32) return launch_fuse<float, true>(a, st);
    return launch_fuse<__nv_bfloat16, true>(a, st);
}

// ---------------------------------------------------------------------------------------------
// DCB_FLAG_DETERMINISTIC: both recipes as one level of the deterministic pyramid's splats (pyramid.cu) and one epilogue
// ---------------------------------------------------------------------------------------------
// The recipe is one pyramid level with flow_f = flow1, flow_b = flow2: field 1 (flow1's footprints) carries image1 and flow2
// (occ_bwd = compute_mask(flow2, flow1)), field 2 (flow2's footprints) carries flow1 (occ_fwd = compute_mask(flow1, flow2)) and,
// in the two-reference recipe, image2. pyramid_det_splats writes the cells; k_recipe_det_fuse does the rest per target pixel.
enum { kRecipeBidir = 2 };   // the third form of k_recipe_det_fuse, next to DCB_RECIPE_DATASET and DCB_RECIPE_WRAPPER

struct RecipeDetArgs {
    View flow1, flow2, gt;
    PyrCells cells;          // C <= 3: one channel quad, so every cell of pixel p sits at index p
    float *fused, *residual, *occ_fwd, *occ_bwd;
    unsigned total, HW;
    int C, W;
};

// Each step is the arithmetic of the composition of deterministic single ops (residual_utils._composed / _composed_bidir):
// warps divided as k_normalize divides, masks by occlusion() (compute_mask), fusion by the k_recipe_fuse weights or
// bidir_soft_fuse (bidir_fuse on the valid masks), residual = gt - fused.
template <int KIND>
__global__ void __launch_bounds__(256) k_recipe_det_fuse(const RecipeDetArgs a) {
    pdl_wait();
    const unsigned p = blockIdx.x * 256 + threadIdx.x;
    if (p >= a.total) return;
    const unsigned n = p / a.HW, r = p - n * a.HW;
    const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
    const PyrCells& c = a.cells;
    const float* f1 = (const float*)a.flow1.p + n * a.flow1.sN + (long long)y * a.flow1.sH + (long long)x * a.flow1.sW;
    const float* f2 = (const float*)a.flow2.p + n * a.flow2.sN + (long long)y * a.flow2.sH + (long long)x * a.flow2.sW;
    const float4 mf = ((const float4*)c.acc_mf)[p], mb = ((const float4*)c.acc_mb)[p];
    const float of = occlusion(mf.x, mf.y, c.dacc_mf[p], f2[0], f2[a.flow2.sC]);
    const float ob = occlusion(mb.x, mb.y, c.dacc_mb[p], f1[0], f1[a.flow1.sC]);
    if (a.occ_fwd) a.occ_fwd[p] = of;
    if (a.occ_bwd) a.occ_bwd[p] = ob;
    // normalisers of softsplat.py:256-258 ('soft' = add 1e-7)
    const float d1 = add_rn(c.dacc_f[p], 0.0000001f);
    const float4 s1 = ((const float4*)c.acc_f)[p];
    const float v1[3] = {s1.x, s1.y, s1.z};
    float v2[3] = {0.f, 0.f, 0.f}, d2 = 1.f;
    if constexpr (KIND == kRecipeBidir) {
        const float4 s2 = ((const float4*)c.acc_b)[p];
        v2[0] = s2.x; v2[1] = s2.y; v2[2] = s2.z;
        d2 = add_rn(c.dacc_b[p], 0.0000001f);
    }
    float w0 = 0.f, w1 = 0.f;
    bool hole = false;
    if constexpr (KIND != kRecipeBidir) {
        recipe_weights(KIND, of, ob, w0, w1);
        hole = KIND == DCB_RECIPE_WRAPPER && add_rn(of, ob) > 1.5f;
    }
    const float* gp = (const float*)a.gt.p + n * a.gt.sN + (long long)y * a.gt.sH + (long long)x * a.gt.sW;
    float* fo = a.fused + (size_t)n * a.C * a.HW + r;
    float* ro = a.residual + (size_t)n * a.C * a.HW + r;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        if (ch >= a.C) break;
        const float A = v1[ch] / d1;
        float f;
        if constexpr (KIND == kRecipeBidir) {
            f = bidir_soft_fuse(A, v2[ch] / d2, of, ob);
        } else {
            f = hole ? mul_rn(0.5f, add_rn(A, A)) : add_rn(mul_rn(w0, A), mul_rn(w1, A));   // warped2 is warped1 (SURVEY.md B-6)
        }
        st_stream(fo + (size_t)ch * a.HW, f);
        st_stream(ro + (size_t)ch * a.HW, sub_rn(ld<float>(gp + (long long)ch * a.gt.sC), f));
    }
}

static DcbPyramidLevel recipe_level(const DcbTensor* first) {
    DcbPyramidLevel lv = {};
    lv.first = first;
    return lv;
}

// sized for the two-reference recipe (C channels on both fields); the one-reference recipe uses the same layout
long long recipe_det_workspace(long long N, long long C, long long H, long long W) {
    DcbTensor t = {};
    t.dtype = DCB_F32;
    t.size[0] = N; t.size[1] = C; t.size[2] = H; t.size[3] = W;
    const DcbPyramidLevel lv = recipe_level(&t);
    return pyramid_det_workspace(&lv, 1);
}

// image2 NULL: the one-reference recipe (`variant`); else the two-reference recipe. Shapes and dtypes checked by the caller.
int residual_det_impl(const DcbTensor* image1, const DcbTensor* image2, const DcbTensor* flow1, const DcbTensor* flow2,
                      const DcbTensor* gt, const DcbTensor* fused, const DcbTensor* residual, const DcbTensor* occ_fwd,
                      const DcbTensor* occ_bwd, void* ws, long long ws_bytes, int variant, cudaStream_t st) {
    const long long N = image1->size[0], C = image1->size[1], H = image1->size[2], W = image1->size[3];
    if (image1->dtype != DCB_F32)
        return set_error(DCB_E_DTYPE, "residual(deterministic): F32 only, got %d", image1->dtype);
    if (N * H * W == 0) return DCB_OK;
    if (8 * N * H * W >= (1ll << 31))
        return set_error(DCB_E_LIMIT, "residual(deterministic): 8 keys per pixel, 8*N*H*W must stay below 2^31 (got %lld)", 8 * N * H * W);
    const long long need = recipe_det_workspace(N, C, H, W);
    if (!ws || ws_bytes < need || ((uintptr_t)ws & 255))
        return set_error(DCB_E_WORKSPACE, "residual(deterministic): workspace of %lld bytes (256 B aligned) required, got %lld", need, ws_bytes);
    DcbPyramidLevel lv = recipe_level(image1);
    lv.last = image2; lv.flow_f = flow1; lv.flow_b = flow2;
    RecipeDetArgs a;
    int rc = pyramid_det_splats(&lv, 1, ws, true, &a.cells, st);
    if (rc != DCB_OK) return rc;
    a.flow1 = make_view(flow1); a.flow2 = make_view(flow2); a.gt = make_view(gt);
    a.fused = (float*)fused->ptr; a.residual = (float*)residual->ptr;
    a.occ_fwd = occ_fwd ? (float*)occ_fwd->ptr : nullptr; a.occ_bwd = occ_bwd ? (float*)occ_bwd->ptr : nullptr;
    a.HW = (unsigned)(H * W); a.total = (unsigned)(N * H * W);
    a.C = (int)C; a.W = (int)W;
    const dim3 grid((a.total + 255) / 256);
    if (image2) DCB_CHECK_CUDA(launch_pdl(k_recipe_det_fuse<kRecipeBidir>, grid, dim3(256), 0, st, a));
    else if (variant == DCB_RECIPE_DATASET) DCB_CHECK_CUDA(launch_pdl(k_recipe_det_fuse<DCB_RECIPE_DATASET>, grid, dim3(256), 0, st, a));
    else DCB_CHECK_CUDA(launch_pdl(k_recipe_det_fuse<DCB_RECIPE_WRAPPER>, grid, dim3(256), 0, st, a));
    count_launch();
    return DCB_OK;
}

}  // namespace dcb
