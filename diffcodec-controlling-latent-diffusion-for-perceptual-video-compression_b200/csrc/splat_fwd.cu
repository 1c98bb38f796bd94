// splat_fwd.cu -- forward splat: dispatch, plus the plain two-kernel path (K1 scatter + K2
// normalise) that serves fp64 tensors and the epilogue of the deterministic mode. sm_100a.
//
// Replaces controlnet/softsplat.py:232-274 (mode wrapper: cat / exp / mul pre-ops, eps + divide
// post-ops) and :277-355 (softsplat_func.forward, kernel `softsplat_out`) of the reference.
//
//   fp32 / bf16 / fp16, C + 1 <= 4 (frames, flows, SD latents)  -> splat_pipe.cu   (float4 accumulators)
//   fp32 / bf16 / fp16, more channels (feature maps)             -> splat_planar.cu (channel-quad accumulators),
//                                      and >= 16 MB of them -> splat_lists.cu  (per-target lists + gather)
//   fp64 (the reference supports double; gradcheck uses it) -> this file
//
// The plain path: one thread per SOURCE PIXEL (flow read once, weights computed once per pixel;
// the reference does both once per channel), the appended channel (1 | m | exp(m)) and the
// in*g(m) product formed in registers, double-precision atomics into planar accumulators, then a
// normalise kernel that applies the eps rule, the TRUE division of softsplat.py:270, the optional
// (1 - mask) product and the cast.
#include "dcb_common.cuh"

namespace dcb {

constexpr int kThreads = 256;

struct FwdArgs {
    View in, flow, metric, mask;
    void* acc;       // planar accumulators (workspace, or `out` itself for SUM)
    void* out;       // [N,C,H,W] contiguous
    void* norm;      // optional [N,1,H,W] accumulator-typed
    unsigned total;  // N*H*W
    unsigned HW;
    int N, C, H, W;
    int Cacc;        // channels held by the accumulators: C (SUM) or C+1
    int cgroup;      // channels per blockIdx.y
    int mode, eps;
    int rezero;      // K2 leaves the accumulators zeroed
};

// ---------------------------------------------------------------------------------------------
// K1: planar accumulators, any C. grid = (ceil(total/256), ceil(Cacc/cgroup)).
// ---------------------------------------------------------------------------------------------
template <class T, class TF>
__global__ void __launch_bounds__(kThreads) k_scatter_planar(const FwdArgs a) {
    using A = typename Acc<T>::type;
    const unsigned p = blockIdx.x * kThreads + threadIdx.x;
    if (p >= a.total) return;
    const unsigned n = p / a.HW, r = p - n * a.HW;
    const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);

    const TF* fp = (const TF*)a.flow.p + n * a.flow.sN + y * a.flow.sH + x * a.flow.sW;
    const Foot<A> f = make_foot<A>(x, y, ld<A>(fp), ld<A>(fp + a.flow.sC));
    if (!f.finite) return;                                        // softsplat.py:301-302

    const int W = a.W, H = a.H;
    const int x1 = (int)((unsigned)f.x0 + 1u), y1 = (int)((unsigned)f.y0 + 1u);
    const bool vx0 = (unsigned)f.x0 < (unsigned)W, vx1 = (unsigned)x1 < (unsigned)W;
    const bool vy0 = (unsigned)f.y0 < (unsigned)H, vy1 = (unsigned)y1 < (unsigned)H;
    const bool bnw = vx0 && vy0, bne = vx1 && vy0, bsw = vx0 && vy1, bse = vx1 && vy1;
    if (!(bnw || bne || bsw || bse)) return;
    const long long onw = (long long)f.y0 * W + f.x0;             // only dereferenced for in-range corners

    A g = (A)1;                                                   // g(m) of softsplat.py:240-247
    if (a.mode == DCB_MODE_LINEAR || a.mode == DCB_MODE_SOFT) {
        const T* mp = (const T*)a.metric.p + n * a.metric.sN + y * a.metric.sH + x * a.metric.sW;
        const A m = ld<A>(mp);
        g = a.mode == DCB_MODE_SOFT ? exp_t(m) : m;
    }

    const int c0 = blockIdx.y * a.cgroup;
    const int c1 = min(a.Cacc, c0 + a.cgroup);
    const T* ip = (const T*)a.in.p + n * a.in.sN + y * a.in.sH + x * a.in.sW + c0 * a.in.sC;
    A* acc = (A*)a.acc + ((long long)n * a.Cacc + c0) * a.HW + onw;
    for (int c = c0; c < c1; ++c, ip += a.in.sC, acc += a.HW) {
        A v;
        if (c < a.C) {
            v = ld<A>(ip);
            if (a.mode >= DCB_MODE_LINEAR) v = mul_rn(v, g);      // in * m  /  in * exp(m)
        } else {
            v = g;                                                // appended channel
        }
        if (bnw) red_add(acc, mul_rn(v, f.wnw));
        if (bne) red_add(acc + 1, mul_rn(v, f.wne));
        if (bsw) red_add(acc + W, mul_rn(v, f.wsw));
        if (bse) red_add(acc + W + 1, mul_rn(v, f.wse));
    }
}

// normaliser rule of softsplat.py:256-266
template <class A> __device__ __forceinline__ A apply_eps(A d, int eps) {
    if (eps == DCB_EPS_ADD) return add_rn(d, (A)0.0000001);
    if (eps == DCB_EPS_ZERO) return d == (A)0 ? (A)1 : d;
    return d < (A)0.0000001 ? (A)0.0000001 : d;      // clip(1e-7, None); NaN propagates like torch.clip
}

// ---------------------------------------------------------------------------------------------
// K2: normalise + cast (+ mask, + save normaliser, + re-zero). One thread per TARGET pixel.
// For SUM the "normaliser" is absent: plain cast/copy.
// ---------------------------------------------------------------------------------------------
template <class T>
__global__ void __launch_bounds__(kThreads) k_normalize(const FwdArgs a) {
    using A = typename Acc<T>::type;
    const unsigned p = blockIdx.x * kThreads + threadIdx.x;
    if (p >= a.total) return;
    const unsigned n = p / a.HW, r = p - n * a.HW;
    const bool normalised = a.mode != DCB_MODE_SUM;

    A keep = (A)1;
    if (a.mask.p) {
        const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
        const T* mp = (const T*)a.mask.p + n * a.mask.sN + y * a.mask.sH + x * a.mask.sW;
        keep = sub_rn((A)1, ld<A>(mp));                           // control_utils.py:69-70
    }
    T* out = (T*)a.out + (long long)n * a.C * a.HW + r;
    A* ap = (A*)a.acc + (long long)n * a.Cacc * a.HW + r;
    A d = (A)1;
    if (normalised) {
        d = apply_eps<A>(ap[(long long)a.C * a.HW], a.eps);
        if (a.norm) ((A*)a.norm)[p] = d;
        if (a.rezero) ap[(long long)a.C * a.HW] = (A)0;
    }
    for (int c = 0; c < a.C; ++c) {
        A* q = ap + (long long)c * a.HW;
        A o = normalised ? *q / d : *q;
        if (a.mask.p) o = mul_rn(o, keep);
        st<T, A>(out + (long long)c * a.HW, o);
        if (a.rezero) *q = (A)0;
    }
}

// ---------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------
// implemented in splat_pipe.cu
long long pipe_workspace(long long N, long long H, long long W);
int splat_pipe_impl(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const DcbTensor* out,
                    const DcbTensor* norm, const DcbTensor* mask, void* ws, int mode, int eps, bool ws_clean,
                    cudaStream_t st, bool ones_metric = false, const DcbTensor* mask_out = nullptr);
bool pipe_supported(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric);
// implemented in splat_planar.cu
long long planar_workspace(long long N, long long C, long long H, long long W, int dtype, int mode);
int splat_planar_impl(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const DcbTensor* out,
                      const DcbTensor* norm, const DcbTensor* mask, void* ws, int mode, int eps, bool ws_clean,
                      cudaStream_t st);

// implemented in splat_owner.cu
long long owner_workspace(long long N, long long H, long long W);
bool owner_supported(long long C, int mode, long long H, long long W);
int splat_owner_impl(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const DcbTensor* out,
                     const DcbTensor* norm, const DcbTensor* mask, void* ws, int mode, int eps, cudaStream_t st,
                     bool ones_metric = false, const DcbTensor* mask_out = nullptr);

// implemented in splat_lists.cu
long long lists_workspace(long long N, long long H, long long W);
bool lists_supported(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, int mode);
int splat_lists_impl(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const DcbTensor* out,
                     const DcbTensor* norm, const DcbTensor* mask, void* ws, int mode, int eps, bool leave_clean,
                     cudaStream_t st);

// the shape-only part of lists_supported (the workspace query has no strides)
static bool lists_shape(int dtype, int mode, long long N, long long C, long long H, long long W) {
    DcbTensor t{};
    t.dtype = dtype;
    t.size[0] = N; t.size[1] = C; t.size[2] = H; t.size[3] = W;
    t.stride[3] = 1; t.stride[2] = W; t.stride[1] = H * W; t.stride[0] = C * H * W;
    return lists_supported(&t, nullptr, nullptr, mode);
}

// C+1 <= 4 channels in fp32 / bf16: float4 accumulators (splat_pipe.cu)
static bool use_pipe(int dtype, int mode, long long C) {
    return dtype != DCB_F64 && C + (mode == DCB_MODE_SUM ? 0 : 1) <= 4;
}

// dcb_set_option("fwd_path"): 0 = automatic, 1 = accumulator pipelines only (no cluster kernel for small frames), 2 = target-tile
// owner wherever it applies
int g_fwd_path = 0;

// small frames: one launch, one thread-block cluster per frame (splat_small.cu)
bool use_cluster(int dtype, int mode, long long N, long long C, long long H, long long W);
long long cluster_workspace(long long N, long long C, long long H, long long W, int mode);
int splat_cluster_impl(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const DcbTensor* out,
                       const DcbTensor* norm, const DcbTensor* mask, void* ws, int mode, int eps, bool ws_clean,
                       cudaStream_t st, bool ones_metric, const DcbTensor* mask_out);
bool small_frames(int dtype, int mode, long long N, long long C, long long H, long long W) {
    return g_fwd_path == 0 && use_cluster(dtype, mode, N, C, H, W);
}

// C+1 <= 8 channels in fp32 / bf16: target-tile ownership, accumulators in shared memory (splat_owner.cu)
// Opt-in only: measured on B200 (profiles/r02/NOTES.md) it needs 2-3x the instructions of the accumulator pipeline and loses
// at every size, so the automatic dispatch never picks it. It has no fp16 instantiation: fp16 stays on the pipelines.
bool use_owner(int dtype, int mode, long long C, long long H, long long W) {
    if (dtype == DCB_F64 || dtype == DCB_F16 || g_fwd_path != 2) return false;
    return owner_supported(C, mode, H, W);
}

// Is the forward's workspace plain scratch at these sizes (nothing in it has to be all-zero on entry or is left all-zero)?
// True for the owner kernels and for the per-target list path: its lists are rebuilt by every call and only its counters are
// zeroed (by the call itself), so sharing the kept-zero accumulator buffer would cost a memset of the whole list area
// (40 B per pixel) behind every call. A strided view of these sizes that falls back to the planar accumulators zeroes them itself.
bool fwd_ws_is_scratch(long long N, long long C, long long H, long long W, int dtype, int mode) {
    if (use_owner(dtype, mode, C, H, W)) return true;
    if (small_frames(dtype, mode, N, C, H, W) || use_pipe(dtype, mode, C) || dtype == DCB_F64) return false;
    return lists_shape(dtype, mode, N, C, H, W);
}

long long splat_fwd_workspace(long long N, long long C, long long H, long long W, int dtype, int mode) {
    if (use_owner(dtype, mode, C, H, W)) return owner_workspace(N, H, W);
    if (small_frames(dtype, mode, N, C, H, W)) return cluster_workspace(N, C, H, W, mode);
    if (use_pipe(dtype, mode, C)) return pipe_workspace(N, H, W);
    if (dtype != DCB_F64) {
        const long long planar = planar_workspace(N, C, H, W, dtype, mode);
        if (!lists_shape(dtype, mode, N, C, H, W)) return planar;
        const long long lists = lists_workspace(N, H, W);         // strides may still send the call to the planar path
        return lists > planar ? lists : planar;
    }
    if (mode == DCB_MODE_SUM) return 0;                           // fp64 reds go straight into `out`
    return align_up(N * (C + 1) * H * W * 8, 256);
}

static void fill_args(FwdArgs& a, const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric,
                      const DcbTensor* mask, const DcbTensor* out, const DcbTensor* norm, int mode, int eps) {
    a.in = make_view(in); a.flow = make_view(flow); a.metric = make_view(metric); a.mask = make_view(mask);
    a.N = (int)in->size[0]; a.C = (int)in->size[1]; a.H = (int)in->size[2]; a.W = (int)in->size[3];
    a.HW = (unsigned)(in->size[2] * in->size[3]);
    a.total = (unsigned)(in->size[0] * in->size[2] * in->size[3]);
    a.Cacc = a.C + (mode == DCB_MODE_SUM ? 0 : 1);
    a.cgroup = a.Cacc;
    a.mode = mode; a.eps = eps;
    a.out = out->ptr;
    a.norm = norm ? norm->ptr : nullptr;
    a.acc = nullptr;
    a.rezero = 0;
}

// epilogue-only entry used by the deterministic path (det.cu): planar accumulators -> out, true division
int normalize_planar_launch(int dtype, const DcbTensor* in, const DcbTensor* out, const DcbTensor* norm,
                            const DcbTensor* mask, void* acc, int mode, int eps, cudaStream_t st) {
    FwdArgs a;
    fill_args(a, in, nullptr, nullptr, mask, out, norm, mode, eps);
    a.acc = acc;
    const unsigned blocks = (a.total + kThreads - 1) / kThreads;
    switch (dtype) {
        case DCB_F32: k_normalize<float><<<blocks, kThreads, 0, st>>>(a); break;
        case DCB_F64: k_normalize<double><<<blocks, kThreads, 0, st>>>(a); break;
        case DCB_BF16: k_normalize<__nv_bfloat16><<<blocks, kThreads, 0, st>>>(a); break;
        case DCB_F16: k_normalize<__half><<<blocks, kThreads, 0, st>>>(a); break;
        default: return set_error(DCB_E_DTYPE, "normalize: unsupported dtype %d", dtype);
    }
    DCB_CHECK_LAUNCH("k_normalize");
    return DCB_OK;
}

static int splat_fwd_f64(FwdArgs& a, const DcbTensor* out, void* ws, long long ws_bytes, int mode, bool ws_clean,
                         bool has_mask, cudaStream_t st) {
    const bool acc_is_out = mode == DCB_MODE_SUM && !has_mask;
    const long long acc_bytes = (long long)a.total * a.Cacc * 8;
    if (acc_is_out) {
        a.acc = out->ptr;
    } else {
        if (!ws || ws_bytes < acc_bytes || ((uintptr_t)ws & 255))
            return set_error(DCB_E_WORKSPACE, "splat_fwd: workspace of %lld bytes (256 B aligned) required, got %lld", acc_bytes, ws_bytes);
        a.acc = ws;
    }
    const bool clean = ws_clean && !acc_is_out;
    a.rezero = clean ? 1 : 0;
    if (!clean) DCB_CHECK_CUDA(cudaMemsetAsync(a.acc, 0, (size_t)acc_bytes, st));
    // split channels over blockIdx.y when there are too few pixels to fill 148 SMs
    const unsigned blocks = (a.total + kThreads - 1) / kThreads;
    int groups = 1;
    while (groups < a.Cacc && (long long)a.total * groups < 148LL * 8 * kThreads && groups < 64) groups *= 2;
    a.cgroup = (a.Cacc + groups - 1) / groups;
    k_scatter_planar<double, double><<<dim3(blocks, (a.Cacc + a.cgroup - 1) / a.cgroup), kThreads, 0, st>>>(a);
    DCB_CHECK_LAUNCH("k_scatter_planar");
    if (!acc_is_out) {
        k_normalize<double><<<blocks, kThreads, 0, st>>>(a);
        DCB_CHECK_LAUNCH("k_normalize");
    }
    return DCB_OK;
}

int splat_fwd_impl(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const DcbTensor* out,
                   const DcbTensor* norm, const DcbTensor* mask, void* ws, long long ws_bytes, int mode, int eps,
                   int flags, cudaStream_t st) {
    const long long N = in->size[0], C = in->size[1], H = in->size[2], W = in->size[3];
    if (N * H * W == 0 || C == 0) return DCB_OK;
    const bool ws_clean = (flags & DCB_FLAG_WS_CLEAN) != 0;
    if (in->dtype == DCB_F64) {
        FwdArgs a;
        fill_args(a, in, flow, metric, mask, out, norm, mode, eps);
        return splat_fwd_f64(a, out, ws, ws_bytes, mode, ws_clean, mask != nullptr, st);
    }
    if (in->dtype != DCB_F32 && !is_half_storage(in->dtype)) return set_error(DCB_E_DTYPE, "splat_fwd: unsupported dtype %d", in->dtype);
    if (use_owner(in->dtype, mode, C, H, W)) {
        if (!pipe_supported(in, flow, metric))
            return set_error(DCB_E_LIMIT, "splat_fwd: tensor spans beyond 2^31 elements are not supported (32-bit in-frame offsets)");
        const long long need = owner_workspace(N, H, W);
        if (need > 0 && (!ws || ws_bytes < need || ((uintptr_t)ws & 255)))
            return set_error(DCB_E_WORKSPACE, "splat_fwd: workspace of %lld bytes (256 B aligned) required, got %lld", need, ws_bytes);
        const int rc = splat_owner_impl(in, flow, metric, out, norm, mask, ws, mode, eps, st);
        // the flag promises an all-zero workspace on exit; callers that ask dcb_splat_fwd_workspace_is_scratch() never pass it here
        if (rc == DCB_OK && ws_clean && need > 0) DCB_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)need, st));
        return rc;
    }
    if (small_frames(in->dtype, mode, N, C, H, W)) {
        const long long need = cluster_workspace(N, C, H, W, mode);
        if (!ws || ws_bytes < need || ((uintptr_t)ws & 255))
            return set_error(DCB_E_WORKSPACE, "splat_fwd: workspace of %lld bytes (256 B aligned) required, got %lld", need, ws_bytes);
        return splat_cluster_impl(in, flow, metric, out, norm, mask, ws, mode, eps, ws_clean, st, false, nullptr);
    }
    const bool pipe = use_pipe(in->dtype, mode, C);
    if (pipe && !pipe_supported(in, flow, metric))
        return set_error(DCB_E_LIMIT, "splat_fwd: tensor spans beyond 2^31 elements are not supported by the float4 path");
    const long long need = splat_fwd_workspace(N, C, H, W, in->dtype, mode);
    if (need > 0 && (!ws || ws_bytes < need || ((uintptr_t)ws & 255)))
        return set_error(DCB_E_WORKSPACE, "splat_fwd: workspace of %lld bytes (256 B aligned) required, got %lld", need, ws_bytes);
    if (pipe) return splat_pipe_impl(in, flow, metric, out, norm, mask, ws, mode, eps, ws_clean, st);
    if (lists_supported(in, flow, metric, mode)) return splat_lists_impl(in, flow, metric, out, norm, mask, ws, mode, eps, ws_clean, st);
    return splat_planar_impl(in, flow, metric, out, norm, mask, ws, mode, eps, ws_clean, st);
}

}  // namespace dcb
