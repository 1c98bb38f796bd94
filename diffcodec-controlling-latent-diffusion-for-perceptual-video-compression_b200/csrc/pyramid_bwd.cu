// pyramid_bwd.cu -- the backward of dcb_bidir_pyramid_fwd (masks + holes, or NO_HOLES) for a WHOLE pyramid in two launches
// (sm_100a), with gradients w.r.t. both feature maps, both flows and both metrics.
//
// Per level and direction (f shown, b symmetric), with G = grad_fused, A = warped_f (the saved forward output, rounded to T),
// D = norm_f (eps included), occ = occ_f and k0 = hole ? 0.5 : w0 the fusion weight of the target pixel:
//   fused = k0 A + k1 B, A = splat(first, flow_f, metric_f) * (1 - occ) / D, so the gradient reaching A is k0 G and the splat
//   backward's target scalars (splat_bwd.cu) with the fusion weight folded in are
//       a'(t) = k0 (1 - occ) / D            T'(t) = -k0 sum_c G_c A_c / D
//   and the source pass is exactly k_bwd_source's with gradOut = G. The fusion-confidence gradient of a pixel (the dca / dcb
//   of k_bidir_fuse_bwd, fuse.cu; 0 at holes) needs the same two dot products sum_c G_c A_c, sum_c G_c B_c as T'.
//
//   launch A  k_pyr_bwd_target : every target pixel of every level; G, A and B are read once for both directions. Writes
//                                (a', T') of both directions and both confidence gradients: 24 bytes per pixel of workspace.
//   launch B  k_pyr_bwd_source : one job per (level, direction) through a job table; the device code is k_bwd_source's
//                                (bwd_source_body, splat_bwd.cuh); the confidence gradient is added to grad_metric before
//                                its single store.
// A pure gather: no atomics, no cross-CTA partial sums, the same bits on every run. The masks carry no gradient (compute_mask
// thresholds, as in the reference).
#include "splat_bwd.cuh"

namespace dcb {

constexpr int kBwdMaxLevels = 4;

// ---------------------------------------------------------------------------------------------
// launch A: target scalars of both directions + fusion-confidence gradients
// ---------------------------------------------------------------------------------------------
struct PyrBwdTarget {
    View g, metric_f, metric_b;                   // metric.p == nullptr: all-ones
    const void *warped_f, *warped_b, *occ_f, *occ_b;
    const float *norm_f, *norm_b;
    float *ts_f, *ts_b;                           // [N*H*W][2] (a', T')
    float *conf_f, *conf_b;                       // [N*H*W] or null when that metric gradient is not wanted
    int C, W;
    unsigned HW, total;
    int px, cs;                                   // px pixels x cs channel slices per 256-thread CTA
    unsigned block0;
};
struct PyrBwdTargetArgs {
    PyrBwdTarget lv[kBwdMaxLevels];
    int n_levels;
    int holes;
};

template <class T>
__global__ void __launch_bounds__(256) k_pyr_bwd_target(const __grid_constant__ PyrBwdTargetArgs a) {
    __shared__ float red[2 * 256];                // [cs][px][2] when cs > 1
    pdl_wait();
    int l = 0;
    while (l + 1 < a.n_levels && blockIdx.x >= a.lv[l + 1].block0) ++l;
    const PyrBwdTarget& L = a.lv[l];
    const int px = L.px, cs = L.cs;
    const int tx = (int)threadIdx.x % px, ty = (int)threadIdx.x / px;
    const unsigned p = (blockIdx.x - L.block0) * px + tx;
    const bool live = p < L.total;
    const unsigned pc = live ? p : 0;
    const unsigned n = pc / L.HW, r = pc - n * L.HW;
    const int y = (int)(r / (unsigned)L.W), x = (int)(r - (unsigned)y * (unsigned)L.W);
    const T* gp = (const T*)L.g.p + n * L.g.sN + (long long)y * L.g.sH + (long long)x * L.g.sW;
    const size_t fb = (size_t)n * L.C * L.HW + r;
    const T* ap = (const T*)L.warped_f + fb;
    const T* bp = (const T*)L.warped_b + fb;
    float da = 0.f, db = 0.f;                     // sum_c G_c A_c, sum_c G_c B_c
    constexpr int U = 4;                          // 12 loads in flight per thread
    for (int c0 = ty; c0 < L.C; c0 += U * cs) {
        float gv[U], av[U], bv[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int c = c0 + j * cs;
            const bool in = c < L.C;
            gv[j] = in ? ld<float>(gp + (long long)c * L.g.sC) : 0.f;
            av[j] = in ? ld<float>(ap + (size_t)c * L.HW) : 0.f;
            bv[j] = in ? ld<float>(bp + (size_t)c * L.HW) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < U; ++j) { da = fmaf(gv[j], av[j], da); db = fmaf(gv[j], bv[j], db); }
    }
    if (cs > 1) {
        red[2 * threadIdx.x] = da; red[2 * threadIdx.x + 1] = db;
        __syncthreads();
        if (ty != 0) return;
        for (int s = 1; s < cs; ++s) { da += red[2 * (s * px + tx)]; db += red[2 * (s * px + tx) + 1]; }
    }
    if (!live) return;
    // the fusion weights as the forward computed them (k_pyr_fuse; extractors.py:298-306)
    float ra = 1.f, rb = 1.f;
    if (L.metric_f.p) ra = ld<float>((const T*)L.metric_f.p + n * L.metric_f.sN + (long long)y * L.metric_f.sH + (long long)x * L.metric_f.sW);
    if (L.metric_b.p) rb = ld<float>((const T*)L.metric_b.p + n * L.metric_b.sN + (long long)y * L.metric_b.sH + (long long)x * L.metric_b.sW);
    const float ca = fmaxf(ra, 0.f), cb = fmaxf(rb, 0.f);
    const float s = add_rn(add_rn(ca, cb), 0.000001f);
    const float of = ld<float>((const T*)L.occ_f + p), ob = ld<float>((const T*)L.occ_b + p);
    const bool hole = a.holes && add_rn(of, ob) > 1.5f;
    const float k0 = hole ? 0.5f : ca / s, k1 = hole ? 0.5f : cb / s;
    const float df = L.norm_f[p], dbn = L.norm_b[p];
    ((float2*)L.ts_f)[p] = make_float2(k0 * sub_rn(1.f, of) / df, -(k0 * da) / df);
    ((float2*)L.ts_b)[p] = make_float2(k1 * sub_rn(1.f, ob) / dbn, -(k1 * db) / dbn);
    if (L.conf_f || L.conf_b) {
        // k_bidir_fuse_bwd (fuse.cu): the `where` routes the gradient of a hole to the average; clamp(min=0) passes it where
        // the metric is >= 0
        const float gw0 = hole ? 0.f : da, gw1 = hole ? 0.f : db;
        const float is = 1.f / s, is2 = is * is;
        if (L.conf_f) L.conf_f[p] = ra >= 0.f ? gw0 * (is - ca * is2) - gw1 * cb * is2 : 0.f;
        if (L.conf_b) L.conf_b[p] = rb >= 0.f ? gw1 * (is - cb * is2) - gw0 * ca * is2 : 0.f;
    }
}

// ---------------------------------------------------------------------------------------------
// launch B: the source-side gather of every (level, direction)
// ---------------------------------------------------------------------------------------------
struct PyrBwdJob {
    BwdArgs a;
    const float* gadd;                            // confidence gradient added to grad_metric, or null
    unsigned block0;
};
struct PyrBwdSourceArgs {
    PyrBwdJob job[2 * kBwdMaxLevels];
    int n_jobs;
};

template <class T>
__global__ void __launch_bounds__(256, DCB_BS_MINCTAS) k_pyr_bwd_source(const __grid_constant__ PyrBwdSourceArgs a) {
    __shared__ float red[256 * 4];                // [cs][px][4] when cs > 1
    pdl_wait();
    int j = 0;
    while (j + 1 < a.n_jobs && blockIdx.x >= a.job[j + 1].block0) ++j;
    const PyrBwdJob& b = a.job[j];
    bwd_source_body<T, T, int, true>(b.a, blockIdx.x - b.block0, (int)threadIdx.x % b.a.px, (int)threadIdx.x / b.a.px, red, b.gadd);
}

// ---------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------
static long long level_bwd_bytes(const DcbTensor* f) { return align_up(f->size[0] * f->size[2] * f->size[3] * 24, 256); }

long long pyramid_bwd_workspace(const DcbPyramidBwdLevel* lv, int n) {
    long long total = 0;
    for (int l = 0; l < n; ++l)
        if (lv[l].first) total += level_bwd_bytes(lv[l].first);
    return total;
}

template <class T>
static int launch_pyramid_bwd(const PyrBwdTargetArgs& ta, unsigned t_blocks, const PyrBwdSourceArgs& sa, unsigned s_blocks, cudaStream_t st) {
    DCB_CHECK_CUDA(launch_pdl(k_pyr_bwd_target<T>, dim3(t_blocks), dim3(256), 0, st, ta));
    count_launch();
    DCB_CHECK_CUDA(launch_pdl(k_pyr_bwd_source<T>, dim3(s_blocks), dim3(256), 0, st, sa));
    count_launch();
    return DCB_OK;
}

// Preconditions (checked by the caller): 1 <= n <= kBwdMaxLevels, one dtype (F32 / BF16 / F16) for all tensors, shapes consistent,
// the six saved forward outputs present, ws holds pyramid_bwd_workspace() bytes, 256-byte aligned.
int bidir_pyramid_bwd_impl(const DcbPyramidBwdLevel* lv, int n, void* ws, bool holes, cudaStream_t st) {
    PyrBwdTargetArgs ta; PyrBwdSourceArgs sa;
    ta.n_levels = 0; ta.holes = holes ? 1 : 0; sa.n_jobs = 0;
    unsigned t_blocks = 0, s_blocks = 0;
    char* wsp = (char*)ws;
    const int pf_dist = device_sm_count() * DCB_BS_MINCTAS;
    for (int l = 0; l < n; ++l) {
        const DcbPyramidBwdLevel& d = lv[l];
        const long long N = d.first->size[0], C = d.first->size[1], H = d.first->size[2], W = d.first->size[3], P = N * H * W;
        float* ts_f = (float*)wsp;
        float* ts_b = ts_f + 2 * P;
        float* conf_f = ts_b + 2 * P;
        float* conf_b = conf_f + P;
        wsp += level_bwd_bytes(d.first);
        const bool want_f = d.grad_first || d.grad_flow_f || d.grad_metric_f, want_b = d.grad_last || d.grad_flow_b || d.grad_metric_b;
        if (N * C * H * W == 0 || !(want_f || want_b)) continue;
        // gradOut offsets inside one plane are formed in 32 bits (k_bwd_source's IX = int)
        const long long span = (H - 1) * (d.grad_fused->stride[2] < 0 ? -d.grad_fused->stride[2] : d.grad_fused->stride[2]) +
                               (W - 1) * (d.grad_fused->stride[3] < 0 ? -d.grad_fused->stride[3] : d.grad_fused->stride[3]);
        if (span >= (1ll << 30)) return set_error(DCB_E_LIMIT, "bidir_pyramid_bwd: level %d: grad_fused spans 2^30 elements per plane or more", l);

        PyrBwdTarget& L = ta.lv[ta.n_levels++];
        L.g = make_view(d.grad_fused); L.metric_f = make_view(d.metric_f); L.metric_b = make_view(d.metric_b);
        L.warped_f = d.warped_f; L.warped_b = d.warped_b; L.occ_f = d.occ_f; L.occ_b = d.occ_b;
        L.norm_f = (const float*)d.norm_f; L.norm_b = (const float*)d.norm_b;
        L.ts_f = ts_f; L.ts_b = ts_b;
        L.conf_f = d.grad_metric_f ? conf_f : nullptr; L.conf_b = d.grad_metric_b ? conf_b : nullptr;
        L.C = (int)C; L.W = (int)W; L.HW = (unsigned)(H * W); L.total = (unsigned)P;
        int ct = 1;                               // channel slices when pixels are scarce, as k_bwd_target
        while (ct < 32 && ct * 2 * 8 <= C && P * ct < 148LL * 2048) ct *= 2;
        L.cs = ct; L.px = 256 / ct;
        L.block0 = t_blocks;
        t_blocks += (unsigned)((P + L.px - 1) / L.px);

        int cs = 1;                               // as launch_bwd (splat_bwd.cu)
        while (cs < 32 && cs * 2 <= C && P * cs < 148LL * 2048) cs *= 2;
        auto add_job = [&](const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const float* tscal, void* gin, void* gflow,
                           void* gmetric, const float* gadd) {
            PyrBwdJob& j = sa.job[sa.n_jobs++];
            BwdArgs& b = j.a;
            b = BwdArgs{};
            b.gout = make_view(d.grad_fused); b.in = make_view(in); b.flow = make_view(flow); b.metric = make_view(metric);
            b.tscal = (void*)tscal; b.gin = gin; b.gflow = gflow; b.gmetric = gmetric;
            b.total = (unsigned)P; b.HW = (unsigned)(H * W);
            b.N = (int)N; b.C = (int)C; b.H = (int)H; b.W = (int)W;
            b.mode = DCB_MODE_SOFT; b.eps = DCB_EPS_ADD;
            b.cs = cs; b.px = 256 / cs;
            b.pf_dist = (unsigned)pf_dist;
            j.gadd = gmetric ? gadd : nullptr;
            j.block0 = s_blocks;
            s_blocks += (unsigned)((P + b.px - 1) / b.px);
        };
        if (want_f) add_job(d.first, d.flow_f, d.metric_f, ts_f, d.grad_first, d.grad_flow_f, d.grad_metric_f, conf_f);
        if (want_b) add_job(d.last, d.flow_b, d.metric_b, ts_b, d.grad_last, d.grad_flow_b, d.grad_metric_b, conf_b);
    }
    if (ta.n_levels == 0) return DCB_OK;
    switch (lv[0].first->dtype) {
        case DCB_F32: return launch_pyramid_bwd<float>(ta, t_blocks, sa, s_blocks, st);
        case DCB_BF16: return launch_pyramid_bwd<__nv_bfloat16>(ta, t_blocks, sa, s_blocks, st);
        case DCB_F16: return launch_pyramid_bwd<__half>(ta, t_blocks, sa, s_blocks, st);
    }
    return set_error(DCB_E_DTYPE, "bidir_pyramid_bwd: unsupported dtype %d", lv[0].first->dtype);
}

}  // namespace dcb
