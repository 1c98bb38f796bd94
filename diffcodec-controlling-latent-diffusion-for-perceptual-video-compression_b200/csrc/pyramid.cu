// pyramid.cu -- the motion compensation of a WHOLE conditioning pyramid in two launches (sm_100a).
// SURVEY.md section 8: row f-1 as the survey defines it (<= 2 launches per scale), the batched multi-tensor entry for
// the 16 splats of one ControlNet forward, and row f-4 (the multi-scale conditioning pyramid of the notebook).
//
// Replaces, for all scales of one forward at once:
//   * controlnet/extractors.py:282-310 (Bi_Dir_FeatureExtractor.forward between the conv stacks): per scale two
//     compute_mask() calls (control_utils.py:11-17), two FeatureWarperSoftsplat splats with (1 - mask)
//     (control_utils.py:61-72), the confidence fusion and the double-hole fill with its `holes.any()` host sync --
//     4 scales x ~45 eager kernels + 16 NVRTC cache lookups + 4 device->host stalls in the reference; 36 launches through
//     dcb_bidir_block_fwd (block.cu);
//   * improv_experiments.ipynb cell 5 (soft splat of both resized frames at 128 / 64 / 32 and soft_fuse with identity
//     masks, cell 3) -- flag DCB_PYRAMID_NO_MASKS;
//   * the bilinear resampling in front of both (resize_and_normalize_flow_batched, control_utils.py:74-97;
//     F.interpolate of frames and flows, notebook cell 5 and extractors.py:182-183): dcb_resample_batch, ONE launch for
//     every (tensor, scale) pair.
//
//   launch A  k_pyr_scatter : every scatter job of every scale -- per scale the two flow-by-flow splats behind the
//                             occlusion masks (2 channels, all-ones metric) and the two feature splats (C channels,
//                             learned metric); the device code is the register-merged channel-quad scatter of
//                             splat_planar.cuh; jobs are independent, their accumulators disjoint;
//   launch B  k_pyr_fuse    : per target pixel: both occlusion tests, both normalisers, (1 - mask), the confidence
//                             weights and the double-hole test ONCE, then the channel quads of both directions stream
//                             through: normalise, mask, fuse, store. The warped maps never reach memory unless the
//                             caller asks for them (the backward does).
//   one cudaMemsetAsync re-zeroes the per-pixel planes that several warps read (48 B per pixel); the channel-quad
//   accumulators are re-zeroed by their only reader. The workspace follows the DCB_FLAG_WS_CLEAN protocol.
#include "splat_planar.cuh"

namespace dcb {

constexpr int kMaxLevels = 4;            // kernel parameters stay below 4 KB
constexpr int kMaxJobs = 4 * kMaxLevels;
constexpr int kMaxResample = 16;

// ---------------------------------------------------------------------------------------------
// batched bilinear resampling (torch's upsample_bilinear2d arithmetic, see flow_ingest.cu)
// ---------------------------------------------------------------------------------------------
struct ResampleJob {
    View src;                // [N,C,H,W] any strides
    void* dst;               // [N,C,th,tw] contiguous
    int N, C, H, W, th, tw;
    int align, op;           // align_corners; DCB_RESAMPLE_*
    int src_st, dst_st;      // storage of src / dst: kStF32, kStBF16 or kStF16
    float sx, sy, f0, f1;    // source-index scales; post factor of channel 0 / of every other channel
    unsigned block0, blocks; // 256-thread blocks of this job inside the launch
};
struct ResampleArgs {
    ResampleJob job[kMaxResample];
    int n_jobs;
};

// storage of a resample tensor; a batch with any F16 tensor runs k_resample_batch_f16, which knows all three codes
enum { kStF32 = 0, kStBF16 = 1, kStF16 = 2 };
static int storage_code(int dtype) { return dtype == DCB_BF16 ? kStBF16 : (dtype == DCB_F16 ? kStF16 : kStF32); }
template <bool F16> __device__ __forceinline__ float ld_rt(const void* p, long long i, int code) {
    if (F16 && code == kStF16) return __half2float(((const __half*)p)[i]);
    return code ? __bfloat162float(((const __nv_bfloat16*)p)[i]) : ((const float*)p)[i];
}
template <bool F16> __device__ __forceinline__ void st_rt(void* p, long long i, int code, float v) {
    if (F16 && code == kStF16) ((__half*)p)[i] = __float2half_rn(v);
    else if (code) ((__nv_bfloat16*)p)[i] = __float2bfloat16_rn(v); else ((float*)p)[i] = v;
}
__device__ __forceinline__ float src_index_rt(float scale, int dst, bool align) {
    if (align) return mul_rn(scale, (float)dst);
    const float s = sub_rn(mul_rn(scale, add_rn((float)dst, 0.5f)), 0.5f);          // torch: scale * (dst + 0.5) - 0.5, clamped at 0
    return s < 0.f ? 0.f : s;
}

template <bool F16> __device__ __forceinline__ void resample_batch(const ResampleArgs& a) {
    pdl_wait();
    int j = 0;
    while (j + 1 < a.n_jobs && blockIdx.x >= a.job[j + 1].block0) ++j;
    const ResampleJob& b = a.job[j];
    const long long total = (long long)b.N * b.th * b.tw;
    const long long p = (long long)(blockIdx.x - b.block0) * 256 + threadIdx.x;
    if (p >= total) return;
    const int x = (int)(p % b.tw), y = (int)((p / b.tw) % b.th), n = (int)(p / ((long long)b.tw * b.th));
    const float fy = src_index_rt(b.sy, y, b.align), fx = src_index_rt(b.sx, x, b.align);
    const int iy = (int)fy, ix = (int)fx;
    const int py = iy < b.H - 1 ? 1 : 0, px = ix < b.W - 1 ? 1 : 0;
    const float ly1 = sub_rn(fy, (float)iy), ly0 = sub_rn(1.f, ly1), lx1 = sub_rn(fx, (float)ix), lx0 = sub_rn(1.f, lx1);
    const long long base = (long long)n * b.src.sN + (long long)iy * b.src.sH + (long long)ix * b.src.sW;
    const long long plane = (long long)b.th * b.tw;
    for (int c = 0; c < b.C; ++c) {
        const long long q = base + c * b.src.sC;
        const float v00 = ld_rt<F16>(b.src.p, q, b.src_st), v01 = ld_rt<F16>(b.src.p, q + px * b.src.sW, b.src_st);
        const float v10 = ld_rt<F16>(b.src.p, q + py * b.src.sH, b.src_st), v11 = ld_rt<F16>(b.src.p, q + py * b.src.sH + px * b.src.sW, b.src_st);
        // torch: h0lambda * (w0lambda * v00 + w1lambda * v01) + h1lambda * (w0lambda * v10 + w1lambda * v11)
        const float top = add_rn(mul_rn(lx0, v00), mul_rn(lx1, v01)), bot = add_rn(mul_rn(lx0, v10), mul_rn(lx1, v11));
        float r = add_rn(mul_rn(ly0, top), mul_rn(ly1, bot));
        const float f = c == 0 ? b.f0 : b.f1;
        if (b.op == DCB_RESAMPLE_MUL) r = mul_rn(r, f);
        else if (b.op == DCB_RESAMPLE_DIV) r = r / f;
        st_rt<F16>(b.dst, ((long long)n * b.C + c) * plane + (long long)y * b.tw + x, b.dst_st, r);
    }
}
__global__ void __launch_bounds__(256) k_resample_batch(const __grid_constant__ ResampleArgs a) { resample_batch<false>(a); }
__global__ void __launch_bounds__(256) k_resample_batch_f16(const __grid_constant__ ResampleArgs a) { resample_batch<true>(a); }

int resample_batch_impl(const DcbResampleJob* jobs, int n_jobs, cudaStream_t st) {
    for (int j0 = 0; j0 < n_jobs; j0 += kMaxResample) {
        ResampleArgs a;
        a.n_jobs = 0;
        unsigned blocks = 0;
        for (int j = j0; j < n_jobs && j < j0 + kMaxResample; ++j) {
            const DcbTensor* s = jobs[j].src; const DcbTensor* d = jobs[j].dst;
            const long long total = d->size[0] * d->size[2] * d->size[3];
            if (total == 0 || d->size[1] == 0) continue;
            ResampleJob& b = a.job[a.n_jobs++];
            b.src = make_view(s); b.dst = d->ptr;
            b.N = (int)d->size[0]; b.C = (int)d->size[1]; b.H = (int)s->size[2]; b.W = (int)s->size[3];
            b.th = (int)d->size[2]; b.tw = (int)d->size[3];
            b.align = jobs[j].align_corners ? 1 : 0; b.op = jobs[j].op;
            b.src_st = storage_code(s->dtype); b.dst_st = storage_code(d->dtype);
            // torch area_pixel_compute_scale<float>
            b.sy = b.align ? (b.th > 1 ? (float)(b.H - 1) / (float)(b.th - 1) : 0.f) : (float)b.H / (float)b.th;
            b.sx = b.align ? (b.tw > 1 ? (float)(b.W - 1) / (float)(b.tw - 1) : 0.f) : (float)b.W / (float)b.tw;
            b.f0 = jobs[j].factor0; b.f1 = jobs[j].factor1;
            b.block0 = blocks; b.blocks = (unsigned)((total + 255) / 256);
            blocks += b.blocks;
        }
        if (a.n_jobs == 0) continue;
        bool f16 = false;
        for (int j = 0; j < a.n_jobs; ++j) f16 = f16 || a.job[j].src_st == kStF16 || a.job[j].dst_st == kStF16;
        DCB_CHECK_CUDA(launch_pdl(f16 ? k_resample_batch_f16 : k_resample_batch, dim3(blocks), dim3(256), 0, st, a));
        count_launch();
    }
    return DCB_OK;
}

// ---------------------------------------------------------------------------------------------
// launch A: every scatter job of the pyramid
// ---------------------------------------------------------------------------------------------
struct PyrJob {              // one soft splat of `in` by `flow` into its own accumulators
    View in, flow, metric;   // metric.p == nullptr: all-ones, never materialised
    float* acc;              // [N][Cq][HW] float4, all-zero
    float* dacc;             // [N][HW] weights, all-zero
    int C, Cq, H, W;
    unsigned HW;
    int tiles_x, ts;         // strips of 32 x 4 per frame
    int cg, ncg;             // channel quads per item, items per strip
    unsigned item0, items;
    int vec_in;              // channels-last input: one vector load per channel quad
};
struct PyrScatterArgs {
    PyrJob job[kMaxJobs];
    int n_jobs;
};

template <class T>
__global__ void __launch_bounds__(32, 16) k_pyr_scatter(const __grid_constant__ PyrScatterArgs a) {
    pdl_wait();
    int j = 0;
    while (j + 1 < a.n_jobs && blockIdx.x >= a.job[j + 1].item0) ++j;
    const PyrJob& b = a.job[j];
    const unsigned item = blockIdx.x - b.item0;
    if (item >= b.items) return;
    const unsigned per = (unsigned)b.ts * b.ncg;
    const int fi = item / per, q = item % per;
    const int strip = q % b.ts, cgi = q / b.ts;
    PlanarArgs pa;                                   // only the fields planar_scatter_strip reads
    pa.in = b.in; pa.flow = b.flow; pa.metric = b.metric;
    pa.C = b.C; pa.Cq = b.Cq; pa.H = b.H; pa.W = b.W; pa.HW = b.HW;
    pa.tiles_x = b.tiles_x; pa.mode = DCB_MODE_SOFT; pa.ones = b.metric.p == nullptr; pa.vec_in = b.vec_in;
    float* acc = b.acc + (size_t)fi * b.Cq * b.HW * 4;
    float* dplane = b.dacc + (size_t)fi * b.HW;
    const int q0 = cgi * b.cg, q1 = min(b.Cq, (cgi + 1) * b.cg);
    planar_scatter_strip<T, T>(pa, fi, strip, q0, q1, cgi == 0, acc, dplane, threadIdx.x & 31);
}

// ---------------------------------------------------------------------------------------------
// launch B: masks, normalisation, (1 - mask), confidence fusion, hole fill
// ---------------------------------------------------------------------------------------------
struct PyrLevel {
    View flow_f, flow_b, metric_f, metric_b;
    float *acc_mf, *dacc_mf, *acc_mb, *dacc_mb;   // flow-by-flow splats behind the masks: [N][HW] float4 (x, y, -, -), [N][HW]
    float *acc_f, *dacc_f, *acc_b, *dacc_b;       // feature splats: [N][Cq][HW] float4, [N][HW]
    void *fused, *warped_f, *warped_b, *occ_f, *occ_b;
    float *norm_f, *norm_b;
    int C, Cq, W;
    unsigned HW;
    int tn;                  // chunks of 128 target pixels per frame
    int cg, ncg;             // channel quads per item, items per chunk
    unsigned item0, items;
};
struct PyrFuseArgs {
    PyrLevel lv[kMaxLevels];
    int n_levels;
    int masks;               // 0: identity masks (notebook cell 5): no occlusion test, no (1 - mask), no holes
    int holes;               // 0: no double-hole fill (DCB_PYRAMID_NO_HOLES; extractors.py:193-199)
};

template <class T>
__global__ void __launch_bounds__(32, 16) k_pyr_fuse(const __grid_constant__ PyrFuseArgs a) {
    pdl_wait();
    int l = 0;
    while (l + 1 < a.n_levels && blockIdx.x >= a.lv[l + 1].item0) ++l;
    const PyrLevel& L = a.lv[l];
    const unsigned item = blockIdx.x - L.item0;
    if (item >= L.items) return;
    const int lane = threadIdx.x & 31;
    const unsigned per = (unsigned)L.tn * L.ncg;
    const unsigned fi = item / per, q = item % per;
    const unsigned chunk = q % L.tn, cgi = q / L.tn;
    constexpr int kPer = kPChunk / 32;
    const unsigned base = chunk * kPChunk + lane;
    const size_t fpix = (size_t)fi * L.HW;
    float sf[kPer], sb[kPer], w0[kPer], w1[kPer];
    bool hole[kPer];
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
        const unsigned r = base + i * 32;
        sf[i] = sb[i] = w0[i] = w1[i] = 0.f; hole[i] = false;
        if (r >= L.HW) continue;
        const int y = (int)(r / (unsigned)L.W), x = (int)(r - (unsigned)y * (unsigned)L.W);
        float of = 0.f, ob = 0.f;
        if (a.masks) {
            // occ_fwd = compute_mask(flow_f, flow_b): flow_f splatted by flow_b, compared with flow_b   (extractors.py:290)
            const float4 mf = __ldcg((const float4*)L.acc_mf + fpix + r), mb = __ldcg((const float4*)L.acc_mb + fpix + r);
            const float dmf = __ldcg(L.dacc_mf + fpix + r), dmb = __ldcg(L.dacc_mb + fpix + r);
            const T* pf = (const T*)L.flow_f.p + fi * L.flow_f.sN + (long long)y * L.flow_f.sH + (long long)x * L.flow_f.sW;
            const T* pb = (const T*)L.flow_b.p + fi * L.flow_b.sN + (long long)y * L.flow_b.sH + (long long)x * L.flow_b.sW;
            of = occlusion(mf.x, mf.y, dmf, ld<float>(pb), ld<float>(pb + L.flow_b.sC));
            ob = occlusion(mb.x, mb.y, dmb, ld<float>(pf), ld<float>(pf + L.flow_f.sC));
        }
        // normalisers of both feature splats: softsplat.py:256-258 ('soft' = add 1e-7), one reciprocal per pixel
        const float df = add_rn(__ldcg(L.dacc_f + fpix + r), 0.0000001f), db = add_rn(__ldcg(L.dacc_b + fpix + r), 0.0000001f);
        sf[i] = __frcp_rn(df); sb[i] = __frcp_rn(db);
        if (a.masks) { sf[i] = mul_rn(sf[i], sub_rn(1.f, of)); sb[i] = mul_rn(sb[i], sub_rn(1.f, ob)); }   // control_utils.py:69-70
        // confidences = the warpers' metrics (extractors.py:298-303)
        float ca = 1.f, cb = 1.f;
        if (L.metric_f.p) ca = ld<float>((const T*)L.metric_f.p + fi * L.metric_f.sN + (long long)y * L.metric_f.sH + (long long)x * L.metric_f.sW);
        if (L.metric_b.p) cb = ld<float>((const T*)L.metric_b.p + fi * L.metric_b.sN + (long long)y * L.metric_b.sH + (long long)x * L.metric_b.sW);
        ca = fmaxf(ca, 0.f); cb = fmaxf(cb, 0.f);
        const float s = add_rn(add_rn(ca, cb), 0.000001f);
        w0[i] = ca / s; w1[i] = cb / s;
        hole[i] = a.masks && a.holes && add_rn(of, ob) > 1.5f;                                                        // extractors.py:306
        if (cgi == 0) {
            if (L.occ_f) st<T, float>((T*)L.occ_f + fpix + r, of);
            if (L.occ_b) st<T, float>((T*)L.occ_b + fpix + r, ob);
            if (L.norm_f) L.norm_f[fpix + r] = df;
            if (L.norm_b) L.norm_b[fpix + r] = db;
        }
    }
    const int C = L.C;
    const size_t fbase = (size_t)fi * C * L.HW;
    T* fo = (T*)L.fused + fbase;
    T* wf = L.warped_f ? (T*)L.warped_f + fbase : nullptr;
    T* wb = L.warped_b ? (T*)L.warped_b + fbase : nullptr;
    const int q0 = cgi * L.cg, q1 = min(L.Cq, (int)(cgi + 1) * L.cg);
    for (int qq = q0; qq < q1; ++qq) {
        float4* pf = (float4*)L.acc_f + ((size_t)fi * L.Cq + qq) * L.HW;
        float4* pb = (float4*)L.acc_b + ((size_t)fi * L.Cq + qq) * L.HW;
        float4 vf[kPer], vb[kPer];
#pragma unroll
        for (int i = 0; i < kPer; ++i) {
            const unsigned r = base + i * 32;
            vf[i] = vb[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < L.HW) { vf[i] = __ldcg(pf + r); vb[i] = __ldcg(pb + r); }
        }
#pragma unroll
        for (int i = 0; i < kPer; ++i) {
            const unsigned r = base + i * 32;
            if (r >= L.HW) continue;
            __stcg(pf + r, make_float4(0.f, 0.f, 0.f, 0.f));
            __stcg(pb + r, make_float4(0.f, 0.f, 0.f, 0.f));
            const float af[4] = {vf[i].x, vf[i].y, vf[i].z, vf[i].w}, ab[4] = {vb[i].x, vb[i].y, vb[i].z, vb[i].w};
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
                const int c = 4 * qq + jj;
                if (c >= C) break;
                // the warped maps as the unfused path stores them (rounded to T), then extractors.py:303-310
                const float A = round_as<T>(mul_rn(af[jj], sf[i])), B = round_as<T>(mul_rn(ab[jj], sb[i]));
                const float v = hole[i] ? mul_rn(0.5f, add_rn(A, B)) : add_rn(mul_rn(w0[i], A), mul_rn(w1[i], B));
                st_stream(fo + (size_t)c * L.HW + r, v);
                if (wf) st_stream(wf + (size_t)c * L.HW + r, A);
                if (wb) st_stream(wb + (size_t)c * L.HW + r, B);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------
static long long level_shared_bytes(long long N, long long H, long long W) { return align_up(N * H * W * 48, 256); }
static long long level_feat_bytes(long long N, long long C, long long H, long long W) { return align_up(2 * N * ((C + 3) / 4) * H * W * 16, 256); }

long long pyramid_workspace(const DcbPyramidLevel* lv, int n) {
    long long total = 0;
    for (int l = 0; l < n; ++l) {
        const DcbTensor* f = lv[l].first;
        if (!f) continue;
        total += level_shared_bytes(f->size[0], f->size[2], f->size[3]) + level_feat_bytes(f->size[0], f->size[1], f->size[2], f->size[3]);
    }
    return total;
}

// channel quads per item so that small levels still spread over the machine
static void split_quads(long long items, int quads, int* cg, int* ncg) {
    const long long want = 148ll * 16;
    long long n = items > 0 ? (want + items - 1) / items : 1;
    if (n > quads) n = quads;
    if (n < 1) n = 1;
    *cg = (int)((quads + n - 1) / n);
    *ncg = (quads + *cg - 1) / *cg;
}

template <class T>
static int launch_pyramid(const PyrScatterArgs& sa, unsigned s_items, const PyrFuseArgs& fa, unsigned f_items, cudaStream_t st) {
    DCB_CHECK_CUDA(launch_pdl(k_pyr_scatter<T>, dim3(s_items), dim3(32), 0, st, sa));
    count_launch();
    DCB_CHECK_CUDA(launch_pdl(k_pyr_fuse<T>, dim3(f_items), dim3(32), 0, st, fa));
    count_launch();
    return DCB_OK;
}

// Preconditions (checked by the caller): 1 <= n <= kMaxLevels, all tensors of one dtype (F32 / BF16 / F16), shapes consistent,
// ws holds pyramid_workspace() bytes, 256-byte aligned, all-zero if DCB_FLAG_WS_CLEAN.
int bidir_pyramid_fwd_impl(const DcbPyramidLevel* lv, int n, void* ws, int flags, cudaStream_t st) {
    PyrScatterArgs sa; PyrFuseArgs fa;
    sa.n_jobs = 0; fa.n_levels = 0;
    fa.masks = (flags & DCB_PYRAMID_NO_MASKS) ? 0 : 1;
    fa.holes = (flags & DCB_PYRAMID_NO_HOLES) ? 0 : 1;
    long long shared_total = 0;
    for (int l = 0; l < n; ++l) shared_total += level_shared_bytes(lv[l].first->size[0], lv[l].first->size[2], lv[l].first->size[3]);
    const long long total = pyramid_workspace(lv, n);
    if (!(flags & DCB_FLAG_WS_CLEAN)) DCB_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)total, st));
    char* shared = (char*)ws;
    char* feat = (char*)ws + shared_total;
    unsigned s_items = 0, f_items = 0;
    const int dt = lv[0].first->dtype;
    for (int l = 0; l < n; ++l) {
        const DcbPyramidLevel& d = lv[l];
        const long long N = d.first->size[0], C = d.first->size[1], H = d.first->size[2], W = d.first->size[3];
        if (N * C * H * W == 0) continue;
        const long long HW = H * W, Cq = (C + 3) / 4;
        float* acc_mf = (float*)shared;              float* acc_mb = acc_mf + N * HW * 4;
        float* dacc_mf = acc_mb + N * HW * 4;        float* dacc_mb = dacc_mf + N * HW;
        float* dacc_f = dacc_mb + N * HW;            float* dacc_b = dacc_f + N * HW;
        float* acc_f = (float*)feat;                 float* acc_b = acc_f + N * Cq * HW * 4;
        shared += level_shared_bytes(N, H, W);
        feat += level_feat_bytes(N, C, H, W);
        const int tiles_x = (int)((W + 31) / 32), ts = tiles_x * (int)((H + kPRows - 1) / kPRows);
        auto add_job = [&](const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, float* acc, float* dacc, long long Cj) {
            PyrJob& b = sa.job[sa.n_jobs++];
            b.in = make_view(in); b.flow = make_view(flow); b.metric = make_view(metric);
            b.acc = acc; b.dacc = dacc;
            b.C = (int)Cj; b.Cq = (int)((Cj + 3) / 4); b.H = (int)H; b.W = (int)W; b.HW = (unsigned)HW;
            b.tiles_x = tiles_x; b.ts = ts;
            b.vec_in = planar_vec_ok(in) ? 1 : 0;
            split_quads(N * ts, b.Cq, &b.cg, &b.ncg);
            b.item0 = s_items; b.items = (unsigned)(N * ts * b.ncg);
            s_items += b.items;
        };
        if (fa.masks) {
            add_job(d.flow_f, d.flow_b, nullptr, acc_mf, dacc_mf, 2);        // compute_mask(flow_f, flow_b)
            add_job(d.flow_b, d.flow_f, nullptr, acc_mb, dacc_mb, 2);        // compute_mask(flow_b, flow_f)
        }
        add_job(d.first, d.flow_f, d.metric_f, acc_f, dacc_f, C);
        add_job(d.last, d.flow_b, d.metric_b, acc_b, dacc_b, C);
        PyrLevel& L = fa.lv[fa.n_levels++];
        L.flow_f = make_view(d.flow_f); L.flow_b = make_view(d.flow_b);
        L.metric_f = make_view(d.metric_f); L.metric_b = make_view(d.metric_b);
        L.acc_mf = acc_mf; L.dacc_mf = dacc_mf; L.acc_mb = acc_mb; L.dacc_mb = dacc_mb;
        L.acc_f = acc_f; L.dacc_f = dacc_f; L.acc_b = acc_b; L.dacc_b = dacc_b;
        L.fused = d.fused; L.warped_f = d.warped_f; L.warped_b = d.warped_b; L.occ_f = d.occ_f; L.occ_b = d.occ_b;
        L.norm_f = (float*)d.norm_f; L.norm_b = (float*)d.norm_b;
        L.C = (int)C; L.Cq = (int)Cq; L.W = (int)W; L.HW = (unsigned)HW;
        L.tn = (int)((HW + kPChunk - 1) / kPChunk);
        split_quads(N * L.tn, L.Cq, &L.cg, &L.ncg);
        L.item0 = f_items; L.items = (unsigned)(N * L.tn * L.ncg);
        f_items += L.items;
    }
    if (fa.n_levels == 0) return DCB_OK;
    int rc;
    switch (dt) {
        case DCB_F32: rc = launch_pyramid<float>(sa, s_items, fa, f_items, st); break;
        case DCB_BF16: rc = launch_pyramid<__nv_bfloat16>(sa, s_items, fa, f_items, st); break;
        case DCB_F16: rc = launch_pyramid<__half>(sa, s_items, fa, f_items, st); break;
        default: return set_error(DCB_E_DTYPE, "bidir_pyramid_fwd: unsupported dtype %d", dt);
    }
    if (rc != DCB_OK) return rc;
    // the per-pixel planes have several readers (one warp per channel group): re-zeroed behind the kernel
    DCB_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)shared_total, st));
    return DCB_OK;
}

}  // namespace dcb
