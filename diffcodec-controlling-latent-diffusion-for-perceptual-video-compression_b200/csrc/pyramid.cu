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
//
// DCB_FLAG_DETERMINISTIC replaces launch A by the sort-then-reduce of det.cu, over every splat of the pyramid at once:
//   k_pyr_det_emit   : one key per (source, corner) of every footprint field (level x direction), see PyrDetField
//   sort             : ONE cub::DeviceRadixSort over all keys (det_sort_keys, det.cu)
//   k_pyr_det_reduce : per (target, channel quad) the contributions in ascending source order, with k_det_reduce's
//                      arithmetic (det_add), written into the cells launch B reads
//   k_pyr_fuse<T, 1> : launch B dividing as k_normalize does; nothing is re-zeroed, the workspace is plain scratch.
// The outputs are then bit-identical, run to run, to the composition of deterministic single ops (compute_mask, the masked
// soft splat, bidir_fuse) in fp32.
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

// DET: the cells come from k_pyr_det_reduce. The division and the (1 - mask) product are those of k_normalize (o = S / d,
// then o * (1 - mask), one rounding to T), and the cells are plain scratch: nothing is re-zeroed.
template <class T, bool DET>
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
    float kf[kPer], kb[kPer];                        // DET: the (1 - mask) factors
    bool hole[kPer];
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
        const unsigned r = base + i * 32;
        sf[i] = sb[i] = w0[i] = w1[i] = 0.f; hole[i] = false;
        if constexpr (DET) kf[i] = kb[i] = 1.f;
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
        if constexpr (DET) {
            sf[i] = df; sb[i] = db;
            if (a.masks) { kf[i] = sub_rn(1.f, of); kb[i] = sub_rn(1.f, ob); }
        } else {
            sf[i] = __frcp_rn(df); sb[i] = __frcp_rn(db);
            if (a.masks) { sf[i] = mul_rn(sf[i], sub_rn(1.f, of)); sb[i] = mul_rn(sb[i], sub_rn(1.f, ob)); }   // control_utils.py:69-70
        }
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
            if constexpr (!DET) {
                __stcg(pf + r, make_float4(0.f, 0.f, 0.f, 0.f));
                __stcg(pb + r, make_float4(0.f, 0.f, 0.f, 0.f));
            }
            const float af[4] = {vf[i].x, vf[i].y, vf[i].z, vf[i].w}, ab[4] = {vb[i].x, vb[i].y, vb[i].z, vb[i].w};
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
                const int c = 4 * qq + jj;
                if (c >= C) break;
                // the warped maps as the unfused path stores them (rounded to T), then extractors.py:303-310
                float A, B;
                if constexpr (DET) {
                    A = af[jj] / sf[i]; B = ab[jj] / sb[i];
                    if (a.masks) { A = mul_rn(A, kf[i]); B = mul_rn(B, kb[i]); }
                    A = round_as<T>(A); B = round_as<T>(B);
                } else {
                    A = round_as<T>(mul_rn(af[jj], sf[i])); B = round_as<T>(mul_rn(ab[jj], sb[i]));
                }
                const float v = hole[i] ? mul_rn(0.5f, add_rn(A, B)) : add_rn(mul_rn(w0[i], A), mul_rn(w1[i], B));
                st_stream(fo + (size_t)c * L.HW + r, v);
                if (wf) st_stream(wf + (size_t)c * L.HW + r, A);
                if (wb) st_stream(wb + (size_t)c * L.HW + r, B);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// DCB_FLAG_DETERMINISTIC: emit + sort + reduce in place of launch A
// ---------------------------------------------------------------------------------------------
// A footprint field is one (level, direction): every source pixel of every frame of the level, landing where its flow
// (flow_f forward, flow_b backward) takes it. The feature splat of the direction (first by flow_f, last by flow_b) and the
// mask splat by the same flow (flow_b by flow_f behind occ_b, flow_f by flow_b behind occ_f) land on the same footprints, so
// they share one key set. The targets of all fields are numbered one after the other (global target); a key is
// global_target << s | source_in_frame with 2^s >= the largest H*W, so within a target the keys ascend with the source index:
// the order of k_det_reduce (key = target * HW + source).
struct PyrDetField {
    View flow, in, metric, mflow;    // footprint flow; feature input, its metric (NULL: all-ones); the mask splat's input
    float *acc, *dacc;               // feature cells [N][Cq][HW] float4, normaliser [N][HW]
    float *acc_m, *dacc_m;           // mask cells [N][HW] float4 (x, y, 0, 0), normaliser [N][HW]
    int C, Cq, H, W;
    unsigned HW, NHW;
    unsigned src0, tgt0;             // first source (emit thread, key group of 4) and first global target of the field
    long long item0;                 // first reduce thread of the field: NHW * Cq threads, channel quad major
};
struct PyrDetArgs {
    PyrDetField f[2 * kMaxLevels];
    int n_fields, masks, s;
    unsigned long long* keys;
    const unsigned long long* sorted;
    long long nkeys;
    unsigned long long invalid;      // sorts behind every real key
};

template <class T>
__global__ void __launch_bounds__(256) k_pyr_det_emit(const __grid_constant__ PyrDetArgs a) {
    pdl_wait();
    const unsigned p = blockIdx.x * 256 + threadIdx.x;
    int j = 0;
    while (j + 1 < a.n_fields && p >= a.f[j + 1].src0) ++j;
    const PyrDetField& F = a.f[j];
    const unsigned q = p - F.src0;
    if (q >= F.NHW) return;
    const unsigned n = q / F.HW, r = q - n * F.HW;
    const int y = (int)(r / (unsigned)F.W), x = (int)(r - (unsigned)y * (unsigned)F.W);
    const T* fp = (const T*)F.flow.p + n * F.flow.sN + (long long)y * F.flow.sH + (long long)x * F.flow.sW;
    const Foot<float> f = make_foot<float>(x, y, ld<float>(fp), ld<float>(fp + F.flow.sC));
    const int x1 = (int)((unsigned)f.x0 + 1u), y1 = (int)((unsigned)f.y0 + 1u);
    const bool vx0 = (unsigned)f.x0 < (unsigned)F.W, vx1 = (unsigned)x1 < (unsigned)F.W;
    const bool vy0 = (unsigned)f.y0 < (unsigned)F.H, vy1 = (unsigned)y1 < (unsigned)F.H;
    const bool b[4] = {f.finite && vx0 && vy0, f.finite && vx1 && vy0, f.finite && vx0 && vy1, f.finite && vx1 && vy1};
    const long long t0 = (long long)F.tgt0 + (long long)n * F.HW + (long long)f.y0 * F.W + f.x0;
    const long long off[4] = {0, 1, F.W, (long long)F.W + 1};
#pragma unroll
    for (int k = 0; k < 4; ++k)
        a.keys[4ull * p + k] = b[k] ? ((unsigned long long)(t0 + off[k]) << a.s) | r : a.invalid;
}

template <class T>
__global__ void __launch_bounds__(256) k_pyr_det_reduce(const __grid_constant__ PyrDetArgs a) {
    pdl_wait();
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    int j = 0;
    while (j + 1 < a.n_fields && i >= a.f[j + 1].item0) ++j;
    const PyrDetField& F = a.f[j];
    const long long it = i - F.item0;
    if (it >= (long long)F.NHW * F.Cq) return;
    const unsigned qd = (unsigned)(it / F.NHW), t = (unsigned)(it - (long long)qd * F.NHW);   // channel quad, target
    const unsigned n = t / F.HW, r = t - n * F.HW;
    const int ty = (int)(r / (unsigned)F.W), tx = (int)(r - (unsigned)ty * (unsigned)F.W);
    const unsigned long long lo_key = (unsigned long long)(F.tgt0 + t) << a.s, hi_key = lo_key + (1ull << a.s);
    long long lo = 0, hi = a.nkeys;                       // lower_bound(lo_key)
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (a.sorted[mid] < lo_key) lo = mid + 1; else hi = mid;
    }
    const bool cells = qd == 0;                           // quad 0 also owns the normalisers and the mask cells
    const bool masks = cells && a.masks;
    const float g1 = exp_det_t(1.f);                      // the all-ones metric of compute_mask and of a NULL metric
    const int c0 = 4 * (int)qd;
    float sum[4] = {0.f, 0.f, 0.f, 0.f}, d = 0.f, mx = 0.f, my = 0.f, dm = 0.f;
    for (long long k = lo; k < a.nkeys; ++k) {
        const unsigned long long key = a.sorted[k];
        if (key >= hi_key) break;
        const unsigned src = (unsigned)(key - lo_key);
        const int y = (int)(src / (unsigned)F.W), x = (int)(src - (unsigned)y * (unsigned)F.W);
        const T* fp = (const T*)F.flow.p + n * F.flow.sN + (long long)y * F.flow.sH + (long long)x * F.flow.sW;
        const Foot<float> f = make_foot<float>(x, y, ld<float>(fp), ld<float>(fp + F.flow.sC));
        const int kx = tx - f.x0, ky = ty - f.y0;         // which of the source's corners this target is: 0 or 1 each
        const float w = ky == 0 ? (kx == 0 ? f.wnw : f.wne) : (kx == 0 ? f.wsw : f.wse);
        float g = g1;
        if (F.metric.p) g = exp_det_t(ld<float>((const T*)F.metric.p + n * F.metric.sN + (long long)y * F.metric.sH + (long long)x * F.metric.sW));
        const T* ip = (const T*)F.in.p + n * F.in.sN + (long long)y * F.in.sH + (long long)x * F.in.sW + (long long)c0 * F.in.sC;
#pragma unroll
        for (int jj = 0; jj < 4; ++jj)
            if (c0 + jj < F.C) sum[jj] = det_add(sum[jj], mul_rn(ld<float>(ip + jj * F.in.sC), g), w);
        if (cells) d = det_add(d, g, w);
        if (masks) {
            const T* mp = (const T*)F.mflow.p + n * F.mflow.sN + (long long)y * F.mflow.sH + (long long)x * F.mflow.sW;
            mx = det_add(mx, mul_rn(ld<float>(mp), g1), w);
            my = det_add(my, mul_rn(ld<float>(mp + F.mflow.sC), g1), w);
            dm = det_add(dm, g1, w);
        }
    }
    ((float4*)F.acc)[((size_t)n * F.Cq + qd) * F.HW + r] = make_float4(sum[0], sum[1], sum[2], sum[3]);
    if (cells) F.dacc[t] = d;
    if (masks) {
        ((float4*)F.acc_m)[t] = make_float4(mx, my, 0.f, 0.f);
        F.dacc_m[t] = dm;
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

// deterministic workspace: keys | sorted keys | cub temp | the cells of pyramid_workspace()
struct PyrDetLayout {
    long long nsrc, nkeys, sorted_off, temp_off, cells_off, total_bytes;
    size_t temp_bytes;
    int s, end_bit;
};

static PyrDetLayout pyr_det_layout(const DcbPyramidLevel* lv, int n) {
    PyrDetLayout L;
    long long nhw = 0, max_hw = 1;
    for (int l = 0; l < n; ++l) {
        const DcbTensor* f = lv[l].first;
        if (!f || f->size[0] * f->size[1] * f->size[2] * f->size[3] <= 0) continue;
        nhw += f->size[0] * f->size[2] * f->size[3];
        if (f->size[2] * f->size[3] > max_hw) max_hw = f->size[2] * f->size[3];
    }
    L.nsrc = 2 * nhw;                                  // two footprint fields per level; as many targets as sources
    L.nkeys = 4 * L.nsrc;
    L.s = 0;
    while ((1ll << L.s) < max_hw) ++L.s;
    L.end_bit = key_bits(L.nsrc, 1ll << L.s);
    L.temp_bytes = L.nkeys > 0 && L.nkeys < (1ll << 31) ? cub_temp_bytes(L.nkeys, L.end_bit) : 0;
    L.sorted_off = align_up(L.nkeys * 8, 256);
    L.temp_off = L.sorted_off + align_up(L.nkeys * 8, 256);
    L.cells_off = L.temp_off + align_up((long long)L.temp_bytes, 256);
    L.total_bytes = L.cells_off + pyramid_workspace(lv, n);
    return L;
}

long long pyramid_det_keys(const DcbPyramidLevel* lv, int n) { return pyr_det_layout(lv, n).nkeys; }
long long pyramid_det_workspace(const DcbPyramidLevel* lv, int n) { return pyr_det_layout(lv, n).total_bytes; }

template <class T>
static int launch_pyramid(const PyrScatterArgs& sa, unsigned s_items, const PyrFuseArgs& fa, unsigned f_items, cudaStream_t st) {
    DCB_CHECK_CUDA(launch_pdl(k_pyr_scatter<T>, dim3(s_items), dim3(32), 0, st, sa));
    count_launch();
    DCB_CHECK_CUDA(launch_pdl(k_pyr_fuse<T, false>, dim3(f_items), dim3(32), 0, st, fa));
    count_launch();
    return DCB_OK;
}

template <class T>
static int launch_pyramid_det(const PyrDetArgs& da, const PyrDetLayout& D, char* ws, long long r_items, const PyrFuseArgs& fa,
                              unsigned f_items, cudaStream_t st) {
    DCB_CHECK_CUDA(launch_pdl(k_pyr_det_emit<T>, dim3((unsigned)((D.nsrc + 255) / 256)), dim3(256), 0, st, da));
    count_launch();
    const int rc = det_sort_keys(ws + D.temp_off, D.temp_bytes, da.keys, (unsigned long long*)da.sorted, D.nkeys, D.end_bit, st);
    if (rc != DCB_OK) return rc;
    DCB_CHECK_CUDA(launch_pdl(k_pyr_det_reduce<T>, dim3((unsigned)((r_items + 255) / 256)), dim3(256), 0, st, da));
    count_launch();
    DCB_CHECK_CUDA(launch_pdl(k_pyr_fuse<T, true>, dim3(f_items), dim3(32), 0, st, fa));
    count_launch();
    return DCB_OK;
}

// Preconditions (checked by the caller): 1 <= n <= kMaxLevels, all tensors of one dtype (F32 / BF16 / F16), shapes consistent,
// ws holds pyramid_workspace() bytes, 256-byte aligned, all-zero if DCB_FLAG_WS_CLEAN; with DCB_FLAG_DETERMINISTIC (never with
// WS_CLEAN) ws is plain scratch of pyramid_det_workspace() bytes and pyramid_det_keys() < 2^31.
int bidir_pyramid_fwd_impl(const DcbPyramidLevel* lv, int n, void* ws, int flags, cudaStream_t st) {
    PyrScatterArgs sa; PyrFuseArgs fa; PyrDetArgs da;
    sa.n_jobs = 0; fa.n_levels = 0; da.n_fields = 0;
    fa.masks = (flags & DCB_PYRAMID_NO_MASKS) ? 0 : 1;
    fa.holes = (flags & DCB_PYRAMID_NO_HOLES) ? 0 : 1;
    const bool det = (flags & DCB_FLAG_DETERMINISTIC) != 0;
    long long shared_total = 0;
    for (int l = 0; l < n; ++l) shared_total += level_shared_bytes(lv[l].first->size[0], lv[l].first->size[2], lv[l].first->size[3]);
    const long long total = pyramid_workspace(lv, n);
    PyrDetLayout D = {};
    char* cells = (char*)ws;
    if (det) {
        D = pyr_det_layout(lv, n);
        cells += D.cells_off;
        da.masks = fa.masks; da.s = D.s; da.nkeys = D.nkeys;
        da.keys = (unsigned long long*)ws;
        da.sorted = (const unsigned long long*)((char*)ws + D.sorted_off);
        da.invalid = (unsigned long long)D.nsrc << D.s;
    } else if (!(flags & DCB_FLAG_WS_CLEAN)) {
        DCB_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)total, st));
    }
    char* shared = cells;
    char* feat = cells + shared_total;
    unsigned s_items = 0, f_items = 0, d_src = 0, d_tgt = 0;
    long long r_items = 0;
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
        auto add_field = [&](const DcbTensor* flow, const DcbTensor* in, const DcbTensor* metric, const DcbTensor* mflow, float* acc,
                             float* dacc, float* acc_m, float* dacc_m) {
            PyrDetField& F = da.f[da.n_fields++];
            F.flow = make_view(flow); F.in = make_view(in); F.metric = make_view(metric); F.mflow = make_view(mflow);
            F.acc = acc; F.dacc = dacc; F.acc_m = acc_m; F.dacc_m = dacc_m;
            F.C = (int)C; F.Cq = (int)Cq; F.H = (int)H; F.W = (int)W;
            F.HW = (unsigned)HW; F.NHW = (unsigned)(N * HW);
            F.src0 = d_src; F.tgt0 = d_tgt; F.item0 = r_items;
            d_src += F.NHW; d_tgt += F.NHW; r_items += (long long)F.NHW * F.Cq;
        };
        if (det) {
            add_field(d.flow_f, d.first, d.metric_f, d.flow_b, acc_f, dacc_f, acc_mb, dacc_mb);   // compute_mask(flow_b, flow_f)
            add_field(d.flow_b, d.last, d.metric_b, d.flow_f, acc_b, dacc_b, acc_mf, dacc_mf);    // compute_mask(flow_f, flow_b)
        } else {
            if (fa.masks) {
                add_job(d.flow_f, d.flow_b, nullptr, acc_mf, dacc_mf, 2);        // compute_mask(flow_f, flow_b)
                add_job(d.flow_b, d.flow_f, nullptr, acc_mb, dacc_mb, 2);        // compute_mask(flow_b, flow_f)
            }
            add_job(d.first, d.flow_f, d.metric_f, acc_f, dacc_f, C);
            add_job(d.last, d.flow_b, d.metric_b, acc_b, dacc_b, C);
        }
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
    if (det) {
        if ((r_items + 255) / 256 >= (1ll << 31))
            return set_error(DCB_E_LIMIT, "bidir_pyramid_fwd(deterministic): %lld (pixel, channel quad) cells exceed the grid", r_items);
        switch (dt) {
            case DCB_F32: return launch_pyramid_det<float>(da, D, (char*)ws, r_items, fa, f_items, st);
            case DCB_BF16: return launch_pyramid_det<__nv_bfloat16>(da, D, (char*)ws, r_items, fa, f_items, st);
            case DCB_F16: return launch_pyramid_det<__half>(da, D, (char*)ws, r_items, fa, f_items, st);
            default: return set_error(DCB_E_DTYPE, "bidir_pyramid_fwd: unsupported dtype %d", dt);
        }
    }
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
