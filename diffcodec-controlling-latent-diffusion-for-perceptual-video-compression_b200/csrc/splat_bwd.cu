// splat_bwd.cu -- backward of the forward splat (K3) for sm_100a.
//
// Replaces softsplat_func.backward (kernels `softsplat_ingrad` controlnet/softsplat.py:368-435 and
// `softsplat_flowgrad` :439-524) AND the autograd of the eager ops around it (exp, mul, cat,
// slice, eps, div -- softsplat.py:240-270; (1 - mask) product -- control_utils.py:69-70).
//
// Closed form (SURVEY.md Appendix A-4), with G the upstream gradient, D the saved normaliser,
// out the saved output, g(m) in {1, m, exp(m)}:
//   target side (K3a, one thread per target pixel):
//       a = (1 - mask) / D              T = -(sum_c G_c * out_c) / D
//   source side (K3b, gather; no atomics), corners k = NW, NE, SW, SE with bilinear weights w_k:
//       A_k      = sum_c G_c(k) * in_c
//       gradIn_c = g * sum_k w_k a_k G_c(k)
//       B_k      = a_k A_k + T_k                     (B_k = A_k for 'sum')
//       gradMetric = g'(m) * sum_k w_k B_k           (g' = exp(m) | 1)
//       gradFlow_x = g * [(B_NE - B_NW)(y1 - fy) + (B_SE - B_SW)(fy - y0)]
//       gradFlow_y = g * [(B_SW - B_NW)(x1 - fx) + (B_SE - B_NE)(fx - x0)]
// The reference reads every gradOut corner 1 + 2*C' times per pixel (ingrad thread + two flowgrad
// threads); here each corner is read once per channel and feeds all three gradients.
//
// Thread layout: blockDim = (PX, CS): PX source pixels, CS channel slices per pixel. CS > 1 is
// chosen when there are too few pixels to fill the machine (8x8 .. 64x64 ControlNet pyramids with
// hundreds of channels); the A_k partials are then reduced through shared memory.
#include "splat_bwd.cuh"

#include <type_traits>

namespace dcb {

// K3a -- target-side scalars. blockDim = (px, cs) like K3b: cs channel slices per pixel when pixels are scarce
// (one thread per pixel walked the 1280 channels of an 8x8 pyramid level in 160 dependent steps: 175 us).
// 8 channels (16 loads) in flight per thread.
template <class T>
__global__ void __launch_bounds__(256) k_bwd_target(const BwdArgs a) {
    using A = typename Acc<T>::type;
    extern __shared__ unsigned char smem_raw[];
    A* red = (A*)smem_raw;                                        // [cs][px] when cs > 1
    const int tx = threadIdx.x, ty = threadIdx.y, cs = blockDim.y, npx = blockDim.x;
    const unsigned p = blockIdx.x * npx + tx;
    const bool live = p < a.total;
    const unsigned pc = live ? p : 0;
    const unsigned n = pc / a.HW, r = pc - n * a.HW;
    const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
    const T* gp = (const T*)a.gout.p + n * a.gout.sN + y * a.gout.sH + x * a.gout.sW;
    const T* op = (const T*)a.out + (long long)n * a.C * a.HW + r;
    A dot = (A)0;
    constexpr int U = 8;
    for (int c0 = ty; c0 < a.C; c0 += U * cs) {
        A gv[U], ov[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int c = c0 + j * cs;
            const bool in = c < a.C;
            gv[j] = in ? ld<A>(gp + (long long)c * a.gout.sC) : (A)0;
            ov[j] = in ? ld<A>(op + (long long)c * a.HW) : (A)0;
        }
#pragma unroll
        for (int j = 0; j < U; ++j) dot += gv[j] * ov[j];
    }
    if (cs > 1) {
        red[(size_t)ty * npx + tx] = dot;
        __syncthreads();
        if (ty != 0) return;
        for (int s = 1; s < cs; ++s) dot += red[(size_t)s * npx + tx];
    }
    if (!live) return;
    const A d = ((const A*)a.norm)[p];
    A keep = (A)1;
    if (a.mask.p) {
        const T* mp = (const T*)a.mask.p + n * a.mask.sN + y * a.mask.sH + x * a.mask.sW;
        keep = (A)1 - ld<A>(mp);
    }
    A* ts = (A*)a.tscal + 2ll * p;
    ts[0] = keep / d;
    // d(normaliser)/d(S_w) is 0 where clip(1e-7) was active (softsplat.py:266); for zeroeps the
    // replaced entries have out == 0, hence dot == 0, on their own
    const bool clipped = a.eps == DCB_EPS_CLIP && d == (A)0.0000001;
    ts[1] = clipped ? (A)0 : -dot / d;
}

// K3b -- source-side gather (bwd_source_body, splat_bwd.cuh).
template <class T, class TF, class IX>
__global__ void __launch_bounds__(256, DCB_BS_MINCTAS) k_bwd_source(const BwdArgs a) {
    extern __shared__ unsigned char smem_raw[];
    bwd_source_body<T, TF, IX, false>(a, blockIdx.x, threadIdx.x, threadIdx.y, smem_raw, nullptr);
}

// ---------------------------------------------------------------------------------------------
// Few channels (C <= 3: frames, flows, masks) in fp32 / bf16, normalised modes: the target pass packs
// everything the source pass needs from a target pixel into ONE float4
//       P_c = a * G_c  (c < 3, zero-padded),   T
// because  gradIn_c = g * sum_k w_k P_c(k)   and   B_k = a_k A_k + T_k = sum_c P_c(k) in_c + T_k.
// The source pass then gathers one 16-byte cell per corner (4 loads) instead of C gradOut scalars
// plus two scalars (20 loads at C = 3), and neighbouring lanes read neighbouring cells.
// ---------------------------------------------------------------------------------------------
template <class T>
__global__ void __launch_bounds__(256) k_bwd_target4(const BwdArgs a) {
    pdl_wait();                                                   // the packed cells are one slot shared by consecutive frame groups
    const unsigned p = blockIdx.x * 256 + threadIdx.x;
    if (p >= a.total) return;
    const unsigned n = p / a.HW, r = p - n * a.HW;
    const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
    const float d = ld_stream((const float*)a.norm + p);
    const T* gp = (const T*)a.gout.p + n * a.gout.sN + y * a.gout.sH + x * a.gout.sW;
    const T* op = (const T*)a.out + (long long)n * a.C * a.HW + r;
    float gv[3] = {0.f, 0.f, 0.f}, ov[3] = {0.f, 0.f, 0.f};
#pragma unroll
    for (int c = 0; c < 3; ++c)
        if (c < a.C) { gv[c] = ld_stream(gp + (long long)c * a.gout.sC); ov[c] = ld_stream(op + (long long)c * a.HW); }
    float dot = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) dot += gv[c] * ov[c];
    float keep = 1.f;
    if (a.mask.p) {
        const T* mp = (const T*)a.mask.p + n * a.mask.sN + y * a.mask.sH + x * a.mask.sW;
        keep = 1.f - ld<float>(mp);
    }
    const float av = keep / d;
    const bool clipped = a.eps == DCB_EPS_CLIP && d == 0.0000001f;     // see k_bwd_target
    __stcg((float4*)a.tscal + p, make_float4(av * gv[0], av * gv[1], av * gv[2], clipped ? 0.f : -dot / d));
}

#ifndef DCB_B4_PF
#define DCB_B4_PF 1
#endif
// grid = (32-pixel tile columns, 8-row tile rows, frames): no integer division anywhere; one 64-bit base per tensor and
// frame, every in-frame offset in 32 bits (checked by the host: views whose in-frame span does not fit are refused, as in the
// forward). 32 x 8 pixel tiles: the packed cells gathered by vertically adjacent pixels are the same rows (L1).
// CT = 0: any strides, channel count and mode at run time. CT = 1..3: C = CT and mode = MT at compile time, `in`, `flow` and
// `metric` NCHW-contiguous inside a frame, all three gradients wanted (the autograd call on frames / flows / latents): every
// load offset is the pixel index plus a multiple of H*W, and the per-channel / per-mode tests disappear.
template <class T, class TF, int CT, int MT>
__global__ void __launch_bounds__(256) k_bwd_source4(const BwdArgs a) {
    pdl_wait();
    constexpr bool kFlat = CT != 0;
    const int C = kFlat ? CT : a.C, mode = kFlat ? MT : a.mode;
    const int W = a.W, H = a.H;
    const unsigned n = blockIdx.z;
    const int x = (int)(blockIdx.x * 32 + (threadIdx.x & 31)), y = (int)(blockIdx.y * 8 + (threadIdx.x >> 5));
#if DCB_B4_PF
    {   // L2 prefetch for the tile one wave ahead (pf_rows tile rows further down, wrapping into the next frame): flow (2),
        // metric, in (3) and the packed cells at the zero-flow position; 8 rows x 12 planes, one line per thread
        unsigned pty = blockIdx.y + a.pf_rows, pn = n;
        if (pty >= gridDim.y) { pty -= gridDim.y; ++pn; }
        const int py = (int)(pty * 8 + (threadIdx.x & 7)), px0 = (int)(blockIdx.x * 32);
        const int plane = threadIdx.x >> 3;
        if (pn < gridDim.z && pty < gridDim.y && py < H) {
            const void* q = nullptr;
            if (plane < 2) q = (const TF*)a.flow.p + (pn * a.flow.sN + plane * a.flow.sC) + (py * (int)a.flow.sH + px0 * (int)a.flow.sW);
            else if (plane == 2 && a.metric.p) q = (const T*)a.metric.p + pn * a.metric.sN + (py * (int)a.metric.sH + px0 * (int)a.metric.sW);
            else if (plane >= 4 && plane < 4 + a.C) q = (const T*)a.in.p + (pn * a.in.sN + (plane - 4) * a.in.sC) + (py * (int)a.in.sH + px0 * (int)a.in.sW);
            else if (plane >= 8 && plane < 12) q = (const float4*)a.tscal + (size_t)pn * a.HW + (unsigned)(py * W + px0 + (plane - 8) * 8);
            if (q) asm volatile("prefetch.global.L2 [%0];" ::"l"(q));
        }
    }
#endif
    if (x >= W || y >= H) return;
    const unsigned r = (unsigned)y * (unsigned)W + (unsigned)x, p = n * a.HW + r;
    const TF* fp = (const TF*)a.flow.p + n * a.flow.sN + (kFlat ? (int)r : y * (int)a.flow.sH + x * (int)a.flow.sW);
    const Foot<float> f = make_foot<float>(x, y, (float)ld_stream(fp), (float)ld_stream(fp + (kFlat ? (long long)a.HW : a.flow.sC)));
    const int x1 = (int)((unsigned)f.x0 + 1u), y1 = (int)((unsigned)f.y0 + 1u);
    const bool vx0 = (unsigned)f.x0 < (unsigned)W, vx1 = (unsigned)x1 < (unsigned)W;
    const bool vy0 = (unsigned)f.y0 < (unsigned)H, vy1 = (unsigned)y1 < (unsigned)H;
    const bool ok = f.finite;                                     // softsplat.py:389-390, 460-461
    const bool b[4] = {ok && vx0 && vy0, ok && vx1 && vy0, ok && vx0 && vy1, ok && vx1 && vy1};
    const bool any = b[0] || b[1] || b[2] || b[3];
    const float w[4] = {f.wnw, f.wne, f.wsw, f.wse};

    float g = 1.f, gprime = 1.f;
    if (mode == DCB_MODE_LINEAR || mode == DCB_MODE_SOFT) {
        const T* mp = (const T*)a.metric.p + n * a.metric.sN + (kFlat ? (int)r : y * (int)a.metric.sH + x * (int)a.metric.sW);
        const float m = ld_stream(mp);
        g = mode == DCB_MODE_SOFT ? expf(m) : m;
        gprime = mode == DCB_MODE_SOFT ? g : 1.f;
    }
    // the four target cells: one 16-byte gather each (element 0 of the frame stands in for a corner out of range)
    const float4* cell = (const float4*)a.tscal + (size_t)n * a.HW;
    const int o0 = f.y0 * W + f.x0;
    const int co[4] = {b[0] ? o0 : 0, b[1] ? o0 + 1 : 0, b[2] ? o0 + W : 0, b[3] ? o0 + W + 1 : 0};
    float4 P[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) P[k] = __ldcg(cell + co[k]);
    const T* ip = (const T*)a.in.p + n * a.in.sN + (kFlat ? (int)r : y * (int)a.in.sH + x * (int)a.in.sW);
    float v[3] = {0.f, 0.f, 0.f};
    const bool need_A = kFlat || (a.gflow != nullptr) || (a.gmetric != nullptr);
    if (need_A) {
#pragma unroll
        for (int c = 0; c < 3; ++c)
            if (c < C) v[c] = ld_stream(ip + (kFlat ? c * (int)a.HW : c * (int)a.in.sC));
    }
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (!b[k]) P[k] = make_float4(0.f, 0.f, 0.f, 0.f);

    if (kFlat || a.gin) {
        T* gi = (T*)a.gin + (long long)n * C * a.HW + r;
        // a dropped corner carries P = 0, but its weight may be inf (huge finite flow): keep 0 * inf out
        const float wz[4] = {b[0] ? w[0] : 0.f, b[1] ? w[1] : 0.f, b[2] ? w[2] : 0.f, b[3] ? w[3] : 0.f};
        const float s0 = fma_rn(P[3].x, wz[3], fma_rn(P[2].x, wz[2], fma_rn(P[1].x, wz[1], mul_rn(P[0].x, wz[0]))));
        const float s1 = fma_rn(P[3].y, wz[3], fma_rn(P[2].y, wz[2], fma_rn(P[1].y, wz[1], mul_rn(P[0].y, wz[0]))));
        const float s2 = fma_rn(P[3].z, wz[3], fma_rn(P[2].z, wz[2], fma_rn(P[1].z, wz[1], mul_rn(P[0].z, wz[0]))));
        st_stream(gi, (any ? s0 : 0.f) * g);
        if (C > 1) st_stream(gi + a.HW, (any ? s1 : 0.f) * g);
        if (C > 2) st_stream(gi + 2ll * a.HW, (any ? s2 : 0.f) * g);
    }
    if (!need_A) return;
    float B[4];
#pragma unroll
    for (int k = 0; k < 4; ++k)
        B[k] = b[k] ? fma_rn(P[k].x, v[0], fma_rn(P[k].y, v[1], fma_rn(P[k].z, v[2], P[k].w))) : 0.f;
    if (kFlat ? mode != DCB_MODE_AVG : a.gmetric != nullptr) {
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) if (b[k]) s = fma_rn(w[k], B[k], s);
        st<T, float>((T*)a.gmetric + p, any ? s * gprime : 0.f);
    }
    if (kFlat || a.gflow) {
        const float ey = sub_rn((float)y1, f.fy), dy = sub_rn(f.fy, (float)f.y0);      // d w / d flow, softsplat.py:477-487
        const float ex = sub_rn((float)x1, f.fx), dx = sub_rn(f.fx, (float)f.x0);
        float gx = (B[1] - B[0]) * ey + (B[3] - B[2]) * dy;
        float gy = (B[2] - B[0]) * ex + (B[3] - B[1]) * dx;
        if (!any) { gx = 0.f; gy = 0.f; }
        TF* gf = (TF*)a.gflow + (long long)n * 2 * a.HW + r;
        st<TF, float>(gf, gx * g);
        st<TF, float>(gf + a.HW, gy * g);
    }
}

// dcb_set_option("bwd_group_bytes"): packed cells per frame group of the C <= 3 backward; 0 restores the default = ONE group.
// Measured on 16 x 1080p (profiles/scripts/run_frames_bwd.py, us per frame, backward only): one frame per group (cells stay in
// L2, two launches per frame) 52.5; 2 frames 51.3; 4 frames 49.7; all frames in one group (cells round-trip through HBM) 48.6 --
// the launch boundaries cost more than the 32 B/px of DRAM traffic they save, the same lesson as the forward's tails.
// dcb_set_option("bwd_flat", 0): A/B switch, always the run-time (strided) form of the packed source pass
int g_bwd_flat = 1;
void bwd_set_flat(long long v) { g_bwd_flat = v != 0; }
constexpr long long kBwdOneGroup = 1ll << 50;
long long g_bwd_group_bytes = kBwdOneGroup;
void bwd_set_group_bytes(long long b) { g_bwd_group_bytes = b > 0 ? b : kBwdOneGroup; }

static bool packed_bwd(int C, int dtype, int mode) { return C <= 3 && mode != DCB_MODE_SUM && dtype != DCB_F64; }

// ---------------------------------------------------------------------------------------------
long long splat_bwd_workspace(long long N, long long C, long long H, long long W, int dtype, int mode) {
    if (mode == DCB_MODE_SUM) return 0;
    if (packed_bwd((int)(C > 3 ? 4 : C), dtype, mode)) {                                          // one float4 per target pixel of ONE frame group
        long long G = g_bwd_group_bytes / (H * W * 16 > 0 ? H * W * 16 : 1);
        if (G < 1) G = 1;
        return align_up((N < G ? N : G) * H * W * 16, 256);
    }
    return align_up(N * H * W * 2 * (dtype == DCB_F64 ? 8 : 4), 256);
}

template <class T, class TF, int CT>
static cudaError_t launch_source4_c(const BwdArgs& g, const dim3& grid, cudaStream_t st) {
    switch (g.mode) {
        case DCB_MODE_AVG: return launch_pdl(k_bwd_source4<T, TF, CT, DCB_MODE_AVG>, grid, dim3(256), 0, st, g);
        case DCB_MODE_LINEAR: return launch_pdl(k_bwd_source4<T, TF, CT, DCB_MODE_LINEAR>, grid, dim3(256), 0, st, g);
        default: return launch_pdl(k_bwd_source4<T, TF, CT, DCB_MODE_SOFT>, grid, dim3(256), 0, st, g);
    }
}

template <class T, class TF>
static cudaError_t launch_source4(const BwdArgs& g, bool flat, cudaStream_t st) {
    const dim3 grid(g.tiles_x, g.tiles / g.tiles_x, (unsigned)g.N);
    if (flat) {
        if (g.C == 1) return launch_source4_c<T, TF, 1>(g, grid, st);
        if (g.C == 2) return launch_source4_c<T, TF, 2>(g, grid, st);
        if (g.C == 3) return launch_source4_c<T, TF, 3>(g, grid, st);
    }
    return launch_pdl(k_bwd_source4<T, TF, 0, 0>, grid, dim3(256), 0, st, g);
}

template <class T, class TF>
static int launch_bwd(BwdArgs& a, int dtype, cudaStream_t st) {
    using A = typename Acc<T>::type;
    if constexpr (!std::is_same<T, double>::value) {
        if (packed_bwd(a.C, dtype, a.mode)) {
            // Frame groups (dcb_set_option("bwd_group_bytes"); default: one group = all frames): target pass and source pass
            // alternate on one slot of packed cells, chained by programmatic dependent launch.
            a.tiles_x = (unsigned)(a.W + 31) / 32;
            a.tiles = a.tiles_x * ((unsigned)(a.H + 7) / 8);
            a.pf_dist = (unsigned)(device_sm_count() * 5);      // 48 registers: 5 CTAs per SM
            a.pf_rows = a.pf_dist / a.tiles_x > 0 ? a.pf_dist / a.tiles_x : 1;
            {   // in-frame element offsets are formed in 32 bits
                auto fits = [&](const View& v, long long ch) {
                    if (!v.p) return true;
                    auto ab = [](long long q) { return q < 0 ? -q : q; };
                    return (ch - 1) * ab(v.sC) + (long long)(a.H - 1) * ab(v.sH) + (long long)(a.W - 1) * ab(v.sW) < (1ll << 31);
                };
                if (!fits(a.in, a.C) || !fits(a.flow, 2) || !fits(a.metric, 1) || (long long)a.tiles / a.tiles_x > 65535)
                    return set_error(DCB_E_LIMIT, "splat_bwd: tensor spans beyond 2^31 elements (or more than 524280 rows) are not supported by the packed path");
            }
            long long G = g_bwd_group_bytes / ((long long)a.HW * 16 > 0 ? (long long)a.HW * 16 : 1);
            if (G < 1) G = 1;
            if (G > 65535) G = 65535;                           // gridDim.z of the source pass
            const int es = (int)sizeof(T), fs = (int)sizeof(TF);
            // the compile-time form: frames contiguous inside (NCHW), every gradient wanted (a metric gradient exists in the
            // linear / soft modes only)
            auto plane_contig = [&](const View& v, long long ch) { return v.sW == 1 && v.sH == a.W && (ch == 1 || v.sC == (long long)a.HW); };
            const bool has_metric = a.mode == DCB_MODE_LINEAR || a.mode == DCB_MODE_SOFT;
            const bool flat = g_bwd_flat && plane_contig(a.in, a.C) && plane_contig(a.flow, 2) && (!has_metric || plane_contig(a.metric, 1)) &&
                              a.gin && a.gflow && (has_metric ? a.gmetric != nullptr : a.gmetric == nullptr);
            for (long long f0 = 0; f0 < a.N; f0 += G) {
                const long long nf = a.N - f0 < G ? a.N - f0 : G;
                BwdArgs g = a;
                auto adv = [&](View& v, int e) { if (v.p) v.p = (const char*)v.p + f0 * v.sN * e; };
                adv(g.gout, es); adv(g.in, es); adv(g.flow, fs); adv(g.metric, es); adv(g.mask, es);
                if (a.out) g.out = (const char*)a.out + (size_t)f0 * a.C * a.HW * es;
                if (a.norm) g.norm = (const char*)a.norm + (size_t)f0 * a.HW * sizeof(float);
                if (a.gin) g.gin = (char*)a.gin + (size_t)f0 * a.C * a.HW * es;
                if (a.gflow) g.gflow = (char*)a.gflow + (size_t)f0 * 2 * a.HW * fs;
                if (a.gmetric) g.gmetric = (char*)a.gmetric + (size_t)f0 * a.HW * es;
                g.N = (int)nf; g.total = (unsigned)(nf * a.HW);
                DCB_CHECK_CUDA(launch_pdl(k_bwd_target4<T>, dim3((g.total + 255) / 256), dim3(256), 0, st, g));
                count_launch();
                DCB_CHECK_CUDA((launch_source4<T, TF>(g, flat, st)));
                count_launch();
            }
            return DCB_OK;
        }
    }
    // channel slices: fill ~148 SMs x 8 CTAs when pixels are scarce
#ifndef DCB_BS_FILL
#define DCB_BS_FILL 2048
#endif
    int cs = 1;
    while (cs < 32 && cs * 2 <= a.C && (long long)a.total * cs < 148LL * DCB_BS_FILL) cs *= 2;
    if (a.mode != DCB_MODE_SUM) {
        int ct = 1;                                               // the target pass keeps 8 channels per slice in flight
        while (ct < 32 && ct * 2 * 8 <= a.C && (long long)a.total * ct < 148LL * 2048) ct *= 2;
        const int tpx = 256 / ct;
        k_bwd_target<T><<<(a.total + tpx - 1) / tpx, dim3(tpx, ct), ct > 1 ? (size_t)256 * sizeof(A) : 0, st>>>(a);
        DCB_CHECK_LAUNCH("k_bwd_target");
    }
    a.cs = cs;
    a.px = 256 / cs;
    a.pf_dist = (unsigned)(device_sm_count() * DCB_BS_MINCTAS);
    dim3 block(a.px, cs);
    const unsigned blocks = (a.total + a.px - 1) / a.px;
    const size_t smem = cs > 1 ? (size_t)256 * 4 * sizeof(A) : 0;
    // plane-relative gradOut offsets in 32 bits whenever the view allows it
    const long long span = (long long)(a.H - 1) * (a.gout.sH < 0 ? -a.gout.sH : a.gout.sH) +
                           (long long)(a.W - 1) * (a.gout.sW < 0 ? -a.gout.sW : a.gout.sW);
    if (span < (1ll << 30))
        k_bwd_source<T, TF, int><<<blocks, block, smem, st>>>(a);
    else
        k_bwd_source<T, TF, long long><<<blocks, block, smem, st>>>(a);
    DCB_CHECK_LAUNCH("k_bwd_source");
    return DCB_OK;
}

int splat_bwd_impl(const DcbTensor* gout, const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric,
                   const DcbTensor* out, const DcbTensor* norm, const DcbTensor* mask, const DcbTensor* gin,
                   const DcbTensor* gflow, const DcbTensor* gmetric, void* ws, long long ws_bytes, int mode,
                   int eps, cudaStream_t st) {
    BwdArgs a;
    a.gout = make_view(gout);
    a.in = make_view(in);
    a.flow = make_view(flow);
    a.metric = make_view(metric);
    a.mask = make_view(mask);
    a.out = out ? out->ptr : nullptr;
    a.norm = norm ? norm->ptr : nullptr;
    a.gin = gin ? gin->ptr : nullptr;
    a.gflow = gflow ? gflow->ptr : nullptr;
    a.gmetric = gmetric ? gmetric->ptr : nullptr;
    a.N = (int)in->size[0]; a.C = (int)in->size[1]; a.H = (int)in->size[2]; a.W = (int)in->size[3];
    a.HW = (unsigned)(in->size[2] * in->size[3]);
    a.total = (unsigned)(in->size[0] * in->size[2] * in->size[3]);
    a.mode = mode;
    a.eps = eps;
    a.tscal = nullptr;
    if (a.total == 0) return DCB_OK;
    if (!a.gin && !a.gflow && !a.gmetric) return DCB_OK;
    if (mode != DCB_MODE_SUM) {
        const long long need = splat_bwd_workspace(a.N, a.C, a.H, a.W, in->dtype, mode);
        if (!ws || ws_bytes < need || ((uintptr_t)ws & 255))
            return set_error(DCB_E_WORKSPACE, "splat_bwd: workspace of %lld bytes (256 B aligned) required, got %lld",
                             need, ws_bytes);
        a.tscal = ws;
    }
    const bool flow_f32 = flow->dtype == DCB_F32;
    switch (in->dtype) {
        case DCB_F32: return launch_bwd<float, float>(a, DCB_F32, st);
        case DCB_F64: return launch_bwd<double, double>(a, DCB_F64, st);
        case DCB_BF16:
            return flow_f32 ? launch_bwd<__nv_bfloat16, float>(a, DCB_BF16, st) : launch_bwd<__nv_bfloat16, __nv_bfloat16>(a, DCB_BF16, st);
    }
    return set_error(DCB_E_DTYPE, "splat_bwd: unsupported dtype %d", in->dtype);
}

}  // namespace dcb
