// backwarp.cu -- bilinear backward warp (+ fused residual) and its backward (K4 / K4b), sm_100a.
//
// Replaces WarpingLayerBWFlow.forward, cmp/models/modules/warp.py:9-25: the reference allocates
// zeros_like(flow), two linspace grids, a cat, an H2D copy, an add and a permute (five extra
// full-tensor passes) and then calls torch's grid_sample. Here the normalised grid value is
// formed in registers with the same fp32 operation sequence, so no grid tensor exists:
//     t    = flow_x / ((W-1)/2)                                     warp.py:11
//     lin  = linspace(-1, 1, W)[x]   (torch: fma(step, i, -1) below W/2, fma(-step, W-1-i, 1) above)
//     g    = lin + t                                                warp.py:24
//     sx   = ((g + 1) * W - 1) / 2          align_corners = 0   (grid_sample default, as executed)
//     sx   = ((g + 1) / 2) * (W - 1)        align_corners = 1
// followed by grid_sample's bilinear footprint with zeros padding. The optional residual
// (gt - warped, controlnet/residual_utils.py:199) is fused into the same pass.
#include "dcb_common.cuh"

namespace dcb {

struct WarpArgs {
    View image, flow, gt, gout;
    void* warped;        // [N,C,H,W] contiguous
    void* residual;      // [N,C,H,W] contiguous or null
    void* gimage;        // [N,C,H,W] contiguous (zeroed before the launch) or null
    void* gflow;         // [N,2,H,W] contiguous or null
    unsigned total, HW;
    int N, C, H, W;
    int align;
};

template <class A> struct Tap {
    int x0, y0;
    A wnw, wne, wsw, wse;
    A ex, ey, dx, dy;    // (x1 - sx), (y1 - sy), (sx - x0), (sy - y0)
    bool b[4];
};

// Per-launch constants of the grid arithmetic, evaluated once on the host with the same IEEE
// operations (a division per pixel costs ~10 instructions plus a range check on the device).
template <class A> struct TapConst {
    A stepx, stepy;      // linspace step 2 / (n - 1)
    A divx, divy;        // (n - 1) / 2, the divisor of warp.py:11-12
};

template <class A> static TapConst<A> make_tap_const(int W, int H) {
    TapConst<A> k;
    k.stepx = W > 1 ? (A)2 / (A)(W - 1) : (A)0;
    k.stepy = H > 1 ? (A)2 / (A)(H - 1) : (A)0;
    k.divx = (A)((W - 1.0) / 2.0);
    k.divy = (A)((H - 1.0) / 2.0);
    return k;
}

template <class A> __device__ __forceinline__ A linspace_pm1(int i, int n, A step) {
    if (n == 1) return (A)-1;
    return i < n / 2 ? fma_rn(step, (A)i, (A)-1) : fma_rn(-step, (A)(n - 1 - i), (A)1);
}

template <class A> __device__ __forceinline__ A unnormalize(A g, int size, int align) {
    if (align) return ((g + (A)1) / (A)2) * (A)(size - 1);
    return fma_rn(g + (A)1, (A)size, (A)-1) / (A)2;
}

template <class A>
__device__ __forceinline__ Tap<A> make_tap(int x, int y, A flow_x, A flow_y, int W, int H, int align, const TapConst<A>& k) {
    Tap<A> t;
    const A gx = linspace_pm1<A>(x, W, k.stepx) + flow_x / k.divx;
    const A gy = linspace_pm1<A>(y, H, k.stepy) + flow_y / k.divy;
    const A sx = unnormalize<A>(gx, W, align), sy = unnormalize<A>(gy, H, align);
    const A x0f = floor_t(sx), y0f = floor_t(sy);
    t.x0 = to_int_sat(x0f);
    t.y0 = to_int_sat(y0f);
    t.ex = (x0f + (A)1) - sx; t.ey = (y0f + (A)1) - sy;
    t.dx = sx - x0f; t.dy = sy - y0f;
    t.wnw = mul_rn(t.ex, t.ey); t.wne = mul_rn(t.dx, t.ey);
    t.wsw = mul_rn(t.ex, t.dy); t.wse = mul_rn(t.dx, t.dy);
    const bool fin = finite_t(sx) && finite_t(sy);
    const int x1 = (int)((unsigned)t.x0 + 1u), y1 = (int)((unsigned)t.y0 + 1u);
    const bool vx0 = fin && (unsigned)t.x0 < (unsigned)W, vx1 = fin && (unsigned)x1 < (unsigned)W;
    const bool vy0 = (unsigned)t.y0 < (unsigned)H, vy1 = (unsigned)y1 < (unsigned)H;
    t.b[0] = vx0 && vy0; t.b[1] = vx1 && vy0; t.b[2] = vx0 && vy1; t.b[3] = vx1 && vy1;
    return t;
}

// K4: one thread per OUTPUT pixel, loop over channels (gather, coalesced for smooth flow).
template <class T, class TF>
__global__ void __launch_bounds__(256) k_backwarp_fwd(const WarpArgs a, const TapConst<typename Acc<T>::type> kc) {
    using A = typename Acc<T>::type;
    const unsigned p = blockIdx.x * 256 + threadIdx.x;
    if (p >= a.total) return;
    const unsigned n = p / a.HW, r = p - n * a.HW;
    const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
    const TF* fp = (const TF*)a.flow.p + n * a.flow.sN + y * a.flow.sH + x * a.flow.sW;
    const Tap<A> t = make_tap<A>(x, y, (A)ld_stream(fp), (A)ld_stream(fp + a.flow.sC), a.W, a.H, a.align, kc);

    // tap offsets inside one (n, c) plane; an out-of-range tap reads element 0 and is zeroed by its weight
    const long long o0 = (long long)t.y0 * a.image.sH + (long long)t.x0 * a.image.sW;
    const long long to[4] = {t.b[0] ? o0 : 0, t.b[1] ? o0 + a.image.sW : 0, t.b[2] ? o0 + a.image.sH : 0,
                             t.b[3] ? o0 + a.image.sH + a.image.sW : 0};
    const A tw[4] = {t.wnw, t.wne, t.wsw, t.wse};
    const T* im = (const T*)a.image.p + n * a.image.sN;
    const T* gt = a.gt.p ? (const T*)a.gt.p + n * a.gt.sN + y * a.gt.sH + x * a.gt.sW : nullptr;
    T* wp = (T*)a.warped + (long long)n * a.C * a.HW + r;
    T* rp = a.residual ? (T*)a.residual + (long long)n * a.C * a.HW + r : nullptr;
    constexpr int U = 4;                                  // channels in flight: 16 taps + 4 gt loads
    for (int c0 = 0; c0 < a.C; c0 += U) {
        A v[U][4], gv[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int c = c0 + j < a.C ? c0 + j : a.C - 1;
            const T* pl = im + (long long)c * a.image.sC;
#pragma unroll
            for (int k = 0; k < 4; ++k) v[j][k] = ld<A>(pl + to[k]);      // the image is re-read by neighbours: keep it cached
            gv[j] = gt ? (A)ld_stream(gt + (long long)c * a.gt.sC) : (A)0;
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            if (c0 + j < a.C) {
                A acc = (A)0;
#pragma unroll
                for (int k = 0; k < 4; ++k) acc = t.b[k] ? fma_rn(v[j][k], tw[k], acc) : acc;   // grid_sample's tap order and fma chain
                st_stream(wp + (long long)(c0 + j) * a.HW, acc);
                // residual of the value as stored (rounded to T), like `gt - warped` on the stored tensor
                if (rp) st_stream(rp + (long long)(c0 + j) * a.HW, sub_rn(gv[j], round_as<T>(acc)));
            }
        }
    }
}

// K4, fast path for unit-stride rows (fp32 or bf16): two consecutive output pixels per thread, paired
// loads of flow / gt and paired stores of warped / residual, 32-bit element offsets, 8-row x 64-column
// CTA tiles, one channel in flight (48 registers -> 40 warps per SM), L2 prefetch one wave ahead. The
// per-pixel arithmetic is the same sequence as above, so the results are bit-identical to the generic kernel.
#ifndef DCB_BW_MINCTAS
#define DCB_BW_MINCTAS 5
#endif
#ifndef DCB_BW_PF
#define DCB_BW_PF 1          // L2 prefetch one wave of CTAs ahead (0 = off)
#endif

struct WarpRowsArgs {
    const void *image, *flow, *gt;
    void *warped, *residual;
    int isN, isC, isH, isW;      // image strides (elements)
    int fsN, fsC, fsH;           // flow strides; sW == 1
    int gsN, gsC, gsH;           // gt strides; sW == 1
    unsigned tiles_x, pf_dist;   // CTAs per tile row; prefetch distance = resident CTAs
    unsigned pf_rows;            // ... in tile rows
    int C, H, W, HW, align;
};

__device__ __forceinline__ void ld2_stream(const float* p, float (&o)[2]) { const float2 v = __ldcs((const float2*)p); o[0] = v.x; o[1] = v.y; }
__device__ __forceinline__ void ld2_stream(const __nv_bfloat16* p, float (&o)[2]) {
    const __nv_bfloat162 v = __ldcs((const __nv_bfloat162*)p);
    o[0] = __low2float(v); o[1] = __high2float(v);
}
__device__ __forceinline__ void st2_stream(float* p, float a, float b) { __stcs((float2*)p, make_float2(a, b)); }
__device__ __forceinline__ void st2_stream(__nv_bfloat16* p, float a, float b) { __stcs((__nv_bfloat162*)p, __floats2bfloat162_rn(a, b)); }

template <class T, class TF>
__global__ void __launch_bounds__(256, DCB_BW_MINCTAS) k_backwarp_rows(const WarpRowsArgs a, const TapConst<float> kc) {
    constexpr int PX = 2;
    // a CTA covers 8 rows x 64 columns: the two image rows a warp gathers from are the rows its
    // neighbours in the CTA gather from too, so they are served by this SM's L1
    // grid = (tile columns, tile rows, frames): no integer division in front of the first load
    const unsigned tx = blockIdx.x, ty = blockIdx.y;
    const unsigned n = blockIdx.z;
    const int y = (int)(ty * 8 + (threadIdx.x >> 5));
    const int x = (int)((tx * 32 + (threadIdx.x & 31)) * PX);
#if DCB_BW_PF
    {   // L2 prefetch of the rows a CTA one wave ahead (pf_rows tile rows further down, wrapping into the next frame) will
        // stream: one line per lane
        unsigned pty = ty + a.pf_rows, pn = n;
        if (pty >= gridDim.y) { pty -= gridDim.y; ++pn; }
        if (pn < gridDim.z && pty < gridDim.y) {
            const int px0 = (int)(tx * 32 * PX), py = (int)(pty * 8 + (threadIdx.x >> 5));
            const int lane = threadIdx.x & 31;
            const int plane = lane >> 1, pxl = px0 + (lane & 1) * 32;      // two lines of 32 elements per row segment
            if (py < a.H && pxl < a.W) {
                const void* q = nullptr;
                if (plane < 2) q = (const TF*)a.flow + (int)pn * a.fsN + plane * a.fsC + py * a.fsH + pxl;
                else if (plane < 2 + a.C && a.gt) q = (const T*)a.gt + (int)pn * a.gsN + (plane - 2) * a.gsC + py * a.gsH + pxl;
                else if (plane >= 8 && plane < 8 + a.C) q = (const T*)a.image + (int)pn * a.isN + (plane - 8) * a.isC + py * a.isH + pxl * a.isW;
                if (q) asm volatile("prefetch.global.L2 [%0];" ::"l"(q));
            }
        }
    }
#endif
    if (y >= a.H || x >= a.W) return;
    const TF* fp = (const TF*)a.flow + (int)n * a.fsN + y * a.fsH + x;
    float fx[PX], fy[PX];
    ld2_stream(fp, fx); ld2_stream(fp + a.fsC, fy);
    // the gt row does not depend on the flow: put the first channel's load in flight before the taps
    const T* gt = a.gt ? (const T*)a.gt + (int)n * a.gsN + y * a.gsH + x : nullptr;
    float g[PX] = {0.f, 0.f};
    if (gt) ld2_stream(gt, g);

    int to[PX][4];
    float tw[PX][4];
    unsigned valid = 0;
#pragma unroll
    for (int j = 0; j < PX; ++j) {
        const Tap<float> t = make_tap<float>(x + j, y, fx[j], fy[j], a.W, a.H, a.align, kc);
        const int o0 = t.y0 * a.isH + t.x0 * a.isW;        // only used when the tap is valid
        to[j][0] = t.b[0] ? o0 : 0;
        to[j][1] = t.b[1] ? o0 + a.isW : 0;
        to[j][2] = t.b[2] ? o0 + a.isH : 0;
        to[j][3] = t.b[3] ? o0 + a.isH + a.isW : 0;
        tw[j][0] = t.wnw; tw[j][1] = t.wne; tw[j][2] = t.wsw; tw[j][3] = t.wse;
#pragma unroll
        for (int k = 0; k < 4; ++k) valid |= (t.b[k] ? 1u : 0u) << (j * 4 + k);
    }
    const T* im = (const T*)a.image + (int)n * a.isN;
    const int oo = ((int)n * a.C) * a.HW + y * a.W + x;
    T* wp = (T*)a.warped + oo;
    T* rp = a.residual ? (T*)a.residual + oo : nullptr;
    for (int c = 0; c < a.C; ++c, im += a.isC, wp += a.HW) {
        float v[PX][4];
#pragma unroll
        for (int j = 0; j < PX; ++j)
#pragma unroll
            for (int k = 0; k < 4; ++k) v[j][k] = ld<float>(im + to[j][k]);      // the image is re-read by neighbours: keep it cached
        if (c > 0 && gt) ld2_stream(gt + c * a.gsC, g);
        float acc[PX];
#pragma unroll
        for (int j = 0; j < PX; ++j) {
            acc[j] = 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                acc[j] = (valid >> (j * 4 + k)) & 1u ? fma_rn(v[j][k], tw[j][k], acc[j]) : acc[j];   // grid_sample's tap order and fma chain
        }
        st2_stream(wp, acc[0], acc[1]);
        if (rp) {
            // residual of the value as stored (rounded to T), like `gt - warped` on the stored tensor
            st2_stream(rp, sub_rn(g[0], round_as<T>(acc[0])), sub_rn(g[1], round_as<T>(acc[1])));
            rp += a.HW;
        }
    }
}

// K4b: gradImage by scatter (reds into the zeroed planar buffer), gradFlow by gather.
template <class T, class TF>
__global__ void __launch_bounds__(256) k_backwarp_bwd(const WarpArgs a, const TapConst<typename Acc<T>::type> kc,
                                                      typename Acc<T>::type* gimage_acc) {
    using A = typename Acc<T>::type;
    const unsigned p = blockIdx.x * 256 + threadIdx.x;
    if (p >= a.total) return;
    const unsigned n = p / a.HW, r = p - n * a.HW;
    const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
    const TF* fp = (const TF*)a.flow.p + n * a.flow.sN + y * a.flow.sH + x * a.flow.sW;
    const Tap<A> t = make_tap<A>(x, y, ld<A>(fp), ld<A>(fp + a.flow.sC), a.W, a.H, a.align, kc);

    const T* im = (const T*)a.image.p + n * a.image.sN + (long long)t.y0 * a.image.sH + (long long)t.x0 * a.image.sW;
    const long long o1 = a.image.sW, o2 = a.image.sH, o3 = a.image.sH + a.image.sW;
    const T* gp = (const T*)a.gout.p + n * a.gout.sN + y * a.gout.sH + x * a.gout.sW;
    A* gi = gimage_acc ? gimage_acc + (long long)n * a.C * a.HW + (long long)t.y0 * a.W + t.x0 : nullptr;
    A gx = (A)0, gy = (A)0;
    for (int c = 0; c < a.C; ++c, im += a.image.sC) {
        const A g = ld<A>(gp + c * a.gout.sC);
        if (gi) {
            A* q = gi + (long long)c * a.HW;
            if (t.b[0]) red_add(q, mul_rn(g, t.wnw));
            if (t.b[1]) red_add(q + 1, mul_rn(g, t.wne));
            if (t.b[2]) red_add(q + a.W, mul_rn(g, t.wsw));
            if (t.b[3]) red_add(q + a.W + 1, mul_rn(g, t.wse));
        }
        if (a.gflow) {
            const A vnw = t.b[0] ? ld<A>(im) : (A)0, vne = t.b[1] ? ld<A>(im + o1) : (A)0;
            const A vsw = t.b[2] ? ld<A>(im + o2) : (A)0, vse = t.b[3] ? ld<A>(im + o3) : (A)0;
            gx += g * ((vne - vnw) * t.ey + (vse - vsw) * t.dy);
            gy += g * ((vsw - vnw) * t.ex + (vse - vne) * t.dx);
        }
    }
    if (a.gflow) {
        // chain through the un-normalisation (W/2 or (W-1)/2) and warp.py:11-12 (1 / ((W-1)/2))
        const A kx = a.align ? (A)1 : (A)a.W / (A)(a.W - 1);
        const A ky = a.align ? (A)1 : (A)a.H / (A)(a.H - 1);
        TF* gf = (TF*)a.gflow + (long long)n * 2 * a.HW + r;
        st<TF, A>(gf, gx * kx);
        st<TF, A>(gf + a.HW, gy * ky);
    }
}

// cast an accumulator-typed planar buffer to T (only needed for bf16 gradImage)
__global__ void __launch_bounds__(256) k_cast_f32_bf16(const float* src, __nv_bfloat16* dst, long long n) {
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    if (i < n) dst[i] = __float2bfloat16_rn(src[i]);
}

static void fill(WarpArgs& a, const DcbTensor* image) {
    a.N = (int)image->size[0]; a.C = (int)image->size[1]; a.H = (int)image->size[2]; a.W = (int)image->size[3];
    a.HW = (unsigned)(image->size[2] * image->size[3]);
    a.total = (unsigned)(image->size[0] * image->size[2] * image->size[3]);
}

template <class T, class TF> static int launch_warp_fwd(const WarpArgs& a, cudaStream_t st) {
    k_backwarp_fwd<T, TF><<<(a.total + 255) / 256, 256, 0, st>>>(a, make_tap_const<typename Acc<T>::type>(a.W, a.H));
    DCB_CHECK_LAUNCH("k_backwarp_fwd");
    return DCB_OK;
}

// largest element offset a [N,C,H,W] view can address, or -1 when it does not fit 31 bits
static long long max_offset31(const DcbTensor* t) {
    long long m = 0;
    for (int d = 0; d < 4; ++d) {
        if (t->size[d] == 0) return 0;
        const long long s = t->stride[d];
        if (s < 0) return -1;
        m += (t->size[d] - 1) * s;
    }
    return m < (1ll << 31) ? m : -1;
}

static bool rows_vec(const DcbTensor* t) {      // paired loads along x are legal
    const int es = elem_size(t->dtype);
    return t->dtype != DCB_F64 && t->stride[3] == 1 && t->stride[0] % 2 == 0 && t->stride[1] % 2 == 0 &&
           t->stride[2] % 2 == 0 && ((uintptr_t)t->ptr & (uintptr_t)(2 * es - 1)) == 0 && max_offset31(t) >= 0;
}

static bool rows_supported(const DcbTensor* image, const DcbTensor* flow, const DcbTensor* gt, const DcbTensor* warped,
                           const DcbTensor* residual) {
    if (image->size[0] > 65535 || image->dtype == DCB_F64 || image->size[3] % 2 != 0 || max_offset31(image) < 0) return false;
    if (image->size[0] * image->size[1] * image->size[2] * image->size[3] >= (1ll << 31)) return false;
    if (image->size[0] > 65535 || (image->size[2] + 7) / 8 > 65535) return false;      // frames on gridDim.z, tile rows on gridDim.y
    if (!rows_vec(flow) || (gt && (!rows_vec(gt) || gt->dtype != image->dtype))) return false;
    if (flow->dtype != image->dtype && !(image->dtype == DCB_BF16 && flow->dtype == DCB_F32)) return false;
    const uintptr_t m = (uintptr_t)(2 * elem_size(image->dtype) - 1);
    if (((uintptr_t)warped->ptr & m) || (residual && ((uintptr_t)residual->ptr & m))) return false;
    return true;
}

static int launch_warp_rows(const DcbTensor* image, const DcbTensor* flow, const DcbTensor* gt, const DcbTensor* warped,
                            const DcbTensor* residual, int align, cudaStream_t st) {
    WarpRowsArgs a{};
    a.image = image->ptr; a.flow = flow->ptr; a.gt = gt ? gt->ptr : nullptr;
    a.warped = warped->ptr; a.residual = residual ? residual->ptr : nullptr;
    a.isN = (int)image->stride[0]; a.isC = (int)image->stride[1]; a.isH = (int)image->stride[2]; a.isW = (int)image->stride[3];
    a.fsN = (int)flow->stride[0]; a.fsC = (int)flow->stride[1]; a.fsH = (int)flow->stride[2];
    if (gt) { a.gsN = (int)gt->stride[0]; a.gsC = (int)gt->stride[1]; a.gsH = (int)gt->stride[2]; }
    a.C = (int)image->size[1]; a.H = (int)image->size[2]; a.W = (int)image->size[3];
    a.HW = a.H * a.W; a.align = align;
    a.tiles_x = (unsigned)(a.W / 2 + 31) / 32;
    a.pf_dist = (unsigned)(device_sm_count() * DCB_BW_MINCTAS);
    a.pf_rows = a.pf_dist / a.tiles_x > 0 ? a.pf_dist / a.tiles_x : 1;
    const dim3 grid(a.tiles_x, (unsigned)((a.H + 7) / 8), (unsigned)image->size[0]);
    const TapConst<float> kc = make_tap_const<float>(a.W, a.H);
    if (image->dtype == DCB_F32) k_backwarp_rows<float, float><<<grid, 256, 0, st>>>(a, kc);
    else if (flow->dtype == DCB_F32) k_backwarp_rows<__nv_bfloat16, float><<<grid, 256, 0, st>>>(a, kc);
    else k_backwarp_rows<__nv_bfloat16, __nv_bfloat16><<<grid, 256, 0, st>>>(a, kc);
    DCB_CHECK_LAUNCH("k_backwarp_rows");
    return DCB_OK;
}

int backwarp_fwd_impl(const DcbTensor* image, const DcbTensor* flow, const DcbTensor* gt, const DcbTensor* warped,
                      const DcbTensor* residual, int align, cudaStream_t st) {
    WarpArgs a{};
    a.image = make_view(image); a.flow = make_view(flow); a.gt = make_view(gt);
    a.warped = warped->ptr; a.residual = residual ? residual->ptr : nullptr;
    a.align = align;
    fill(a, image);
    // no fp16 kernels here: every dispatch below reads a 16-bit tensor as bf16
    if (image->dtype == DCB_F16 || flow->dtype == DCB_F16) return set_error(DCB_E_DTYPE, "backwarp_fwd: F16 is not supported");
    if (a.total == 0 || a.C == 0) return DCB_OK;
    if (rows_supported(image, flow, gt, warped, residual)) return launch_warp_rows(image, flow, gt, warped, residual, align, st);
    const bool ff = flow->dtype == DCB_F32;
    switch (image->dtype) {
        case DCB_F32: return launch_warp_fwd<float, float>(a, st);
        case DCB_F64: return launch_warp_fwd<double, double>(a, st);
        case DCB_BF16: return ff ? launch_warp_fwd<__nv_bfloat16, float>(a, st) : launch_warp_fwd<__nv_bfloat16, __nv_bfloat16>(a, st);
    }
    return set_error(DCB_E_DTYPE, "backwarp_fwd: unsupported dtype %d", image->dtype);
}

template <class T, class TF> static int launch_warp_bwd(const WarpArgs& a, void* acc, cudaStream_t st) {
    using A = typename Acc<T>::type;
    k_backwarp_bwd<T, TF><<<(a.total + 255) / 256, 256, 0, st>>>(a, make_tap_const<A>(a.W, a.H), (A*)acc);
    DCB_CHECK_LAUNCH("k_backwarp_bwd");
    return DCB_OK;
}

long long backwarp_bwd_workspace(long long N, long long C, long long H, long long W, int dtype) {
    return dtype == DCB_BF16 ? align_up(N * C * H * W * 4, 256) : 0;
}

int backwarp_bwd_impl(const DcbTensor* gout, const DcbTensor* image, const DcbTensor* flow, const DcbTensor* gimage,
                      const DcbTensor* gflow, int align, void* ws, long long ws_bytes, cudaStream_t st) {
    WarpArgs a{};
    a.image = make_view(image); a.flow = make_view(flow); a.gout = make_view(gout);
    a.gimage = gimage ? gimage->ptr : nullptr;
    a.gflow = gflow ? gflow->ptr : nullptr;
    a.align = align;
    fill(a, image);
    if (image->dtype == DCB_F16 || flow->dtype == DCB_F16) return set_error(DCB_E_DTYPE, "backwarp_bwd: F16 is not supported");
    if (a.total == 0 || a.C == 0 || (!a.gimage && !a.gflow)) return DCB_OK;
    const long long nelem = (long long)a.total * a.C;
    void* acc = a.gimage;
    if (a.gimage) {
        if (image->dtype == DCB_BF16) {
            const long long need = backwarp_bwd_workspace(a.N, a.C, a.H, a.W, DCB_BF16);
            if (!ws || ws_bytes < need || ((uintptr_t)ws & 255))
                return set_error(DCB_E_WORKSPACE, "backwarp_bwd: workspace of %lld bytes required, got %lld", need, ws_bytes);
            acc = ws;
        }
        DCB_CHECK_CUDA(cudaMemsetAsync(acc, 0, (size_t)nelem * (image->dtype == DCB_F64 ? 8 : 4), st));
    }
    const bool ff = flow->dtype == DCB_F32;
    int rc;
    switch (image->dtype) {
        case DCB_F32: rc = launch_warp_bwd<float, float>(a, acc, st); break;
        case DCB_F64: rc = launch_warp_bwd<double, double>(a, acc, st); break;
        case DCB_BF16:
            rc = ff ? launch_warp_bwd<__nv_bfloat16, float>(a, acc, st) : launch_warp_bwd<__nv_bfloat16, __nv_bfloat16>(a, acc, st);
            break;
        default: return set_error(DCB_E_DTYPE, "backwarp_bwd: unsupported dtype %d", image->dtype);
    }
    if (rc != DCB_OK) return rc;
    if (a.gimage && image->dtype == DCB_BF16) {
        k_cast_f32_bf16<<<(unsigned)((nelem + 255) / 256), 256, 0, st>>>((const float*)acc, (__nv_bfloat16*)a.gimage, nelem);
        DCB_CHECK_LAUNCH("k_cast_f32_bf16");
    }
    return DCB_OK;
}

}  // namespace dcb
