// fuse.cu -- confidence fusion of the two warped feature maps of a bi-directional block (f-1), sm_100a.
//
// Replaces controlnet/extractors.py:298-310 (and :193-205; residual_utils.py:181-193): cat, clamp,
// sum, add-eps, divide, two products, add, the `holes` compare, a DEVICE->HOST SYNC (`holes.any()`,
// extractors.py:308) and a `where` -- 10 eager kernels and one stall per scale -- by one
// elementwise kernel (and one for its backward into both feature maps and both confidences).
#include "dcb_common.cuh"

namespace dcb {

struct FuseBArgs {
    View A, B, ca, cb, oa, ob, g;
    void* fused;                      // [N,C,H,W]
    void *gA, *gB, *gca, *gcb;        // backward outputs (any may be null)
    unsigned total, HW;
    int C, W;
};

template <class T> struct FuseW { float w0, w1, ca, cb, s; bool hole; };

template <class T>
__device__ __forceinline__ FuseW<T> fuse_weights(const FuseBArgs& a, unsigned n, int y, int x) {
    FuseW<T> f;
    const float ra = ld<float>((const T*)a.ca.p + n * a.ca.sN + (long long)y * a.ca.sH + (long long)x * a.ca.sW);
    const float rb = ld<float>((const T*)a.cb.p + n * a.cb.sN + (long long)y * a.cb.sH + (long long)x * a.cb.sW);
    f.ca = fmaxf(ra, 0.f); f.cb = fmaxf(rb, 0.f);                       // torch.clamp(conf, min=0)
    f.s = add_rn(add_rn(f.ca, f.cb), 0.000001f);                        // conf.sum(1) + 1e-6
    f.w0 = f.ca / f.s; f.w1 = f.cb / f.s;
    f.hole = false;
    if (a.oa.p) {
        const float oa = ld<float>((const T*)a.oa.p + n * a.oa.sN + (long long)y * a.oa.sH + (long long)x * a.oa.sW);
        const float ob = ld<float>((const T*)a.ob.p + n * a.ob.sN + (long long)y * a.ob.sH + (long long)x * a.ob.sW);
        f.hole = add_rn(oa, ob) > 1.5f;                                 // both occluded
    }
    return f;
}

// Thread layout (both kernels): blockDim = (PX, CS): PX pixels, CS channel slices per pixel. CS > 1 when
// there are too few pixels to fill the machine (8x8 .. 64x64 pyramid levels with hundreds of channels: one
// thread per pixel would walk 1280 channels one dependent round trip at a time). Four channels in flight.
constexpr int kFU = 4;

template <class T>
__global__ void __launch_bounds__(256) k_bidir_fuse_fwd(const FuseBArgs a) {
    const int tx = threadIdx.x, ty = threadIdx.y, cs = blockDim.y;
    const unsigned p = blockIdx.x * blockDim.x + tx;
    if (p >= a.total) return;
    const unsigned n = p / a.HW, r = p - n * a.HW;
    const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
    const FuseW<T> f = fuse_weights<T>(a, n, y, x);
    const T* pa = (const T*)a.A.p + n * a.A.sN + (long long)y * a.A.sH + (long long)x * a.A.sW;
    const T* pb = (const T*)a.B.p + n * a.B.sN + (long long)y * a.B.sH + (long long)x * a.B.sW;
    T* po = (T*)a.fused + (long long)n * a.C * a.HW + r;
    for (int c0 = ty; c0 < a.C; c0 += kFU * cs) {
        float va[kFU], vb[kFU];
#pragma unroll
        for (int j = 0; j < kFU; ++j) {
            const int c = c0 + j * cs;
            const bool in = c < a.C;
            va[j] = in ? ld_stream(pa + (long long)c * a.A.sC) : 0.f;
            vb[j] = in ? ld_stream(pb + (long long)c * a.B.sC) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < kFU; ++j) {
            const int c = c0 + j * cs;
            if (c < a.C) {
                const float v = f.hole ? mul_rn(0.5f, add_rn(va[j], vb[j])) : add_rn(mul_rn(f.w0, va[j]), mul_rn(f.w1, vb[j]));
                st_stream(po + (long long)c * a.HW, v);
            }
        }
    }
}

template <class T>
__global__ void __launch_bounds__(256) k_bidir_fuse_bwd(const FuseBArgs a) {
    extern __shared__ float red[];                                         // [cs][px][2] when cs > 1
    const int tx = threadIdx.x, ty = threadIdx.y, cs = blockDim.y, px = blockDim.x;
    const unsigned p = blockIdx.x * px + tx;
    const bool live = p < a.total;
    const unsigned pc = live ? p : 0;
    const unsigned n = pc / a.HW, r = pc - n * a.HW;
    const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
    const FuseW<T> f = fuse_weights<T>(a, n, y, x);
    const T* pa = (const T*)a.A.p + n * a.A.sN + (long long)y * a.A.sH + (long long)x * a.A.sW;
    const T* pb = (const T*)a.B.p + n * a.B.sN + (long long)y * a.B.sH + (long long)x * a.B.sW;
    const T* pg = (const T*)a.g.p + n * a.g.sN + (long long)y * a.g.sH + (long long)x * a.g.sW;
    T* ga = (a.gA && live) ? (T*)a.gA + (long long)n * a.C * a.HW + r : nullptr;
    T* gb = (a.gB && live) ? (T*)a.gB + (long long)n * a.C * a.HW + r : nullptr;
    const float k0 = f.hole ? 0.5f : f.w0, k1 = f.hole ? 0.5f : f.w1;
    const bool need_w = a.gca || a.gcb;
    float gw0 = 0.f, gw1 = 0.f;
    for (int c0 = ty; c0 < a.C; c0 += kFU * cs) {
        float g[kFU], va[kFU], vb[kFU];
#pragma unroll
        for (int j = 0; j < kFU; ++j) {
            const int c = c0 + j * cs;
            const bool in = c < a.C;
            g[j] = in ? ld_stream(pg + (long long)c * a.g.sC) : 0.f;
            va[j] = (in && need_w) ? ld_stream(pa + (long long)c * a.A.sC) : 0.f;
            vb[j] = (in && need_w) ? ld_stream(pb + (long long)c * a.B.sC) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < kFU; ++j) {
            const int c = c0 + j * cs;
            if (c < a.C) {
                if (ga) st_stream(ga + (long long)c * a.HW, g[j] * k0);
                if (gb) st_stream(gb + (long long)c * a.HW, g[j] * k1);
            }
            gw0 = fmaf(g[j], va[j], gw0);
            gw1 = fmaf(g[j], vb[j], gw1);
        }
    }
    if (!need_w) return;
    if (cs > 1) {                                                           // reduce the two dot products over the channel slices
        float* mine = red + ((size_t)ty * px + tx) * 2;
        mine[0] = gw0; mine[1] = gw1;
        __syncthreads();
        if (ty != 0) return;
        for (int s = 1; s < cs; ++s) { gw0 += red[((size_t)s * px + tx) * 2]; gw1 += red[((size_t)s * px + tx) * 2 + 1]; }
    }
    if (!live) return;
    if (f.hole) { gw0 = 0.f; gw1 = 0.f; }                                   // the `where` routes the gradient to the average
    const float is = 1.f / f.s, is2 = is * is;
    const float dca = gw0 * (is - f.ca * is2) - gw1 * f.cb * is2;
    const float dcb = gw1 * (is - f.cb * is2) - gw0 * f.ca * is2;
    // clamp(min=0) passes the gradient where the input is >= 0
    const float ra = ld<float>((const T*)a.ca.p + n * a.ca.sN + (long long)y * a.ca.sH + (long long)x * a.ca.sW);
    const float rb = ld<float>((const T*)a.cb.p + n * a.cb.sN + (long long)y * a.cb.sH + (long long)x * a.cb.sW);
    if (a.gca) st<T, float>((T*)a.gca + p, ra >= 0.f ? dca : 0.f);
    if (a.gcb) st<T, float>((T*)a.gcb + p, rb >= 0.f ? dcb : 0.f);
}

// channel slices per pixel: fill ~148 SMs x 2048 threads when pixels are scarce
static int channel_slices(unsigned total, int C) {
    int cs = 1;
    while (cs < 32 && cs * 2 * kFU <= C && (long long)total * cs < 148LL * 2048) cs *= 2;
    return cs;
}

static void fill(FuseBArgs& a, const DcbTensor* A) {
    a.C = (int)A->size[1]; a.W = (int)A->size[3];
    a.HW = (unsigned)(A->size[2] * A->size[3]);
    a.total = (unsigned)(A->size[0] * A->size[2] * A->size[3]);
}

int bidir_fuse_fwd_impl(const DcbTensor* A, const DcbTensor* B, const DcbTensor* ca, const DcbTensor* cb,
                        const DcbTensor* oa, const DcbTensor* ob, const DcbTensor* fused, cudaStream_t st) {
    FuseBArgs a{};
    a.A = make_view(A); a.B = make_view(B); a.ca = make_view(ca); a.cb = make_view(cb); a.oa = make_view(oa); a.ob = make_view(ob);
    a.fused = fused->ptr;
    fill(a, A);
    if (a.total == 0 || a.C == 0) return DCB_OK;
    const int cs = channel_slices(a.total, a.C), px = 256 / cs;
    const dim3 block(px, cs);
    const unsigned blocks = (a.total + px - 1) / px;
    if (A->dtype == DCB_F32) k_bidir_fuse_fwd<float><<<blocks, block, 0, st>>>(a);
    else if (A->dtype == DCB_BF16) k_bidir_fuse_fwd<__nv_bfloat16><<<blocks, block, 0, st>>>(a);
    else if (A->dtype == DCB_F16) k_bidir_fuse_fwd<__half><<<blocks, block, 0, st>>>(a);
    else return set_error(DCB_E_DTYPE, "bidir_fuse: F32, BF16 or F16 only, got %d", A->dtype);
    DCB_CHECK_LAUNCH("k_bidir_fuse_fwd");
    return DCB_OK;
}

int bidir_fuse_bwd_impl(const DcbTensor* g, const DcbTensor* A, const DcbTensor* B, const DcbTensor* ca, const DcbTensor* cb,
                        const DcbTensor* oa, const DcbTensor* ob, const DcbTensor* gA, const DcbTensor* gB,
                        const DcbTensor* gca, const DcbTensor* gcb, cudaStream_t st) {
    FuseBArgs a{};
    a.A = make_view(A); a.B = make_view(B); a.ca = make_view(ca); a.cb = make_view(cb); a.oa = make_view(oa); a.ob = make_view(ob);
    a.g = make_view(g);
    a.gA = gA ? gA->ptr : nullptr; a.gB = gB ? gB->ptr : nullptr;
    a.gca = gca ? gca->ptr : nullptr; a.gcb = gcb ? gcb->ptr : nullptr;
    fill(a, A);
    if (a.total == 0) return DCB_OK;
    const int cs = channel_slices(a.total, a.C), px = 256 / cs;
    const dim3 block(px, cs);
    const unsigned blocks = (a.total + px - 1) / px;
    const size_t smem = cs > 1 ? (size_t)256 * 2 * sizeof(float) : 0;
    if (A->dtype == DCB_F32) k_bidir_fuse_bwd<float><<<blocks, block, smem, st>>>(a);
    else if (A->dtype == DCB_BF16) k_bidir_fuse_bwd<__nv_bfloat16><<<blocks, block, smem, st>>>(a);
    else if (A->dtype == DCB_F16) k_bidir_fuse_bwd<__half><<<blocks, block, smem, st>>>(a);
    else return set_error(DCB_E_DTYPE, "bidir_fuse: F32, BF16 or F16 only, got %d", A->dtype);
    DCB_CHECK_LAUNCH("k_bidir_fuse_bwd");
    return DCB_OK;
}

}  // namespace dcb
