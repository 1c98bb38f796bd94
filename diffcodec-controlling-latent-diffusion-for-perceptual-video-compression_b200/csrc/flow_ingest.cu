// flow_ingest.cu -- the step immediately before the hot path (SURVEY.md section 8, row f-2), on the device (sm_100a).
//
// The reference prepares its flows on the host and with eager torch ops:
//   * Middlebury .flo payload (h * w * 2 float32, (u, v) INTERLEAVED per pixel) -> controlnet/utils.py:10-19; the dataset
//     reader reshapes the same payload as planar (2, h, w) with np.resize (controlnet/dataset.py:15-24, SURVEY.md App. B-9);
//   * resize_flow_to: bilinear, align_corners=True, vectors rescaled by (tw / W, th / H) -> controlnet/utils.py:21-28;
//   * fast_downsample_flow: adaptive average pooling, vectors NOT rescaled               -> controlnet/dataset.py:43-50;
//   * resize_and_normalize_flow_batched: bilinear, align_corners=False, then u /= (tw-1)/2, v /= (th-1)/2
//                                                                                         -> controlnet/control_utils.py:74-97.
// Here the raw payload is uploaded as it is and ONE kernel reads it through a strided view (interleaved or the planar
// quirk: only the strides differ), resamples and writes the planar [N,2,th,tw] tensor the splat kernels take. The index
// and weight arithmetic restates what torch's upsample_bilinear2d / adaptive_avg_pool2d compute (fp32, same operation
// order), so the results agree with the reference's callees to rounding.
#include "dcb_common.cuh"

namespace dcb {

struct IngestArgs {
    View flow;            // [N,2,H,W] any strides (elements)
    void* out;            // [N,2,th,tw] contiguous
    int N, H, W, th, tw;
    int mode;             // DCB_FLOW_*
    float sx, sy;         // bilinear source-index scales (torch: area_pixel_compute_scale)
    float mu, mv;         // post factors: u * mu, v * mv  (BILINEAR_RESCALE) ; u / mu, v / mv (BILINEAR_NORMALIZE)
};

__device__ __forceinline__ float src_index(float scale, int dst, bool align) {
    if (align) return mul_rn(scale, (float)dst);
    const float s = sub_rn(mul_rn(scale, add_rn((float)dst, 0.5f)), 0.5f);          // torch: scale * (dst + 0.5) - 0.5, clamped at 0
    return s < 0.f ? 0.f : s;
}

template <class T, class TO>
__global__ void __launch_bounds__(256) k_flow_ingest(const IngestArgs a) {
    pdl_wait();
    const long long total = (long long)a.N * a.th * a.tw;
    const long long p = (long long)blockIdx.x * 256 + threadIdx.x;
    if (p >= total) return;
    const int x = (int)(p % a.tw), y = (int)((p / a.tw) % a.th), n = (int)(p / ((long long)a.tw * a.th));
    const T* base = (const T*)a.flow.p + (long long)n * a.flow.sN;
    float r[2];
    if (a.mode == DCB_FLOW_ADAPTIVE_AVG) {
        // torch adaptive_avg_pool2d: window [floor(o * in / out), ceil((o + 1) * in / out)), sum in fp32, divided by the count
        const int y0 = (int)(((long long)y * a.H) / a.th), y1 = (int)((((long long)y + 1) * a.H + a.th - 1) / a.th);
        const int x0 = (int)(((long long)x * a.W) / a.tw), x1 = (int)((((long long)x + 1) * a.W + a.tw - 1) / a.tw);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            float sum = 0.f;
            for (int yy = y0; yy < y1; ++yy)
                for (int xx = x0; xx < x1; ++xx)
                    sum = add_rn(sum, ld<float>(base + c * a.flow.sC + (long long)yy * a.flow.sH + (long long)xx * a.flow.sW));
            r[c] = sum / (float)((y1 - y0) * (x1 - x0));
        }
    } else {
        const bool align = a.mode == DCB_FLOW_BILINEAR_RESCALE;
        const float fy = src_index(a.sy, y, align), fx = src_index(a.sx, x, align);
        const int iy = (int)fy, ix = (int)fx;
        const int py = iy < a.H - 1 ? 1 : 0, px = ix < a.W - 1 ? 1 : 0;
        const float ly1 = sub_rn(fy, (float)iy), ly0 = sub_rn(1.f, ly1), lx1 = sub_rn(fx, (float)ix), lx0 = sub_rn(1.f, lx1);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            const T* q = base + c * a.flow.sC + (long long)iy * a.flow.sH + (long long)ix * a.flow.sW;
            const float v00 = ld<float>(q), v01 = ld<float>(q + px * a.flow.sW);
            const float v10 = ld<float>(q + py * a.flow.sH), v11 = ld<float>(q + py * a.flow.sH + px * a.flow.sW);
            // torch: h0lambda * (w0lambda * v00 + w1lambda * v01) + h1lambda * (w0lambda * v10 + w1lambda * v11)
            const float top = add_rn(mul_rn(lx0, v00), mul_rn(lx1, v01)), bot = add_rn(mul_rn(lx0, v10), mul_rn(lx1, v11));
            r[c] = add_rn(mul_rn(ly0, top), mul_rn(ly1, bot));
        }
        if (a.mode == DCB_FLOW_BILINEAR_RESCALE) { r[0] = mul_rn(r[0], a.mu); r[1] = mul_rn(r[1], a.mv); }
        else { r[0] = r[0] / a.mu; r[1] = r[1] / a.mv; }
    }
    TO* o = (TO*)a.out + ((long long)n * 2 * a.th + y) * a.tw + x;
    st<TO, float>(o, r[0]);
    st<TO, float>(o + (long long)a.th * a.tw, r[1]);
}

template <class T, class TO> static int launch_ingest(const IngestArgs& a, cudaStream_t st) {
    const long long total = (long long)a.N * a.th * a.tw;
    DCB_CHECK_CUDA(launch_pdl(k_flow_ingest<T, TO>, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, a));
    count_launch();
    return DCB_OK;
}

int flow_ingest_impl(const DcbTensor* flow, const DcbTensor* out, int mode, cudaStream_t st) {
    IngestArgs a;
    a.flow = make_view(flow);
    a.out = out->ptr;
    a.N = (int)flow->size[0]; a.H = (int)flow->size[2]; a.W = (int)flow->size[3];
    a.th = (int)out->size[2]; a.tw = (int)out->size[3];
    a.mode = mode;
    if ((long long)a.N * a.th * a.tw == 0) return DCB_OK;
    const bool align = mode == DCB_FLOW_BILINEAR_RESCALE;
    // torch area_pixel_compute_scale<float>
    a.sy = align ? (a.th > 1 ? (float)(a.H - 1) / (float)(a.th - 1) : 0.f) : (float)a.H / (float)a.th;
    a.sx = align ? (a.tw > 1 ? (float)(a.W - 1) / (float)(a.tw - 1) : 0.f) : (float)a.W / (float)a.tw;
    if (mode == DCB_FLOW_BILINEAR_RESCALE) {            // utils.py:26-27: ft[:, 0] *= target_w / max(W, 1)
        a.mu = (float)((double)a.tw / (double)(a.W > 1 ? a.W : 1)); a.mv = (float)((double)a.th / (double)(a.H > 1 ? a.H : 1));
    } else {                                            // control_utils.py:90-95: u / ((w - 1) / 2.0)
        a.mu = (float)((double)(a.tw - 1) / 2.0); a.mv = (float)((double)(a.th - 1) / 2.0);
    }
    if (out->dtype != DCB_F32 && out->dtype != DCB_BF16) return set_error(DCB_E_DTYPE, "flow_resize: out must be F32 or BF16, got %d", out->dtype);
    const bool of32 = out->dtype == DCB_F32;
    if (flow->dtype == DCB_F32) return of32 ? launch_ingest<float, float>(a, st) : launch_ingest<float, __nv_bfloat16>(a, st);
    if (flow->dtype == DCB_BF16) return of32 ? launch_ingest<__nv_bfloat16, float>(a, st) : launch_ingest<__nv_bfloat16, __nv_bfloat16>(a, st);
    return set_error(DCB_E_DTYPE, "flow_resize: F32 or BF16 flows only, got %d", flow->dtype);
}

}  // namespace dcb
