// tile_merge.cu -- Hann-window merge of overlapping latent tiles (K8), sm_100a.
//
// Replaces merge_latent_tiles_from_pixel_coords(), patch_utils.py:83-174: the reference maps every
// tile's pixel rectangle to a latent rectangle, optionally resizes the tile to it (bilinear,
// align_corners=False), builds a 2-d Hann mask, and runs `out[rect] += tile * mask;
// weight[rect] += mask` tile after tile (6-8 eager kernels and three temporaries per tile, on two
// canvas-sized accumulators), then divides. Here ONE gather kernel: a thread owns an output pixel,
// walks the tiles in list order (so the fp32 additions happen in the reference's order), forms the
// mask value and the (possibly resampled) tile value in registers and writes the normalised result
// once. No atomics, no accumulators, no temporaries; up to 48 tiles per launch travel as kernel
// parameters (a 1080p frame in 512^2 tiles with 64 px overlap is 15), longer lists are chained
// through an fp32 canvas in the caller's workspace.
#include "dcb_common.cuh"

#include <math.h>

namespace dcb {

constexpr int kMaxTiles = 48;
constexpr int kCB = 4;                 // channels per pass

struct TileDesc {
    const void* p;                     // [1,C,th,tw], any strides
    long long sC, sH, sW;
    int th, tw;                        // stored size
    int y0, x0, h, w;                  // latent rectangle (clamped; h, w > 0)
    float ky, kx;                      // Hann phase step 2*pi / (n - 1) (0 for n == 1)
    float denom;                       // max of the window product + 1e-12  (patch_utils.py:131)
    float ry, rx;                      // resize scale th / h, tw / w (1 when no resize)
    int resize;
};

struct MergeArgs {
    TileDesc t[kMaxTiles];
    int n;
    void* out;                         // [N,C,H,W] contiguous
    float* canvas;                     // [(C+1),H,W] fp32 partial sums of earlier launches, or null
    int N, C, H, W;
    unsigned HW;
    float eps;
    int first, last;
};

// torch.hann_window(n, periodic=False): 0.5 - 0.5 * cos(i * 2*pi/(n-1)); ones for n <= 1 (patch_utils.py:122-129)
__device__ __forceinline__ float hann(int i, int n, float k) {
    return n <= 1 ? 1.f : add_rn(mul_rn(cosf(mul_rn((float)i, k)), -0.5f), 0.5f);
}

// torch upsample_bilinear2d, align_corners=False: source index and the two taps of one axis
__device__ __forceinline__ void bilinear_axis(int dst, float scale, int in_size, int& i0, int& step, float& l1) {
    float s = fmaf(scale, (float)dst + 0.5f, -0.5f);
    s = s < 0.f ? 0.f : s;
    i0 = (int)s;
    if (i0 > in_size - 1) i0 = in_size - 1;
    step = i0 < in_size - 1 ? 1 : 0;
    l1 = s - (float)i0;
}

template <class T>
__global__ void __launch_bounds__(256) k_tile_merge(const __grid_constant__ MergeArgs a) {
    const unsigned r = blockIdx.x * 256 + threadIdx.x;
    // which tiles touch this CTA's 256 pixels at all? two ballots, kept as bit masks so that the
    // tiles are still visited in list order (typically 1-4 of them instead of all 15-48)
    __shared__ unsigned live_mask[2];
    if (threadIdx.x < 64) {
        const unsigned r0 = blockIdx.x * 256, r1 = min(r0 + 255u, a.HW - 1);
        const int ya = (int)(r0 / (unsigned)a.W), yb = (int)(r1 / (unsigned)a.W);
        const int xa = ya == yb ? (int)(r0 - (unsigned)ya * (unsigned)a.W) : 0;
        const int xb = ya == yb ? (int)(r1 - (unsigned)ya * (unsigned)a.W) : a.W - 1;
        const int i = threadIdx.x;
        bool hit = false;
        if (i < a.n) {
            const TileDesc& t = a.t[i];
            hit = t.y0 <= yb && t.y0 + t.h > ya && t.x0 <= xb && t.x0 + t.w > xa;
        }
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if ((threadIdx.x & 31) == 0) live_mask[threadIdx.x >> 5] = m;
    }
    __syncthreads();
    if (r >= a.HW) return;
    const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
    float wsum = 0.f;
    for (int c0 = 0; c0 < a.C; c0 += kCB) {
        float acc[kCB];
#pragma unroll
        for (int j = 0; j < kCB; ++j) acc[j] = 0.f;
        if (!a.first) {
#pragma unroll
            for (int j = 0; j < kCB; ++j)
                if (c0 + j < a.C) acc[j] = a.canvas[(size_t)(c0 + j) * a.HW + r];
            if (c0 == 0) wsum = a.canvas[(size_t)a.C * a.HW + r];
        }
        unsigned long long todo = ((unsigned long long)live_mask[1] << 32) | live_mask[0];
        while (todo) {
            const int i = __ffsll((long long)todo) - 1;
            todo &= todo - 1;
            const TileDesc& t = a.t[i];
            const int ty = y - t.y0, tx = x - t.x0;
            if ((unsigned)ty >= (unsigned)t.h || (unsigned)tx >= (unsigned)t.w) continue;
            const float m = mul_rn(hann(ty, t.h, t.ky), hann(tx, t.w, t.kx)) / t.denom;     // patch_utils.py:130-132
            if (c0 == 0) wsum = add_rn(wsum, m);                                           // weight[rect] += mask
            const T* p = (const T*)t.p + (long long)c0 * t.sC;
            if (!t.resize) {
                p += (long long)ty * t.sH + (long long)tx * t.sW;
#pragma unroll
                for (int j = 0; j < kCB; ++j)
                    if (c0 + j < a.C) acc[j] = add_rn(acc[j], mul_rn(ld<float>(p + (long long)j * t.sC), m));   // out[rect] += tile * mask
            } else {
                int y0, ys, x0, xs;
                float ly, lx;
                bilinear_axis(ty, t.ry, t.th, y0, ys, ly);
                bilinear_axis(tx, t.rx, t.tw, x0, xs, lx);
                const float hy = 1.f - ly, hx = 1.f - lx;
                const T* q = p + (long long)y0 * t.sH + (long long)x0 * t.sW;
                const long long dy = (long long)ys * t.sH, dx = (long long)xs * t.sW;
#pragma unroll
                for (int j = 0; j < kCB; ++j) {
                    if (c0 + j < a.C) {
                        const T* qc = q + (long long)j * t.sC;
                        const float v = hy * (hx * ld<float>(qc) + lx * ld<float>(qc + dx)) +
                                        ly * (hx * ld<float>(qc + dy) + lx * ld<float>(qc + dy + dx));
                        acc[j] = add_rn(acc[j], mul_rn(round_as<T>(v), m));
                    }
                }
            }
        }
        if (!a.last) {
#pragma unroll
            for (int j = 0; j < kCB; ++j)
                if (c0 + j < a.C) a.canvas[(size_t)(c0 + j) * a.HW + r] = acc[j];
        } else {
            // merged = out / max(weight, eps), patch_utils.py:172-173 (wsum is complete after the first channel pass)
            const float d = wsum > a.eps ? wsum : a.eps;
#pragma unroll
            for (int j = 0; j < kCB; ++j) {
                if (c0 + j < a.C) {
                    const float v = acc[j] / d;
                    for (int n = 0; n < a.N; ++n) st_stream((T*)a.out + ((size_t)n * a.C + c0 + j) * a.HW + r, v);
                }
            }
        }
    }
    if (!a.last) a.canvas[(size_t)a.C * a.HW + r] = wsum;
}

long long tile_merge_workspace(long long C, long long H, long long W, int n_tiles) {
    return n_tiles > kMaxTiles ? align_up((C + 1) * H * W * 4, 256) : 0;
}

// int(round(v)) of Python: round-half-to-even on a double
static long long py_round(double v) { return (long long)nearbyint(v); }

int tile_merge_impl(const DcbTensor* tiles, const long long* pixel_coords, int n_tiles, const DcbTensor* out, long long H_px,
                    long long W_px, double eps, void* ws, long long ws_bytes, cudaStream_t st) {
    const long long N = out->size[0], C = out->size[1], H = out->size[2], W = out->size[3];
    if (N * C * H * W == 0) return DCB_OK;
    const long long need = tile_merge_workspace(C, H, W, n_tiles);
    if (need > 0 && (!ws || ws_bytes < need || ((uintptr_t)ws & 255)))
        return set_error(DCB_E_WORKSPACE, "tile_merge: workspace of %lld bytes (256 B aligned) required, got %lld", need, ws_bytes);
    MergeArgs a;
    a.out = out->ptr; a.canvas = (float*)ws;
    a.N = (int)N; a.C = (int)C; a.H = (int)H; a.W = (int)W; a.HW = (unsigned)(H * W);
    a.eps = (float)eps;                                           // torch.tensor(eps, dtype=dtype), patch_utils.py:172
    a.first = 1;
    a.n = 0;
    const unsigned blocks = (a.HW + 255) / 256;
    auto flush = [&](int last) -> int {
        a.last = last;
        if (out->dtype == DCB_F32) k_tile_merge<float><<<blocks, 256, 0, st>>>(a);
        else if (out->dtype == DCB_BF16) k_tile_merge<__nv_bfloat16><<<blocks, 256, 0, st>>>(a);
        else k_tile_merge<__half><<<blocks, 256, 0, st>>>(a);
        DCB_CHECK_LAUNCH("k_tile_merge");
        a.first = 0;
        a.n = 0;
        return DCB_OK;
    };
    const double ry = (double)H / (double)H_px, rx = (double)W / (double)W_px;
    for (int i = 0; i < n_tiles; ++i) {
        const DcbTensor* t = tiles + i;
        // the tuple is unpacked as (x1, x2, y1, y2), patch_utils.py:135: positions 2,3 scale with the height
        long long ly1 = py_round((double)pixel_coords[4 * i + 2] * ry), ly2 = py_round((double)pixel_coords[4 * i + 3] * ry);
        long long lx1 = py_round((double)pixel_coords[4 * i + 0] * rx), lx2 = py_round((double)pixel_coords[4 * i + 1] * rx);
        ly1 = ly1 < 0 ? 0 : (ly1 > H ? H : ly1); ly2 = ly2 < 0 ? 0 : (ly2 > H ? H : ly2);
        lx1 = lx1 < 0 ? 0 : (lx1 > W ? W : lx1); lx2 = lx2 < 0 ? 0 : (lx2 > W ? W : lx2);
        const long long h = ly2 - ly1, w = lx2 - lx1;
        if (h <= 0 || w <= 0) continue;                           // patch_utils.py:149-151
        if (a.n == kMaxTiles) {
            const int rc = flush(0);
            if (rc != DCB_OK) return rc;
        }
        TileDesc& d = a.t[a.n++];
        d.p = t->ptr; d.sC = t->stride[1]; d.sH = t->stride[2]; d.sW = t->stride[3];
        d.th = (int)t->size[2]; d.tw = (int)t->size[3];
        d.y0 = (int)ly1; d.x0 = (int)lx1; d.h = (int)h; d.w = (int)w;
        // torch.hann_window: arange(n) * (2*pi / (n - 1)) with the factor rounded to the tensor's dtype
        d.ky = h > 1 ? (float)(6.283185307179586476925286766559 / (double)(h - 1)) : 0.f;
        d.kx = w > 1 ? (float)(6.283185307179586476925286766559 / (double)(w - 1)) : 0.f;
        // max of the outer product = product of the 1-d maxima (rounding is monotonic)
        auto wmax = [](long long n, float k) {
            if (n <= 1) return 1.f;
            float best = 0.f;
            for (long long i = (n - 1) / 2; i <= n / 2; ++i) {
                const float v = -0.5f * cosf((float)i * k) + 0.5f;
                best = v > best ? v : best;
            }
            return best;
        };
        d.denom = wmax(h, d.ky) * wmax(w, d.kx) + 1e-12f;
        d.resize = (d.th != d.h || d.tw != d.w) ? 1 : 0;
        d.ry = (float)d.th / (float)d.h;                          // area_pixel_compute_scale, align_corners = False
        d.rx = (float)d.tw / (float)d.w;
    }
    return flush(1);
}

}  // namespace dcb
