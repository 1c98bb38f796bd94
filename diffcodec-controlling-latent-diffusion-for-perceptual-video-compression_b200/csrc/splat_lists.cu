// splat_lists.cu -- forward splat for MANY channels on LARGE tensors (fp32 / bf16 / fp16): per-target
// contribution lists built once per flow field, then ONE gather pass per channel. sm_100a.
//
// Replaces controlnet/softsplat.py:240-270 (pre/post ops) + :281-345 (zero-init + softsplat_out)
// for C + 1 > 4 when the tensor is big enough that accumulate-then-normalise is bound by the
// accumulators (splat_planar.cu: the reduction target of a 64-channel batch is as large as the
// batch itself, it does not stay in L2, and every element crosses L2 four times).
//
// A splat scatters: each source pixel adds into four targets. The four (target, weight) pairs of a
// pixel do not depend on the channel, so with many channels it pays to invert the map once:
//
//   K7a count   one thread per source pixel: cursor[target] += 1 for every in-range corner
//   K7b alloc   one thread per target: a block-wide prefix sum of the counts plus ONE atomicAdd per
//               CTA on a global cursor hands every target a contiguous range: start[t], cursor[t] = start
//   K7c fill    one thread per source pixel: slot = cursor[target]++ ; entries[slot] =
//               (offset of the source inside an input plane, g(metric) * bilinear weight)
//               -- afterwards cursor[t] is the end of target t's list
//   K7d gather  one thread per TARGET pixel: normaliser = sum of g * w over its list; then for
//               blocks of channels: out_c = (sum over the list of in_c[src] * (g * w)) * 1/D
//
// No atomics on the data, no accumulators, no normalise pass, `in` is read through L1/L2 (each
// source is used by ~4 neighbouring targets) and `out` is written exactly once. The normaliser is
// the reference's sum of rounded g * w products; a value term is fma(in, g * w, acc), i.e. within
// 1.5 ulp of the reference's round(round(in * g) * w) (softsplat.py:244-247, 320-334) -- the same
// size as the run-to-run reordering of the reference's own atomicAdd, far inside the 1e-5 contract.
// Frames are processed in groups whose lists (32 B per pixel) stay L2-resident.
//
// Channels-last (NHWC) input takes its own gather (k_list_gather_nhwc): eight lanes walk the CHANNELS of one target, so a
// list entry is one 16-byte (fp32) / 8-byte (bf16, fp16) load per lane and channel quad, 128 contiguous bytes per group, and there
// is one address computation per four channels; the entries of a list are read once and reused for all channels. The NCHW output the
// reference's callers expect is written through a shared-memory transpose, 128 contiguous bytes per store.
#include "dcb_common.cuh"

namespace dcb {

#ifndef DCB_LCB
#define DCB_LCB 16            // channels per gather block (accumulators + loads in flight per thread)
#endif
#ifndef DCB_LMINCTAS
#define DCB_LMINCTAS 3
#endif
#ifndef DCB_LGROUP_MB
#define DCB_LGROUP_MB 32      // list bytes per frame group
#endif

// read-only global load with the address space spelled out: ld.global.nc is not ordered against
// the kernel's stores and keeps the loads of a whole channel block in flight (plain loads: +25 %
// kernel time)
__device__ __forceinline__ float ld_global_ro(const float* p) {
    float v;
    asm("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float ld_global_ro(const __nv_bfloat16* p) {
    unsigned short v;
    asm("ld.global.nc.u16 %0, [%1];" : "=h"(v) : "l"(p));
    return __uint_as_float((unsigned)v << 16);
}
__device__ __forceinline__ float ld_global_ro(const __half* p) {
    unsigned short v;
    asm("ld.global.nc.u16 %0, [%1];" : "=h"(v) : "l"(p));
    return __half2float(__ushort_as_half(v));
}

// dcb_set_option("lists_nhwc", 0): A/B switch, channels-last input through the NCHW gather (strided scalar loads)
int g_lists_nhwc = 1;
void lists_set_nhwc(long long v) { g_lists_nhwc = (int)v; }      // 0 off | 1 on | 8 on, always eight lanes per target (A/B)

struct ListArgs {
    View in, flow, metric, mask;
    int* cursor;             // [gtotal]: counts -> starts -> ends
    int* start;              // [gtotal]: first entry of each target's list
    int* total;              // one counter: entries handed out so far
    int2* entries;           // [4 * gtotal]: (source offset in a plane, g(metric) * bilinear weight)
    void* out;               // [N,C,H,W]
    void* norm;              // [N,1,H,W] fp32 or null
    int C, H, W;
    unsigned HW, gtotal;     // pixels per frame, pixels in this frame group
    unsigned tiles_x, tiles; // gather: 32 x 8 target tiles per row / per frame
    unsigned q_tiles_x, row_tiles;   // channels-last gather: (256 / G) x 1 target tiles per row / per frame
    int frame0;              // first frame of the group
    int mode, eps;
    int nhwc;                // channels-last input whose channel quads are aligned: k_list_gather_nhwc
};

// the four corners of a source pixel: target index inside the group, weight, in range or not
template <class TF>
__device__ __forceinline__ void corners(const ListArgs& a, unsigned p, unsigned& n, int& y, int& x, unsigned (&tgt)[4], float (&w)[4],
                                        bool (&ok)[4]) {
    n = p / a.HW;
    const unsigned r = p - n * a.HW;
    y = (int)(r / (unsigned)a.W); x = (int)(r - (unsigned)y * (unsigned)a.W);
    const TF* fp = (const TF*)a.flow.p + (long long)(a.frame0 + n) * a.flow.sN + (long long)y * a.flow.sH + (long long)x * a.flow.sW;
    const Foot<float> f = make_foot<float>(x, y, (float)ld_stream(fp), (float)ld_stream(fp + a.flow.sC));
    const int x1 = (int)((unsigned)f.x0 + 1u), y1 = (int)((unsigned)f.y0 + 1u);
    const bool vx0 = f.finite && (unsigned)f.x0 < (unsigned)a.W, vx1 = f.finite && (unsigned)x1 < (unsigned)a.W;   // softsplat.py:301-302
    const bool vy0 = (unsigned)f.y0 < (unsigned)a.H, vy1 = (unsigned)y1 < (unsigned)a.H;
    const unsigned t0 = n * a.HW + (unsigned)(f.y0 * a.W + f.x0);  // only used for in-range corners
    tgt[0] = t0; tgt[1] = t0 + 1; tgt[2] = t0 + a.W; tgt[3] = t0 + a.W + 1;
    w[0] = f.wnw; w[1] = f.wne; w[2] = f.wsw; w[3] = f.wse;
    ok[0] = vx0 && vy0; ok[1] = vx1 && vy0; ok[2] = vx0 && vy1; ok[3] = vx1 && vy1;
}

template <class TF>
__global__ void __launch_bounds__(256) k_list_count(const ListArgs a) {
    pdl_wait();
    const unsigned p = blockIdx.x * 256 + threadIdx.x;
    if (p >= a.gtotal) return;
    unsigned n, tgt[4]; int y, x; float w[4]; bool ok[4];
    corners<TF>(a, p, n, y, x, tgt, w, ok);
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (ok[i]) atomicAdd(a.cursor + tgt[i], 1);
}

// contiguous list ranges without a global scan: the order of the CTAs' ranges does not matter
__global__ void __launch_bounds__(256) k_list_alloc(const ListArgs a) {
    __shared__ int warp_sum[8];
    __shared__ int cta_base;
    pdl_wait();
    const unsigned t = blockIdx.x * 256 + threadIdx.x;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int cnt = t < a.gtotal ? __ldcg(a.cursor + t) : 0;
    int inc = cnt;                                                // inclusive prefix inside the warp
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int up = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += up;
    }
    if (lane == 31) warp_sum[wid] = inc;
    __syncthreads();
    if (threadIdx.x == 0) {
        int s = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) { const int v = warp_sum[i]; warp_sum[i] = s; s += v; }
        cta_base = atomicAdd(a.total, s);
    }
    __syncthreads();
    if (t < a.gtotal) {
        const int first = cta_base + warp_sum[wid] + inc - cnt;
        __stcg(a.start + t, first);
        __stcg(a.cursor + t, first);
    }
}

template <class T, class TF>
__global__ void __launch_bounds__(256) k_list_fill(const ListArgs a) {
    pdl_wait();
    const unsigned p = blockIdx.x * 256 + threadIdx.x;
    if (p >= a.gtotal) return;
    unsigned n, tgt[4]; int y, x; float w[4]; bool ok[4];
    corners<TF>(a, p, n, y, x, tgt, w, ok);
    if (!(ok[0] || ok[1] || ok[2] || ok[3])) return;
    float g = 1.f;                                                // g(m) of softsplat.py:240-247
    if (a.mode == DCB_MODE_LINEAR || a.mode == DCB_MODE_SOFT) {
        const T* mp = (const T*)a.metric.p + (long long)(a.frame0 + n) * a.metric.sN + (long long)y * a.metric.sH + (long long)x * a.metric.sW;
        const float m = ld_stream(mp);
        g = a.mode == DCB_MODE_SOFT ? expf(m) : m;
    }
    const int src = (int)((long long)y * a.in.sH + (long long)x * a.in.sW);
    int slot[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) slot[i] = ok[i] ? atomicAdd(a.cursor + tgt[i], 1) : 0;   // four independent round trips
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (ok[i]) __stcg(a.entries + slot[i], make_int2(src, __float_as_int(mul_rn(g, w[i]))));
}

template <class T>
__global__ void __launch_bounds__(256, DCB_LMINCTAS) k_list_gather(const ListArgs a) {
    constexpr int CB = DCB_LCB;
    pdl_wait();
    // a CTA owns a 32 x 8 tile of targets: the sources of vertically adjacent targets are the same
    // rows of `in`, so they are served by this SM's L1 instead of L2
    // grid = (tile columns, tile rows, frames of the group): no integer division in front of the first load
    const unsigned n = blockIdx.z;
    const unsigned tx = blockIdx.x, ty = blockIdx.y;
    const unsigned x = tx * 32 + (threadIdx.x & 31), y = ty * 8 + (threadIdx.x >> 5);
    if (x >= (unsigned)a.W || y >= (unsigned)a.H) return;
    const unsigned r = y * a.W + x, t = n * a.HW + r;
    const int frame = a.frame0 + (int)n;
    const int beg = __ldcg(a.start + t), end = __ldcg(a.cursor + t);
    const bool normalised = a.mode != DCB_MODE_SUM;

    float scale = 1.f;
    if (normalised) {
        float d = 0.f;
        for (int e = beg; e < end; ++e) d = add_rn(d, __int_as_float(__ldcg(a.entries + e).y));   // the appended channel, softsplat.py:243-247
        // softsplat.py:256-266
        if (a.eps == DCB_EPS_ADD) d = add_rn(d, 0.0000001f);
        else if (a.eps == DCB_EPS_ZERO) d = (d == 0.f) ? 1.f : d;
        else d = (d < 0.0000001f) ? 0.0000001f : d;
        if (a.norm) __stcs((float*)a.norm + (long long)frame * a.HW + r, d);
        scale = __frcp_rn(d);                                     // <= 1 ulp from the true quotient of softsplat.py:270
    }
    if (a.mask.p) {
        const T* mp = (const T*)a.mask.p + (long long)frame * a.mask.sN + (long long)y * a.mask.sH + (long long)x * a.mask.sW;
        scale = mul_rn(scale, sub_rn(1.f, ld<float>(mp)));        // control_utils.py:69-70
    }
    const bool scaled = normalised || a.mask.p != nullptr;

    // all offsets inside one frame are unsigned 32-bit (lists_supported): one IMAD.WIDE.U32 per load
    const T* ibase = (const T*)a.in.p + (long long)frame * a.in.sN;
    T* obase = (T*)a.out + (long long)frame * a.C * a.HW;
    const unsigned sC = (unsigned)a.in.sC;
    // optimisation barrier: without it the compiler re-derives frame * sN inside every load's
    // address (7 integer instructions per element instead of 2; +20 % kernel time)
    asm volatile("" : "+l"(ibase));
    for (int c0 = 0; c0 < a.C; c0 += CB) {
        float acc[CB];
        unsigned jo[CB];                                          // channel offsets of this block; a short last block re-reads its first plane
        const int live = min(CB, a.C - c0);
#pragma unroll
        for (int j = 0; j < CB; ++j) {
            acc[j] = 0.f;
            jo[j] = (unsigned)(c0 + (j < live ? j : 0)) * sC;
        }
        int2 nxt = beg < end ? __ldcg(a.entries + beg) : make_int2(0, 0);
        for (int e = beg; e < end; ++e) {
            const int2 en = nxt;
            if (e + 1 < end) nxt = __ldcg(a.entries + e + 1);     // the next entry is in flight while this one's loads are
            const float gw = __int_as_float(en.y);
            const unsigned src = (unsigned)en.x;
            float v[CB];
#pragma unroll
            for (int j = 0; j < CB; ++j) v[j] = ld_global_ro(ibase + (src + jo[j]));
#pragma unroll
            for (int j = 0; j < CB; ++j) acc[j] = fma_rn(v[j], gw, acc[j]);
        }
        const unsigned o0 = (unsigned)c0 * a.HW + r;
        if (live == CB) {
#pragma unroll
            for (int j = 0; j < CB; ++j) st_stream(obase + (o0 + (unsigned)j * a.HW), scaled ? mul_rn(acc[j], scale) : acc[j]);
        } else {
#pragma unroll
            for (int j = 0; j < CB; ++j)
                if (j < live) st_stream(obase + (o0 + (unsigned)j * a.HW), scaled ? mul_rn(acc[j], scale) : acc[j]);
        }
    }
}

// the four channels of a quad of a channels-last tensor in one read-only load
__device__ __forceinline__ void ld_quad_ro(const float* p, float (&o)[4]) {
    asm("ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(o[0]), "=f"(o[1]), "=f"(o[2]), "=f"(o[3]) : "l"(p));
}
__device__ __forceinline__ void ld_quad_ro(const __nv_bfloat16* p, float (&o)[4]) {
    unsigned lo, hi;
    asm("ld.global.nc.v2.u32 {%0,%1}, [%2];" : "=r"(lo), "=r"(hi) : "l"(p));
    o[0] = __uint_as_float(lo << 16); o[1] = __uint_as_float(lo & 0xffff0000u);
    o[2] = __uint_as_float(hi << 16); o[3] = __uint_as_float(hi & 0xffff0000u);
}
__device__ __forceinline__ void ld_quad_ro(const __half* p, float (&o)[4]) {
    unsigned lo, hi;
    asm("ld.global.nc.v2.u32 {%0,%1}, [%2];" : "=r"(lo), "=r"(hi) : "l"(p));
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&lo)), b = __half22float2(*reinterpret_cast<const __half2*>(&hi));
    o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y;
}

#ifndef DCB_LQ_CBLK
#define DCB_LQ_CBLK 64        // channels per pass through the transpose tile (8.25 KB of shared memory; measured: 64 beats 32 and 128 at C = 64)
#endif
#ifndef DCB_LQ_U
#define DCB_LQ_U 4            // list entries whose loads are in flight together
#endif

// K7d for channels-last input. G lanes share a target (8, or 4 when whole 64-channel blocks make every lane's four quads
// live): a CTA owns 256 / G consecutive targets of one row, one pass per CTA; a lane owns the channel quads q = lane,
// lane + G, ... of the block (G x 16 contiguous bytes per group and load). The entries of a list are read once per chunk
// of U and reused for every quad; the normaliser is summed in the same pass. Output: NCHW-contiguous, through the
// transpose tile (row pitch chosen so that neither its writes nor its reads conflict).
template <class T, int G>
__global__ void __launch_bounds__(256) k_list_gather_nhwc(const ListArgs a) {
    constexpr int CBLK = DCB_LQ_CBLK, U = DCB_LQ_U, QPL = CBLK / 4 / G, TT = 256 / G, PITCH = TT + (G == 8 ? 1 : 2);
    __shared__ float tile[CBLK][PITCH];
    pdl_wait();
    // grid = (tile columns, rows, frames of the group): no integer division in front of the first load
    const unsigned n = blockIdx.z;
    const unsigned tx = blockIdx.x, y = blockIdx.y;
    const unsigned x0 = tx * TT;
    const int frame = a.frame0 + (int)n;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ql = lane % G;
    const int tt = warp * (32 / G) + lane / G;                    // this group's target inside the tile
    const unsigned x = x0 + (unsigned)tt;
    const bool live = x < (unsigned)a.W;
    const bool normalised = a.mode != DCB_MODE_SUM;
    const T* ibase = (const T*)a.in.p + (long long)frame * a.in.sN;
    T* obase = (T*)a.out + (long long)frame * a.C * a.HW + (size_t)y * a.W + x0;
    const unsigned r = y * (unsigned)a.W + (live ? x : 0u), t = n * a.HW + r;
    int beg = 0, end = 0;
    if (live) { beg = __ldcg(a.start + t); end = __ldcg(a.cursor + t); }
    float mscale = 1.f;
    if (live && a.mask.p) {
        const T* mp = (const T*)a.mask.p + (long long)frame * a.mask.sN + (long long)y * a.mask.sH + (long long)x * a.mask.sW;
        mscale = sub_rn(1.f, ld<float>(mp));                      // control_utils.py:69-70
    }

    for (int c0 = 0; c0 < a.C; c0 += CBLK) {
        const int quads = min(CBLK, a.C - c0) >> 2;               // C % 4 == 0 (checked by the host)
        float acc[QPL][4];
#pragma unroll
        for (int i = 0; i < QPL; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
        float d = 0.f;
        const T* ip = ibase + (c0 + 4 * ql);
        for (int e = beg; e < end; e += U) {
            int2 en[U];
#pragma unroll
            for (int u = 0; u < U; ++u) en[u] = __ldcg(a.entries + min(e + u, end - 1));
            float gw[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                gw[u] = e + u < end ? __int_as_float(en[u].y) : 0.f;                      // a repeated last entry adds nothing
                if (e + u < end) d = add_rn(d, gw[u]);                                    // the appended channel, softsplat.py:243-247
            }
#pragma unroll
            for (int i = 0; i < QPL; ++i) {
                if (ql + i * G < quads) {
                    float v[U][4];
#pragma unroll
                    for (int u = 0; u < U; ++u) ld_quad_ro(ip + ((unsigned)en[u].x + (unsigned)(4 * G * i)), v[u]);
#pragma unroll
                    for (int u = 0; u < U; ++u)
#pragma unroll
                        for (int k = 0; k < 4; ++k) acc[i][k] = fma_rn(v[u][k], gw[u], acc[i][k]);
                }
            }
        }
        float scale = mscale;
        if (normalised) {
            // softsplat.py:256-266
            if (a.eps == DCB_EPS_ADD) d = add_rn(d, 0.0000001f);
            else if (a.eps == DCB_EPS_ZERO) d = (d == 0.f) ? 1.f : d;
            else d = (d < 0.0000001f) ? 0.0000001f : d;
            if (live && a.norm && c0 == 0 && ql == 0) __stcs((float*)a.norm + (long long)frame * a.HW + r, d);
            scale = mul_rn(__frcp_rn(d), mscale);                 // <= 1 ulp from the true quotient of softsplat.py:270 (x 1.0f is exact)
        }
        const bool scaled = normalised || a.mask.p != nullptr;
#pragma unroll
        for (int i = 0; i < QPL; ++i)
            if (ql + i * G < quads)
#pragma unroll
                for (int k = 0; k < 4; ++k) tile[4 * (ql + i * G) + k][tt] = scaled ? mul_rn(acc[i][k], scale) : acc[i][k];
        __syncthreads();
        for (int c = warp; c < 4 * quads; c += 8)
#pragma unroll
            for (int col = lane; col < TT; col += 32)
                if (x0 + (unsigned)col < (unsigned)a.W) st_stream(obase + (size_t)(c0 + c) * a.HW + col, tile[c][col]);
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------
static long long lists_group_frames(long long N, long long H, long long W) {
    const long long per = 32 * H * W;                             // 4 entries of 8 B per pixel
    long long g = ((long long)DCB_LGROUP_MB << 20) / (per > 0 ? per : 1);
    if (g < 1) g = 1;
    if (g > 65535) g = 65535;                                     // the gathers put the group's frames on gridDim.z
    return g > N ? (N < 1 ? 1 : N) : g;
}

struct ListLayout {
    long long total_off, cursor_off, start_off, entries_off, total_bytes;
    long long G;
};

static ListLayout lists_layout(long long N, long long H, long long W) {
    ListLayout L;
    L.G = lists_group_frames(N, H, W);
    const long long gtotal = L.G * H * W;
    L.total_off = 0;                                              // the counter and the counts are zeroed together
    L.cursor_off = 256;
    L.start_off = L.cursor_off + align_up(gtotal * 4, 256);
    L.entries_off = L.start_off + align_up(gtotal * 4, 256);
    L.total_bytes = L.entries_off + align_up(gtotal * 32, 256);
    return L;
}

long long lists_workspace(long long N, long long H, long long W) { return lists_layout(N, H, W).total_bytes; }

// many channels, enough bytes that the accumulate-then-normalise pipeline is accumulator-bound, and
// every offset the kernels form fits 31 bits
bool lists_supported(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, int mode) {
    (void)flow; (void)metric;
    const long long N = in->size[0], C = in->size[1], H = in->size[2], W = in->size[3];
    if (in->dtype != DCB_F32 && !is_half_storage(in->dtype)) return false;
    // building the lists costs about as much as scattering 8-16 channels (measured crossover on
    // 1080p, 540p and 256 x 256 batches with a rough random flow: lists lose at C = 8, win from C = 16)
    if (C < 16) return false;
#ifndef DCB_LMIN_MB
#define DCB_LMIN_MB 16
#endif
    if (N * C * H * W * elem_size(in->dtype) < ((long long)DCB_LMIN_MB << 20)) return false;
    if (N * H * W < 65536) return false;                          // one thread per pixel: few pixels cannot fill the machine
    if (H > 65535) return false;                                  // rows on gridDim.y of the channels-last gather
    const long long G = lists_group_frames(N, H, W);
    if (4 * G * H * W >= (1ll << 31)) return false;
    if (in->stride[2] < 0 || in->stride[3] < 0) return false;
    if (in->stride[1] < 0 || C * H * W >= (1ll << 31)) return false;
    return (C - 1) * in->stride[1] + (H - 1) * in->stride[2] + (W - 1) * in->stride[3] < (1ll << 31);
}

template <class T, class TF>
static int launch_lists(ListArgs& a, const ListLayout& L, char* ws, int N, bool clean, cudaStream_t st) {
    for (int f0 = 0; f0 < N; f0 += (int)L.G) {
        const int frames = N - f0 < (int)L.G ? N - f0 : (int)L.G;
        a.frame0 = f0;
        a.gtotal = (unsigned)frames * a.HW;
        const unsigned blocks = (a.gtotal + 255) / 256;
        if (!clean)
            DCB_CHECK_CUDA(cudaMemsetAsync(ws + L.total_off, 0, (size_t)(L.cursor_off - L.total_off) + (size_t)a.gtotal * 4, st));
        // programmatic dependent launches: each kernel's launch overlaps its predecessor's drain
        DCB_CHECK_CUDA(launch_pdl(k_list_count<TF>, blocks, 256, 0, st, a));
        DCB_CHECK_CUDA(launch_pdl(k_list_alloc, blocks, 256, 0, st, a));
        DCB_CHECK_CUDA(launch_pdl(k_list_fill<T, TF>, blocks, 256, 0, st, a));
        if (a.nhwc) {
            // four lanes per target when every lane's four quads are live (whole 64-channel blocks), else eight
            // measured at C = 64 (profiles/r02/NOTES.md section 9): 8 / 4 / 2 lanes per target = 151 / 127 / 147 us (fp32)
            const bool g4 = a.C % DCB_LQ_CBLK == 0 && g_lists_nhwc != 8;
            const unsigned tt = g4 ? 64u : 32u;
            a.q_tiles_x = ((unsigned)a.W + tt - 1) / tt;
            a.row_tiles = a.q_tiles_x * (unsigned)a.H;
            const dim3 grid(a.q_tiles_x, (unsigned)a.H, (unsigned)frames);
            if (g4) DCB_CHECK_CUDA(launch_pdl(k_list_gather_nhwc<T, 4>, grid, dim3(256), 0, st, a));
            else DCB_CHECK_CUDA(launch_pdl(k_list_gather_nhwc<T, 8>, grid, dim3(256), 0, st, a));
        } else {
            DCB_CHECK_CUDA(launch_pdl(k_list_gather<T>, dim3(a.tiles_x, a.tiles / a.tiles_x, (unsigned)frames), dim3(256), 0, st, a));
        }
        count_launch(4);
        // a shared all-zero workspace is handed back all-zero: one memset behind the gather (zeroing
        // the cells inside the kernel that reads them cost 10-60 % of its speed: the stores order
        // the loads behind them)
        if (clean) DCB_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)L.entries_off + (size_t)a.gtotal * 32, st));
    }
    return DCB_OK;
}

// `ws` must hold lists_workspace() bytes. With `clean` (DCB_FLAG_WS_CLEAN: the caller shares an
// all-zero workspace with the accumulator paths) it is all-zero on entry and all-zero again when the
// last kernel has run; otherwise its contents on entry do not matter.
int splat_lists_impl(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const DcbTensor* out,
                     const DcbTensor* norm, const DcbTensor* mask, void* ws, int mode, int eps, bool clean,
                     cudaStream_t st) {
    ListArgs a;
    a.in = make_view(in); a.flow = make_view(flow); a.metric = make_view(metric); a.mask = make_view(mask);
    const int N = (int)in->size[0];
    a.C = (int)in->size[1]; a.H = (int)in->size[2]; a.W = (int)in->size[3];
    a.HW = (unsigned)(in->size[2] * in->size[3]);
    a.mode = mode; a.eps = eps;
    a.tiles_x = (unsigned)(a.W + 31) / 32;
    a.tiles = a.tiles_x * ((unsigned)(a.H + 7) / 8);
    a.q_tiles_x = a.tiles_x; a.row_tiles = a.tiles_x * (unsigned)a.H;
    {   // channels-last: unit channel stride, whole quads, every quad aligned to its vector load
        const long long es = elem_size(in->dtype);
        a.nhwc = (g_lists_nhwc && in->stride[1] == 1 && a.C % 4 == 0 && a.C >= 32 && ((uintptr_t)in->ptr % (uintptr_t)(4 * es)) == 0 &&
                  in->stride[0] % 4 == 0 && in->stride[2] % 4 == 0 && in->stride[3] % 4 == 0) ? 1 : 0;
    }
    a.out = out->ptr;
    a.norm = norm ? norm->ptr : nullptr;
    const ListLayout L = lists_layout(N, a.H, a.W);
    char* base = (char*)ws;
    a.total = (int*)(base + L.total_off);
    a.cursor = (int*)(base + L.cursor_off);
    a.start = (int*)(base + L.start_off);
    a.entries = (int2*)(base + L.entries_off);
    const bool ff = flow->dtype == DCB_F32;
    int rc;
    if (in->dtype == DCB_F32) rc = launch_lists<float, float>(a, L, base, N, clean, st);
    else if (in->dtype == DCB_BF16)
        rc = ff ? launch_lists<__nv_bfloat16, float>(a, L, base, N, clean, st) : launch_lists<__nv_bfloat16, __nv_bfloat16>(a, L, base, N, clean, st);
    else if (in->dtype == DCB_F16)
        rc = ff ? launch_lists<__half, float>(a, L, base, N, clean, st) : launch_lists<__half, __half>(a, L, base, N, clean, st);
    else return set_error(DCB_E_DTYPE, "splat_lists: unsupported dtype %d", in->dtype);
    return rc;
}

}  // namespace dcb
