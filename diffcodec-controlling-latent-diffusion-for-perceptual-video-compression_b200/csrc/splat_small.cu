// splat_small.cu -- the forward splat of SMALL few-channel frames (pyramid-level flows, thumbnails) in ONE launch:
// a thread-block CLUSTER of eight CTAs owns one frame (sm_100a).
//
// The accumulate-then-normalise forward needs "every contribution has landed" between its two halves. For big tensors
// that point is a kernel boundary (splat_pipe.cu / splat_planar.cu: two launches per frame group). A thumbnail-sized call
// (the flow-by-flow splats behind compute_mask at the pyramid resolutions, few-channel frames up to ~90 x 90) is bound by
// exactly those two dependent launches; a software grid barrier was measured slower than the boundary it replaces
// (profiles/r01/NOTES.md section 7). Here the dependency is confined to ONE frame and the frame to ONE cluster:
//
//   * a frame's source pixels are spread over the 8 x 512 threads of a cluster; each thread scatters its pixels with
//     `red.global.add.v4.f32` into channel-quad accumulators [frame][quad][H*W] (the appended weight channel is simply
//     channel C) -- a splat never leaves its frame, so no other cluster ever touches these cells;
//   * `barrier.cluster` (hardware barrier across the eight co-scheduled CTAs, release / acquire) behind a gpu-scope fence is
//     the "all landed" point: no global counter, no polling, no second launch;
//   * the same threads then normalise the frame out of L2 (eps rule, reciprocal, (1 - mask), cast, saved normaliser, or the
//     occlusion test of compute_mask) and re-zero what they read (DCB_FLAG_WS_CLEAN protocol).
//
// Replaces controlnet/softsplat.py:240-270 (pre/post ops) + :281-345 (zero-init + softsplat_out) for small frames, and the
// splat inside compute_mask (controlnet/control_utils.py:11-17).
#include "dcb_common.cuh"

namespace dcb {

constexpr int kClusterCtas = 8;              // portable maximum
constexpr int kSmallThreads = 512;
constexpr int kClusterThreads = kClusterCtas * kSmallThreads;
constexpr int kSmallBatch = 2;               // pixels per thread in flight
constexpr float kExp1s = 2.7182817459106445f;   // expf(1.0f)

struct SmallArgs {
    View in, flow, metric, mask, epi_flow;
    float* acc;              // [N][Cq][HW] float4, all-zero on entry and on exit
    void* out;               // [N,C,H,W]
    void* norm;              // [N,1,H,W] fp32 or null
    void* mask_out;          // epilogue 1: [N,1,H,W] in T
    int N, C, CA, Cq, H, W;
    unsigned HW;
    int mode, eps, ones, epi;
};

__device__ __forceinline__ void cluster_barrier() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

__device__ __forceinline__ float quad_comp(const float4& v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w)); }

template <class T, class TF>
__global__ void __cluster_dims__(kClusterCtas, 1, 1) __launch_bounds__(kSmallThreads) k_splat_cluster(const __grid_constant__ SmallArgs a) {
    pdl_wait();
    const unsigned frame = blockIdx.x / kClusterCtas;                    // clusters are consecutive CTAs along x
    const unsigned tid = (blockIdx.x % kClusterCtas) * kSmallThreads + threadIdx.x;
    const int W = a.W, H = a.H, C = a.C, CA = a.CA;
    const unsigned HW = a.HW;
    float4* acc = (float4*)a.acc + (size_t)frame * a.Cq * HW;
    const TF* fbase = (const TF*)a.flow.p + frame * a.flow.sN;
    const T* ibase = (const T*)a.in.p + frame * a.in.sN;
    const T* mbase = (a.mode >= DCB_MODE_LINEAR && !a.ones) ? (const T*)a.metric.p + frame * a.metric.sN : nullptr;

    // ---- scatter: kSmallBatch pixels per thread per round, their loads in flight together ----
    for (unsigned p0 = tid; p0 < HW; p0 += kSmallBatch * kClusterThreads) {
        Foot<float> f[kSmallBatch];
        float g[kSmallBatch];
        long long ioff[kSmallBatch];
        bool live[kSmallBatch];
#pragma unroll
        for (int b = 0; b < kSmallBatch; ++b) {
            const unsigned p = p0 + b * kClusterThreads;
            live[b] = p < HW;
            const unsigned pc = live[b] ? p : 0;
            const int y = (int)(pc / (unsigned)W), x = (int)(pc - (unsigned)y * (unsigned)W);
            const TF* fp = fbase + (long long)y * a.flow.sH + (long long)x * a.flow.sW;
            f[b] = make_foot<float>(x, y, (float)ld_stream(fp), (float)ld_stream(fp + a.flow.sC));     // softsplat.py:298-318
            float m = 1.f;
            if (mbase) m = ld_stream(mbase + (long long)y * a.metric.sH + (long long)x * a.metric.sW);
            g[b] = a.mode == DCB_MODE_SOFT ? (a.ones ? kExp1s : expf(m)) : (a.mode == DCB_MODE_LINEAR ? m : 1.f);
            ioff[b] = (long long)y * a.in.sH + (long long)x * a.in.sW;
            live[b] = live[b] && f[b].finite;                                                          // softsplat.py:301-302
        }
        for (int q = 0; q < a.Cq; ++q) {
            float v[kSmallBatch][4];
#pragma unroll
            for (int b = 0; b < kSmallBatch; ++b)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int c = 4 * q + j;
                    float t = 0.f;
                    if (c < C) {
                        t = live[b] ? ld_stream(ibase + ioff[b] + (long long)c * a.in.sC) : 0.f;
                        if (a.mode >= DCB_MODE_LINEAR) t = mul_rn(t, g[b]);                            // softsplat.py:244,247
                    } else if (c == C && CA > C) {
                        t = g[b];                                                                      // appended channel: 1 | m | exp(m)
                    }
                    v[b][j] = t;
                }
#pragma unroll
            for (int b = 0; b < kSmallBatch; ++b) {
                if (!live[b]) continue;
                const int x0 = f[b].x0, y0 = f[b].y0;
                const int x1 = (int)((unsigned)x0 + 1u), y1 = (int)((unsigned)y0 + 1u);
                const bool vx0 = (unsigned)x0 < (unsigned)W, vx1 = (unsigned)x1 < (unsigned)W;
                const bool vy0 = (unsigned)y0 < (unsigned)H, vy1 = (unsigned)y1 < (unsigned)H;
                float4* base = acc + (size_t)q * HW;
                const float w4[4] = {f[b].wnw, f[b].wne, f[b].wsw, f[b].wse};
                const bool ok[4] = {vx0 && vy0, vx1 && vy0, vx0 && vy1, vx1 && vy1};
                const int cell[4] = {y0 * W + x0, y0 * W + x1, y1 * W + x0, y1 * W + x1};
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (ok[k])
                        red_add_v4((float*)(base + cell[k]), mul_rn(v[b][0], w4[k]), mul_rn(v[b][1], w4[k]), mul_rn(v[b][2], w4[k]), mul_rn(v[b][3], w4[k]));
            }
        }
    }

    // ---- every contribution of this frame has landed: gpu-scope fence, then the cluster's hardware barrier ----
    __threadfence();
    cluster_barrier();

    // ---- normalise (or occlusion test), re-zero ----
    const int qd = C >> 2, jd = C & 3;                                   // where the weight channel lives
    for (unsigned p = tid; p < HW; p += kClusterThreads) {
        const int y = (int)(p / (unsigned)W), x = (int)(p - (unsigned)y * (unsigned)W);
        if (a.epi == 1) {                                                // compute_mask: accumulators hold (x*e, y*e, e, -)
            const float4 s = __ldcg(acc + p);
            __stcg(acc + p, make_float4(0.f, 0.f, 0.f, 0.f));
            const T* fp = (const T*)a.epi_flow.p + frame * a.epi_flow.sN + (long long)y * a.epi_flow.sH + (long long)x * a.epi_flow.sW;
            st<T, float>((T*)a.mask_out + (size_t)frame * HW + p, occlusion(s.x, s.y, s.z, ld<float>(fp), ld<float>(fp + a.epi_flow.sC)));
            continue;
        }
        float scale = 1.f;
        float4 wq = make_float4(0.f, 0.f, 0.f, 0.f);
        if (a.mode != DCB_MODE_SUM) {
            wq = __ldcg(acc + (size_t)qd * HW + p);
            float d = quad_comp(wq, jd);
            // softsplat.py:256-266
            if (a.eps == DCB_EPS_ADD) d = add_rn(d, 0.0000001f);
            else if (a.eps == DCB_EPS_ZERO) d = (d == 0.f) ? 1.f : d;
            else d = (d < 0.0000001f) ? 0.0000001f : d;
            if (a.norm) ((float*)a.norm)[(size_t)frame * HW + p] = d;
            scale = __frcp_rn(d);                                        // <= 1 ulp from the quotient of softsplat.py:270, as the other paths
        }
        if (a.mask.p) {
            const T* mp = (const T*)a.mask.p + frame * a.mask.sN + (long long)y * a.mask.sH + (long long)x * a.mask.sW;
            scale = mul_rn(scale, sub_rn(1.f, ld<float>(mp)));          // control_utils.py:69-70
        }
        const bool scaled = a.mode != DCB_MODE_SUM || a.mask.p != nullptr;
        T* o = (T*)a.out + (size_t)frame * C * HW + p;
        for (int q = 0; q < a.Cq; ++q) {
            float4* cellp = acc + (size_t)q * HW + p;
            const float4 s = (q == qd && a.mode != DCB_MODE_SUM) ? wq : __ldcg(cellp);
            __stcg(cellp, make_float4(0.f, 0.f, 0.f, 0.f));
            const float sv[4] = {s.x, s.y, s.z, s.w};
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (4 * q + j < C) st_stream(o + (size_t)(4 * q + j) * HW, scaled ? mul_rn(sv[j], scale) : sv[j]);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------
// dcb_set_option("small_path"): 1 (default) = small frames take the single-launch cluster kernel, 0 = never
int g_small_path = 1;
void small_set_enabled(long long v) { g_small_path = v ? 1 : 0; }

static long long small_quads(long long C, int mode) { return (C + (mode == DCB_MODE_SUM ? 0 : 1) + 3) / 4; }

// One cluster walks one frame, so a frame has 8 SMs at most: worth it while a frame is one or two rounds of the cluster's 4096
// threads. Measured (profiles/scripts/r02_small.py, CUDA-graph replay, us per call, cluster kernel / two pipeline launches):
// flow-by-flow splat + occlusion test 2x2x8x8 6.2 / 8.2, 2x2x16x16 6.3 / 10.3, 2x2x32x32 8.2 / 12.3, 2x2x64x64 8.2 / 12.3;
// but 4x4x135x240 latents (8 rounds per frame, 32 of 148 SMs busy) 45.6 / 16.4 and 4x3x256x256 47.6 / 12.3: bigger frames stay
// on the pipelines, whose two launches spread a frame over the whole machine.
bool use_cluster(int dtype, int mode, long long N, long long C, long long H, long long W) {
    if (!g_small_path || (dtype != DCB_F32 && !is_half_storage(dtype))) return false;
    const long long P = H * W;
    return P > 0 && P <= 8192 && small_quads(C, mode) <= 2 && N <= 64;
}

long long cluster_workspace(long long N, long long C, long long H, long long W, int mode) {
    return align_up(N * small_quads(C, mode) * H * W * 16, 256);
}

template <class T, class TF> static int launch_small(const SmallArgs& a, cudaStream_t st) {
    DCB_CHECK_CUDA(launch_pdl(k_splat_cluster<T, TF>, dim3((unsigned)a.N * kClusterCtas), dim3(kSmallThreads), 0, st, a));
    count_launch();
    return DCB_OK;
}

// Same contract as splat_pipe_impl; `ws` holds cluster_workspace() bytes.
int splat_cluster_impl(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const DcbTensor* out,
                       const DcbTensor* norm, const DcbTensor* mask, void* ws, int mode, int eps, bool ws_clean,
                       cudaStream_t st, bool ones_metric, const DcbTensor* mask_out) {
    SmallArgs a;
    a.in = make_view(in); a.flow = make_view(flow); a.metric = make_view(metric); a.mask = make_view(mask);
    a.epi = mask_out ? 1 : 0;
    a.epi_flow = make_view(mask_out ? flow : nullptr);
    a.mask_out = mask_out ? mask_out->ptr : nullptr;
    a.N = (int)in->size[0]; a.C = (int)in->size[1]; a.H = (int)in->size[2]; a.W = (int)in->size[3];
    a.HW = (unsigned)(in->size[2] * in->size[3]);
    a.CA = a.C + (mode == DCB_MODE_SUM ? 0 : 1);
    a.Cq = (a.CA + 3) / 4;
    a.mode = mode; a.eps = eps; a.ones = ones_metric ? 1 : 0;
    a.out = out ? out->ptr : nullptr;
    a.norm = norm ? norm->ptr : nullptr;
    a.acc = (float*)ws;
    if (!ws_clean) DCB_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)cluster_workspace(a.N, a.C, a.H, a.W, mode), st));
    const bool ff = flow->dtype == DCB_F32;
    if (in->dtype == DCB_F32) return launch_small<float, float>(a, st);
    if (in->dtype == DCB_BF16)
        return ff ? launch_small<__nv_bfloat16, float>(a, st) : launch_small<__nv_bfloat16, __nv_bfloat16>(a, st);
    if (in->dtype == DCB_F16) return ff ? launch_small<__half, float>(a, st) : launch_small<__half, __half>(a, st);
    return set_error(DCB_E_DTYPE, "splat_cluster: unsupported dtype %d", in->dtype);
}

}  // namespace dcb
