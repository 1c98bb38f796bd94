// splat_planar.cuh -- device code of the many-channel forward splat shared by splat_planar.cu (the step pipeline)
// and pyramid.cu (all scatter jobs of a conditioning pyramid in one launch). See splat_planar.cu for the design.
#pragma once
#include "dcb_common.cuh"

namespace dcb {

#ifndef DCB_PTHREADS
#define DCB_PTHREADS 32
#endif
#ifndef DCB_PGROUP_MB
#define DCB_PGROUP_MB 34
#endif
#ifndef DCB_PMINCTAS
#define DCB_PMINCTAS 24
#endif
constexpr int kPThreads = DCB_PTHREADS;
constexpr int kPWarps = kPThreads / 32;
constexpr int kPRows = 4;                         // strip: 32 columns x 4 rows
constexpr int kPChunk = 128;                      // normalise item: 128 target pixels (4 per lane)
constexpr long long kPGroupBytes = (long long)DCB_PGROUP_MB << 20;    // accumulator bytes per ring slot


struct PlanarArgs {
    View in, flow, metric, mask;
    float* acc;              // channel quads: 2 slots x G frames x Cq x HW float4
    float* dacc;             // normaliser planes: 3 slots x G frames x HW floats (read by several warps, re-zeroed one step later)
    void* out;               // [N,C,H,W]
    void* norm;              // [N,1,H,W] fp32 or null
    int N, C, Cq, H, W;      // Cq = ceil(C / 4) channel quads
    unsigned HW;
    int mode, eps;
    int G;
    int tiles_x, ts, tn;
    int cg_s, ncg_s;         // scatter: channel quads per item, items per strip
    int cg_n, ncg_n;         // normalise: channel quads per item, items per chunk
    int tz;                  // re-zero items per frame (1024 normaliser cells each)
    int step;                // pipeline step k: scatter group k, normalise group k-1, re-zero normaliser slot (k+1) % 3
    int s_frame0, s_frames, n_frame0, n_frames;
    int ones;                // the metric is all-ones and not materialised (compute_mask, warpers without metric_net)
    int vec_in;              // channels-last input (stride[1] == 1, C % 4 == 0, 16-byte aligned quads): one vector load per quad
    unsigned* bar;           // single-launch kernel (k_planar_one): arrive / depart counters in the workspace, zero between calls
};

// the four channels of a quad of a channels-last (NHWC) tensor in one load: 16 bytes fp32, 8 bytes bf16 / fp16
__device__ __forceinline__ void ld_quad(const float* p, float (&o)[4]) {
    const float4 t = __ldcs((const float4*)p);
    o[0] = t.x; o[1] = t.y; o[2] = t.z; o[3] = t.w;
}
__device__ __forceinline__ void ld_quad(const __nv_bfloat16* p, float (&o)[4]) {
    const uint2 u = __ldcs((const uint2*)p);
    o[0] = __uint_as_float(u.x << 16); o[1] = __uint_as_float(u.x & 0xffff0000u);
    o[2] = __uint_as_float(u.y << 16); o[3] = __uint_as_float(u.y & 0xffff0000u);
}
__device__ __forceinline__ void ld_quad(const __half* p, float (&o)[4]) {
    const uint2 u = __ldcs((const uint2*)p);
    const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&u.x)), hi = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
    o[0] = lo.x; o[1] = lo.y; o[2] = hi.x; o[3] = hi.y;
}

// host: can `in` ([N,C,H,W] view) be read quad-wise?
inline bool planar_vec_ok(const DcbTensor* in) {
    const long long es = elem_size(in->dtype);
    if (in->dtype != DCB_F32 && !is_half_storage(in->dtype)) return false;
    if (in->stride[1] != 1 || in->size[1] % 4 != 0 || in->size[1] < 4) return false;
    if (((uintptr_t)in->ptr) % (uintptr_t)(4 * es)) return false;
    return in->stride[0] % 4 == 0 && in->stride[2] % 4 == 0 && in->stride[3] % 4 == 0;
}

__device__ __forceinline__ void red1_if(bool p, float* addr, float v) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.s32 q, %0, 0;\n\t"
        "@q red.global.add.f32 [%1], %2;\n\t}"
        ::"r"((int)p), "l"(addr), "f"(v) : "memory");
}

__device__ __forceinline__ void red4p_if(bool p, float4* addr, const float (&v)[4]) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.s32 q, %0, 0;\n\t"
        "@q red.global.add.v4.f32 [%1], {%2, %3, %4, %5};\n\t}"
        ::"r"((int)p), "l"(addr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]) : "memory");
}

template <class T, class TF>
__device__ __forceinline__ void planar_scatter_strip(const PlanarArgs& a, int frame, int tile, int q_begin, int q_end,
                                                     bool with_weight, float* acc, float* dplane, int lane) {
    const int tx = tile % a.tiles_x, ty = tile / a.tiles_x;
    const int x = tx * 32 + lane, yb = ty * kPRows;
    const int W = a.W, H = a.H, C = a.C;
    const bool xin = x < W;
    const int rows = min(kPRows, H - yb);
    const unsigned full = 0xffffffffu;
    constexpr int kDead = -7;
    const int pitch = W + 2;
    const int xs = xin ? x : 0;

    // ---- footprints of the strip's 4 pixels per lane: computed once, reused for every channel ----
    float wnw[kPRows], wne[kPRows], wsw[kPRows], wse[kPRows], g[kPRows];
    int off[kPRows];
    bool take[kPRows], e_n[kPRows], e_s[kPRows], join[kPRows], n_ok[kPRows], flush_prev[kPRows];
    bool last_ok = false;
    int last_off = 0;
    {
        const TF* fbase = (const TF*)a.flow.p + frame * a.flow.sN + (long long)xs * a.flow.sW;
        const T* mbase = a.metric.p ? (const T*)a.metric.p + frame * a.metric.sN + (long long)xs * a.metric.sW : nullptr;
        int pend_key = kDead;
        bool pend_ok = false;
#pragma unroll
        for (int r = 0; r < kPRows; ++r) {
            const bool in_img = xin && r < rows;
            const long long y = yb + r;
            float flx = 0.f, fly = 0.f, m = 0.f;
            if (in_img) {
                const TF* fp = fbase + y * a.flow.sH;
                flx = ld_stream(fp); fly = ld_stream(fp + a.flow.sC);
                if (mbase) m = ld_stream(mbase + y * a.metric.sH);
            }
            const float fx = add_rn((float)x, flx), fy = add_rn((float)(yb + r), fly);       // softsplat.py:298-299
            const float x0f = floorf(fx), y0f = floorf(fy);
            const int x0 = __float2int_rz(x0f), y0 = __float2int_rz(y0f);
            const bool alive = in_img && fabsf(fx) < 3.0e38f && fabsf(fy) < 3.0e38f &&
                               ((unsigned)x0 + 1u) <= (unsigned)W && ((unsigned)y0 + 1u) <= (unsigned)H;
            const float ex = sub_rn(add_rn(x0f, 1.f), fx), ey = sub_rn(add_rn(y0f, 1.f), fy);  // softsplat.py:315-318
            const float dx = sub_rn(fx, x0f), dy = sub_rn(fy, y0f);
            wnw[r] = mul_rn(ex, ey); wne[r] = mul_rn(dx, ey); wsw[r] = mul_rn(ex, dy); wse[r] = mul_rn(dx, dy);
            // expf(1.0f) as a constant: what tenMetric.exp() yields for an all-ones metric
            g[r] = a.mode == DCB_MODE_SOFT ? (a.ones ? 2.7182817459106445f : expf(m)) : (a.mode == DCB_MODE_LINEAR ? (a.ones ? 1.f : m) : 1.f);
            const int key = alive ? (y0 + 1) * pitch + (x0 + 1) : kDead;
            off[r] = y0 * W + x0;
            const bool vx0 = x0 >= 0, vx1 = x0 < W - 1, vy0 = y0 >= 0, vy1 = y0 < H - 1;
            const int lkey = __shfl_up_sync(full, key, 1);
            take[r] = lane > 0 && alive && lkey != kDead && lkey + 1 == key;
            const bool given = (__shfl_down_sync(full, (int)take[r], 1) != 0) && lane < 31;
            const bool east = alive && !given && vx1;
            e_n[r] = east && vy0; e_s[r] = east && vy1;
            join[r] = pend_key == key && alive;
            flush_prev[r] = pend_ok && !join[r];
            n_ok[r] = alive && vx0 && vy0;
            pend_key = alive ? key + pitch : kDead;
            pend_ok = alive && vx0 && vy1;
        }
        last_ok = pend_ok;
        last_off = off[kPRows - 1] + W;
    }

    // ---- stream the channel quads through the footprints ----
    const T* ibase = (const T*)a.in.p + frame * a.in.sN + (long long)xs * a.in.sW + (long long)yb * a.in.sH;
    for (int q = q_begin; q < q_end; ++q) {
        float v[kPRows][4];
        if (a.vec_in) {                                      // warp-uniform: NHWC, the quad is contiguous
#pragma unroll
            for (int r = 0; r < kPRows; ++r) {
                v[r][0] = v[r][1] = v[r][2] = v[r][3] = 0.f;
                if (xin && r < rows) ld_quad(ibase + 4 * q + (long long)r * a.in.sH, v[r]);
            }
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = 4 * q + j;
                const T* ip = ibase + (long long)(c < C ? c : 0) * a.in.sC;
#pragma unroll
                for (int r = 0; r < kPRows; ++r) {
                    v[r][j] = 0.f;
                    if (c < C && xin && r < rows) v[r][j] = ld_stream(ip + (long long)r * a.in.sH);
                }
            }
        }
        float4* plane = (float4*)acc + (size_t)q * a.HW;
        float pend[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int r = 0; r < kPRows; ++r) {
            float nw[4], ne[4], sw[4], se[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float t = (a.mode >= DCB_MODE_LINEAR) ? mul_rn(v[r][j], g[r]) : v[r][j];        // softsplat.py:244,247
                nw[j] = mul_rn(t, wnw[r]); ne[j] = mul_rn(t, wne[r]); sw[j] = mul_rn(t, wsw[r]); se[j] = mul_rn(t, wse[r]);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float en = __shfl_up_sync(full, ne[j], 1), es = __shfl_up_sync(full, se[j], 1);
                nw[j] = take[r] ? add_rn(nw[j], en) : nw[j];
                sw[j] = take[r] ? add_rn(sw[j], es) : sw[j];
            }
            red4p_if(e_n[r], plane + off[r] + 1, ne);
            red4p_if(e_s[r], plane + off[r] + W + 1, se);
            if (r > 0) red4p_if(flush_prev[r], plane + off[r - 1] + W, pend);
#pragma unroll
            for (int j = 0; j < 4; ++j) nw[j] = join[r] ? add_rn(nw[j], pend[j]) : nw[j];
            red4p_if(n_ok[r], plane + off[r], nw);
#pragma unroll
            for (int j = 0; j < 4; ++j) pend[j] = sw[j];
        }
        red4p_if(last_ok, plane + last_off, pend);
    }
    // ---- the appended weight channel (1 | m | exp(m)): its own plane, scalar reds ----
    if (with_weight) {
        float pend = 0.f;
#pragma unroll
        for (int r = 0; r < kPRows; ++r) {
            float nw = mul_rn(g[r], wnw[r]), sw = mul_rn(g[r], wsw[r]);
            const float ne = mul_rn(g[r], wne[r]), se = mul_rn(g[r], wse[r]);
            const float en = __shfl_up_sync(full, ne, 1), es = __shfl_up_sync(full, se, 1);
            nw = take[r] ? add_rn(nw, en) : nw;
            sw = take[r] ? add_rn(sw, es) : sw;
            red1_if(e_n[r], dplane + off[r] + 1, ne);
            red1_if(e_s[r], dplane + off[r] + W + 1, se);
            if (r > 0) red1_if(flush_prev[r], dplane + off[r - 1] + W, pend);
            nw = join[r] ? add_rn(nw, pend) : nw;
            red1_if(n_ok[r], dplane + off[r], nw);
            pend = sw;
        }
        red1_if(last_ok, dplane + last_off, pend);
    }
}

}  // namespace dcb
