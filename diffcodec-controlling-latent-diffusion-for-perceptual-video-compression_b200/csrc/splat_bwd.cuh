// splat_bwd.cuh -- the source-side gather of the splat backward (K3b, see splat_bwd.cu for the closed form), shared by
// k_bwd_source (splat_bwd.cu) and the pyramid backward (pyramid_bwd.cu).
#pragma once
#include "dcb_common.cuh"

namespace dcb {

struct BwdArgs {
    View gout, in, flow, metric, mask;
    const void* out;     // [N,C,H,W] contiguous (forward output)
    const void* norm;    // [N,1,H,W] accumulator-typed (forward normaliser)
    void* tscal;         // workspace: [N*H*W][2] accumulator-typed (a, T)
    void* gin;           // [N,C,H,W] contiguous or null
    void* gflow;         // [N,2,H,W] contiguous or null
    void* gmetric;       // [N,1,H,W] contiguous or null
    unsigned total, HW;
    int N, C, H, W;
    int mode, eps;
    int px, cs;          // block shape
    unsigned pf_dist;    // source pass: L2 prefetch distance in CTAs (one wave)
    unsigned tiles_x, tiles;   // packed source pass: 32 x 8 pixel tiles per row / per frame
    unsigned pf_rows;          // packed source pass: prefetch distance in tile rows
};

#ifndef DCB_BS_PF
#define DCB_BS_PF 1
#endif
// K3b -- source-side gather. blockDim = (px, cs): px source pixels, cs channel slices per pixel.
// Loads are unconditional from always-valid addresses (an out-of-range corner reads element 0 of
// its plane and is then zeroed by a select): no branches in the channel loop, 3 channels = 15
// loads in flight per thread.
#ifndef DCB_BS_U
#define DCB_BS_U 3           // channels in flight per thread (5 loads each); 64 registers -> 4 CTAs per SM (measured best of 1..6)
#endif
#ifndef DCB_BS_MINCTAS
#define DCB_BS_MINCTAS 4
#endif
// IX: type of the element offsets inside one gradOut plane (int when they fit 31 bits: one
// IMAD.WIDE per load instead of a 64-bit multiply-add chain).
// The body is shared with the pyramid backward (pyramid_bwd.cu), which runs one such pass per (level, direction) inside one
// launch: `bx` / `tx` / `ty` are the CTA and thread coordinates inside the pass. PYR = true adds what only the pyramid needs,
// and compiles to nothing for k_bwd_source: a NULL metric is the all-ones metric (g = exp(1)), and `gadd` (F32 [N*H*W] or
// null) is added to the metric gradient before its single store (the fusion-confidence term of the same pixel).
template <class T, class TF, class IX, bool PYR>
__device__ __forceinline__ void bwd_source_body(const BwdArgs& a, unsigned bx, int tx, int ty, void* smem, const float* gadd) {
    using A = typename Acc<T>::type;
    A* red = (A*)smem;                                            // [cs][px][4] when cs > 1

#if DCB_BS_PF
    if (a.cs == 1) {
        // L2 prefetch of the rows the CTA one wave ahead will stream (flow, metric, and up to 8 channels of
        // `in` and gradOut at the zero-flow position): one 128-byte line per thread
        const unsigned q0 = (bx + a.pf_dist) * 256u;
        if (q0 < a.total) {
            const unsigned qn = q0 / a.HW, qr = q0 - qn * a.HW;
            const int qy = (int)(qr / (unsigned)a.W), qx = (int)(qr - (unsigned)qy * (unsigned)a.W);
            const int line = tx & 7, plane = tx >> 3;                      // 8 lines of 32 pixels, 32 planes
            const int cmax = a.C < 8 ? a.C : 8;
            const int px = qx + line * 32;
            if (px < a.W) {
                const void* q = nullptr;
                if (plane < 2) q = (const TF*)a.flow.p + qn * a.flow.sN + plane * a.flow.sC + qy * a.flow.sH + px * a.flow.sW;
                else if (plane == 2 && a.metric.p) q = (const T*)a.metric.p + qn * a.metric.sN + qy * a.metric.sH + px * a.metric.sW;
                else if (plane >= 8 && plane < 8 + cmax) q = (const T*)a.in.p + qn * a.in.sN + (plane - 8) * a.in.sC + qy * a.in.sH + px * a.in.sW;
                else if (plane >= 16 && plane < 16 + cmax) q = (const T*)a.gout.p + qn * a.gout.sN + (plane - 16) * a.gout.sC + qy * a.gout.sH + px * a.gout.sW;
                if (q) asm volatile("prefetch.global.L2 [%0];" ::"l"(q));
            }
        }
    }
#endif
    const unsigned p = bx * a.px + tx;
    const bool live = p < a.total;
    const unsigned pc = live ? p : 0;
    const unsigned n = pc / a.HW, r = pc - n * a.HW;
    const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
    const int W = a.W, H = a.H;
    const bool normalised = a.mode != DCB_MODE_SUM;

    const TF* fp = (const TF*)a.flow.p + n * a.flow.sN + y * a.flow.sH + x * a.flow.sW;
    const Foot<A> f = make_foot<A>(x, y, ld<A>(fp), ld<A>(fp + a.flow.sC));
    const int x1 = (int)((unsigned)f.x0 + 1u), y1 = (int)((unsigned)f.y0 + 1u);
    const bool vx0 = (unsigned)f.x0 < (unsigned)W, vx1 = (unsigned)x1 < (unsigned)W;
    const bool vy0 = (unsigned)f.y0 < (unsigned)H, vy1 = (unsigned)y1 < (unsigned)H;
    const bool ok = live && f.finite;                             // softsplat.py:389-390, 460-461
    const bool b[4] = {ok && vx0 && vy0, ok && vx1 && vy0, ok && vx0 && vy1, ok && vx1 && vy1};
    const bool any = b[0] || b[1] || b[2] || b[3];
    const A w[4] = {f.wnw, f.wne, f.wsw, f.wse};
    // gradOut element offsets of the four corners inside one (n, c) plane; 0 when out of range
    IX go[4];
    {
        const IX sH = (IX)a.gout.sH, sW = (IX)a.gout.sW;
        const IX o0 = (IX)f.y0 * sH + (IX)f.x0 * sW;              // only used when the corner is in range
        go[0] = b[0] ? o0 : (IX)0;
        go[1] = b[1] ? o0 + sW : (IX)0;
        go[2] = b[2] ? o0 + sH : (IX)0;
        go[3] = b[3] ? o0 + sH + sW : (IX)0;
    }

    A g = (A)1, gprime = (A)1;
    if (PYR && !a.metric.p) {
        g = gprime = (A)2.7182817459106445f;                      // expf(1.0f), as the forward's all-ones metric (splat_planar.cuh)
    } else if (a.mode == DCB_MODE_LINEAR || a.mode == DCB_MODE_SOFT) {
        const T* mp = (const T*)a.metric.p + n * a.metric.sN + y * a.metric.sH + x * a.metric.sW;
        const A m = ld<A>(mp);
        g = a.mode == DCB_MODE_SOFT ? exp_t(m) : m;
        gprime = a.mode == DCB_MODE_SOFT ? g : (A)1;
    }

    A ak[4] = {(A)1, (A)1, (A)1, (A)1}, tk[4] = {(A)0, (A)0, (A)0, (A)0};
    if (normalised) {
        const A* ts = (const A*)a.tscal + 2ll * ((long long)n * a.HW + (long long)f.y0 * W + f.x0);
        const long long to[4] = {0, 2, 2ll * W, 2ll * W + 2};
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (b[k]) { ak[k] = ts[to[k]]; tk[k] = ts[to[k] + 1]; }
    }
    A wa[4];                                                      // weight * (1 - mask) / D, 0 for dropped corners
#pragma unroll
    for (int k = 0; k < 4; ++k) wa[k] = b[k] ? w[k] * ak[k] : (A)0;

    const bool need_A = (a.gflow != nullptr) || (a.gmetric != nullptr);
    // moving plane pointers: one 64-bit add per channel, corner loads are base + 32-bit offset
    const long long gstep = (long long)a.cs * a.gout.sC, istep = (long long)a.cs * a.in.sC, ostep = (long long)a.cs * a.HW;
    const T* gc = (const T*)a.gout.p + n * a.gout.sN + (long long)ty * a.gout.sC;
    const T* ic = (const T*)a.in.p + n * a.in.sN + y * a.in.sH + x * a.in.sW + (long long)ty * a.in.sC;
    T* gi = (a.gin && live) ? (T*)a.gin + (long long)n * a.C * a.HW + r + (long long)ty * a.HW : nullptr;

    A Ak[4] = {(A)0, (A)0, (A)0, (A)0};
    constexpr int U = DCB_BS_U;
    int c = ty;
    for (; c + (U - 1) * a.cs < a.C; c += U * a.cs) {
        A gk[U][4], v[U];
        const T* gcj = gc;
        const T* icj = ic;
#pragma unroll
        for (int j = 0; j < U; ++j, gcj += gstep, icj += istep) {
#pragma unroll
            for (int k = 0; k < 4; ++k) gk[j][k] = ld<A>(gcj + go[k]);
            v[j] = need_A ? ld<A>(icj) : (A)0;
        }
        gc = gcj; ic = icj;
#pragma unroll
        for (int j = 0; j < U; ++j) {
#pragma unroll
            for (int k = 0; k < 4; ++k) gk[j][k] = b[k] ? gk[j][k] : (A)0;
            if (gi) {
                A s = (A)0;
#pragma unroll
                for (int k = 0; k < 4; ++k) s = fma_rn(gk[j][k], wa[k], s);
                st<T, A>(gi, s * g);
                gi += ostep;
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) Ak[k] = fma_rn(gk[j][k], v[j], Ak[k]);
        }
    }
    for (; c < a.C; c += a.cs, gc += gstep, ic += istep) {
        A gk[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { gk[k] = ld<A>(gc + go[k]); gk[k] = b[k] ? gk[k] : (A)0; }
        if (gi) {
            A s = (A)0;
#pragma unroll
            for (int k = 0; k < 4; ++k) s = fma_rn(gk[k], wa[k], s);
            st<T, A>(gi, s * g);
            gi += ostep;
        }
        if (need_A) {
            const A v = ld<A>(ic);
#pragma unroll
            for (int k = 0; k < 4; ++k) Ak[k] = fma_rn(gk[k], v, Ak[k]);
        }
    }
    if (!need_A) return;

    if (a.cs > 1) {                                               // reduce A_k over the channel slices
        A* mine = red + ((size_t)ty * a.px + tx) * 4;
#pragma unroll
        for (int k = 0; k < 4; ++k) mine[k] = Ak[k];
        __syncthreads();
        if (ty != 0) return;
        for (int s = 1; s < a.cs; ++s) {
            const A* o = red + ((size_t)s * a.px + tx) * 4;
#pragma unroll
            for (int k = 0; k < 4; ++k) Ak[k] += o[k];
        }
    }
    if (!live) return;

    A B[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) B[k] = b[k] ? (normalised ? fma_rn(ak[k], Ak[k], tk[k]) : Ak[k]) : (A)0;

    if (a.gmetric) {
        A s = (A)0;
#pragma unroll
        for (int k = 0; k < 4; ++k) if (b[k]) s = fma_rn(w[k], B[k], s);
        A gm = any ? s * gprime : (A)0;
        if (PYR && gadd) gm += (A)gadd[p];
        st<T, A>((T*)a.gmetric + p, gm);
    }
    if (a.gflow) {
        // d w / d flow, softsplat.py:477-487
        const A ey = sub_rn((A)y1, f.fy), dy = sub_rn(f.fy, (A)f.y0);
        const A ex = sub_rn((A)x1, f.fx), dx = sub_rn(f.fx, (A)f.x0);
        A gx = (B[1] - B[0]) * ey + (B[3] - B[2]) * dy;
        A gy = (B[2] - B[0]) * ex + (B[3] - B[1]) * dx;
        if (!any) { gx = (A)0; gy = (A)0; }                       // a huge finite flow gives inf weights with no corner in range
        TF* gf = (TF*)a.gflow + (long long)n * 2 * a.HW + r;      // gradFlow has the dtype of the flow tensor
        st<TF, A>(gf, gx * g);
        st<TF, A>(gf + a.HW, gy * g);
    }
}

}  // namespace dcb
