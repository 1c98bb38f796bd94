// splat_pipe.cu -- the forward splat for C+1 <= 4 channels (frames, flows, SD latents) as a
// software pipeline of plain, synchronisation-free kernels (sm_100a).
//
// Why (measured on B200, profiles/r01/, profiles/r02/): an L2 reduction occupies its slice for ~2.4 clocks per 32-byte
// sector-op whether it carries one 16-byte cell or two (~150 G sector-ops/s over the chip), so the reference's 4 corner
// adds per pixel (~3 sector-ops/px on realistic flow) cap a scatter at ~50 Gpx/s; fp32 accumulators that round-trip through HBM
// triple the DRAM traffic (only ~1.5 frames of 1080p accumulators stay L2-resident next to the
// streaming inputs). Two persistent-kernel variants (CTA-granular with TMA-staged tiles, and
// warp-granular with global tickets) were built and measured first: their in-kernel dependency
// tracking (gpu-scope fences, acquire polling, bar.sync) cost more than it saved
// (profiles/r01/NOTES.md). What survived:
//
//  1. the KERNEL BOUNDARY is the only synchronisation: a frame group is scattered by one launch (k_splat_step) and
//     normalised by the next (k_splat_epilogue), chained by programmatic dependent launch; the in-order stream gives
//     "normalise(g) after all of scatter(g)" and "scatter(g+1) after all of normalise(g)" for free. (Round 1 ran
//     normalise(g-1) and scatter(g) in ONE launch on a ring of two slots: dcb_set_option("pipe_ring_slots", 2).)
//  2. the fp32 accumulators stay L2-RESIDENT: ONE slot of one frame group (a group is ~32 MB: one 1080p frame, or dozens
//     of latents), re-zeroed by the normalise pass that reads it, so there is no memset and no accumulator traffic to
//     HBM (measured: the scatter launch reads exactly the compulsory bytes, profiles/r02/ncu_step_slots.txt; two slots
//     did not stay resident next to the streaming inputs and outputs);
//  3. one 16-byte `red.global.add.v4.f32` per corner carries all C+1 channels, and corner pieces
//     are merged IN REGISTERS before they reach L2: the east column of lane i is handed to lane
//     i+1 by shuffle when their footprints abut, the south row of a pixel is carried to the next
//     row of the same thread when they abut vertically (~1.2 reds per pixel instead of 4 on smooth
//     flow; any flow stays correct -- an unmatched piece is simply issued alone);
//  4. all loads of 4 rows are in flight before the first use; the pre-op (1 | m | exp(m), in*g)
//     and the post-op (eps rule, divide, (1 - mask), cast, saved normaliser) never touch memory;
//  5. epilogues besides the normalise: the occlusion test of compute_mask, and the conditioning recipe's second pass
//     (KIND = 1: a 2-channel rider scattered with the same footprints into float2 cells, one epilogue that normalises,
//     tests occlusion, fuses and subtracts) -- two pixels per lane with 256-bit cell loads where the layout allows; the
//     two-reference recipe runs the same rider scatter twice (KIND = 2, 3: bidir_chunk epilogues).
//  What bounds it (DESIGN.md section 4.1): the scatter launch's time is its reduction sector-ops x ~2.4 L2 slice clocks.
//
// Replaces controlnet/softsplat.py:240-270 (pre/post ops) + :281-345 (zero-init + softsplat_out).
#include "dcb_common.cuh"

#include <stdlib.h>

namespace dcb {

constexpr int kPipeThreads = 32;            // one warp per CTA: the item index is blockIdx-uniform, so every shuffle is provably convergent
constexpr int kWarpsPerCta = kPipeThreads / 32;
#ifndef DCB_KROWS
#define DCB_KROWS 4
#endif
#ifndef DCB_NORM_V
#define DCB_NORM_V 2         // normalise stage: 0 = one pixel per lane (any layout), 2 = two pixels per lane with 256-bit accesses, 4 = four
#endif
#ifndef DCB_KPASSES
#define DCB_KPASSES 2
#endif
#ifndef DCB_MINCTAS
#define DCB_MINCTAS 32
#endif
constexpr int kRows = DCB_KROWS;            // rows loaded at once by a warp
constexpr int kPasses = DCB_KPASSES;        // consecutive row groups per strip (the vertical carry spans them)
constexpr int kMinCtas = DCB_MINCTAS;       // register budget: 64 per thread -> 32 warps per SM
constexpr int kMinCtasRecipe = 24;          // the recipe pass carries two more channels and a wider epilogue: 80 registers
constexpr int kStripH = kRows * kPasses;    // a scatter item: 32 columns x 16 rows
#ifndef DCB_NPER
#define DCB_NPER 8
#endif
#ifndef DCB_TAIL_PERCENT
#define DCB_TAIL_PERCENT 0
#endif
#ifndef DCB_NBATCH
#define DCB_NBATCH (DCB_KROWS * DCB_KPASSES / DCB_NPER)
#endif
constexpr int kNPer = DCB_NPER;             // normalise: pixels per lane per batch
constexpr int kNBatches = DCB_NBATCH;
static_assert(kNBatches >= 1 && kNPer % 4 == 0, "a normalise item covers the pixels of one scatter strip");
constexpr int kChunk = 32 * kNPer * kNBatches;   // a normalise item: 512 target pixels
constexpr float kExp1 = 2.7182817459106445f;     // expf(1.0f): what tenMetric.exp() yields for an all-ones metric
constexpr long long kGroupBytes = 34ll << 20;    // accumulator bytes per ring slot (one 1080p frame = 31.6 MiB)

struct PipeArgs {
    View in, flow, metric, mask;
    float* acc;              // 2 slots x G frames x HW x 4 floats, all-zero on entry and on exit
    void* out;               // [N,C,H,W]
    void* norm;              // [N,1,H,W] fp32 or null
    int N, C, H, W;
    unsigned HW;
    int eps;
    int G;                   // frames per group (per accumulator slot)
    int tiles_x, tiles_y, ts, tn;   // scatter strips per row / per column / per frame, normalise chunks per frame
    int s_frame0, s_frames;  // this step scatters frames [s_frame0, s_frame0 + s_frames)
    int n_frame0, n_frames;  // ... and normalises frames [n_frame0, n_frame0 + n_frames)
    View epi_flow;           // epilogue 1 (occlusion mask): the motion field compared with the splatted one
    void* mask_out;          // epilogue 1: [N,1,H,W] in T
    int epi;                 // 0 = normalise (softsplat), 1 = occlusion mask (control_utils.py:15-16)
    int ones;                // metric is all-ones and not materialised (compute_mask, dataset wrappers)
    float* acc_s;            // accumulator slot of the frame group this launch scatters (frame s_frame0 at offset 0)
    float* acc_n;            // ... and of the group it normalises
    int vec4;                // H*W % 4 == 0 and out / norm 16-byte aligned: the normalise stage works on 4 pixels per lane
    int ny_big;              // strip rows of full height (kStripH); the rows below them are single-pass strips (kRows)
    // conditioning recipe (recipe_pipe_impl): a 2-channel RIDER splatted by the same flow with the same weights, and the
    // tensors of the two recipe epilogues (epi 2, 3)
    View in2;                // rider input [N,2,H,W] (flow2 riding on flow1)
    float* acc2_s;           // rider accumulators of the group this launch scatters: float2 cells [frame][HW]
    float* acc2_n;           // ... and of the group it normalises
    View gt;                 // epi 3: ground truth
    void* residual;          // epi 3: [N,C,H,W]
    const void* occ_other;   // epi 3: the occlusion plane computed by epi 2, [N,1,H,W] in T
    int variant;             // epi 3: DCB_RECIPE_*
    int flat2;               // epi 1, 3: two-pixel epilogue (even H*W; the tensors it reads are plain contiguous planes, pair-aligned)
};

// ---------------------------------------------------------------------------------------------
// scatter of one 32 x (kRows * kPasses) strip.  CA = accumulated channels (C, or C + 1 with the
// appended weight channel) is a template parameter: no per-channel runtime tests in the hot loop.
// ---------------------------------------------------------------------------------------------
// predicated vector reduction: no branch, the address is formed unconditionally but only used if p
__device__ __forceinline__ void red4_if(bool p, float* acc, int off, const float (&v)[4]) {
    float* addr = acc + (long long)off * 4;
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.s32 q, %0, 0;\n\t"
        "@q red.global.add.v4.f32 [%1], {%2, %3, %4, %5};\n\t}"
        ::"r"((int)p), "l"(addr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]) : "memory");
}

__device__ __forceinline__ void red2_if(bool p, float* acc2, int off, const float (&v)[2]) {
    float* addr = acc2 + (long long)off * 2;
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.s32 q, %0, 0;\n\t"
        "@q red.global.add.v2.f32 [%1], {%2, %3};\n\t}"
        ::"r"((int)p), "l"(addr), "f"(v[0]), "f"(v[1]) : "memory");
}

// RIDER: two more channels (a.in2) ride on the same footprints into float2 cells (acc2): the conditioning recipe splats
// image1 AND flow2 by flow1 with the same all-ones metric, so flow, weights, merge decisions and the weight channel are shared
template <class T, class TF, int MODE, int CA, bool RIDER>
__device__ __forceinline__ void scatter_strip(const PipeArgs& a, int frame, int tx, int y_first, int passes, float* acc, float* acc2, int lane) {
    constexpr int C = CA - (MODE != DCB_MODE_SUM ? 1 : 0);
    const int x = tx * 32 + lane;
    const int W = a.W, H = a.H;
    const bool xin = x < W;
    const unsigned full = 0xffffffffu;
    constexpr int kDead = -7;
    const int pitch = W + 2;                       // key = (y0 + 1) * pitch + (x0 + 1) identifies a footprint

    float pend[4] = {0.f, 0.f, 0.f, 0.f};
    float pend2[2] = {0.f, 0.f};
    int pend_key = kDead, pend_off = 0;
    bool pend_ok = false;
    // The diagonal joins / hand-overs below cost ~35 instructions per pixel and only pay where neighbouring footprints often
    // fail to abut (rough flow: the launch is bound by reduction sector-ops). `rough_pass` (warp-uniform, per group of kRows
    // rows) selects them when the flow of the group's first row jumps by more than a quarter pixel between at least
    // kRoughLanes neighbouring lanes; smooth flow runs the plain form (abutting footprints only) and never pays for them.
    constexpr int kRoughLanes = 5;

    const int xs = xin ? x : 0;
    const TF* fbase = (const TF*)a.flow.p + frame * a.flow.sN;
    const T* ibase = (const T*)a.in.p + frame * a.in.sN;
    const T* mbase = (MODE >= DCB_MODE_LINEAR && !a.ones) ? (const T*)a.metric.p + frame * a.metric.sN : nullptr;
    // element offsets fit 32 bits (checked by the host)
    const int f_sH = (int)a.flow.sH, f_sC = (int)a.flow.sC, i_sH = (int)a.in.sH, i_sC = (int)a.in.sC, m_sH = (int)a.metric.sH;
    const int f_x = xs * (int)a.flow.sW, i_x = xs * (int)a.in.sW, m_x = xs * (int)a.metric.sW;
    const TF* rbase = RIDER ? (const TF*)a.in2.p + frame * a.in2.sN : nullptr;
    const int r_sH = (int)a.in2.sH, r_sC = (int)a.in2.sC, r_x = xs * (int)a.in2.sW;

#pragma unroll 1
    for (int pass = 0; pass < passes; ++pass) {
        const int yb = y_first + pass * kRows;
        if (yb >= H) break;                                              // warp-uniform
        const int rows = min(kRows, H - yb);
        // ---- every load of the pass in flight before the first use ----
        float flx[kRows], fly[kRows], mv[kRows], iv[kRows][C > 0 ? C : 1], rv[kRows][2];
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
            const bool on = xin && r < rows;
            const int y = yb + r;
            flx[r] = fly[r] = 0.f; mv[r] = 0.f;
            rv[r][0] = rv[r][1] = 0.f;
            if (RIDER && on) { const TF* rp = rbase + (y * r_sH + r_x); rv[r][0] = ld_stream(rp); rv[r][1] = ld_stream(rp + r_sC); }
#pragma unroll
            for (int c = 0; c < C; ++c) iv[r][c] = 0.f;
            if (on) {
                const TF* fp = fbase + (y * f_sH + f_x);
                flx[r] = ld_stream(fp); fly[r] = ld_stream(fp + f_sC);
                if (MODE >= DCB_MODE_LINEAR && !a.ones) mv[r] = ld_stream(mbase + (y * m_sH + m_x));
                const T* ip = ibase + (y * i_sH + i_x);
#pragma unroll
                for (int c = 0; c < C; ++c) iv[r][c] = ld_stream(ip + c * i_sC);
            }
        }
        bool rough_pass;
        {
            const float dfx = fabsf(flx[0] - __shfl_up_sync(full, flx[0], 1)), dfy = fabsf(fly[0] - __shfl_up_sync(full, fly[0], 1));
            rough_pass = __popc(__ballot_sync(full, lane > 0 && (dfx > 0.25f || dfy > 0.25f))) >= kRoughLanes;
        }
#pragma unroll
        for (int r = 0; r < kRows; ++r) {
            const bool in_img = xin && r < rows;
            const float fx = add_rn((float)x, flx[r]), fy = add_rn((float)(yb + r), fly[r]);   // softsplat.py:298-299
            const float x0f = floorf(fx), y0f = floorf(fy);
            const int x0 = __float2int_rz(x0f), y0 = __float2int_rz(y0f);
            // finite landing point (softsplat.py:301-302) with at least one corner inside the frame
            const bool alive = in_img && fabsf(fx) < 3.0e38f && fabsf(fy) < 3.0e38f &&
                               ((unsigned)x0 + 1u) <= (unsigned)W && ((unsigned)y0 + 1u) <= (unsigned)H;
            const float ex = sub_rn(add_rn(x0f, 1.f), fx), ey = sub_rn(add_rn(y0f, 1.f), fy);  // softsplat.py:315-318
            const float dx = sub_rn(fx, x0f), dy = sub_rn(fy, y0f);
            const float wnw = mul_rn(ex, ey), wne = mul_rn(dx, ey), wsw = mul_rn(ex, dy), wse = mul_rn(dx, dy);

            float g = 1.f;
            if (MODE == DCB_MODE_LINEAR) g = a.ones ? 1.f : mv[r];
            if (MODE == DCB_MODE_SOFT) g = a.ones ? kExp1 : expf(mv[r]);
            float nw[4] = {0.f, 0.f, 0.f, 0.f}, ne[4] = {0.f, 0.f, 0.f, 0.f}, sw[4] = {0.f, 0.f, 0.f, 0.f}, se[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int c = 0; c < CA; ++c) {
                float v;
                if (c < C) v = (MODE >= DCB_MODE_LINEAR) ? mul_rn(iv[r][c < C ? c : 0], g) : iv[r][c < C ? c : 0];   // softsplat.py:244,247
                else v = g;                                                                     // appended channel
                nw[c] = mul_rn(v, wnw); ne[c] = mul_rn(v, wne);
                sw[c] = mul_rn(v, wsw); se[c] = mul_rn(v, wse);
            }
            float nw2[2] = {0.f, 0.f}, ne2[2] = {0.f, 0.f}, sw2[2] = {0.f, 0.f}, se2[2] = {0.f, 0.f};
            if (RIDER) {
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    const float v = (MODE >= DCB_MODE_LINEAR) ? mul_rn(rv[r][c], g) : rv[r][c];
                    nw2[c] = mul_rn(v, wnw); ne2[c] = mul_rn(v, wne); sw2[c] = mul_rn(v, wsw); se2[c] = mul_rn(v, wse);
                }
            }
            const int key = alive ? (y0 + 1) * pitch + (x0 + 1) : kDead;
            const int off = y0 * W + x0;
            const bool vx0 = x0 >= 0, vx1 = x0 < W - 1, vy0 = y0 >= 0, vy1 = y0 < H - 1;

            if (rough_pass) {
                // ---- vertical carry (before the hand-over, whose shuffles must see it): the previous row's south-west piece
                // joins my NW piece if the footprints abut vertically, my NE piece if I sit one row down and one cell LEFT, my SW
                // piece if my footprint is the same one again (bench flow: 54 % / 9 % / 9 % of the row steps) ----
                const bool join = pend_key == key && alive;            // kDead never equals a live key
                const bool join_e = pend_key == key + 1 && alive;
                const bool join_s = pend_key == key + pitch && alive;   // the SAME footprint again: the piece stays my SW piece (carried on)
    #pragma unroll
                for (int c = 0; c < CA; ++c) nw[c] = join ? add_rn(nw[c], pend[c]) : nw[c];
                if (RIDER) {
    #pragma unroll
                    for (int c = 0; c < 2; ++c) nw2[c] = join ? add_rn(nw2[c], pend2[c]) : nw2[c];
                }
                // the two rarer joins sit behind a warp-uniform test: smooth flow (where they never fire) does not pay for them
                if (__any_sync(full, join_e || join_s)) {
    #pragma unroll
                    for (int c = 0; c < CA; ++c) {
                        ne[c] = join_e ? add_rn(ne[c], pend[c]) : ne[c];
                        sw[c] = join_s ? add_rn(sw[c], pend[c]) : sw[c];
                    }
                    if (RIDER) {
    #pragma unroll
                        for (int c = 0; c < 2; ++c) {
                            ne2[c] = join_e ? add_rn(ne2[c], pend2[c]) : ne2[c];
                            sw2[c] = join_s ? add_rn(sw2[c], pend2[c]) : sw2[c];
                        }
                    }
                }
                const bool lone = pend_ok && !join && !join_e && !join_s;
                red4_if(lone, acc, pend_off, pend);
                if (RIDER) red2_if(lone, acc2, pend_off, pend2);
                // ---- horizontal hand-over: my east pieces go to lane + 1 wherever they fall on its west column ----
                // footprints abut (lane + 1 sits one cell to the right, same row): NE -> its NW, SE -> its SW;
                // one to the right and one row DOWN: my SE is its NW; one to the right and one row UP: my NE is its SW
                // (bench flow: 53 % / 9 % / 9 % of the neighbour pairs). The shuffled values are the east pieces after the vertical
                // joins, and the hand-over only modifies west pieces, so chains of hand-overs need no ordering.
                // (the kernel is bound by L2 reduction sector-ops, not by issue slots: profiles/r02/NOTES.md)
                const int lkey = __shfl_up_sync(full, key, 1);
                const bool nb = lane > 0 && alive && lkey != kDead;
                const bool t_ab = nb && lkey + 1 == key, t_dn = nb && lkey + 1 + pitch == key, t_up = nb && lkey + 1 - pitch == key;
                const int took = (t_ab ? 3 : 0) | (t_up ? 1 : 0) | (t_dn ? 2 : 0);          // bit 0: the left lane's NE, bit 1: its SE
                const int right = __shfl_down_sync(full, took, 1);
                const int gone = lane < 31 ? right : 0;                                       // which of my east pieces the right lane took
                const bool diag = __any_sync(full, t_dn || t_up);
    #pragma unroll
                for (int c = 0; c < CA; ++c) {
                    const float en = __shfl_up_sync(full, ne[c], 1), es = __shfl_up_sync(full, se[c], 1);
                    nw[c] = t_ab ? add_rn(nw[c], en) : nw[c];
                    sw[c] = t_ab ? add_rn(sw[c], es) : sw[c];
                    if (diag) {
                        nw[c] = t_dn ? add_rn(nw[c], es) : nw[c];
                        sw[c] = t_up ? add_rn(sw[c], en) : sw[c];
                    }
                }
                if (RIDER) {
    #pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        const float en = __shfl_up_sync(full, ne2[c], 1), es = __shfl_up_sync(full, se2[c], 1);
                        nw2[c] = t_ab ? add_rn(nw2[c], en) : (t_dn ? add_rn(nw2[c], es) : nw2[c]);
                        sw2[c] = t_ab ? add_rn(sw2[c], es) : (t_up ? add_rn(sw2[c], en) : sw2[c]);
                    }
                }
                const bool east = alive && vx1;
                const bool e_n = east && vy0 && !(gone & 1), e_s = east && vy1 && !(gone & 2);
                red4_if(e_n, acc, off + 1, ne);
                red4_if(e_s, acc, off + W + 1, se);
                if (RIDER) { red2_if(e_n, acc2, off + 1, ne2); red2_if(e_s, acc2, off + W + 1, se2); }
                red4_if(alive && vx0 && vy0, acc, off, nw);
                if (RIDER) {
                    red2_if(alive && vx0 && vy0, acc2, off, nw2);
                    pend2[0] = sw2[0]; pend2[1] = sw2[1];
                }
            } else {
                // ---- horizontal hand-over: my east column goes to lane + 1 if our footprints abut ----
                // (the kernel is bound by L2 reduction sectors, not by issue slots: 12 shuffles per pixel
                //  buy ~20 % fewer sectors on rough flow and ~45 % on smooth flow -- profiles/r01/NOTES.md)
                const int lkey = __shfl_up_sync(full, key, 1);
                const bool take = lane > 0 && alive && lkey != kDead && lkey + 1 == key;
                const bool given = (__shfl_down_sync(full, (int)take, 1) != 0) && lane < 31;
    #pragma unroll
                for (int c = 0; c < CA; ++c) {
                    const float en = __shfl_up_sync(full, ne[c], 1), es = __shfl_up_sync(full, se[c], 1);
                    nw[c] = take ? add_rn(nw[c], en) : nw[c];
                    sw[c] = take ? add_rn(sw[c], es) : sw[c];
                }
                if (RIDER) {
    #pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        const float en = __shfl_up_sync(full, ne2[c], 1), es = __shfl_up_sync(full, se2[c], 1);
                        nw2[c] = take ? add_rn(nw2[c], en) : nw2[c];
                        sw2[c] = take ? add_rn(sw2[c], es) : sw2[c];
                    }
                }
                const bool east = alive && !given && vx1;
                red4_if(east && vy0, acc, off + 1, ne);
                red4_if(east && vy1, acc, off + W + 1, se);
                if (RIDER) { red2_if(east && vy0, acc2, off + 1, ne2); red2_if(east && vy1, acc2, off + W + 1, se2); }
                // ---- vertical carry: the previous row's south piece joins my north piece if they abut ----
                const bool join = pend_key == key && alive;            // kDead never equals a live key
    #pragma unroll
                for (int c = 0; c < CA; ++c) nw[c] = join ? add_rn(nw[c], pend[c]) : nw[c];
                red4_if(pend_ok && !join, acc, pend_off, pend);
                red4_if(alive && vx0 && vy0, acc, off, nw);
                if (RIDER) {
    #pragma unroll
                    for (int c = 0; c < 2; ++c) nw2[c] = join ? add_rn(nw2[c], pend2[c]) : nw2[c];
                    red2_if(pend_ok && !join, acc2, pend_off, pend2);
                    red2_if(alive && vx0 && vy0, acc2, off, nw2);
                    pend2[0] = sw2[0]; pend2[1] = sw2[1];
                }
            }
#pragma unroll
            for (int c = 0; c < CA; ++c) pend[c] = sw[c];
            pend_key = alive ? key + pitch : kDead;
            pend_off = off + W;
            pend_ok = alive && vx0 && vy1;
        }
    }
    red4_if(pend_ok, acc, pend_off, pend);
    if (RIDER) red2_if(pend_ok, acc2, pend_off, pend2);
}

// ---------------------------------------------------------------------------------------------
// normalise chunk: eps rule, divide, (1 - mask), cast, save normaliser, re-zero
// ---------------------------------------------------------------------------------------------
template <class T, int MODE, int CA>
__device__ __forceinline__ void normalize_chunk(const PipeArgs& a, int frame, int chunk, float* acc, int lane) {
    constexpr int C = CA - (MODE != DCB_MODE_SUM ? 1 : 0);
    T* out = (T*)a.out + (long long)frame * C * a.HW;
    const bool plain = a.norm == nullptr && a.mask.p == nullptr;        // warp-uniform
#pragma unroll 1
    for (int b = 0; b < kNBatches; ++b) {
        const unsigned base = (unsigned)chunk * kChunk + b * (32 * kNPer) + lane;
        if (base - lane >= a.HW) break;
        float4 s[kNPer];
#pragma unroll
        for (int i = 0; i < kNPer; ++i) {                                // all L2 reads in flight first
            const unsigned r = base + i * 32;
            s[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < a.HW) s[i] = __ldcg((const float4*)acc + r);         // written by other SMs' reds: L2 is the point of coherence
        }
#pragma unroll
        for (int i = 0; i < kNPer; ++i) {
            const unsigned r = base + i * 32;
            if (r < a.HW) {
                __stcg((float4*)acc + r, make_float4(0.f, 0.f, 0.f, 0.f));   // accumulators leave the kernel all-zero
                const float sv[4] = {s[i].x, s[i].y, s[i].z, s[i].w};
                float scale = 1.f;
                if (MODE != DCB_MODE_SUM) {
                    float d = sv[C];
                    // softsplat.py:256-266
                    if (a.eps == DCB_EPS_ADD) d = add_rn(d, 0.0000001f);
                    else if (a.eps == DCB_EPS_ZERO) d = (d == 0.f) ? 1.f : d;
                    else d = (d < 0.0000001f) ? 0.0000001f : d;
                    // one correctly-rounded reciprocal and C multiplies instead of C IEEE divisions
                    // (<= 1 ulp from softsplat.py:270; the deterministic path divides exactly)
                    scale = __frcp_rn(d);
                    if (!plain && a.norm) __stcs((float*)a.norm + (long long)frame * a.HW + r, d);
                }
                if (!plain && a.mask.p) {
                    const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
                    const T* mp = (const T*)a.mask.p + frame * a.mask.sN + (long long)y * a.mask.sH + (long long)x * a.mask.sW;
                    scale = mul_rn(scale, sub_rn(1.f, ld<float>(mp)));   // control_utils.py:69-70
                }
                T* o = out + r;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const float val = (MODE != DCB_MODE_SUM) ? mul_rn(sv[c], scale) : ((!plain && a.mask.p) ? mul_rn(sv[c], scale) : sv[c]);
                    st_stream(o + (size_t)c * a.HW, val);
                }
            }
        }
    }
}

// four consecutive pixels per lane: 128-bit accumulator loads, re-zero stores and output stores (one per channel
// for FOUR pixels instead of one per channel per pixel): 60 -> ~18 instructions per pixel
__device__ __forceinline__ void st_stream4(float* p, float a, float b, float c, float d) { __stcs((float4*)p, make_float4(a, b, c, d)); }
__device__ __forceinline__ void st_stream4(__nv_bfloat16* p, float a, float b, float c, float d) {
    const __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
    uint2 u; u.x = *reinterpret_cast<const unsigned*>(&lo); u.y = *reinterpret_cast<const unsigned*>(&hi);
    __stcs((uint2*)p, u);
}
__device__ __forceinline__ void st_stream4(__half* p, float a, float b, float c, float d) {
    const __half2 lo = __floats2half2_rn(a, b), hi = __floats2half2_rn(c, d);
    uint2 u; u.x = *reinterpret_cast<const unsigned*>(&lo); u.y = *reinterpret_cast<const unsigned*>(&hi);
    __stcs((uint2*)p, u);
}

template <class T, int MODE, int CA>
__device__ __forceinline__ void normalize_chunk_v4(const PipeArgs& a, int frame, int chunk, float* acc, int lane) {
    constexpr int C = CA - (MODE != DCB_MODE_SUM ? 1 : 0);
    constexpr int kGroups = kNPer / 4;                                   // groups of 4 pixels per lane per batch
    T* out = (T*)a.out + (long long)frame * C * a.HW;
    float* normp = a.norm ? (float*)a.norm + (long long)frame * a.HW : nullptr;
#pragma unroll 1
    for (int b = 0; b < kNBatches; ++b) {
        const unsigned base = (unsigned)chunk * kChunk + b * (32 * kNPer);
        if (base >= a.HW) break;
        float4 s[kGroups][4];
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {                              // all L2 reads in flight first
            const unsigned r = base + g * 128 + lane * 4;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                s[g][i] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (r < a.HW) s[g][i] = __ldcg((const float4*)acc + r + i);
            }
        }
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            const unsigned r = base + g * 128 + lane * 4;
            if (r < a.HW) {
                float scale[4], dn[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    __stcg((float4*)acc + r + i, make_float4(0.f, 0.f, 0.f, 0.f));   // accumulators leave the kernel all-zero
                    scale[i] = 1.f; dn[i] = 1.f;
                    if (MODE != DCB_MODE_SUM) {
                        float d = C == 0 ? s[g][i].x : (C == 1 ? s[g][i].y : (C == 2 ? s[g][i].z : s[g][i].w));
                        // softsplat.py:256-266
                        if (a.eps == DCB_EPS_ADD) d = add_rn(d, 0.0000001f);
                        else if (a.eps == DCB_EPS_ZERO) d = (d == 0.f) ? 1.f : d;
                        else d = (d < 0.0000001f) ? 0.0000001f : d;
                        scale[i] = __frcp_rn(d);
                        dn[i] = d;
                    }
                }
                if (MODE != DCB_MODE_SUM && normp) __stcs((float4*)(normp + r), make_float4(dn[0], dn[1], dn[2], dn[3]));
                if (C > 0) st_stream4(out + r, MODE != DCB_MODE_SUM ? mul_rn(s[g][0].x, scale[0]) : s[g][0].x, MODE != DCB_MODE_SUM ? mul_rn(s[g][1].x, scale[1]) : s[g][1].x,
                                      MODE != DCB_MODE_SUM ? mul_rn(s[g][2].x, scale[2]) : s[g][2].x, MODE != DCB_MODE_SUM ? mul_rn(s[g][3].x, scale[3]) : s[g][3].x);
                if (C > 1) st_stream4(out + (size_t)a.HW + r, MODE != DCB_MODE_SUM ? mul_rn(s[g][0].y, scale[0]) : s[g][0].y, MODE != DCB_MODE_SUM ? mul_rn(s[g][1].y, scale[1]) : s[g][1].y,
                                      MODE != DCB_MODE_SUM ? mul_rn(s[g][2].y, scale[2]) : s[g][2].y, MODE != DCB_MODE_SUM ? mul_rn(s[g][3].y, scale[3]) : s[g][3].y);
                if (C > 2) st_stream4(out + 2 * (size_t)a.HW + r, MODE != DCB_MODE_SUM ? mul_rn(s[g][0].z, scale[0]) : s[g][0].z, MODE != DCB_MODE_SUM ? mul_rn(s[g][1].z, scale[1]) : s[g][1].z,
                                      MODE != DCB_MODE_SUM ? mul_rn(s[g][2].z, scale[2]) : s[g][2].z, MODE != DCB_MODE_SUM ? mul_rn(s[g][3].z, scale[3]) : s[g][3].z);
                if (C > 3) st_stream4(out + 3 * (size_t)a.HW + r, s[g][0].w, s[g][1].w, s[g][2].w, s[g][3].w);      // SUM mode only
            }
        }
    }
}

// two consecutive pixels per lane: ONE 256-bit load fetches both accumulator cells (a full 32-byte sector per lane, the
// same L2 sectors per warp as the scalar layout), one 256-bit store re-zeroes them, one 64-bit store per channel
__device__ __forceinline__ void ld_cells2(const float* p, float4& a, float4& b) {
    asm volatile("ld.global.cg.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w) : "l"(p));
}
__device__ __forceinline__ void zero_cells2(float* p) {
    asm volatile("st.global.cg.v8.f32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1};" :: "l"(p), "f"(0.f) : "memory");
}
__device__ __forceinline__ void st_stream2(float* p, float a, float b) { __stcs((float2*)p, make_float2(a, b)); }
__device__ __forceinline__ void st_stream2(__nv_bfloat16* p, float a, float b) {
    const __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    __stcs((unsigned*)p, *reinterpret_cast<const unsigned*>(&v));
}
__device__ __forceinline__ void st_stream2(__half* p, float a, float b) {
    const __half2 v = __floats2half2_rn(a, b);
    __stcs((unsigned*)p, *reinterpret_cast<const unsigned*>(&v));
}
__device__ __forceinline__ float comp(const float4& v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w)); }

template <class T, int MODE, int CA>
__device__ __forceinline__ void normalize_chunk_v2(const PipeArgs& a, int frame, int chunk, float* acc, int lane) {
    constexpr int C = CA - (MODE != DCB_MODE_SUM ? 1 : 0);
    constexpr int kGroups = kNPer / 2;                                   // groups of 2 pixels per lane per batch
    T* out = (T*)a.out + (long long)frame * C * a.HW;
    float* normp = a.norm ? (float*)a.norm + (long long)frame * a.HW : nullptr;
#pragma unroll 1
    for (int b = 0; b < kNBatches; ++b) {
        const unsigned base = (unsigned)chunk * kChunk + b * (32 * kNPer);
        if (base >= a.HW) break;
        float4 s[kGroups][2];
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {                              // all L2 reads in flight first
            const unsigned r = base + g * 64 + lane * 2;
            s[g][0] = s[g][1] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < a.HW) ld_cells2(acc + (size_t)r * 4, s[g][0], s[g][1]);
        }
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            const unsigned r = base + g * 64 + lane * 2;
            if (r < a.HW) {
                zero_cells2(acc + (size_t)r * 4);                        // accumulators leave the kernel all-zero
                float scale[2] = {1.f, 1.f}, dn[2] = {1.f, 1.f};
                if (MODE != DCB_MODE_SUM) {
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        float d = comp(s[g][i], C);
                        // softsplat.py:256-266
                        if (a.eps == DCB_EPS_ADD) d = add_rn(d, 0.0000001f);
                        else if (a.eps == DCB_EPS_ZERO) d = (d == 0.f) ? 1.f : d;
                        else d = (d < 0.0000001f) ? 0.0000001f : d;
                        scale[i] = __frcp_rn(d);
                        dn[i] = d;
                    }
                    if (normp) __stcs((float2*)(normp + r), make_float2(dn[0], dn[1]));
                }
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const float v0 = comp(s[g][0], c), v1 = comp(s[g][1], c);
                    st_stream2(out + (size_t)c * a.HW + r, MODE != DCB_MODE_SUM ? mul_rn(v0, scale[0]) : v0, MODE != DCB_MODE_SUM ? mul_rn(v1, scale[1]) : v1);
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// occlusion epilogue (compute_mask, controlnet/control_utils.py:11-17): the accumulators hold the
// soft splat of a 2-channel flow (x*e, y*e, e); mask = (||motion + splat/(norm + 1e-7)||_2 > 0.3)
// ---------------------------------------------------------------------------------------------
// occlusion(): dcb_common.cuh

template <class T>
__device__ __forceinline__ void mask_chunk(const PipeArgs& a, int frame, int chunk, float* acc, int lane) {
    T* out = (T*)a.mask_out + (long long)frame * a.HW;
#pragma unroll 1
    for (int b = 0; b < kNBatches; ++b) {
        const unsigned base = (unsigned)chunk * kChunk + b * (32 * kNPer) + lane;
        if (base - lane >= a.HW) break;
        float4 s[kNPer];
#pragma unroll
        for (int i = 0; i < kNPer; ++i) {
            const unsigned r = base + i * 32;
            s[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < a.HW) s[i] = __ldcg((const float4*)acc + r);
        }
#pragma unroll
        for (int i = 0; i < kNPer; ++i) {
            const unsigned r = base + i * 32;
            if (r < a.HW) {
                __stcg((float4*)acc + r, make_float4(0.f, 0.f, 0.f, 0.f));
                const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
                const T* fp = (const T*)a.epi_flow.p + frame * a.epi_flow.sN + (long long)y * a.epi_flow.sH + (long long)x * a.epi_flow.sW;
                st<T, float>(out + r, occlusion(s[i].x, s[i].y, s[i].z, ld<float>(fp), ld<float>(fp + a.epi_flow.sC)));
            }
        }
    }
}

// two consecutive pixels per lane (a.flat2: even H*W, the compared flow is a plain [N,2,H,W] plane pair whose pixel pairs are
// aligned): one 256-bit accumulator load, one 64-bit load per flow plane, one paired store -- and no row / column arithmetic
template <class T>
__device__ __forceinline__ void mask_chunk_v2(const PipeArgs& a, int frame, int chunk, float* acc, int lane) {
    constexpr int kGroups = 2;                                            // 4 pixels per lane in flight (register budget of the step kernel)
    T* out = (T*)a.mask_out + (long long)frame * a.HW;
    const T* fbase = (const T*)a.epi_flow.p + frame * a.epi_flow.sN;
#pragma unroll 1
    for (int b = 0; b < kChunk / (64 * kGroups); ++b) {
        const unsigned base = (unsigned)chunk * kChunk + b * (64 * kGroups);
        if (base >= a.HW) break;
        float4 s[kGroups][2]; float2 mx[kGroups], my[kGroups];
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            const unsigned r = base + g * 64 + lane * 2;
            s[g][0] = s[g][1] = make_float4(0.f, 0.f, 0.f, 0.f); mx[g] = my[g] = make_float2(0.f, 0.f);
            if (r < a.HW) {
                ld_cells2(acc + (size_t)r * 4, s[g][0], s[g][1]);
                mx[g] = ld2_stream(fbase + r); my[g] = ld2_stream(fbase + a.epi_flow.sC + r);
            }
        }
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            const unsigned r = base + g * 64 + lane * 2;
            if (r < a.HW) {
                zero_cells2(acc + (size_t)r * 4);
                st_stream2(out + r, occlusion(s[g][0].x, s[g][0].y, s[g][0].z, mx[g].x, my[g].x),
                           occlusion(s[g][1].x, s[g][1].y, s[g][1].z, mx[g].y, my[g].y));
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// conditioning-recipe epilogue (dataset.py:233-265, residual_utils.py:159-199): the float4 cells hold the soft splat of
// image1 by flow1 (C channels + weight), the float2 cells the soft splat of flow2 by the same flow1 (the weight is shared).
// One pass per target pixel: warped = S / (D + 1e-7); occ_bwd = compute_mask(flow2, flow1); fusion weights from occ_fwd
// (computed by the pass before) and occ_bwd; optional double-hole fill; fused and residual = gt - fused stored once.
// ---------------------------------------------------------------------------------------------
constexpr int kRPer = 4;                          // pixels per lane in flight
template <class T, int CA>
__device__ __forceinline__ void recipe_chunk(const PipeArgs& a, int frame, int chunk, float* acc, float* acc2, int lane) {
    constexpr int C = CA - 1;
    T* fo = (T*)a.out + (long long)frame * C * a.HW;
    T* ro = (T*)a.residual + (long long)frame * C * a.HW;
    const T* oo = (const T*)a.occ_other + (long long)frame * a.HW;
    T* mo = a.mask_out ? (T*)a.mask_out + (long long)frame * a.HW : nullptr;
    const T* fbase = (const T*)a.epi_flow.p + frame * a.epi_flow.sN;
    const T* gbase = (const T*)a.gt.p + frame * a.gt.sN;
#pragma unroll 1
    for (int b = 0; b < kChunk / (32 * kRPer); ++b) {
        const unsigned base = (unsigned)chunk * kChunk + b * (32 * kRPer) + lane;
        if (base - lane >= a.HW) break;
        float4 s[kRPer]; float2 q[kRPer]; float mx[kRPer], my[kRPer], of[kRPer], gv[kRPer][C > 0 ? C : 1];
#pragma unroll
        for (int i = 0; i < kRPer; ++i) {                                // every load of the batch in flight first
            const unsigned r = base + i * 32;
            s[i] = make_float4(0.f, 0.f, 0.f, 0.f); q[i] = make_float2(0.f, 0.f);
            mx[i] = my[i] = of[i] = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) gv[i][c] = 0.f;
            if (r < a.HW) {
                s[i] = __ldcg((const float4*)acc + r);
                q[i] = __ldcg((const float2*)acc2 + r);
                const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
                const T* fp = fbase + (long long)y * a.epi_flow.sH + (long long)x * a.epi_flow.sW;
                mx[i] = ld<float>(fp); my[i] = ld<float>(fp + a.epi_flow.sC);
                of[i] = ld_stream(oo + r);
                const T* gp = gbase + (long long)y * a.gt.sH + (long long)x * a.gt.sW;
#pragma unroll
                for (int c = 0; c < C; ++c) gv[i][c] = ld_stream(gp + (long long)c * a.gt.sC);
            }
        }
#pragma unroll
        for (int i = 0; i < kRPer; ++i) {
            const unsigned r = base + i * 32;
            if (r < a.HW) {
                __stcg((float4*)acc + r, make_float4(0.f, 0.f, 0.f, 0.f));   // accumulators leave the kernel all-zero
                __stcg((float2*)acc2 + r, make_float2(0.f, 0.f));
                const float sv[4] = {s[i].x, s[i].y, s[i].z, s[i].w};
                const float d = sv[C];
                const float ob = occlusion(q[i].x, q[i].y, d, mx[i], my[i]);          // control_utils.py:15-16
                if (mo) st<T, float>(mo + r, ob);
                const float scale = __frcp_rn(add_rn(d, 0.0000001f));                 // softsplat.py:256-258, :270
                float w0, w1;
                if (a.variant == DCB_RECIPE_DATASET) {        // dataset.py:255-259: masks are the confidences
                    const float ws = add_rn(add_rn(of[i], ob), 0.000001f);
                    w0 = of[i] / ws; w1 = ob / ws;
                } else {                                      // residual_utils.py:181-185: ones are the confidences
                    const float ws = add_rn(2.f, 0.000001f);
                    w0 = 1.f / ws; w1 = w0;
                }
                const bool hole = a.variant == DCB_RECIPE_WRAPPER && add_rn(of[i], ob) > 1.5f;   // residual_utils.py:190-193
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const float wv = round_as<T>(mul_rn(sv[c], scale));               // warped1 == warped2 (SURVEY.md B-6)
                    float fused = add_rn(mul_rn(w0, wv), mul_rn(w1, wv));
                    if (hole) fused = mul_rn(0.5f, add_rn(wv, wv));
                    st_stream(fo + (size_t)c * a.HW + r, fused);
                    st_stream(ro + (size_t)c * a.HW + r, sub_rn(gv[i][c], round_as<T>(fused)));   // residual of the stored (rounded) value
                }
            }
        }
    }
}

// the recipe epilogue on two consecutive pixels per lane (a.flat2: see mask_chunk_v2; gt is a plain [N,C,H,W] tensor too)
template <class T, int C> __device__ __forceinline__ void recipe_pixel(const PipeArgs& a, const float (&sv)[4], float qx, float qy, float mx, float my,
                                                                      float of, const float* gv, float& ob, float* fused, float* resid) {
    const float d = sv[C];
    ob = occlusion(qx, qy, d, mx, my);                                   // control_utils.py:15-16
    const float scale = __frcp_rn(add_rn(d, 0.0000001f));                // softsplat.py:256-258, :270
    // masks are 0 or 1, so conf / (conf.sum() + 1e-6) takes one of three values: 0, 1 / (1 + 1e-6), 1 / (2 + 1e-6) -- the two
    // quotients are IEEE divisions of constants (folded at compile time), exactly what the per-pixel division would give
    const float one_of_one = 1.f / (1.f + 0.000001f), one_of_two = 1.f / (2.f + 0.000001f);
    float w0, w1;
    if (a.variant == DCB_RECIPE_DATASET) {            // dataset.py:255-259: masks are the confidences
        const bool both = of != 0.f && ob != 0.f;
        w0 = of != 0.f ? (both ? one_of_two : one_of_one) : 0.f;
        w1 = ob != 0.f ? (both ? one_of_two : one_of_one) : 0.f;
    } else {                                          // residual_utils.py:181-185: ones are the confidences
        w0 = one_of_two; w1 = one_of_two;
    }
    const bool hole = a.variant == DCB_RECIPE_WRAPPER && of != 0.f && ob != 0.f;   // residual_utils.py:190-193: (occ_fwd + occ_bwd) > 1.5
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const float wv = round_as<T>(mul_rn(sv[c], scale));              // warped1 == warped2 (SURVEY.md B-6)
        float f = add_rn(mul_rn(w0, wv), mul_rn(w1, wv));
        if (hole) f = mul_rn(0.5f, add_rn(wv, wv));
        fused[c] = f;
        resid[c] = sub_rn(gv[c], round_as<T>(f));                        // residual of the stored (rounded) value
    }
}

template <class T, int CA>
__device__ __forceinline__ void recipe_chunk_v2(const PipeArgs& a, int frame, int chunk, float* acc, float* acc2, int lane) {
    constexpr int C = CA - 1;
    constexpr int kGroups = kRPer / 2;
    T* fo = (T*)a.out + (long long)frame * C * a.HW;
    T* ro = (T*)a.residual + (long long)frame * C * a.HW;
    const T* oo = (const T*)a.occ_other + (long long)frame * a.HW;
    T* mo = a.mask_out ? (T*)a.mask_out + (long long)frame * a.HW : nullptr;
    const T* fbase = (const T*)a.epi_flow.p + frame * a.epi_flow.sN;
    const T* gbase = (const T*)a.gt.p + frame * a.gt.sN;
#pragma unroll 1
    for (int b = 0; b < kChunk / (32 * kRPer); ++b) {
        const unsigned base = (unsigned)chunk * kChunk + b * (32 * kRPer);
        if (base >= a.HW) break;
        float4 s[kGroups][2], q[kGroups]; float2 mx[kGroups], my[kGroups], of[kGroups], gv[kGroups][C > 0 ? C : 1];
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {                               // every load of the batch in flight first
            const unsigned r = base + g * 64 + lane * 2;
            s[g][0] = s[g][1] = q[g] = make_float4(0.f, 0.f, 0.f, 0.f);
            mx[g] = my[g] = of[g] = make_float2(0.f, 0.f);
#pragma unroll
            for (int c = 0; c < C; ++c) gv[g][c] = make_float2(0.f, 0.f);
            if (r < a.HW) {
                ld_cells2(acc + (size_t)r * 4, s[g][0], s[g][1]);
                q[g] = __ldcg((const float4*)(acc2 + (size_t)r * 2));
                mx[g] = ld2_stream(fbase + r); my[g] = ld2_stream(fbase + a.epi_flow.sC + r);
                of[g] = ld2_stream(oo + r);
#pragma unroll
                for (int c = 0; c < C; ++c) gv[g][c] = ld2_stream(gbase + (long long)c * a.gt.sC + r);
            }
        }
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            const unsigned r = base + g * 64 + lane * 2;
            if (r < a.HW) {
                zero_cells2(acc + (size_t)r * 4);                         // accumulators leave the kernel all-zero
                __stcg((float4*)(acc2 + (size_t)r * 2), make_float4(0.f, 0.f, 0.f, 0.f));
                const float s0[4] = {s[g][0].x, s[g][0].y, s[g][0].z, s[g][0].w}, s1[4] = {s[g][1].x, s[g][1].y, s[g][1].z, s[g][1].w};
                float g0[C > 0 ? C : 1], g1[C > 0 ? C : 1], f0[C > 0 ? C : 1], f1[C > 0 ? C : 1], r0[C > 0 ? C : 1], r1[C > 0 ? C : 1], ob0, ob1;
#pragma unroll
                for (int c = 0; c < C; ++c) { g0[c] = gv[g][c].x; g1[c] = gv[g][c].y; }
                recipe_pixel<T, C>(a, s0, q[g].x, q[g].y, mx[g].x, my[g].x, of[g].x, g0, ob0, f0, r0);
                recipe_pixel<T, C>(a, s1, q[g].z, q[g].w, mx[g].y, my[g].y, of[g].y, g1, ob1, f1, r1);
                if (mo) st_stream2(mo + r, ob0, ob1);
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    st_stream2(fo + (size_t)c * a.HW + r, f0[c], f1[c]);
                    st_stream2(ro + (size_t)c * a.HW + r, r0[c], r1[c]);
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// two-reference recipe (dcb_residual_bidir): the rider scatter above, run twice with the roles of the frames swapped.
//   pass A (KIND 2): image2 splatted by flow2, flow1 riding. Epilogue: warped2 = S / (D + 1e-7), parked (rounded to T) in the
//                    caller's `fused` buffer; occ_fwd = compute_mask(flow1, flow2), tested against flow2 at the target
//   pass B (KIND 3): image1 splatted by flow1, flow2 riding. Epilogue: warped1; occ_bwd = compute_mask(flow2, flow1), tested
//                    against flow1; soft_fuse(warped1, warped2, 1 - occ_fwd, 1 - occ_bwd); fused and gt - fused stored once
// Pass B reads what pass A's epilogues wrote (warped2 in `fused`, the occ_fwd plane), as the one-reference recipe reads its
// mask plane: every launch of the chain waits (griddepcontrol.wait) until its predecessor has completed and its writes are
// visible, and that predecessor did the same, so all of pass A is visible to every launch of pass B.
// ---------------------------------------------------------------------------------------------
template <class T, int C>
__device__ __forceinline__ void bidir_pixel(const float (&sv)[4], float qx, float qy, float mx, float my, float& occ, float* warped) {
    const float d = sv[C];
    occ = occlusion(qx, qy, d, mx, my);                                  // control_utils.py:15-16
    const float scale = __frcp_rn(add_rn(d, 0.0000001f));                // softsplat.py:256-258, :270
#pragma unroll
    for (int c = 0; c < C; ++c) warped[c] = round_as<T>(mul_rn(sv[c], scale));
}

template <class T, int CA, bool PASS_B>
__device__ __forceinline__ void bidir_chunk(const PipeArgs& a, int frame, int chunk, float* acc, float* acc2, int lane) {
    constexpr int C = CA - 1;
    T* fo = (T*)a.out + (long long)frame * C * a.HW;                    // pass A: warped2 out; pass B: warped2 in, fused out
    T* ro = (T*)a.residual + (long long)frame * C * a.HW;
    const T* oo = (const T*)a.occ_other + (long long)frame * a.HW;
    T* mo = a.mask_out ? (T*)a.mask_out + (long long)frame * a.HW : nullptr;
    const T* fbase = (const T*)a.epi_flow.p + frame * a.epi_flow.sN;
    const T* gbase = (const T*)a.gt.p + frame * a.gt.sN;
#pragma unroll 1
    for (int b = 0; b < kChunk / (32 * kRPer); ++b) {
        const unsigned base = (unsigned)chunk * kChunk + b * (32 * kRPer) + lane;
        if (base - lane >= a.HW) break;
        float4 s[kRPer]; float2 q[kRPer]; float mx[kRPer], my[kRPer];
#pragma unroll
        for (int i = 0; i < kRPer; ++i) {                                // every load of the batch in flight first
            const unsigned r = base + i * 32;
            s[i] = make_float4(0.f, 0.f, 0.f, 0.f); q[i] = make_float2(0.f, 0.f);
            mx[i] = my[i] = 0.f;
            if (r < a.HW) {
                s[i] = __ldcg((const float4*)acc + r);
                q[i] = __ldcg((const float2*)acc2 + r);
                const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
                const T* fp = fbase + (long long)y * a.epi_flow.sH + (long long)x * a.epi_flow.sW;
                mx[i] = ld<float>(fp); my[i] = ld<float>(fp + a.epi_flow.sC);
            }
        }
#pragma unroll
        for (int i = 0; i < kRPer; ++i) {
            const unsigned r = base + i * 32;
            if (r < a.HW) {
                __stcg((float4*)acc + r, make_float4(0.f, 0.f, 0.f, 0.f));   // accumulators leave the kernel all-zero
                __stcg((float2*)acc2 + r, make_float2(0.f, 0.f));
                const float sv[4] = {s[i].x, s[i].y, s[i].z, s[i].w};
                float occ, wv[C > 0 ? C : 1];
                bidir_pixel<T, C>(sv, q[i].x, q[i].y, mx[i], my[i], occ, wv);
                if (mo) st<T, float>(mo + r, occ);
                if (!PASS_B) {
#pragma unroll
                    for (int c = 0; c < C; ++c) st_stream(fo + (size_t)c * a.HW + r, wv[c]);
                    continue;
                }
                const float of = ld_stream(oo + r);
                const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
                const T* gp = gbase + (long long)y * a.gt.sH + (long long)x * a.gt.sW;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const float f = bidir_soft_fuse(wv[c], ld_stream(fo + (size_t)c * a.HW + r), of, occ);
                    st_stream(fo + (size_t)c * a.HW + r, f);
                    st_stream(ro + (size_t)c * a.HW + r, sub_rn(ld_stream(gp + (long long)c * a.gt.sC), round_as<T>(f)));   // residual of the stored value
                }
            }
        }
    }
}

// two consecutive pixels per lane (a.flat2: every plane the epilogue touches is a plain, pair-aligned [H,W] plane)
template <class T, int CA, bool PASS_B>
__device__ __forceinline__ void bidir_chunk_v2(const PipeArgs& a, int frame, int chunk, float* acc, float* acc2, int lane) {
    constexpr int C = CA - 1;
    constexpr int kGroups = kRPer / 2;
    T* fo = (T*)a.out + (long long)frame * C * a.HW;                    // pass A: warped2 out; pass B: warped2 in, fused out
    T* ro = (T*)a.residual + (long long)frame * C * a.HW;
    const T* oo = (const T*)a.occ_other + (long long)frame * a.HW;
    T* mo = a.mask_out ? (T*)a.mask_out + (long long)frame * a.HW : nullptr;
    const T* fbase = (const T*)a.epi_flow.p + frame * a.epi_flow.sN;
    const T* gbase = (const T*)a.gt.p + frame * a.gt.sN;
#pragma unroll 1
    for (int b = 0; b < kChunk / (32 * kRPer); ++b) {
        const unsigned base = (unsigned)chunk * kChunk + b * (32 * kRPer);
        if (base >= a.HW) break;
        float4 s[kGroups][2], q[kGroups]; float2 mx[kGroups], my[kGroups];
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {                               // accumulator and flow loads of the batch in flight first
            const unsigned r = base + g * 64 + lane * 2;
            s[g][0] = s[g][1] = q[g] = make_float4(0.f, 0.f, 0.f, 0.f);
            mx[g] = my[g] = make_float2(0.f, 0.f);
            if (r < a.HW) {
                ld_cells2(acc + (size_t)r * 4, s[g][0], s[g][1]);
                q[g] = __ldcg((const float4*)(acc2 + (size_t)r * 2));
                mx[g] = ld2_stream(fbase + r); my[g] = ld2_stream(fbase + a.epi_flow.sC + r);
            }
        }
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            const unsigned r = base + g * 64 + lane * 2;
            if (r < a.HW) {
                // pass B: the streamed operands of this pair, issued before the accumulator cells are re-zeroed
                float2 of = make_float2(0.f, 0.f), gv[C > 0 ? C : 1], w2[C > 0 ? C : 1];
                if (PASS_B) {
                    of = ld2_stream(oo + r);
#pragma unroll
                    for (int c = 0; c < C; ++c) { gv[c] = ld2_stream(gbase + (long long)c * a.gt.sC + r); w2[c] = ld2_stream(fo + (size_t)c * a.HW + r); }
                }
                zero_cells2(acc + (size_t)r * 4);                         // accumulators leave the kernel all-zero
                __stcg((float4*)(acc2 + (size_t)r * 2), make_float4(0.f, 0.f, 0.f, 0.f));
                const float s0[4] = {s[g][0].x, s[g][0].y, s[g][0].z, s[g][0].w}, s1[4] = {s[g][1].x, s[g][1].y, s[g][1].z, s[g][1].w};
                float w0v[C > 0 ? C : 1], w1v[C > 0 ? C : 1], ob0, ob1;
                bidir_pixel<T, C>(s0, q[g].x, q[g].y, mx[g].x, my[g].x, ob0, w0v);
                bidir_pixel<T, C>(s1, q[g].z, q[g].w, mx[g].y, my[g].y, ob1, w1v);
                if (mo) st_stream2(mo + r, ob0, ob1);
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    if (!PASS_B) {
                        st_stream2(fo + (size_t)c * a.HW + r, w0v[c], w1v[c]);
                    } else {
                        const float f0 = bidir_soft_fuse(w0v[c], w2[c].x, of.x, ob0), f1 = bidir_soft_fuse(w1v[c], w2[c].y, of.y, ob1);
                        st_stream2(fo + (size_t)c * a.HW + r, f0, f1);
                        st_stream2(ro + (size_t)c * a.HW + r, sub_rn(gv[c].x, round_as<T>(f0)), sub_rn(gv[c].y, round_as<T>(f1)));   // residual of the stored values
                    }
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// the step kernel: warp w of CTA b owns item 4b + w; normalise items first, then scatter items
// ---------------------------------------------------------------------------------------------
// one epilogue item: chunk `chunk` of frame `z` of the group being normalised
template <class T, int MODE, int CA, int KIND>
__device__ __forceinline__ void epilogue_item(const PipeArgs& a, unsigned z, unsigned chunk, int lane) {
    const int f = a.n_frame0 + (int)z;
    float* acc = a.acc_n + z * ((size_t)a.HW * 4);
    if (KIND == 1) {
        if (a.flat2) recipe_chunk_v2<T, CA>(a, f, (int)chunk, acc, a.acc2_n + z * ((size_t)a.HW * 2), lane);
        else recipe_chunk<T, CA>(a, f, (int)chunk, acc, a.acc2_n + z * ((size_t)a.HW * 2), lane);
        return;
    }
    if (KIND == 2 || KIND == 3) {
        if (a.flat2) bidir_chunk_v2<T, CA, KIND == 3>(a, f, (int)chunk, acc, a.acc2_n + z * ((size_t)a.HW * 2), lane);
        else bidir_chunk<T, CA, KIND == 3>(a, f, (int)chunk, acc, a.acc2_n + z * ((size_t)a.HW * 2), lane);
        return;
    }
    if (a.epi == 1) { if (a.flat2) mask_chunk_v2<T>(a, f, (int)chunk, acc, lane); else mask_chunk<T>(a, f, (int)chunk, acc, lane); }
#if DCB_NORM_V == 4
    else if (a.vec4 && a.mask.p == nullptr) normalize_chunk_v4<T, MODE, CA>(a, f, (int)chunk, acc, lane);
#elif DCB_NORM_V == 2
    else if (a.vec4 && a.mask.p == nullptr) normalize_chunk_v2<T, MODE, CA>(a, f, (int)chunk, acc, lane);
#endif
    else normalize_chunk<T, MODE, CA>(a, f, (int)chunk, acc, lane);
}

// An epilogue-only launch (one accumulator slot: every second launch) as CTAs of kEpiWarps warps, one chunk per warp:
// the same per-warp work as in k_splat_step with a quarter of the CTAs to schedule.
#ifndef DCB_EPI_WARPS
#define DCB_EPI_WARPS 4
#endif
#ifndef DCB_EPI_MINCTAS
#define DCB_EPI_MINCTAS (DCB_MINCTAS / DCB_EPI_WARPS)
#endif
constexpr int kEpiWarps = DCB_EPI_WARPS;
template <class T, int MODE, int CA, int KIND>
__global__ void __launch_bounds__(32 * kEpiWarps, KIND ? kMinCtasRecipe / kEpiWarps : DCB_EPI_MINCTAS) k_splat_epilogue(const __grid_constant__ PipeArgs a) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const unsigned chunk = blockIdx.x * kEpiWarps + (threadIdx.x >> 5);
    if (chunk >= (unsigned)a.tn) return;
    epilogue_item<T, MODE, CA, KIND>(a, blockIdx.y, chunk, threadIdx.x & 31);
}

// KIND 0: softsplat / occlusion mask; KIND 1: the conditioning recipe's second pass (rider scatter + recipe epilogue);
// KIND 2, 3: the two passes of the two-reference recipe (rider scatter + bidir_chunk epilogues)
template <class T, class TF, int MODE, int CA, int KIND>
__global__ void __launch_bounds__(kPipeThreads, KIND ? kMinCtasRecipe : kMinCtas) k_splat_step(const __grid_constant__ PipeArgs a) {
    // Programmatic dependent launch: let the next step's grid start being scheduled while this one
    // drains, and wait here until the previous step has completed and flushed (both steps touch
    // the same accumulator ring). The launch latency of 65 dependent launches is thereby hidden.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    // 3-d grid, no integer division anywhere: z < n_frames -> normalise item (frame z of the group, chunk y * gridDim.x + x),
    // else scatter item (frame z - n_frames of its group, strip column x, strip row y); the host passes both slot pointers
    const int lane = threadIdx.x & 31;
    const unsigned z = blockIdx.z;
    const size_t frame_floats = (size_t)a.HW * 4;
    if (z < (unsigned)a.n_frames) {
        const unsigned chunk = blockIdx.y * gridDim.x + blockIdx.x;
        if (chunk >= (unsigned)a.tn) return;
        epilogue_item<T, MODE, CA, KIND>(a, z, chunk, lane);
    } else {
        const unsigned zs = z - (unsigned)a.n_frames;
        if (blockIdx.x >= (unsigned)a.tiles_x || blockIdx.y >= (unsigned)a.tiles_y) return;
        // the bottom rows of a frame (dispatched last) are cut into single-pass strips: the grid's tail drains in finer steps
        const int by = (int)blockIdx.y;
        const int y_first = by < a.ny_big ? by * kStripH : a.ny_big * kStripH + (by - a.ny_big) * kRows;
        scatter_strip<T, TF, MODE, CA, KIND != 0>(a, a.s_frame0 + (int)zs, (int)blockIdx.x, y_first, by < a.ny_big ? kPasses : 1, a.acc_s + zs * frame_floats,
                                                  KIND != 0 ? a.acc2_s + zs * ((size_t)a.HW * 2) : nullptr, lane);
    }
}

// ---------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------
// dcb_set_option("pipe_group_bytes"): tests shrink the ring slots so that small tensors run through many groups
long long g_pipe_group_bytes = 0;
void pipe_set_group_bytes(long long b) { g_pipe_group_bytes = b > 0 ? b : 0; }
// dcb_set_option("pipe_ring_slots"): 1 (default) = one accumulator slot, scatter and normalise of a frame group in
// alternating launches; 2 = round 1's ring (step k normalises group k-1 while it scatters group k). Measured on 1080p
// frames with `ncu --cache-control none` (profiles/r02/): two 33 MB slots do not stay in the 126 MB L2 next to the streaming
// inputs / outputs (131-178 MB of DRAM traffic per 75 MB frame); ONE slot does (50.4 MB read by the scatter launch, 0.2 MB
// read + the output written by the normalise launch: exactly the compulsory bytes), and it is as fast or faster.
int g_pipe_tail_percent = DCB_TAIL_PERCENT;
void pipe_set_tail_percent(long long p) { g_pipe_tail_percent = p < 0 ? DCB_TAIL_PERCENT : (p > 100 ? 100 : (int)p); }
int g_pipe_ring_slots = 1;
void pipe_set_ring_slots(long long n) { g_pipe_ring_slots = n == 1 ? 1 : 2; }

static long long group_frames(long long N, long long H, long long W, long long cell_bytes = 16) {
    // the recipe pass keeps 24 bytes per pixel resident: its slot may be half as large again (one 1080p frame = 47.5 MiB)
    const long long gb = (g_pipe_group_bytes > 0 ? g_pipe_group_bytes : kGroupBytes) * cell_bytes / 16;
    long long g = gb / (H * W * cell_bytes > 0 ? H * W * cell_bytes : 1);
    if (g < 1) g = 1;
    if (g > 32767) g = 32767;                    // gridDim.z = frames normalised + frames scattered <= 65535
    return g > N ? (N < 1 ? 1 : N) : g;
}

long long pipe_acc_bytes(long long N, long long H, long long W) {
    const long long G = group_frames(N, H, W);
    const long long slots = (N > G && g_pipe_ring_slots == 2) ? 2 : 1;
    return align_up(slots * G * H * W * 16, 256);
}

long long pipe_workspace(long long N, long long H, long long W) { return pipe_acc_bytes(N, H, W); }

template <class T, class TF, int MODE, int CA, int KIND = 0> static int launch_steps(PipeArgs& a, cudaStream_t st) {
    const int groups = (a.N + a.G - 1) / a.G;
    const size_t slot_floats = (size_t)a.G * a.HW * 4;
    // both item kinds cover 32 * kStripH pixels, so one (x, y) extent serves the normalise chunks and the scatter strips
    const unsigned gx = (unsigned)a.tiles_x;
    const unsigned rows_n = (unsigned)((a.tn + a.tiles_x - 1) / a.tiles_x);
    const unsigned gy = rows_n > (unsigned)a.tiles_y ? rows_n : (unsigned)a.tiles_y;
    const bool one_slot = g_pipe_ring_slots == 1 || KIND != 0;
    for (int k = 0; k <= (one_slot ? 2 * groups - 1 : groups); ++k) {
        // two slots: launch k = normalise(group k-1) + scatter(group k); one slot: launch 2g = scatter(g), launch 2g+1 = normalise(g)
        const int gs = one_slot ? ((k & 1) ? -1 : k / 2) : (k < groups ? k : -1);
        const int gn = one_slot ? ((k & 1) ? k / 2 : -1) : k - 1;
        a.s_frame0 = gs >= 0 ? gs * a.G : 0;
        a.s_frames = gs >= 0 ? (a.N - a.s_frame0 < a.G ? a.N - a.s_frame0 : a.G) : 0;
        a.n_frame0 = gn >= 0 ? gn * a.G : 0;
        a.n_frames = gn >= 0 ? (a.N - a.n_frame0 < a.G ? a.N - a.n_frame0 : a.G) : 0;
        a.acc_s = a.acc + (one_slot ? 0 : (size_t)(gs & 1) * slot_floats);
        a.acc_n = a.acc + (one_slot ? 0 : (size_t)(gn & 1) * slot_floats);
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(gx, gy, (unsigned)(a.n_frames + a.s_frames)); cfg.blockDim = dim3(kPipeThreads); cfg.dynamicSmemBytes = 0; cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        if (kEpiWarps > 1 && a.s_frames == 0) {          // epilogue-only launch
            cfg.gridDim = dim3((unsigned)((a.tn + kEpiWarps - 1) / kEpiWarps), (unsigned)a.n_frames, 1); cfg.blockDim = dim3(32 * kEpiWarps);
            DCB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, k_splat_epilogue<T, MODE, CA, KIND>, a));
            count_launch();
            continue;
        }
        DCB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, k_splat_step<T, TF, MODE, CA, KIND>, a));
        count_launch();
    }
    return DCB_OK;
}

template <class T, class TF, int MODE> static int launch_mode(PipeArgs& a, cudaStream_t st) {
    const int ca = a.C + (MODE != DCB_MODE_SUM ? 1 : 0);
    switch (ca) {
        case 1: if (MODE == DCB_MODE_SUM) return launch_steps<T, TF, DCB_MODE_SUM, 1>(a, st); break;
        case 2: return launch_steps<T, TF, MODE, 2>(a, st);
        case 3: return launch_steps<T, TF, MODE, 3>(a, st);
        case 4: return launch_steps<T, TF, MODE, 4>(a, st);
    }
    return set_error(DCB_E_LIMIT, "splat_pipe: %d accumulated channels", ca);
}

template <class T, class TF> static int launch_pipe(PipeArgs& a, int mode, cudaStream_t st) {
    switch (mode) {
        case DCB_MODE_SUM: return launch_mode<T, TF, DCB_MODE_SUM>(a, st);
        case DCB_MODE_AVG: return launch_mode<T, TF, DCB_MODE_AVG>(a, st);
        case DCB_MODE_LINEAR: return launch_mode<T, TF, DCB_MODE_LINEAR>(a, st);
        default: return launch_mode<T, TF, DCB_MODE_SOFT>(a, st);
    }
}

// every element offset the kernels form must fit a signed 32-bit integer
static bool offsets_fit32(const DcbTensor* t) {
    if (!t) return true;
    long long span = 0;
    for (int d = 1; d < 4; ++d) span += (t->size[d] - 1) * (t->stride[d] < 0 ? -t->stride[d] : t->stride[d]);
    return span < (1ll << 31);
}
bool pipe_supported(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric) {
    return offsets_fit32(in) && offsets_fit32(flow) && offsets_fit32(metric) && in->size[2] * in->size[3] < (1ll << 28);
}


// a tensor whose H x W planes are contiguous and whose pixel pairs are aligned for one paired load / store
static bool planes_pair_aligned(const DcbTensor* t, long long W) {
    if (!t) return true;
    const long long es = elem_size(t->dtype);
    return t->stride[3] == 1 && t->stride[2] == W && t->stride[1] % 2 == 0 && t->stride[0] % 2 == 0 && ((uintptr_t)t->ptr % (2 * es)) == 0;
}

// Preconditions (checked by the caller): C + (mode != SUM) <= 4, dtype F32/BF16/F16, workspace >= pipe_workspace().
int splat_pipe_impl(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const DcbTensor* out,
                    const DcbTensor* norm, const DcbTensor* mask, void* ws, int mode, int eps, bool ws_clean,
                    cudaStream_t st, bool ones_metric, const DcbTensor* mask_out) {
    PipeArgs a = {};
    a.ones = ones_metric ? 1 : 0;
    a.epi = mask_out ? 1 : 0;
    a.epi_flow = make_view(mask_out ? flow : nullptr);
    a.mask_out = mask_out ? mask_out->ptr : nullptr;
    a.in = make_view(in); a.flow = make_view(flow); a.metric = make_view(metric); a.mask = make_view(mask);
    a.N = (int)in->size[0]; a.C = (int)in->size[1]; a.H = (int)in->size[2]; a.W = (int)in->size[3];
    a.HW = (unsigned)(in->size[2] * in->size[3]);
    a.eps = eps;
    a.G = (int)group_frames(a.N, a.H, a.W);
    a.tiles_x = (a.W + 31) / 32;
    {   // dcb_set_option("pipe_tail_percent"): share of a frame's rows (at the bottom) cut into single-pass strips
        const int rows_fine = (int)((long long)a.H * g_pipe_tail_percent / 100) / kStripH * kStripH;
        a.ny_big = (a.H - rows_fine) / kStripH;
        const int rest = a.H - a.ny_big * kStripH;
        a.tiles_y = a.ny_big + (rest + kRows - 1) / kRows;
    }
    a.ts = a.tiles_x * a.tiles_y;
    a.tn = (int)((a.HW + kChunk - 1) / kChunk);
    a.out = out ? out->ptr : nullptr;
    a.norm = norm ? norm->ptr : nullptr;
    a.acc = (float*)ws;
    a.vec4 = (a.HW % 4 == 0 && out && ((uintptr_t)out->ptr & 15) == 0 && (!norm || ((uintptr_t)norm->ptr & 15) == 0)) ? 1 : 0;
    a.flat2 = (mask_out && a.HW % 2 == 0 && planes_pair_aligned(flow, a.W) && planes_pair_aligned(mask_out, a.W)) ? 1 : 0;
    if (!ws_clean) DCB_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)pipe_workspace(a.N, a.H, a.W), st));
    const bool ff = flow->dtype == DCB_F32;
    if (in->dtype == DCB_F32) return launch_pipe<float, float>(a, mode, st);
    if (in->dtype == DCB_BF16)
        return ff ? launch_pipe<__nv_bfloat16, float>(a, mode, st) : launch_pipe<__nv_bfloat16, __nv_bfloat16>(a, mode, st);
    if (in->dtype == DCB_F16) return ff ? launch_pipe<__half, float>(a, mode, st) : launch_pipe<__half, __half>(a, mode, st);
    return set_error(DCB_E_DTYPE, "splat_pipe: unsupported dtype %d", in->dtype);
}

// ---------------------------------------------------------------------------------------------
// conditioning recipe, second pass: image1 AND flow2 splatted by flow1 in one scatter (shared footprints, shared weight
// channel), then one epilogue that normalises, tests occlusion, fuses and writes fused + residual.
// Workspace: [G frames of float4 cells][G frames of float2 cells], all-zero on entry and on exit.
// ---------------------------------------------------------------------------------------------
long long recipe_pipe_workspace(long long N, long long H, long long W) {
    const long long G = group_frames(N, H, W, 24);
    return align_up(G * H * W * 16, 256) + align_up(G * H * W * 8, 256);
}

template <class T, int KIND> static int launch_recipe(PipeArgs& a, cudaStream_t st) {
    switch (a.C) {
        case 1: return launch_steps<T, T, DCB_MODE_SOFT, 2, KIND>(a, st);
        case 2: return launch_steps<T, T, DCB_MODE_SOFT, 3, KIND>(a, st);
        case 3: return launch_steps<T, T, DCB_MODE_SOFT, 4, KIND>(a, st);
    }
    return set_error(DCB_E_LIMIT, "recipe_pipe: %d image channels", a.C);
}

// the arguments of one rider pass: `in` (C channels) and `rider` (2 channels) splatted together by `flow` with the all-ones
// metric, the occlusion epilogue comparing with `flow` at the target; accumulators [G frames of float4][G frames of float2] in ws
static PipeArgs rider_args(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* rider, const DcbTensor* gt, void* ws) {
    PipeArgs a = {};
    a.ones = 1; a.epi = 3;
    a.in = make_view(in); a.flow = make_view(flow); a.metric = make_view(nullptr); a.mask = make_view(nullptr);
    a.in2 = make_view(rider); a.epi_flow = make_view(flow); a.gt = make_view(gt);
    a.N = (int)in->size[0]; a.C = (int)in->size[1]; a.H = (int)in->size[2]; a.W = (int)in->size[3];
    a.HW = (unsigned)(in->size[2] * in->size[3]);
    a.eps = DCB_EPS_ADD;
    a.G = (int)group_frames(a.N, a.H, a.W, 24);
    a.tiles_x = (a.W + 31) / 32;
    a.ny_big = a.H / kStripH;
    a.tiles_y = a.ny_big + (a.H - a.ny_big * kStripH + kRows - 1) / kRows;
    a.ts = a.tiles_x * a.tiles_y;
    a.tn = (int)((a.HW + kChunk - 1) / kChunk);
    a.norm = nullptr;
    a.vec4 = 0;
    a.acc = (float*)ws;
    a.acc2_s = a.acc2_n = (float*)((char*)ws + align_up((long long)a.G * a.HW * 16, 256));
    return a;
}

// Preconditions (checked by the caller): 1 <= C <= 3, one dtype (F32/BF16) for every tensor, contiguous outputs,
// pipe_supported() for every strided input, workspace >= recipe_pipe_workspace() and all-zero.
int recipe_pipe_impl(const DcbTensor* image1, const DcbTensor* flow1, const DcbTensor* flow2, const DcbTensor* gt,
                     const DcbTensor* fused, const DcbTensor* residual, const DcbTensor* occ_fwd, const DcbTensor* occ_bwd,
                     void* ws, int variant, cudaStream_t st) {
    PipeArgs a = rider_args(image1, flow1, flow2, gt, ws);
    a.out = fused->ptr; a.residual = residual->ptr;
    a.occ_other = occ_fwd->ptr;
    a.mask_out = occ_bwd ? occ_bwd->ptr : nullptr;
    a.variant = variant;
    a.flat2 = (a.HW % 2 == 0 && planes_pair_aligned(flow1, a.W) && planes_pair_aligned(gt, a.W) && planes_pair_aligned(fused, a.W) &&
               planes_pair_aligned(residual, a.W) && planes_pair_aligned(occ_fwd, a.W) && planes_pair_aligned(occ_bwd, a.W) &&
               (((uintptr_t)ws + align_up((long long)a.G * a.HW * 16, 256)) & 15) == 0) ? 1 : 0;
    if (image1->dtype == DCB_F32) return launch_recipe<float, 1>(a, st);
    if (image1->dtype == DCB_BF16) return launch_recipe<__nv_bfloat16, 1>(a, st);
    return set_error(DCB_E_DTYPE, "recipe_pipe: unsupported dtype %d", image1->dtype);
}

// ---------------------------------------------------------------------------------------------
// two-reference recipe: pass A (image2 + rider flow1 by flow2, KIND 2) then pass B (image1 + rider flow2 by flow1, KIND 3),
// four launches per frame group as the one-reference recipe. occ_fwd is required (the caller's plane or a workspace plane:
// pass B reads it); occ_bwd is optional. Preconditions as recipe_pipe_impl.
// ---------------------------------------------------------------------------------------------
int bidir_pipe_impl(const DcbTensor* image1, const DcbTensor* image2, const DcbTensor* flow1, const DcbTensor* flow2,
                    const DcbTensor* gt, const DcbTensor* fused, const DcbTensor* residual, const DcbTensor* occ_fwd,
                    const DcbTensor* occ_bwd, void* ws, cudaStream_t st) {
    PipeArgs a = rider_args(image2, flow2, flow1, gt, ws);
    a.out = fused->ptr; a.residual = residual->ptr;
    a.occ_other = nullptr;
    a.mask_out = occ_fwd->ptr;
    // one layout decision for both passes: every plane either epilogue touches
    a.flat2 = (a.HW % 2 == 0 && planes_pair_aligned(flow1, a.W) && planes_pair_aligned(flow2, a.W) && planes_pair_aligned(gt, a.W) &&
               planes_pair_aligned(fused, a.W) && planes_pair_aligned(residual, a.W) && planes_pair_aligned(occ_fwd, a.W) &&
               planes_pair_aligned(occ_bwd, a.W) && (((uintptr_t)ws + align_up((long long)a.G * a.HW * 16, 256)) & 15) == 0) ? 1 : 0;
    const int dt = image1->dtype;
    if (dt != DCB_F32 && dt != DCB_BF16) return set_error(DCB_E_DTYPE, "bidir_pipe: unsupported dtype %d", dt);
    int rc = dt == DCB_F32 ? launch_recipe<float, 2>(a, st) : launch_recipe<__nv_bfloat16, 2>(a, st);
    if (rc != DCB_OK) return rc;
    const int flat2 = a.flat2;
    a = rider_args(image1, flow1, flow2, gt, ws);
    a.out = fused->ptr; a.residual = residual->ptr;
    a.occ_other = occ_fwd->ptr;
    a.mask_out = occ_bwd ? occ_bwd->ptr : nullptr;
    a.flat2 = flat2;
    return dt == DCB_F32 ? launch_recipe<float, 3>(a, st) : launch_recipe<__nv_bfloat16, 3>(a, st);
}

}  // namespace dcb
