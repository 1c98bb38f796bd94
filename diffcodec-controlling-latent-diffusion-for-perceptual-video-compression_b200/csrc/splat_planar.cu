// splat_planar.cu -- forward splat for MANY channels (feature maps: C = 64 .. 640) in fp32 / bf16 / fp16,
// as the same kernel-per-step software pipeline as splat_pipe.cu, with planar accumulators.
//
// Replaces controlnet/softsplat.py:240-270 (pre/post ops) + :281-345 (zero-init + softsplat_out)
// for C + 1 > 4. The reference runs one thread per (pixel, channel): flow is re-read and the four
// weights recomputed C+1 times per pixel, and every element issues 4 scalar atomics. Here
//
//   * a warp owns a 32-column x 4-row strip of ONE frame for ALL channels: the footprint of every
//     pixel (corner offset, 4 weights, which pieces merge with the lane to the right / the row
//     below) is computed once and kept in registers, then the channels stream through it;
//   * per channel the east column is handed to lane+1 by shuffle and the south row is carried to
//     the next row when footprints abut, so smooth flow costs ~1.2-2 scalar reds per element
//     instead of 4; a warp's reds of one channel fall on one or two 128-byte lines of one plane;
//   * accumulators hold FOUR channels per cell, fp32 [frame][C/4][H*W][4]: one 16-byte
//     `red.global.add.v4.f32` per corner and channel quad instead of four scalar reds (on rough flow
//     a scalar red costs ~0.44 L2 sectors, a v4 red ~0.6 for four times the payload); the weight
//     channel has its own plane; both live in a ring of two L2-sized slots; step k
//     normalises frame group k-1 (and re-zeroes it) while it scatters group k; the kernel boundary
//     is the only synchronisation; inputs/outputs use streaming loads/stores.
#include "splat_planar.cuh"

#include <type_traits>

namespace dcb {

template <class T>
__device__ __forceinline__ void planar_normalize_chunk(const PlanarArgs& a, int frame, int chunk, int q_begin, int q_end,
                                                       float* acc, float* dplane, int lane) {
    const int C = a.C;
    T* out = (T*)a.out + (long long)frame * C * a.HW;
    constexpr int kPer = kPChunk / 32;
    const unsigned base = (unsigned)chunk * kPChunk + lane;
    float scale[kPer];
    const bool normalised = a.mode != DCB_MODE_SUM;
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
        const unsigned r = base + i * 32;
        scale[i] = 1.f;
        if (r < a.HW) {
            if (normalised) {
                float d = __ldcg(dplane + r);     // shared by the warps of every channel group: re-zeroed a step later ...
                if (a.ncg_n == 1) __stcg(dplane + r, 0.f);   // ... unless this warp is its only reader
                // softsplat.py:256-266
                if (a.eps == DCB_EPS_ADD) d = add_rn(d, 0.0000001f);
                else if (a.eps == DCB_EPS_ZERO) d = (d == 0.f) ? 1.f : d;
                else d = (d < 0.0000001f) ? 0.0000001f : d;
                if (a.norm && q_begin == 0) __stcs((float*)a.norm + (long long)frame * a.HW + r, d);
                scale[i] = __frcp_rn(d);          // <= 1 ulp from the true quotient of softsplat.py:270
            }
            if (a.mask.p) {
                const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
                const T* mp = (const T*)a.mask.p + frame * a.mask.sN + (long long)y * a.mask.sH + (long long)x * a.mask.sW;
                scale[i] = mul_rn(scale[i], sub_rn(1.f, ld<float>(mp)));     // control_utils.py:69-70
            }
        }
    }
    const bool scaled = normalised || a.mask.p != nullptr;
    for (int q = q_begin; q < q_end; ++q) {
        float4* plane = (float4*)acc + (size_t)q * a.HW;
        float4 s[kPer];
#pragma unroll
        for (int i = 0; i < kPer; ++i) {
            const unsigned r = base + i * 32;
            s[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < a.HW) s[i] = __ldcg(plane + r);
        }
#pragma unroll
        for (int i = 0; i < kPer; ++i) {
            const unsigned r = base + i * 32;
            if (r < a.HW) {
                __stcg(plane + r, make_float4(0.f, 0.f, 0.f, 0.f));
                const float sv[4] = {s[i].x, s[i].y, s[i].z, s[i].w};
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (4 * q + j < C) st_stream(out + (size_t)(4 * q + j) * a.HW + r, scaled ? mul_rn(sv[j], scale[i]) : sv[j]);
            }
        }
    }
}

template <class T, class TF>
__global__ void __launch_bounds__(kPThreads, DCB_PMINCTAS) k_planar_step(const __grid_constant__ PlanarArgs a) {
    // programmatic dependent launch: see k_splat_step
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int lane = threadIdx.x & 31;
    unsigned item = blockIdx.x * kPWarps + (threadIdx.x >> 5);
    const size_t frame_floats = (size_t)a.Cq * a.HW * 4, slot_floats = (size_t)a.G * frame_floats;
    const size_t dslot = (size_t)a.G * a.HW;
    const unsigned n_items = (unsigned)a.n_frames * a.tn * a.ncg_n;
    const unsigned z_items = a.mode == DCB_MODE_SUM ? 0u : (unsigned)a.G * a.tz;
    if (item < n_items) {                                                 // normalise group step-1
        const unsigned per = (unsigned)a.tn * a.ncg_n;
        const int fi = item / per, q = item % per;
        const int chunk = q % a.tn, cgi = q / a.tn;
        const int f = a.n_frame0 + fi, g = a.step - 1;
        float* acc = a.acc + (size_t)(g & 1) * slot_floats + (size_t)fi * frame_floats;
        float* dplane = a.dacc + (size_t)(g % 3) * dslot + (size_t)fi * a.HW;
        planar_normalize_chunk<T>(a, f, chunk, cgi * a.cg_n, min(a.Cq, (cgi + 1) * a.cg_n), acc, dplane, lane);
        return;
    }
    item -= n_items;
    if (item < z_items) {                                                 // re-zero the normaliser slot of group step+1
        const int fi = item / a.tz, q = item % a.tz;
        float* dplane = a.dacc + (size_t)((a.step + 1) % 3) * dslot + (size_t)fi * a.HW;
        for (unsigned r = (unsigned)q * 1024 + lane; r < min(a.HW, (unsigned)(q + 1) * 1024); r += 32) __stcg(dplane + r, 0.f);
        return;
    }
    item -= z_items;
    const unsigned per = (unsigned)a.ts * a.ncg_s;
    if (item >= (unsigned)a.s_frames * per) return;
    const int fi = item / per, q = item % per;                            // scatter group step
    const int strip = q % a.ts, cgi = q / a.ts;
    const int f = a.s_frame0 + fi;
    float* acc = a.acc + (size_t)(a.step & 1) * slot_floats + (size_t)fi * frame_floats;
    float* dplane = a.dacc + (size_t)(a.step % 3) * dslot + (size_t)fi * a.HW;
    planar_scatter_strip<T, TF>(a, f, strip, cgi * a.cg_s, min(a.Cq, (cgi + 1) * a.cg_s), cgi == 0 && a.mode != DCB_MODE_SUM,
                                acc, dplane, lane);
}

// ---------------------------------------------------------------------------------------------
// ONE launch for a call whose frames fit one group and whose warps are all resident at once (latents, small feature maps):
// every warp scatters its strip, the grid meets at a counter in the workspace, every warp normalises its chunk(s). The second
// launch of the pipeline and its dependency gap disappear -- and yet it is SLOWER on the B200: C2 latents 20.6-22.2 us per call
// under CUDA-graph replay (20 / 200 / 1000 ns back-off in the spin) against 16.4 us for the two programmatically chained
// launches (profiles/r02/NOTES.md section 11; round 1 measured the same with a cooperative launch). Opt-in only:
// dcb_set_option("planar_one_launch", 1).
// Safe because the host launches this kernel only when the whole grid is co-resident (at most half of the machine's CTA
// slots); launch_dependents is issued first, so a dependent grid cannot take slots before every CTA of this one is resident.
// The two counters are back at zero when the kernel ends (workspace protocol).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

#ifndef DCB_BAR_SLEEP
#define DCB_BAR_SLEEP 200
#endif
template <class T, class TF>
__global__ void __launch_bounds__(kPThreads, DCB_PMINCTAS) k_planar_one(const __grid_constant__ PlanarArgs a) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int lane = threadIdx.x & 31;
    const unsigned warps = gridDim.x * kPWarps;
    const unsigned item = blockIdx.x * kPWarps + (threadIdx.x >> 5);
    const size_t frame_floats = (size_t)a.Cq * a.HW * 4;
    {
        const unsigned per = (unsigned)a.ts * a.ncg_s;
        if (item < (unsigned)a.N * per) {
            const int fi = item / per, q = item % per;
            const int strip = q % a.ts, cgi = q / a.ts;
            planar_scatter_strip<T, TF>(a, fi, strip, cgi * a.cg_s, min(a.Cq, (cgi + 1) * a.cg_s), cgi == 0 && a.mode != DCB_MODE_SUM,
                                        a.acc + (size_t)fi * frame_floats, a.dacc + (size_t)fi * a.HW, lane);
        }
    }
    // ---- grid barrier: arrive (release), wait for everybody (acquire) ----
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(a.bar, 1u);
        while (ld_acquire_gpu(a.bar) < gridDim.x) __nanosleep(DCB_BAR_SLEEP);
    }
    __syncthreads();
    {
        const unsigned per = (unsigned)a.tn * a.ncg_n;
        for (unsigned it = item; it < (unsigned)a.N * per; it += warps) {
            const int fi = it / per, q = it % per;
            const int chunk = q % a.tn, cgi = q / a.tn;
            planar_normalize_chunk<T>(a, fi, chunk, cgi * a.cg_n, min(a.Cq, (cgi + 1) * a.cg_n), a.acc + (size_t)fi * frame_floats,
                                      a.dacc + (size_t)fi * a.HW, lane);
        }
    }
    // ---- depart: the last CTA to leave puts both counters back to zero ----
    __syncthreads();
    if (threadIdx.x == 0) {
        if (atomicAdd(a.bar + 1, 1u) == gridDim.x - 1) { a.bar[0] = 0u; a.bar[1] = 0u; }
    }
}

// ---------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------
extern long long g_pipe_group_bytes;      // splat_pipe.cu: dcb_set_option("pipe_group_bytes")

static long long planar_group_frames(long long N, long long C, long long H, long long W) {
    const long long per = (C + 3) / 4 * 16 * H * W;
    long long g = (g_pipe_group_bytes > 0 ? g_pipe_group_bytes : (long long)kPGroupBytes) / (per > 0 ? per : 1);
    if (g < 1) g = 1;
    return g > N ? (N < 1 ? 1 : N) : g;
}

static long long planar_chan_bytes(long long N, long long C, long long H, long long W) {
    const long long G = planar_group_frames(N, C, H, W);
    return align_up((N > G ? 2 : 1) * G * ((C + 3) / 4) * 16 * H * W, 256);
}

long long planar_workspace(long long N, long long C, long long H, long long W, int dtype, int mode) {
    (void)dtype;
    const long long G = planar_group_frames(N, C, H, W);
    const long long dbytes = mode == DCB_MODE_SUM ? 0 : align_up(3 * G * H * W * 4, 256);
    return planar_chan_bytes(N, C, H, W) + dbytes + 256;          // + the two counters of the single-launch kernel
}

// dcb_set_option("planar_one_launch", 1): the single-launch kernel where it applies (measured slower: default off)
int g_planar_one = 0;
void planar_set_one_launch(long long v) { g_planar_one = v != 0; }

// CTA slots of the device for k_planar_one (occupancy x SMs), queried once per instantiation
template <class T, class TF> static long long one_launch_slots() {
    static long long slots = -1;
    if (slots < 0) {
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_planar_one<T, TF>, kPThreads, 0) != cudaSuccess) per_sm = 0;
        slots = (long long)per_sm * device_sm_count();
    }
    return slots;
}

// split channels over several warps when the frames are too small to fill the machine
static void split_channels(long long items, int channels, int min_cg, int* cg, int* ncg) {
    const long long want = 148ll * 24;
    long long n = items > 0 ? (want + items - 1) / items : 1;
    const int max_n = channels / min_cg > 0 ? channels / min_cg : 1;
    if (n > max_n) n = max_n;
    if (n < 1) n = 1;
    *cg = (int)((channels + n - 1) / n);
    *ncg = (channels + *cg - 1) / *cg;
}

template <class T, class TF> static int launch_planar(PlanarArgs& a, cudaStream_t st) {
    const int groups = (a.N + a.G - 1) / a.G;
    const bool normalised = a.mode != DCB_MODE_SUM;
    // the single-launch kernel is opt-in evidence (measured slower) and has no fp16 instantiation
    if constexpr (!std::is_same<T, __half>::value) {
        if (g_planar_one && groups == 1) {
            // every scatter item needs its own warp; the normalise items are looped over. Half of the CTA slots at most.
            const long long s_items = (long long)a.N * a.ts * a.ncg_s;
            const long long ctas = (s_items + kPWarps - 1) / kPWarps;
            if (ctas > 0 && 2 * ctas <= one_launch_slots<T, TF>()) {
                a.step = 0; a.s_frame0 = a.n_frame0 = 0; a.s_frames = a.n_frames = a.N;
                DCB_CHECK_CUDA(launch_pdl(k_planar_one<T, TF>, dim3((unsigned)ctas), dim3(kPThreads), 0, st, a));
                count_launch();
                if (normalised && a.ncg_n > 1) DCB_CHECK_CUDA(cudaMemsetAsync(a.dacc, 0, (size_t)a.G * a.HW * 4, st));
                return DCB_OK;
            }
        }
    }
    for (int k = 0; k <= groups; ++k) {
        a.step = k;
        a.s_frame0 = k * a.G;
        a.s_frames = k < groups ? (a.N - a.s_frame0 < a.G ? a.N - a.s_frame0 : a.G) : 0;
        a.n_frame0 = (k - 1) * a.G;
        a.n_frames = k > 0 ? (a.N - a.n_frame0 < a.G ? a.N - a.n_frame0 : a.G) : 0;
        const long long items = (long long)a.n_frames * a.tn * a.ncg_n + (normalised ? (long long)a.G * a.tz : 0) +
                                (long long)a.s_frames * a.ts * a.ncg_s;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)((items + kPWarps - 1) / kPWarps)); cfg.blockDim = dim3(kPThreads); cfg.dynamicSmemBytes = 0; cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        DCB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, k_planar_step<T, TF>, a));
        count_launch();
    }
    // the normaliser slot read by the last step is the only part of the workspace left non-zero
    // (with one reader per cell the normalise items have zeroed it themselves)
    if (normalised && a.ncg_n > 1)
        DCB_CHECK_CUDA(cudaMemsetAsync(a.dacc + (size_t)((groups - 1) % 3) * a.G * a.HW, 0, (size_t)a.G * a.HW * 4, st));
    return DCB_OK;
}

// fp32 / bf16 / fp16, any channel count. `ws` must hold planar_workspace() bytes (all-zero if ws_clean).
int splat_planar_impl(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const DcbTensor* out,
                      const DcbTensor* norm, const DcbTensor* mask, void* ws, int mode, int eps, bool ws_clean,
                      cudaStream_t st) {
    PlanarArgs a;
    a.ones = 0;
    a.vec_in = planar_vec_ok(in) ? 1 : 0;
    a.in = make_view(in); a.flow = make_view(flow); a.metric = make_view(metric); a.mask = make_view(mask);
    a.N = (int)in->size[0]; a.C = (int)in->size[1]; a.H = (int)in->size[2]; a.W = (int)in->size[3];
    a.Cq = (a.C + 3) / 4;
    a.HW = (unsigned)(in->size[2] * in->size[3]);
    a.mode = mode; a.eps = eps;
    a.G = (int)planar_group_frames(a.N, a.C, a.H, a.W);
    a.tiles_x = (a.W + 31) / 32;
    a.ts = a.tiles_x * ((a.H + kPRows - 1) / kPRows);
    a.tn = (int)((a.HW + kPChunk - 1) / kPChunk);
    a.tz = (int)((a.HW + 1023) / 1024);
    const int frames_per_step = a.N < a.G ? a.N : a.G;
    split_channels((long long)frames_per_step * a.ts, a.Cq, 2, &a.cg_s, &a.ncg_s);
    split_channels((long long)frames_per_step * a.tn, a.Cq, 2, &a.cg_n, &a.ncg_n);
    a.out = out->ptr;
    a.norm = norm ? norm->ptr : nullptr;
    a.acc = (float*)ws;
    a.dacc = (float*)((char*)ws + planar_chan_bytes(a.N, a.C, a.H, a.W));
    a.bar = (unsigned*)((char*)ws + planar_workspace(a.N, a.C, a.H, a.W, in->dtype, mode) - 256);
    if (!ws_clean) DCB_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)planar_workspace(a.N, a.C, a.H, a.W, in->dtype, mode), st));
    const bool ff = flow->dtype == DCB_F32;
    if (in->dtype == DCB_F32) return launch_planar<float, float>(a, st);
    if (in->dtype == DCB_BF16)
        return ff ? launch_planar<__nv_bfloat16, float>(a, st) : launch_planar<__nv_bfloat16, __nv_bfloat16>(a, st);
    if (in->dtype == DCB_F16) return ff ? launch_planar<__half, float>(a, st) : launch_planar<__half, __half>(a, st);
    return set_error(DCB_E_DTYPE, "splat_planar: unsupported dtype %d", in->dtype);
}

}  // namespace dcb
