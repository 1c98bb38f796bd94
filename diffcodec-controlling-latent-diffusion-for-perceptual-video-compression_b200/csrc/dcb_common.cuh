// dcb_common.cuh -- shared device/host helpers for libdiffcodec_b200.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <atomic>

#include "diffcodec_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libdiffcodec_b200 is written for sm_100a (B200) only"
#endif

#define DCB_STR_(x) #x
#define DCB_STR(x) DCB_STR_(x)

namespace dcb {

// ------------------------------------------------------------------------------------------------
// host side: errors, launch accounting
// ------------------------------------------------------------------------------------------------
int set_error(int code, const char* fmt, ...);
extern std::atomic<long long> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// After a <<<>>> launch: convert a launch error into the ABI's positive cudaError_t code.
#define DCB_CHECK_LAUNCH(what)                                                        \
    do {                                                                              \
        cudaError_t e__ = cudaGetLastError();                                         \
        if (e__ != cudaSuccess)                                                       \
            return dcb::set_error((int)e__, "%s: %s", what, cudaGetErrorString(e__)); \
        dcb::count_launch();                                                          \
    } while (0)

#define DCB_CHECK_CUDA(expr)                                                           \
    do {                                                                               \
        cudaError_t e__ = (expr);                                                      \
        if (e__ != cudaSuccess)                                                        \
            return dcb::set_error((int)e__, "%s: %s", #expr, cudaGetErrorString(e__)); \
    } while (0)

// Programmatic dependent launch: the kernel may be scheduled while its predecessor in the stream
// drains; it must call pdl_wait() (device side) before it touches anything the predecessor wrote.
template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Strided 4-d view handed to kernels by value (strides in elements).
struct View {
    const void* p;
    long long sN, sC, sH, sW;
};

inline View make_view(const DcbTensor* t) {
    View v;
    v.p = t ? t->ptr : nullptr;
    v.sN = t ? t->stride[0] : 0;
    v.sC = t ? t->stride[1] : 0;
    v.sH = t ? t->stride[2] : 0;
    v.sW = t ? t->stride[3] : 0;
    return v;
}

inline bool is_contig(const DcbTensor* t) {
    long long e = 1;
    for (int d = 3; d >= 0; --d) {
        if (t->size[d] != 1 && t->stride[d] != e) return false;
        e *= t->size[d];
    }
    return true;
}

inline int elem_size(int dtype) { return dtype == DCB_F64 ? 8 : (dtype == DCB_BF16 ? 2 : 4); }

inline long long align_up(long long v, long long a) { return (v + a - 1) / a * a; }

int device_sm_count();

// ------------------------------------------------------------------------------------------------
// device side
// ------------------------------------------------------------------------------------------------
// let the next kernel of the stream start its launch now; wait until the previous one has completed
// and its writes are visible (both are no-ops for a kernel launched without the PDL attribute)
__device__ __forceinline__ void pdl_wait() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

template <class T> struct Acc { using type = float; };
template <> struct Acc<double> { using type = double; };

template <class A, class T> __device__ __forceinline__ A ld(const T* p) { return (A)(*p); }
template <> __device__ __forceinline__ float ld<float, __nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }

template <class T, class A> __device__ __forceinline__ void st(T* p, A v) { *p = (T)v; }
template <> __device__ __forceinline__ void st<__nv_bfloat16, float>(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

// streaming variants (ld.global.cs / st.global.cs: evict-first in L1 and L2) for data touched once:
// they keep the inputs / outputs from pushing the fp32 accumulators out of L2
__device__ __forceinline__ float ld_stream(const float* p) { return __ldcs(p); }
__device__ __forceinline__ double ld_stream(const double* p) { return __ldcs(p); }
__device__ __forceinline__ void st_stream(double* p, double v) { __stcs(p, v); }
// the value a store of `v` into a T would leave behind
template <class T> __device__ __forceinline__ float round_as(float v) { return v; }
template <> __device__ __forceinline__ float round_as<__nv_bfloat16>(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
template <class T> __device__ __forceinline__ double round_as(double v) { return v; }
__device__ __forceinline__ float ld_stream(const __nv_bfloat16* p) { return __bfloat162float(__ldcs(p)); }
__device__ __forceinline__ void st_stream(float* p, float v) { __stcs(p, v); }
__device__ __forceinline__ void st_stream(__nv_bfloat16* p, float v) { __stcs(p, __float2bfloat16_rn(v)); }

// two neighbouring elements with one load (the address is aligned to the pair)
__device__ __forceinline__ float2 ld2_stream(const float* p) { return __ldcs((const float2*)p); }
__device__ __forceinline__ float2 ld2_stream(const __nv_bfloat16* p) {
    const unsigned u = __ldcs((const unsigned*)p);
    return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u));
}

// rounded (non-contracted) arithmetic: the reference rounds every product before the atomic add
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float sub_rn(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double sub_rn(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float fma_rn(float a, float b, float c) { return __fmaf_rn(a, b, c); }
__device__ __forceinline__ double fma_rn(double a, double b, double c) { return __fma_rn(a, b, c); }

__device__ __forceinline__ float floor_t(float v) { return floorf(v); }
__device__ __forceinline__ double floor_t(double v) { return floor(v); }
__device__ __forceinline__ float exp_t(float v) { return expf(v); }
__device__ __forceinline__ double exp_t(double v) { return exp(v); }
// exp() of the deterministic mode: IEEE double operations only (rint, fma, scalbn), spelled exactly like
// orc_exp_det() in oracle/softsplat_oracle.c, so that the CUDA result and the CPU oracle agree BIT FOR BIT (libm's and
// CUDA's expf differ by an ulp here and there). |relative error| < 2e-16 before the rounding to float.
__device__ __forceinline__ double exp_det(double x) {
    if (!(x == x)) return x;
    if (x > 709.0) return __longlong_as_double(0x7ff0000000000000ll);
    if (x < -745.0) return 0.0;
    const double k = rint(x * 1.4426950408889634);
    double r = fma(-k, 6.93147180369123816490e-01, x);
    r = fma(-k, 1.90821492927058770002e-10, r);
    double p = 1.6059043836821613e-10;                    // 1/13!
    p = fma(p, r, 2.08767569878681e-09);                  // 1/12!
    p = fma(p, r, 2.505210838544172e-08);
    p = fma(p, r, 2.755731922398589e-07);
    p = fma(p, r, 2.7557319223985893e-06);
    p = fma(p, r, 2.48015873015873e-05);
    p = fma(p, r, 0.0001984126984126984);
    p = fma(p, r, 0.001388888888888889);
    p = fma(p, r, 0.008333333333333333);
    p = fma(p, r, 0.041666666666666664);
    p = fma(p, r, 0.16666666666666666);
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    p = fma(p, r, 1.0);
    return scalbn(p, (int)k);
}
__device__ __forceinline__ float exp_det_t(float v) { return (float)exp_det((double)v); }
__device__ __forceinline__ double exp_det_t(double v) { return exp_det(v); }
__device__ __forceinline__ int to_int_sat(float v) { return __float2int_rz(v); }   // cvt.rzi.s32.f32 saturates
__device__ __forceinline__ int to_int_sat(double v) { return __double2int_rz(v); }
__device__ __forceinline__ bool finite_t(float v) { return isfinite(v); }
__device__ __forceinline__ bool finite_t(double v) { return isfinite(v); }

// no-return reductions (REDG); the float4 form is one 16-byte L2 transaction per lane (sm_90+)
__device__ __forceinline__ void red_add(float* p, float v) { atomicAdd(p, v); }
__device__ __forceinline__ void red_add(double* p, double v) { atomicAdd(p, v); }
__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void red_add_v2(float* p, float a, float b) {
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(a), "f"(b) : "memory");
}

// occlusion test of compute_mask (controlnet/control_utils.py:15-16) on the soft splat (wx, wy) / (d + 1e-7) of one motion
// field, compared with the other field (mx, my) at the same pixel: ||m + w|| > 0.3.
// The square root is never taken: sqrt is monotone and correctly rounded, so sqrtf(s) > 0.3f holds exactly when
// s > 0x3DB851ED (0.09000001f, the largest float whose root still rounds to 0.3f or below; checked exhaustively around it).
__device__ __forceinline__ float occlusion(float wx, float wy, float d, float mx, float my) {
    const float n = add_rn(d, 0.0000001f);
    const float ex = add_rn(mx, wx / n), ey = add_rn(my, wy / n);
    return add_rn(mul_rn(ex, ex), mul_rn(ey, ey)) > __uint_as_float(0x3DB851EDu) ? 1.f : 0.f;
}

// soft_fuse (improv_experiments.ipynb cell 3) of two warps on the VALID masks 1 - occ_fwd, 1 - occ_bwd of two binary occlusion
// masks: clamp(M) / (M.sum() + 1e-6) takes one of three values, 0, 1 / (1 + 1e-6) or 1 / (2 + 1e-6) (IEEE divisions of
// constants, folded at compile time: exactly what the per-pixel division gives); where both references are occluded
// (M_fwd + M_bwd < 0.5) the result is 0.5 * (warped1 + warped2). Equal to bidir_fuse(w1, w2, 1 - of, 1 - ob, of, ob).
__device__ __forceinline__ float bidir_soft_fuse(float w1, float w2, float of, float ob) {
    const float one_of_one = 1.f / (1.f + 0.000001f), one_of_two = 1.f / (2.f + 0.000001f);
    const bool v1 = of == 0.f, v2 = ob == 0.f;
    if (!v1 && !v2) return mul_rn(0.5f, add_rn(w1, w2));
    const float k1 = v1 ? (v2 ? one_of_two : one_of_one) : 0.f, k2 = v2 ? (v1 ? one_of_two : one_of_one) : 0.f;
    return add_rn(mul_rn(k1, w1), mul_rn(k2, w2));
}

// Bilinear footprint of one source pixel: softsplat.py:298-318 (and :386-404, :457-470).
template <class A> struct Foot {
    A fx, fy;        // landing position
    int x0, y0;      // north-west corner
    A wnw, wne, wsw, wse;
    bool finite;
};

template <class A> __device__ __forceinline__ Foot<A> make_foot(int x, int y, A flow_x, A flow_y) {
    Foot<A> f;
    f.fx = add_rn((A)x, flow_x);
    f.fy = add_rn((A)y, flow_y);
    f.finite = finite_t(f.fx) && finite_t(f.fy);
    f.x0 = to_int_sat(floor_t(f.fx));
    f.y0 = to_int_sat(floor_t(f.fy));
    // `x0 + 1` wraps on the device exactly like the reference's int arithmetic
    const A x0f = (A)f.x0, y0f = (A)f.y0;
    const A x1f = (A)(int)((unsigned)f.x0 + 1u), y1f = (A)(int)((unsigned)f.y0 + 1u);
    const A ex = sub_rn(x1f, f.fx), ey = sub_rn(y1f, f.fy);   // (SE - f)
    const A dx = sub_rn(f.fx, x0f), dy = sub_rn(f.fy, y0f);   // (f - NW)
    f.wnw = mul_rn(ex, ey);
    f.wne = mul_rn(dx, ey);
    f.wsw = mul_rn(ex, dy);
    f.wse = mul_rn(dx, dy);
    return f;
}

}  // namespace dcb
