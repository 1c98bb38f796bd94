// det.cu -- optional deterministic forward (DCB_FLAG_DETERMINISTIC): sort-then-reduce, sm_100a.
//
// The default forward adds with L2 reductions, so the fp32 summation order (and the last bits
// of the result) change from run to run -- exactly like the reference's atomicAdd
// (controlnet/softsplat.py:320-334). This path reproduces the ONE order a sequential execution
// of the reference kernel would use (linear index ascending: for a target pixel that is
// ascending source index; see oracle/softsplat_oracle.c), so it is bit-identical run to run,
// across GPUs, and to the CPU oracle:
//
//   K6a emit   : every (source pixel, in-range corner) writes key = target * HW + source
//   sort       : 64-bit LSD radix sort of the keys (cub::DeviceRadixSort -- the one library call
//                in this library; it is off the hot path and takes its scratch from the caller's
//                workspace, so the no-allocation contract holds)
//   K6b reduce : one thread per target pixel binary-searches its key range and adds its
//                contributions sequentially, product rounded before each add, starting from +0
//   K2         : the ordinary normalise / cast epilogue (splat_fwd.cu).
#include "dcb_common.cuh"

#include <cub/device/device_radix_sort.cuh>

namespace dcb {

struct DetArgs {
    View in, flow, metric;
    unsigned long long* keys;
    const unsigned long long* sorted;
    void* acc;           // planar accumulators [N,Cacc,H,W] (or `out` for SUM)
    unsigned total, HW;
    long long nkeys;
    int N, C, H, W, Cacc, mode;
};

template <class T, class TF>
__global__ void __launch_bounds__(256) k_det_emit(const DetArgs a) {
    using A = typename Acc<T>::type;
    const unsigned p = blockIdx.x * 256 + threadIdx.x;
    if (p >= a.total) return;
    const unsigned n = p / a.HW, r = p - n * a.HW;
    const int y = (int)(r / (unsigned)a.W), x = (int)(r - (unsigned)y * (unsigned)a.W);
    const TF* fp = (const TF*)a.flow.p + n * a.flow.sN + y * a.flow.sH + x * a.flow.sW;
    const Foot<A> f = make_foot<A>(x, y, ld<A>(fp), ld<A>(fp + a.flow.sC));
    const int x1 = (int)((unsigned)f.x0 + 1u), y1 = (int)((unsigned)f.y0 + 1u);
    const bool vx0 = (unsigned)f.x0 < (unsigned)a.W, vx1 = (unsigned)x1 < (unsigned)a.W;
    const bool vy0 = (unsigned)f.y0 < (unsigned)a.H, vy1 = (unsigned)y1 < (unsigned)a.H;
    const bool b[4] = {f.finite && vx0 && vy0, f.finite && vx1 && vy0, f.finite && vx0 && vy1, f.finite && vx1 && vy1};
    const long long t0 = (long long)n * a.HW + (long long)f.y0 * a.W + f.x0;
    const long long off[4] = {0, 1, a.W, (long long)a.W + 1};
    const unsigned long long invalid = (unsigned long long)a.total * a.HW;   // sorts behind every real key
#pragma unroll
    for (int k = 0; k < 4; ++k)
        a.keys[4ull * p + k] = b[k] ? (unsigned long long)(t0 + off[k]) * a.HW + r : invalid;
}

template <class T, class TF, int CH>
__global__ void __launch_bounds__(256) k_det_reduce(const DetArgs a) {
    using A = typename Acc<T>::type;
    const unsigned p = blockIdx.x * 256 + threadIdx.x;   // target pixel (global over N)
    if (p >= a.total) return;
    const unsigned n = p / a.HW, r = p - n * a.HW;
    const int ty = (int)(r / (unsigned)a.W), tx = (int)(r - (unsigned)ty * (unsigned)a.W);
    const unsigned long long lo_key = (unsigned long long)p * a.HW, hi_key = lo_key + a.HW;
    long long lo = 0, hi = a.nkeys;                       // lower_bound(lo_key)
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (a.sorted[mid] < lo_key) lo = mid + 1; else hi = mid;
    }
    const long long first = lo;
    A* acc = (A*)a.acc + (long long)n * a.Cacc * a.HW + r;
    for (int cb = 0; cb < a.Cacc; cb += CH) {
        A sum[CH];
#pragma unroll
        for (int i = 0; i < CH; ++i) sum[i] = (A)0;
        for (long long q = first; q < a.nkeys; ++q) {
            const unsigned long long key = a.sorted[q];
            if (key >= hi_key) break;
            const unsigned s = (unsigned)(key - lo_key);
            const int y = (int)(s / (unsigned)a.W), x = (int)(s - (unsigned)y * (unsigned)a.W);
            const TF* fp = (const TF*)a.flow.p + n * a.flow.sN + y * a.flow.sH + x * a.flow.sW;
            const Foot<A> f = make_foot<A>(x, y, ld<A>(fp), ld<A>(fp + a.flow.sC));
            // which of the source's corners is this target?
            const int kx = tx - f.x0, ky = ty - f.y0;     // 0 or 1 each
            const A w = ky == 0 ? (kx == 0 ? f.wnw : f.wne) : (kx == 0 ? f.wsw : f.wse);
            A g = (A)1;
            if (a.mode == DCB_MODE_LINEAR || a.mode == DCB_MODE_SOFT) {
                const T* mp = (const T*)a.metric.p + n * a.metric.sN + y * a.metric.sH + x * a.metric.sW;
                const A m = ld<A>(mp);
                g = a.mode == DCB_MODE_SOFT ? exp_det_t(m) : m;     // portable exp: bit-identical to the oracle's orc_exp_det
            }
            const T* ip = (const T*)a.in.p + n * a.in.sN + y * a.in.sH + x * a.in.sW;
#pragma unroll
            for (int i = 0; i < CH; ++i) {
                const int c = cb + i;
                if (c < a.Cacc) {
                    A v;
                    if (c < a.C) {
                        v = ld<A>(ip + c * a.in.sC);
                        if (a.mode >= DCB_MODE_LINEAR) v = mul_rn(v, g);
                    } else {
                        v = g;
                    }
                    sum[i] = det_add(sum[i], v, w);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < CH; ++i)
            if (cb + i < a.Cacc) acc[(long long)(cb + i) * a.HW] = sum[i];
    }
}

size_t cub_temp_bytes(long long nkeys, int end_bit) {
    size_t bytes = 0;
    const cudaError_t e = cub::DeviceRadixSort::SortKeys(nullptr, bytes, (const unsigned long long*)nullptr,
                                                         (unsigned long long*)nullptr, (int)nkeys, 0, end_bit);
    if (e != cudaSuccess) {   // no device (size query on a CPU-only host): conservative bound
        (void)cudaGetLastError();
        bytes = (size_t)nkeys * 8 + (8u << 20);
    }
    return bytes;
}

int key_bits(long long total, long long span) {
    // keys go up to total*span (the "invalid" key) inclusive
    const unsigned long long maxkey = (unsigned long long)total * (unsigned long long)span;
    int bits = 1;
    while (bits < 64 && (maxkey >> bits) != 0) ++bits;
    return bits;
}

int det_sort_keys(void* temp, size_t temp_bytes, const unsigned long long* keys, unsigned long long* sorted, long long nkeys,
                  int end_bit, cudaStream_t st) {
    DCB_CHECK_CUDA(cub::DeviceRadixSort::SortKeys(temp, temp_bytes, keys, sorted, (int)nkeys, 0, end_bit, st));
    count_launch(8);   // histogram + onesweep passes (library kernels)
    return DCB_OK;
}

struct DetLayout {
    long long keys_off, sorted_off, temp_off, acc_off, total_bytes;
    size_t temp_bytes;
};

static DetLayout det_layout(long long N, long long C, long long H, long long W, int dtype, int mode) {
    DetLayout L;
    const long long total = N * H * W, nkeys = 4 * total;
    const long long cacc = C + (mode == DCB_MODE_SUM ? 0 : 1);
    L.temp_bytes = nkeys > 0 && nkeys < (1ll << 31) ? cub_temp_bytes(nkeys, key_bits(total, H * W)) : 0;
    L.keys_off = 0;
    L.sorted_off = align_up(nkeys * 8, 256);
    L.temp_off = L.sorted_off + align_up(nkeys * 8, 256);
    L.acc_off = L.temp_off + align_up((long long)L.temp_bytes, 256);
    const bool acc_is_out = mode == DCB_MODE_SUM && (dtype == DCB_F32 || dtype == DCB_F64);   // 16-bit outputs need the fp32 planes
    L.total_bytes = L.acc_off + (acc_is_out ? 0 : align_up(total * cacc * (dtype == DCB_F64 ? 8 : 4), 256));
    return L;
}

long long det_workspace(long long N, long long C, long long H, long long W, int dtype, int mode) {
    return det_layout(N, C, H, W, dtype, mode).total_bytes;
}

// defined in splat_fwd.cu
int normalize_planar_launch(int dtype, const DcbTensor* in, const DcbTensor* out, const DcbTensor* norm,
                            const DcbTensor* mask, void* acc, int mode, int eps, cudaStream_t st);

template <class T, class TF>
static int launch_det(DetArgs& a, const DetLayout& L, char* ws, cudaStream_t st) {
    const unsigned blocks = (a.total + 255) / 256;
    k_det_emit<T, TF><<<blocks, 256, 0, st>>>(a);
    DCB_CHECK_LAUNCH("k_det_emit");
    const int rc = det_sort_keys(ws + L.temp_off, L.temp_bytes, a.keys, (unsigned long long*)a.sorted, a.nkeys,
                                 key_bits(a.total, a.HW), st);
    if (rc != DCB_OK) return rc;
    k_det_reduce<T, TF, 4><<<blocks, 256, 0, st>>>(a);
    DCB_CHECK_LAUNCH("k_det_reduce");
    return DCB_OK;
}

int splat_fwd_det_impl(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const DcbTensor* out,
                       const DcbTensor* norm, const DcbTensor* mask, void* ws, long long ws_bytes, int mode, int eps,
                       int flags, cudaStream_t st) {
    (void)flags;
    DetArgs a;
    a.in = make_view(in); a.flow = make_view(flow); a.metric = make_view(metric);
    a.N = (int)in->size[0]; a.C = (int)in->size[1]; a.H = (int)in->size[2]; a.W = (int)in->size[3];
    a.HW = (unsigned)(in->size[2] * in->size[3]);
    a.total = (unsigned)(in->size[0] * in->size[2] * in->size[3]);
    a.Cacc = a.C + (mode == DCB_MODE_SUM ? 0 : 1);
    a.mode = mode;
    a.nkeys = 4ll * a.total;
    if (a.total == 0 || a.C == 0) return DCB_OK;
    if (a.nkeys >= (1ll << 31))
        return set_error(DCB_E_LIMIT, "splat_fwd(deterministic): 4*N*H*W must stay below 2^31 (got %lld)", a.nkeys);
    const DetLayout L = det_layout(a.N, a.C, a.H, a.W, in->dtype, mode);
    if (!ws || ws_bytes < L.total_bytes || ((uintptr_t)ws & 255))
        return set_error(DCB_E_WORKSPACE, "splat_fwd(deterministic): workspace of %lld bytes required, got %lld",
                         L.total_bytes, ws_bytes);
    char* base = (char*)ws;
    a.keys = (unsigned long long*)(base + L.keys_off);
    a.sorted = (const unsigned long long*)(base + L.sorted_off);
    const bool acc_is_out = mode == DCB_MODE_SUM && (in->dtype == DCB_F32 || in->dtype == DCB_F64);
    a.acc = acc_is_out ? out->ptr : (void*)(base + L.acc_off);

    const bool ff = flow->dtype == DCB_F32;
    int rc;
    switch (in->dtype) {
        case DCB_F32: rc = launch_det<float, float>(a, L, base, st); break;
        case DCB_F64: rc = launch_det<double, double>(a, L, base, st); break;
        case DCB_BF16:
            rc = ff ? launch_det<__nv_bfloat16, float>(a, L, base, st) : launch_det<__nv_bfloat16, __nv_bfloat16>(a, L, base, st);
            break;
        case DCB_F16: rc = ff ? launch_det<__half, float>(a, L, base, st) : launch_det<__half, __half>(a, L, base, st); break;
        default: return set_error(DCB_E_DTYPE, "splat_fwd(deterministic): unsupported dtype %d", in->dtype);
    }
    if (rc != DCB_OK || acc_is_out) return rc;
    return normalize_planar_launch(in->dtype, in, out, norm, mask, a.acc, mode, eps, st);
}

}  // namespace dcb
