// api.cu -- the C ABI of libdiffcodec_b200.so (include/diffcodec_b200.h): argument validation,
// error reporting, launch accounting. No allocation, no synchronisation, no stream creation.
#include "dcb_common.cuh"

#include <initializer_list>
#include <string.h>

namespace dcb {

std::atomic<long long> g_launches{0};
static thread_local char t_error[512] = "";

int set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(t_error, sizeof(t_error), fmt, ap);
    va_end(ap);
    return code;
}

int device_sm_count() {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
            sms = n;
        else
            sms = 148;
    }
    return sms;
}

// implemented in the kernel translation units
long long splat_fwd_workspace(long long N, long long C, long long H, long long W, int dtype, int mode);
long long splat_bwd_workspace(long long N, long long C, long long H, long long W, int dtype, int mode);
long long det_workspace(long long N, long long C, long long H, long long W, int dtype, int mode);
int splat_fwd_impl(const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*,
                   const DcbTensor*, void*, long long, int, int, int, cudaStream_t);
int splat_fwd_det_impl(const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*,
                       const DcbTensor*, void*, long long, int, int, int, cudaStream_t);
int splat_bwd_impl(const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*,
                   const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, void*,
                   long long, int, int, cudaStream_t);
int backwarp_fwd_impl(const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, int,
                      cudaStream_t);
long long backwarp_bwd_workspace(long long N, long long C, long long H, long long W, int dtype);
int backwarp_bwd_impl(const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, int,
                      void*, long long, cudaStream_t);
long long mask_workspace(long long N, long long H, long long W);
long long recipe_workspace(long long N, long long C, long long H, long long W);
int occlusion_mask_impl(const DcbTensor*, const DcbTensor*, const DcbTensor*, void*, long long, int, cudaStream_t);
int residual_fused_impl(const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*,
                        const DcbTensor*, const DcbTensor*, const DcbTensor*, void*, long long, int, int, cudaStream_t);
int residual_bidir_impl(const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*,
                        const DcbTensor*, const DcbTensor*, const DcbTensor*, void*, long long, int, cudaStream_t);
int bidir_fuse_fwd_impl(const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*,
                        const DcbTensor*, const DcbTensor*, cudaStream_t);
int bidir_fuse_bwd_impl(const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*,
                        const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*,
                        const DcbTensor*, cudaStream_t);

long long block_fwd_acc_bytes(long long N, long long C, long long H, long long W, int dtype);
long long block_fwd_scratch_bytes(long long N, long long C, long long H, long long W, int dtype);
long long block_bwd_scratch_bytes(long long N, long long C, long long H, long long W, int dtype);
int bidir_block_fwd_impl(const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*,
                         const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*,
                         const DcbTensor*, void*, long long, void*, long long, int, cudaStream_t);
int bidir_block_bwd_impl(const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*,
                         const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*,
                         const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, const DcbTensor*, void*, long long,
                         cudaStream_t);
int flow_ingest_impl(const DcbTensor* flow, const DcbTensor* out, int mode, cudaStream_t st);
long long pyramid_workspace(const DcbPyramidLevel* lv, int n);
long long pyramid_det_workspace(const DcbPyramidLevel* lv, int n);
long long pyramid_det_keys(const DcbPyramidLevel* lv, int n);
int bidir_pyramid_fwd_impl(const DcbPyramidLevel* lv, int n, void* ws, int flags, cudaStream_t st);
long long pyramid_bwd_workspace(const DcbPyramidBwdLevel* lv, int n);
int bidir_pyramid_bwd_impl(const DcbPyramidBwdLevel* lv, int n, void* ws, bool holes, cudaStream_t st);
int resample_batch_impl(const DcbResampleJob* jobs, int n_jobs, cudaStream_t st);
int convert_impl(const void* src, int src_dtype, void* dst, int dst_dtype, long long n, float scale, cudaStream_t st);
extern int g_fwd_path;
bool use_owner(int dtype, int mode, long long C, long long H, long long W);
bool fwd_ws_is_scratch(long long N, long long C, long long H, long long W, int dtype, int mode);
void owner_set_group_bytes(long long b);
void pipe_set_group_bytes(long long b);
void pipe_set_ring_slots(long long n);
void bwd_set_group_bytes(long long b);
void pipe_set_tail_percent(long long p);
void lists_set_nhwc(long long v);
void bwd_set_flat(long long v);
void planar_set_one_launch(long long v);

long long tile_merge_workspace(long long C, long long H, long long W, int n_tiles);
int tile_merge_impl(const DcbTensor*, const long long*, int, const DcbTensor*, long long, long long, double, void*, long long,
                    cudaStream_t);

// ---------------------------------------------------------------------------------------------
// validation helpers
// ---------------------------------------------------------------------------------------------
static int check_tensor(const char* fn, const char* name, const DcbTensor* t, bool required) {
    if (!t) return required ? set_error(DCB_E_NULL, "%s: %s is required", fn, name) : DCB_OK;
    if (t->dtype != DCB_F32 && t->dtype != DCB_BF16 && t->dtype != DCB_F16 && t->dtype != DCB_F64)
        return set_error(DCB_E_DTYPE, "%s: %s has unsupported dtype %d", fn, name, t->dtype);
    long long numel = 1;
    for (int d = 0; d < 4; ++d) {
        if (t->size[d] < 0) return set_error(DCB_E_SHAPE, "%s: %s has a negative size", fn, name);
        numel *= t->size[d];
    }
    if (numel > 0 && !t->ptr) return set_error(DCB_E_NULL, "%s: %s has a null data pointer", fn, name);
    if ((uintptr_t)t->ptr % (uintptr_t)elem_size(t->dtype))
        return set_error(DCB_E_ALIGN, "%s: %s is not aligned to its element size", fn, name);
    return DCB_OK;
}

static int check_shape(const char* fn, const char* name, const DcbTensor* t, long long N, long long C, long long H,
                       long long W) {
    if (!t) return DCB_OK;
    if (t->size[0] != N || t->size[1] != C || t->size[2] != H || t->size[3] != W)
        return set_error(DCB_E_SHAPE, "%s: %s is [%lld,%lld,%lld,%lld], expected [%lld,%lld,%lld,%lld]", fn, name,
                         (long long)t->size[0], (long long)t->size[1], (long long)t->size[2], (long long)t->size[3], N,
                         C, H, W);
    return DCB_OK;
}

static int check_out(const char* fn, const char* name, const DcbTensor* t, int dtype, int align) {
    if (!t) return DCB_OK;
    if (t->dtype != dtype) return set_error(DCB_E_DTYPE, "%s: %s has dtype %d, expected %d", fn, name, t->dtype, dtype);
    if (!is_contig(t)) return set_error(DCB_E_SHAPE, "%s: %s must be NCHW-contiguous", fn, name);
    if ((uintptr_t)t->ptr % (uintptr_t)align) return set_error(DCB_E_ALIGN, "%s: %s must be %d-byte aligned", fn, name, align);
    return DCB_OK;
}

static int check_limits(const char* fn, const DcbTensor* t) {
    const long long N = t->size[0], C = t->size[1], H = t->size[2], W = t->size[3];
    if (H * W >= (1ll << 31) || N * H * W >= (1ll << 31) || C >= (1ll << 24) || H >= (1 << 24) || W >= (1 << 24))
        return set_error(DCB_E_LIMIT, "%s: sizes [%lld,%lld,%lld,%lld] exceed kernel index limits (N*H*W < 2^31)", fn, N, C, H, W);
    return DCB_OK;
}

static int flow_dtype_ok(const char* fn, const DcbTensor* in, const DcbTensor* flow) {
    if (flow->dtype == in->dtype) return DCB_OK;
    if (is_half_storage(in->dtype) && flow->dtype == DCB_F32) return DCB_OK;
    return set_error(DCB_E_DTYPE, "%s: flow dtype %d does not go with tensor dtype %d", fn, flow->dtype, in->dtype);
}

// the entries without fp16 kernels (backwarp, occlusion mask, conditioning recipes, flow resize) refuse F16 before any launch
static int refuse_f16(const char* fn, std::initializer_list<const DcbTensor*> ts) {
    for (const DcbTensor* t : ts)
        if (t && t->dtype == DCB_F16) return set_error(DCB_E_DTYPE, "%s: F16 is not supported by this entry", fn);
    return DCB_OK;
}

#define TRY(expr)                  \
    do {                           \
        int rc__ = (expr);         \
        if (rc__ != DCB_OK) return rc__; \
    } while (0)

static int acc_dtype(int dtype) { return dtype == DCB_F64 ? DCB_F64 : DCB_F32; }

}  // namespace dcb

using namespace dcb;

extern "C" {

int dcb_version(void) { return DCB_VERSION; }
const char* dcb_last_error(void) { return t_error; }
int64_t dcb_launch_count(void) { return (int64_t)g_launches.load(); }

const char* dcb_build_info(void) {
    return "libdiffcodec_b200 " __DATE__ " nvcc " DCB_STR(__CUDACC_VER_MAJOR__) "." DCB_STR(__CUDACC_VER_MINOR__)
           " target sm_100a; kernels: k_splat_step k_planar_step k_list_count k_list_alloc k_list_fill k_list_gather k_scatter_planar k_normalize k_bwd_target k_bwd_source "
           "k_backwarp_rows k_backwarp_fwd k_backwarp_bwd k_cast_f32_bf16 k_recipe_fuse k_bidir_fuse_fwd k_bidir_fuse_bwd "
           "k_det_emit k_det_reduce k_tile_merge k_splat_owner k_strip_box k_convert k_flow_ingest k_pyr_scatter k_pyr_fuse k_pyr_det_emit k_pyr_det_reduce k_resample_batch k_splat_cluster";
}

int64_t dcb_splat_fwd_workspace_bytes(int64_t N, int64_t C, int64_t H, int64_t W, int32_t dtype, int32_t mode, int32_t flags) {
    if (N < 0 || C < 0 || H < 0 || W < 0) return 0;
    if (flags & DCB_FLAG_DETERMINISTIC) return (int64_t)det_workspace(N, C, H, W, dtype, mode);
    return (int64_t)splat_fwd_workspace(N, C, H, W, dtype, mode);
}

int32_t dcb_splat_fwd_workspace_is_scratch(int64_t N, int64_t C, int64_t H, int64_t W, int32_t dtype, int32_t mode, int32_t flags) {
    if (flags & DCB_FLAG_DETERMINISTIC) return 1;
    return fwd_ws_is_scratch(N, C, H, W, dtype, mode) ? 1 : 0;
}

int dcb_set_option(const char* name, int64_t value) {
    if (!name) return set_error(DCB_E_NULL, "dcb_set_option: name is required");
    if (!strcmp(name, "fwd_path")) {
        if (value < 0 || value > 2) return set_error(DCB_E_MODE, "dcb_set_option: fwd_path is 0, 1 or 2");
        g_fwd_path = (int)value;
        return DCB_OK;
    }
    if (!strcmp(name, "pipe_group_bytes")) { pipe_set_group_bytes(value); return DCB_OK; }
    if (!strcmp(name, "pipe_ring_slots")) { pipe_set_ring_slots(value); return DCB_OK; }
    if (!strcmp(name, "owner_group_bytes")) { owner_set_group_bytes(value); return DCB_OK; }
    if (!strcmp(name, "bwd_group_bytes")) { bwd_set_group_bytes(value); return DCB_OK; }
    if (!strcmp(name, "pipe_tail_percent")) { pipe_set_tail_percent(value); return DCB_OK; }
    if (!strcmp(name, "lists_nhwc")) { lists_set_nhwc(value); return DCB_OK; }
    if (!strcmp(name, "bwd_flat")) { bwd_set_flat(value); return DCB_OK; }
    if (!strcmp(name, "planar_one_launch")) { planar_set_one_launch(value); return DCB_OK; }
    return set_error(DCB_E_MODE, "dcb_set_option: unknown option '%s'", name);
}

int64_t dcb_splat_bwd_workspace_bytes(int64_t N, int64_t C, int64_t H, int64_t W, int32_t dtype, int32_t mode, int32_t flags) {
    (void)flags;
    if (N < 0 || C < 0 || H < 0 || W < 0) return 0;
    return (int64_t)splat_bwd_workspace(N, C, H, W, dtype, mode);
}

int64_t dcb_splat_workspace_bytes(int64_t N, int64_t C, int64_t H, int64_t W, int32_t dtype, int32_t mode, int32_t flags) {
    const int64_t f = dcb_splat_fwd_workspace_bytes(N, C, H, W, dtype, mode, flags);
    const int64_t b = dcb_splat_bwd_workspace_bytes(N, C, H, W, dtype, mode, flags);
    return f > b ? f : b;
}

int dcb_splat_fwd(const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric, const DcbTensor* out,
                  const DcbTensor* norm, const DcbTensor* mask, void* ws, int64_t ws_bytes, int32_t mode, int32_t eps,
                  int32_t flags, void* stream) {
    const char* fn = "dcb_splat_fwd";
    TRY(check_tensor(fn, "in", in, true));
    TRY(check_tensor(fn, "flow", flow, true));
    TRY(check_tensor(fn, "metric", metric, false));
    TRY(check_tensor(fn, "out", out, true));
    TRY(check_tensor(fn, "norm", norm, false));
    TRY(check_tensor(fn, "mask", mask, false));
    if (mode < DCB_MODE_SUM || mode > DCB_MODE_SOFT) return set_error(DCB_E_MODE, "%s: unknown mode %d", fn, mode);
    if (eps < DCB_EPS_ADD || eps > DCB_EPS_CLIP) return set_error(DCB_E_MODE, "%s: unknown eps rule %d", fn, eps);
    if (flags & ~(DCB_FLAG_DETERMINISTIC | DCB_FLAG_WS_CLEAN)) return set_error(DCB_E_MODE, "%s: unknown flags 0x%x", fn, flags);
    // softsplat.py:235-238
    if ((mode == DCB_MODE_SUM || mode == DCB_MODE_AVG) && metric) return set_error(DCB_E_MODE, "%s: metric must be NULL for sum/avg", fn);
    if ((mode == DCB_MODE_LINEAR || mode == DCB_MODE_SOFT) && !metric) return set_error(DCB_E_MODE, "%s: metric is required for linear/soft", fn);
    if (mode == DCB_MODE_SUM && (mask || norm)) return set_error(DCB_E_MODE, "%s: mask/norm need a normalised mode", fn);
    const long long N = in->size[0], C = in->size[1], H = in->size[2], W = in->size[3];
    TRY(check_limits(fn, in));
    TRY(check_shape(fn, "flow", flow, N, 2, H, W));       // softsplat.py:296
    TRY(check_shape(fn, "metric", metric, N, 1, H, W));
    TRY(check_shape(fn, "out", out, N, C, H, W));
    TRY(check_shape(fn, "norm", norm, N, 1, H, W));
    TRY(check_shape(fn, "mask", mask, N, 1, H, W));
    TRY(flow_dtype_ok(fn, in, flow));
    if (metric && metric->dtype != in->dtype) return set_error(DCB_E_DTYPE, "%s: metric dtype differs from in", fn);
    if (mask && mask->dtype != in->dtype) return set_error(DCB_E_DTYPE, "%s: mask dtype differs from in", fn);
    TRY(check_out(fn, "out", out, in->dtype, elem_size(in->dtype)));
    TRY(check_out(fn, "norm", norm, acc_dtype(in->dtype), elem_size(acc_dtype(in->dtype))));
    if (flags & DCB_FLAG_DETERMINISTIC)
        return splat_fwd_det_impl(in, flow, metric, out, norm, mask, ws, ws_bytes, mode, eps, flags, (cudaStream_t)stream);
    return splat_fwd_impl(in, flow, metric, out, norm, mask, ws, ws_bytes, mode, eps, flags, (cudaStream_t)stream);
}

int dcb_splat_bwd(const DcbTensor* gout, const DcbTensor* in, const DcbTensor* flow, const DcbTensor* metric,
                  const DcbTensor* out, const DcbTensor* norm, const DcbTensor* mask, const DcbTensor* gin,
                  const DcbTensor* gflow, const DcbTensor* gmetric, void* ws, int64_t ws_bytes, int32_t mode,
                  int32_t eps, int32_t flags, void* stream) {
    const char* fn = "dcb_splat_bwd";
    (void)flags;
    TRY(check_tensor(fn, "grad_out", gout, true));
    TRY(check_tensor(fn, "in", in, true));
    TRY(check_tensor(fn, "flow", flow, true));
    TRY(check_tensor(fn, "metric", metric, false));
    TRY(check_tensor(fn, "out", out, false));
    TRY(check_tensor(fn, "norm", norm, false));
    TRY(check_tensor(fn, "mask", mask, false));
    TRY(check_tensor(fn, "grad_in", gin, false));
    TRY(check_tensor(fn, "grad_flow", gflow, false));
    TRY(check_tensor(fn, "grad_metric", gmetric, false));
    if (mode < DCB_MODE_SUM || mode > DCB_MODE_SOFT) return set_error(DCB_E_MODE, "%s: unknown mode %d", fn, mode);
    if (eps < DCB_EPS_ADD || eps > DCB_EPS_CLIP) return set_error(DCB_E_MODE, "%s: unknown eps rule %d", fn, eps);
    if ((mode == DCB_MODE_LINEAR || mode == DCB_MODE_SOFT) && !metric) return set_error(DCB_E_MODE, "%s: metric is required for linear/soft", fn);
    if ((mode == DCB_MODE_SUM || mode == DCB_MODE_AVG) && (metric || gmetric)) return set_error(DCB_E_MODE, "%s: no metric in sum/avg", fn);
    if (mode != DCB_MODE_SUM && (!out || !norm)) return set_error(DCB_E_NULL, "%s: out and norm of the forward are required", fn);
    if (mode == DCB_MODE_SUM && mask) return set_error(DCB_E_MODE, "%s: mask needs a normalised mode", fn);
    const long long N = in->size[0], C = in->size[1], H = in->size[2], W = in->size[3];
    TRY(check_limits(fn, in));
    TRY(check_shape(fn, "grad_out", gout, N, C, H, W));
    TRY(check_shape(fn, "flow", flow, N, 2, H, W));
    TRY(check_shape(fn, "metric", metric, N, 1, H, W));
    TRY(check_shape(fn, "out", out, N, C, H, W));
    TRY(check_shape(fn, "norm", norm, N, 1, H, W));
    TRY(check_shape(fn, "mask", mask, N, 1, H, W));
    TRY(check_shape(fn, "grad_in", gin, N, C, H, W));
    TRY(check_shape(fn, "grad_flow", gflow, N, 2, H, W));
    TRY(check_shape(fn, "grad_metric", gmetric, N, 1, H, W));
    TRY(flow_dtype_ok(fn, in, flow));
    if (gout->dtype != in->dtype) return set_error(DCB_E_DTYPE, "%s: grad_out dtype differs from in", fn);
    if (metric && metric->dtype != in->dtype) return set_error(DCB_E_DTYPE, "%s: metric dtype differs from in", fn);
    if (mask && mask->dtype != in->dtype) return set_error(DCB_E_DTYPE, "%s: mask dtype differs from in", fn);
    TRY(check_out(fn, "out", out, in->dtype, elem_size(in->dtype)));
    TRY(check_out(fn, "norm", norm, acc_dtype(in->dtype), elem_size(acc_dtype(in->dtype))));
    TRY(check_out(fn, "grad_in", gin, in->dtype, elem_size(in->dtype)));
    TRY(check_out(fn, "grad_flow", gflow, flow->dtype, elem_size(flow->dtype)));
    TRY(check_out(fn, "grad_metric", gmetric, in->dtype, elem_size(in->dtype)));
    return splat_bwd_impl(gout, in, flow, metric, out, norm, mask, gin, gflow, gmetric, ws, ws_bytes, mode, eps,
                          (cudaStream_t)stream);
}

int dcb_backwarp_fwd(const DcbTensor* image, const DcbTensor* flow, const DcbTensor* gt, const DcbTensor* warped,
                     const DcbTensor* residual, int32_t align_corners, void* stream) {
    const char* fn = "dcb_backwarp_fwd";
    TRY(refuse_f16(fn, {image, flow, gt, warped, residual}));
    TRY(check_tensor(fn, "image", image, true));
    TRY(check_tensor(fn, "flow", flow, true));
    TRY(check_tensor(fn, "gt", gt, false));
    TRY(check_tensor(fn, "warped", warped, true));
    TRY(check_tensor(fn, "residual", residual, false));
    if ((gt == nullptr) != (residual == nullptr)) return set_error(DCB_E_NULL, "%s: gt and residual go together", fn);
    const long long N = image->size[0], C = image->size[1], H = image->size[2], W = image->size[3];
    TRY(check_limits(fn, image));
    TRY(check_shape(fn, "flow", flow, N, 2, H, W));
    TRY(check_shape(fn, "gt", gt, N, C, H, W));
    TRY(check_shape(fn, "warped", warped, N, C, H, W));
    TRY(check_shape(fn, "residual", residual, N, C, H, W));
    TRY(flow_dtype_ok(fn, image, flow));
    if (gt && gt->dtype != image->dtype) return set_error(DCB_E_DTYPE, "%s: gt dtype differs from image", fn);
    TRY(check_out(fn, "warped", warped, image->dtype, elem_size(image->dtype)));
    TRY(check_out(fn, "residual", residual, image->dtype, elem_size(image->dtype)));
    return backwarp_fwd_impl(image, flow, gt, warped, residual, align_corners ? 1 : 0, (cudaStream_t)stream);
}

int64_t dcb_backwarp_bwd_workspace_bytes(int64_t N, int64_t C, int64_t H, int64_t W, int32_t dtype) {
    return (int64_t)backwarp_bwd_workspace(N, C, H, W, dtype);
}

int dcb_backwarp_bwd(const DcbTensor* gout, const DcbTensor* image, const DcbTensor* flow, const DcbTensor* gimage,
                     const DcbTensor* gflow, int32_t align_corners, void* ws, int64_t ws_bytes, void* stream) {
    const char* fn = "dcb_backwarp_bwd";
    TRY(refuse_f16(fn, {gout, image, flow, gimage, gflow}));
    TRY(check_tensor(fn, "grad_warped", gout, true));
    TRY(check_tensor(fn, "image", image, true));
    TRY(check_tensor(fn, "flow", flow, true));
    TRY(check_tensor(fn, "grad_image", gimage, false));
    TRY(check_tensor(fn, "grad_flow", gflow, false));
    const long long N = image->size[0], C = image->size[1], H = image->size[2], W = image->size[3];
    TRY(check_limits(fn, image));
    TRY(check_shape(fn, "grad_warped", gout, N, C, H, W));
    TRY(check_shape(fn, "flow", flow, N, 2, H, W));
    TRY(check_shape(fn, "grad_image", gimage, N, C, H, W));
    TRY(check_shape(fn, "grad_flow", gflow, N, 2, H, W));
    TRY(flow_dtype_ok(fn, image, flow));
    if (gout->dtype != image->dtype) return set_error(DCB_E_DTYPE, "%s: grad_warped dtype differs from image", fn);
    TRY(check_out(fn, "grad_image", gimage, image->dtype, elem_size(image->dtype)));
    TRY(check_out(fn, "grad_flow", gflow, flow->dtype, elem_size(flow->dtype)));
    return backwarp_bwd_impl(gout, image, flow, gimage, gflow, align_corners ? 1 : 0, ws, ws_bytes, (cudaStream_t)stream);
}

int64_t dcb_occlusion_mask_workspace_bytes(int64_t N, int64_t H, int64_t W) { return (int64_t)mask_workspace(N, H, W); }

int dcb_occlusion_mask(const DcbTensor* flow_a, const DcbTensor* flow_b, const DcbTensor* mask, void* ws, int64_t ws_bytes,
                       int32_t flags, void* stream) {
    const char* fn = "dcb_occlusion_mask";
    TRY(refuse_f16(fn, {flow_a, flow_b, mask}));
    TRY(check_tensor(fn, "flow_a", flow_a, true));
    TRY(check_tensor(fn, "flow_b", flow_b, true));
    TRY(check_tensor(fn, "mask", mask, true));
    const long long N = flow_a->size[0], H = flow_a->size[2], W = flow_a->size[3];
    TRY(check_limits(fn, flow_a));
    TRY(check_shape(fn, "flow_a", flow_a, N, 2, H, W));
    TRY(check_shape(fn, "flow_b", flow_b, N, 2, H, W));
    TRY(check_shape(fn, "mask", mask, N, 1, H, W));
    if (flow_b->dtype != flow_a->dtype) return set_error(DCB_E_DTYPE, "%s: flow dtypes differ", fn);
    TRY(check_out(fn, "mask", mask, flow_a->dtype, elem_size(flow_a->dtype)));
    return occlusion_mask_impl(flow_a, flow_b, mask, ws, ws_bytes, flags, (cudaStream_t)stream);
}

int64_t dcb_residual_workspace_bytes(int64_t N, int64_t C, int64_t H, int64_t W) {
    return (int64_t)recipe_workspace(N, C, H, W);
}

int dcb_residual_fused(const DcbTensor* image1, const DcbTensor* flow1, const DcbTensor* flow2, const DcbTensor* gt,
                       const DcbTensor* fused, const DcbTensor* residual, const DcbTensor* occ_fwd,
                       const DcbTensor* occ_bwd, void* ws, int64_t ws_bytes, int32_t variant, int32_t flags,
                       void* stream) {
    const char* fn = "dcb_residual_fused";
    TRY(refuse_f16(fn, {image1, flow1, flow2, gt, fused, residual, occ_fwd, occ_bwd}));
    TRY(check_tensor(fn, "image1", image1, true));
    TRY(check_tensor(fn, "flow1", flow1, true));
    TRY(check_tensor(fn, "flow2", flow2, true));
    TRY(check_tensor(fn, "gt", gt, true));
    TRY(check_tensor(fn, "fused", fused, true));
    TRY(check_tensor(fn, "residual", residual, true));
    TRY(check_tensor(fn, "occ_fwd", occ_fwd, false));
    TRY(check_tensor(fn, "occ_bwd", occ_bwd, false));
    if (variant != DCB_RECIPE_DATASET && variant != DCB_RECIPE_WRAPPER) return set_error(DCB_E_MODE, "%s: unknown variant %d", fn, variant);
    const long long N = image1->size[0], C = image1->size[1], H = image1->size[2], W = image1->size[3];
    TRY(check_limits(fn, image1));
    if (C < 1 || C > 3) return set_error(DCB_E_LIMIT, "%s: fused recipe handles 1..3 image channels, got %lld", fn, C);
    TRY(check_shape(fn, "flow1", flow1, N, 2, H, W));
    TRY(check_shape(fn, "flow2", flow2, N, 2, H, W));
    TRY(check_shape(fn, "gt", gt, N, C, H, W));
    TRY(check_shape(fn, "fused", fused, N, C, H, W));
    TRY(check_shape(fn, "residual", residual, N, C, H, W));
    TRY(check_shape(fn, "occ_fwd", occ_fwd, N, 1, H, W));
    TRY(check_shape(fn, "occ_bwd", occ_bwd, N, 1, H, W));
    const int dt = image1->dtype;
    if (flow1->dtype != dt || flow2->dtype != dt || gt->dtype != dt) return set_error(DCB_E_DTYPE, "%s: all tensors must share one dtype", fn);
    TRY(check_out(fn, "fused", fused, dt, elem_size(dt)));
    TRY(check_out(fn, "residual", residual, dt, elem_size(dt)));
    TRY(check_out(fn, "occ_fwd", occ_fwd, dt, elem_size(dt)));
    TRY(check_out(fn, "occ_bwd", occ_bwd, dt, elem_size(dt)));
    return residual_fused_impl(image1, flow1, flow2, gt, fused, residual, occ_fwd, occ_bwd, ws, ws_bytes, variant, flags,
                               (cudaStream_t)stream);
}

int dcb_residual_bidir(const DcbTensor* image1, const DcbTensor* image2, const DcbTensor* flow1, const DcbTensor* flow2,
                       const DcbTensor* gt, const DcbTensor* fused, const DcbTensor* residual, const DcbTensor* occ_fwd,
                       const DcbTensor* occ_bwd, void* ws, int64_t ws_bytes, int32_t flags, void* stream) {
    const char* fn = "dcb_residual_bidir";
    TRY(refuse_f16(fn, {image1, image2, flow1, flow2, gt, fused, residual, occ_fwd, occ_bwd}));
    TRY(check_tensor(fn, "image1", image1, true));
    TRY(check_tensor(fn, "image2", image2, true));
    TRY(check_tensor(fn, "flow1", flow1, true));
    TRY(check_tensor(fn, "flow2", flow2, true));
    TRY(check_tensor(fn, "gt", gt, true));
    TRY(check_tensor(fn, "fused", fused, true));
    TRY(check_tensor(fn, "residual", residual, true));
    TRY(check_tensor(fn, "occ_fwd", occ_fwd, false));
    TRY(check_tensor(fn, "occ_bwd", occ_bwd, false));
    if (flags & ~DCB_FLAG_WS_CLEAN) return set_error(DCB_E_MODE, "%s: unknown flags 0x%x", fn, flags);
    const long long N = image1->size[0], C = image1->size[1], H = image1->size[2], W = image1->size[3];
    TRY(check_limits(fn, image1));
    if (C < 1 || C > 3) return set_error(DCB_E_LIMIT, "%s: fused recipe handles 1..3 image channels, got %lld", fn, C);
    TRY(check_shape(fn, "image2", image2, N, C, H, W));
    TRY(check_shape(fn, "flow1", flow1, N, 2, H, W));
    TRY(check_shape(fn, "flow2", flow2, N, 2, H, W));
    TRY(check_shape(fn, "gt", gt, N, C, H, W));
    TRY(check_shape(fn, "fused", fused, N, C, H, W));
    TRY(check_shape(fn, "residual", residual, N, C, H, W));
    TRY(check_shape(fn, "occ_fwd", occ_fwd, N, 1, H, W));
    TRY(check_shape(fn, "occ_bwd", occ_bwd, N, 1, H, W));
    const int dt = image1->dtype;
    if (image2->dtype != dt || flow1->dtype != dt || flow2->dtype != dt || gt->dtype != dt)
        return set_error(DCB_E_DTYPE, "%s: all tensors must share one dtype", fn);
    TRY(check_out(fn, "fused", fused, dt, elem_size(dt)));
    TRY(check_out(fn, "residual", residual, dt, elem_size(dt)));
    TRY(check_out(fn, "occ_fwd", occ_fwd, dt, elem_size(dt)));
    TRY(check_out(fn, "occ_bwd", occ_bwd, dt, elem_size(dt)));
    return residual_bidir_impl(image1, image2, flow1, flow2, gt, fused, residual, occ_fwd, occ_bwd, ws, ws_bytes, flags,
                               (cudaStream_t)stream);
}

static int check_fuse_common(const char* fn, const DcbTensor* A, const DcbTensor* B, const DcbTensor* ca, const DcbTensor* cb,
                             const DcbTensor* oa, const DcbTensor* ob) {
    TRY(check_tensor(fn, "A", A, true));
    TRY(check_tensor(fn, "B", B, true));
    TRY(check_tensor(fn, "conf_a", ca, true));
    TRY(check_tensor(fn, "conf_b", cb, true));
    TRY(check_tensor(fn, "occ_a", oa, false));
    TRY(check_tensor(fn, "occ_b", ob, false));
    if ((oa == nullptr) != (ob == nullptr)) return set_error(DCB_E_NULL, "%s: occ_a and occ_b go together", fn);
    const long long N = A->size[0], C = A->size[1], H = A->size[2], W = A->size[3];
    TRY(check_limits(fn, A));
    TRY(check_shape(fn, "B", B, N, C, H, W));
    TRY(check_shape(fn, "conf_a", ca, N, 1, H, W));
    TRY(check_shape(fn, "conf_b", cb, N, 1, H, W));
    TRY(check_shape(fn, "occ_a", oa, N, 1, H, W));
    TRY(check_shape(fn, "occ_b", ob, N, 1, H, W));
    const int dt = A->dtype;
    if (B->dtype != dt || ca->dtype != dt || cb->dtype != dt || (oa && (oa->dtype != dt || ob->dtype != dt)))
        return set_error(DCB_E_DTYPE, "%s: all tensors must share one dtype", fn);
    return DCB_OK;
}

int dcb_bidir_fuse_fwd(const DcbTensor* A, const DcbTensor* B, const DcbTensor* ca, const DcbTensor* cb,
                       const DcbTensor* oa, const DcbTensor* ob, const DcbTensor* fused, void* stream) {
    const char* fn = "dcb_bidir_fuse_fwd";
    TRY(check_fuse_common(fn, A, B, ca, cb, oa, ob));
    TRY(check_tensor(fn, "fused", fused, true));
    TRY(check_shape(fn, "fused", fused, A->size[0], A->size[1], A->size[2], A->size[3]));
    TRY(check_out(fn, "fused", fused, A->dtype, elem_size(A->dtype)));
    return bidir_fuse_fwd_impl(A, B, ca, cb, oa, ob, fused, (cudaStream_t)stream);
}

int dcb_bidir_fuse_bwd(const DcbTensor* g, const DcbTensor* A, const DcbTensor* B, const DcbTensor* ca, const DcbTensor* cb,
                       const DcbTensor* oa, const DcbTensor* ob, const DcbTensor* gA, const DcbTensor* gB,
                       const DcbTensor* gca, const DcbTensor* gcb, void* stream) {
    const char* fn = "dcb_bidir_fuse_bwd";
    TRY(check_fuse_common(fn, A, B, ca, cb, oa, ob));
    TRY(check_tensor(fn, "grad_fused", g, true));
    const long long N = A->size[0], C = A->size[1], H = A->size[2], W = A->size[3];
    TRY(check_shape(fn, "grad_fused", g, N, C, H, W));
    if (g->dtype != A->dtype) return set_error(DCB_E_DTYPE, "%s: grad_fused dtype differs", fn);
    const DcbTensor* outs[4] = {gA, gB, gca, gcb};
    const char* names[4] = {"grad_A", "grad_B", "grad_conf_a", "grad_conf_b"};
    for (int i = 0; i < 4; ++i) {
        TRY(check_tensor(fn, names[i], outs[i], false));
        TRY(check_shape(fn, names[i], outs[i], N, i < 2 ? C : 1, H, W));
        TRY(check_out(fn, names[i], outs[i], A->dtype, elem_size(A->dtype)));
    }
    return bidir_fuse_bwd_impl(g, A, B, ca, cb, oa, ob, gA, gB, gca, gcb, (cudaStream_t)stream);
}

int64_t dcb_tile_merge_workspace_bytes(int64_t C, int64_t H, int64_t W, int32_t n_tiles) {
    if (C < 0 || H < 0 || W < 0 || n_tiles < 0) return 0;
    return (int64_t)tile_merge_workspace(C, H, W, n_tiles);
}

int dcb_tile_merge(const DcbTensor* tiles, const int64_t* pixel_coords, int32_t n_tiles, const DcbTensor* out, int64_t H_px,
                   int64_t W_px, double eps, void* ws, int64_t ws_bytes, void* stream) {
    const char* fn = "dcb_tile_merge";
    TRY(check_tensor(fn, "out", out, true));
    if (out->dtype != DCB_F32 && !is_half_storage(out->dtype)) return set_error(DCB_E_DTYPE, "%s: F32, BF16 or F16 only, got %d", fn, out->dtype);
    TRY(check_out(fn, "out", out, out->dtype, elem_size(out->dtype)));
    TRY(check_limits(fn, out));
    if (n_tiles < 0) return set_error(DCB_E_SHAPE, "%s: n_tiles = %d", fn, n_tiles);
    if (n_tiles > 0 && (!tiles || !pixel_coords)) return set_error(DCB_E_NULL, "%s: tiles and pixel_coords are required", fn);
    if (H_px <= 0 || W_px <= 0) return set_error(DCB_E_SHAPE, "%s: original image size %lld x %lld", fn, (long long)H_px, (long long)W_px);
    for (int i = 0; i < n_tiles; ++i) {
        const DcbTensor* t = tiles + i;
        TRY(check_tensor(fn, "tile", t, true));
        if (t->dtype != out->dtype) return set_error(DCB_E_DTYPE, "%s: tile %d has dtype %d, canvas %d", fn, i, t->dtype, out->dtype);
        if (t->size[0] != 1 || t->size[1] != out->size[1])                                  // patch_utils.py:155
            return set_error(DCB_E_SHAPE, "%s: tile %d is [%lld,%lld,..], expected [1,%lld,h,w]", fn, i, (long long)t->size[0],
                             (long long)t->size[1], (long long)out->size[1]);
        if (t->size[2] <= 0 || t->size[3] <= 0 || t->size[2] >= (1 << 24) || t->size[3] >= (1 << 24))
            return set_error(DCB_E_SHAPE, "%s: tile %d has an empty or oversized plane", fn, i);
    }
    static_assert(sizeof(long long) == sizeof(int64_t), "int64_t coordinates");
    return tile_merge_impl(tiles, (const long long*)pixel_coords, n_tiles, out, H_px, W_px, eps, ws, ws_bytes, (cudaStream_t)stream);
}

static int check_block_common(const char* fn, const DcbTensor* first, const DcbTensor* last, const DcbTensor* flow_f, const DcbTensor* flow_b,
                              const DcbTensor* metric_f, const DcbTensor* metric_b) {
    TRY(check_tensor(fn, "first", first, true));
    TRY(check_tensor(fn, "last", last, true));
    TRY(check_tensor(fn, "flow_f", flow_f, true));
    TRY(check_tensor(fn, "flow_b", flow_b, true));
    TRY(check_tensor(fn, "metric_f", metric_f, true));
    TRY(check_tensor(fn, "metric_b", metric_b, true));
    const long long N = first->size[0], C = first->size[1], H = first->size[2], W = first->size[3];
    TRY(check_limits(fn, first));
    TRY(check_shape(fn, "last", last, N, C, H, W));
    TRY(check_shape(fn, "flow_f", flow_f, N, 2, H, W));
    TRY(check_shape(fn, "flow_b", flow_b, N, 2, H, W));
    TRY(check_shape(fn, "metric_f", metric_f, N, 1, H, W));
    TRY(check_shape(fn, "metric_b", metric_b, N, 1, H, W));
    const int dt = first->dtype;
    if (dt != DCB_F32 && !is_half_storage(dt)) return set_error(DCB_E_DTYPE, "%s: F32, BF16 or F16 only, got %d", fn, dt);
    if (last->dtype != dt || flow_f->dtype != dt || flow_b->dtype != dt || metric_f->dtype != dt || metric_b->dtype != dt)
        return set_error(DCB_E_DTYPE, "%s: all tensors must share one dtype", fn);
    return DCB_OK;
}

static int check_block_opt(const char* fn, const char* name, const DcbTensor* t, const DcbTensor* first, long long C, int dtype) {
    TRY(check_tensor(fn, name, t, false));
    TRY(check_shape(fn, name, t, first->size[0], C, first->size[2], first->size[3]));
    TRY(check_out(fn, name, t, dtype, elem_size(dtype)));
    return DCB_OK;
}

int64_t dcb_bidir_block_workspace_bytes(int64_t N, int64_t C, int64_t H, int64_t W, int32_t dtype, int32_t which) {
    if (N < 0 || C < 0 || H < 0 || W < 0) return 0;
    if (which == 0) return (int64_t)block_fwd_acc_bytes(N, C, H, W, dtype);
    if (which == 1) return (int64_t)block_fwd_scratch_bytes(N, C, H, W, dtype);
    return (int64_t)block_bwd_scratch_bytes(N, C, H, W, dtype);
}

int dcb_bidir_block_fwd(const DcbTensor* first, const DcbTensor* last, const DcbTensor* flow_f, const DcbTensor* flow_b,
                        const DcbTensor* metric_f, const DcbTensor* metric_b, const DcbTensor* fused, const DcbTensor* warped_f,
                        const DcbTensor* warped_b, const DcbTensor* norm_f, const DcbTensor* norm_b, const DcbTensor* occ_f,
                        const DcbTensor* occ_b, void* ws_acc, int64_t ws_acc_bytes, void* ws_scratch, int64_t ws_scratch_bytes,
                        int32_t flags, void* stream) {
    const char* fn = "dcb_bidir_block_fwd";
    TRY(check_block_common(fn, first, last, flow_f, flow_b, metric_f, metric_b));
    if (flags & ~DCB_FLAG_WS_CLEAN) return set_error(DCB_E_MODE, "%s: unknown flags 0x%x", fn, flags);
    const int dt = first->dtype;
    const long long C = first->size[1];
    TRY(check_tensor(fn, "fused", fused, true));
    TRY(check_block_opt(fn, "fused", fused, first, C, dt));
    TRY(check_block_opt(fn, "warped_f", warped_f, first, C, dt));
    TRY(check_block_opt(fn, "warped_b", warped_b, first, C, dt));
    TRY(check_block_opt(fn, "norm_f", norm_f, first, 1, DCB_F32));
    TRY(check_block_opt(fn, "norm_b", norm_b, first, 1, DCB_F32));
    TRY(check_block_opt(fn, "occ_f", occ_f, first, 1, dt));
    TRY(check_block_opt(fn, "occ_b", occ_b, first, 1, dt));
    return bidir_block_fwd_impl(first, last, flow_f, flow_b, metric_f, metric_b, fused, warped_f, warped_b, norm_f, norm_b, occ_f, occ_b,
                                ws_acc, ws_acc_bytes, ws_scratch, ws_scratch_bytes, flags, (cudaStream_t)stream);
}

int dcb_bidir_block_bwd(const DcbTensor* grad_fused, const DcbTensor* first, const DcbTensor* last, const DcbTensor* flow_f,
                        const DcbTensor* flow_b, const DcbTensor* metric_f, const DcbTensor* metric_b, const DcbTensor* warped_f,
                        const DcbTensor* warped_b, const DcbTensor* norm_f, const DcbTensor* norm_b, const DcbTensor* occ_f,
                        const DcbTensor* occ_b, const DcbTensor* grad_first, const DcbTensor* grad_last,
                        const DcbTensor* grad_metric_f, const DcbTensor* grad_metric_b, void* ws, int64_t ws_bytes, void* stream) {
    const char* fn = "dcb_bidir_block_bwd";
    TRY(check_block_common(fn, first, last, flow_f, flow_b, metric_f, metric_b));
    const int dt = first->dtype;
    const long long N = first->size[0], C = first->size[1], H = first->size[2], W = first->size[3];
    TRY(check_tensor(fn, "grad_fused", grad_fused, true));
    TRY(check_shape(fn, "grad_fused", grad_fused, N, C, H, W));
    if (grad_fused->dtype != dt) return set_error(DCB_E_DTYPE, "%s: grad_fused dtype differs", fn);
    const DcbTensor* req[6] = {warped_f, warped_b, norm_f, norm_b, occ_f, occ_b};
    const char* names[6] = {"warped_f", "warped_b", "norm_f", "norm_b", "occ_f", "occ_b"};
    for (int i = 0; i < 6; ++i) {
        if (!req[i]) return set_error(DCB_E_NULL, "%s: %s of the forward is required", fn, names[i]);
        TRY(check_block_opt(fn, names[i], req[i], first, i < 2 ? C : 1, (i == 2 || i == 3) ? DCB_F32 : dt));
    }
    TRY(check_block_opt(fn, "grad_first", grad_first, first, C, dt));
    TRY(check_block_opt(fn, "grad_last", grad_last, first, C, dt));
    TRY(check_block_opt(fn, "grad_metric_f", grad_metric_f, first, 1, dt));
    TRY(check_block_opt(fn, "grad_metric_b", grad_metric_b, first, 1, dt));
    return bidir_block_bwd_impl(grad_fused, first, last, flow_f, flow_b, metric_f, metric_b, warped_f, warped_b, norm_f, norm_b, occ_f, occ_b,
                                grad_first, grad_last, grad_metric_f, grad_metric_b, ws, ws_bytes, (cudaStream_t)stream);
}

// the inputs of one pyramid level (forward and backward): dtype of every level = dtype of `first0`
struct PyramidInputs { const DcbTensor *first, *last, *flow_f, *flow_b, *metric_f, *metric_b; };
static int check_pyramid_inputs(const char* fn, const PyramidInputs& d, int l, const DcbTensor* first0) {
    TRY(check_tensor(fn, "first", d.first, true));
    TRY(check_tensor(fn, "last", d.last, true));
    TRY(check_tensor(fn, "flow_f", d.flow_f, true));
    TRY(check_tensor(fn, "flow_b", d.flow_b, true));
    TRY(check_tensor(fn, "metric_f", d.metric_f, false));
    TRY(check_tensor(fn, "metric_b", d.metric_b, false));
    const long long N = d.first->size[0], C = d.first->size[1], H = d.first->size[2], W = d.first->size[3];
    TRY(check_limits(fn, d.first));
    TRY(check_shape(fn, "last", d.last, N, C, H, W));
    TRY(check_shape(fn, "flow_f", d.flow_f, N, 2, H, W));
    TRY(check_shape(fn, "flow_b", d.flow_b, N, 2, H, W));
    TRY(check_shape(fn, "metric_f", d.metric_f, N, 1, H, W));
    TRY(check_shape(fn, "metric_b", d.metric_b, N, 1, H, W));
    const int dt = d.first->dtype;
    if (dt != DCB_F32 && !is_half_storage(dt)) return set_error(DCB_E_DTYPE, "%s: F32, BF16 or F16 only, got %d", fn, dt);
    if (dt != first0->dtype || d.last->dtype != dt || d.flow_f->dtype != dt || d.flow_b->dtype != dt ||
        (d.metric_f && d.metric_f->dtype != dt) || (d.metric_b && d.metric_b->dtype != dt))
        return set_error(DCB_E_DTYPE, "%s: all tensors of all levels must share one dtype", fn);
    const DcbTensor* in32[6] = {d.first, d.last, d.flow_f, d.flow_b, d.metric_f, d.metric_b};
    for (int i = 0; i < 6; ++i) {
        if (!in32[i]) continue;
        long long span = 0;
        for (int k = 0; k < 4; ++k) span += (in32[i]->size[k] - 1) * (in32[i]->stride[k] < 0 ? -in32[i]->stride[k] : in32[i]->stride[k]);
        if (span >= (1ll << 31)) return set_error(DCB_E_LIMIT, "%s: level %d: a tensor spans 2^31 elements or more", fn, l);
    }
    return DCB_OK;
}

static int check_pyramid(const char* fn, const DcbPyramidLevel* lv, int32_t n) {
    if (n < 0 || n > 4) return set_error(DCB_E_LIMIT, "%s: %d levels (at most 4 per call)", fn, n);
    if (n > 0 && !lv) return set_error(DCB_E_NULL, "%s: levels is required", fn);
    if (n > 0) TRY(check_tensor(fn, "first", lv[0].first, true));
    for (int l = 0; l < n; ++l) {
        const DcbPyramidLevel& d = lv[l];
        TRY(check_pyramid_inputs(fn, {d.first, d.last, d.flow_f, d.flow_b, d.metric_f, d.metric_b}, l, lv[0].first));
        const long long N = d.first->size[0], C = d.first->size[1], H = d.first->size[2], W = d.first->size[3];
        const int dt = d.first->dtype;
        if (N * C * H * W > 0 && !d.fused) return set_error(DCB_E_NULL, "%s: level %d: fused is required", fn, l);
        void* outs[7] = {d.fused, d.warped_f, d.warped_b, d.norm_f, d.norm_b, d.occ_f, d.occ_b};
        for (int i = 0; i < 7; ++i)                                   // norm_f / norm_b are fp32 whatever the tensor dtype
            if ((uintptr_t)outs[i] % (uintptr_t)((i == 3 || i == 4) ? 4 : elem_size(dt)))
                return set_error(DCB_E_ALIGN, "%s: level %d: output %d is not aligned to its element size", fn, l, i);
    }
    return DCB_OK;
}

int64_t dcb_bidir_pyramid_workspace_bytes(const DcbPyramidLevel* levels, int32_t n_levels) {
    if (!levels || n_levels <= 0 || n_levels > 4) return 0;
    for (int l = 0; l < n_levels; ++l)
        if (!levels[l].first) return 0;
    return (int64_t)pyramid_workspace(levels, n_levels);
}

int64_t dcb_bidir_pyramid_det_workspace_bytes(const DcbPyramidLevel* levels, int32_t n_levels) {
    if (!levels || n_levels <= 0 || n_levels > 4) return 0;
    for (int l = 0; l < n_levels; ++l)
        if (!levels[l].first) return 0;
    return (int64_t)pyramid_det_workspace(levels, n_levels);
}

int dcb_bidir_pyramid_fwd(const DcbPyramidLevel* levels, int32_t n_levels, void* ws, int64_t ws_bytes, int32_t flags, void* stream) {
    const char* fn = "dcb_bidir_pyramid_fwd";
    if (flags & ~(DCB_FLAG_DETERMINISTIC | DCB_FLAG_WS_CLEAN | DCB_PYRAMID_NO_MASKS | DCB_PYRAMID_NO_HOLES))
        return set_error(DCB_E_MODE, "%s: unknown flags 0x%x", fn, flags);
    const bool det = (flags & DCB_FLAG_DETERMINISTIC) != 0;
    if (det && (flags & DCB_FLAG_WS_CLEAN))
        return set_error(DCB_E_MODE, "%s: DCB_FLAG_DETERMINISTIC takes a scratch workspace, not DCB_FLAG_WS_CLEAN", fn);
    TRY(check_pyramid(fn, levels, n_levels));
    if (n_levels == 0) return DCB_OK;
    if (det) {
        const long long nkeys = pyramid_det_keys(levels, n_levels);
        if (nkeys >= (1ll << 31))
            return set_error(DCB_E_LIMIT, "%s(deterministic): 4 x the pixels of all levels and directions must stay below 2^31 (got %lld)",
                             fn, nkeys);
    }
    const long long need = det ? pyramid_det_workspace(levels, n_levels) : pyramid_workspace(levels, n_levels);
    if (need > 0 && (!ws || ws_bytes < need || ((uintptr_t)ws & 255)))
        return set_error(DCB_E_WORKSPACE, "%s: workspace of %lld bytes (256 B aligned) required, got %lld", fn, need, (long long)ws_bytes);
    return bidir_pyramid_fwd_impl(levels, n_levels, ws, flags, (cudaStream_t)stream);
}

int64_t dcb_bidir_pyramid_bwd_workspace_bytes(const DcbPyramidBwdLevel* levels, int32_t n_levels) {
    if (!levels || n_levels <= 0 || n_levels > 4) return 0;
    for (int l = 0; l < n_levels; ++l) {
        const DcbTensor* f = levels[l].first;
        if (!f || f->size[0] < 0 || f->size[1] < 0 || f->size[2] < 0 || f->size[3] < 0) return 0;
    }
    return (int64_t)pyramid_bwd_workspace(levels, n_levels);
}

int dcb_bidir_pyramid_bwd(const DcbPyramidBwdLevel* levels, int32_t n_levels, void* ws, int64_t ws_bytes, int32_t flags, void* stream) {
    const char* fn = "dcb_bidir_pyramid_bwd";
    if (flags & ~DCB_PYRAMID_NO_HOLES) return set_error(DCB_E_MODE, "%s: flags 0x%x (only DCB_PYRAMID_NO_HOLES; NO_MASKS has no backward)", fn, flags);
    if (n_levels < 1 || n_levels > 4) return set_error(DCB_E_LIMIT, "%s: %d levels (1 to 4 per call)", fn, n_levels);
    if (!levels) return set_error(DCB_E_NULL, "%s: levels is required", fn);
    TRY(check_tensor(fn, "first", levels[0].first, true));
    for (int l = 0; l < n_levels; ++l) {
        const DcbPyramidBwdLevel& d = levels[l];
        TRY(check_pyramid_inputs(fn, {d.first, d.last, d.flow_f, d.flow_b, d.metric_f, d.metric_b}, l, levels[0].first));
        const long long N = d.first->size[0], C = d.first->size[1], H = d.first->size[2], W = d.first->size[3];
        const int dt = d.first->dtype;
        TRY(check_tensor(fn, "grad_fused", d.grad_fused, true));
        TRY(check_shape(fn, "grad_fused", d.grad_fused, N, C, H, W));
        if (d.grad_fused->dtype != dt) return set_error(DCB_E_DTYPE, "%s: level %d: grad_fused dtype differs", fn, l);
        if ((d.grad_metric_f && !d.metric_f) || (d.grad_metric_b && !d.metric_b))
            return set_error(DCB_E_MODE, "%s: level %d: a metric gradient for an all-ones (NULL) metric", fn, l);
        const void* saved[6] = {d.warped_f, d.warped_b, d.norm_f, d.norm_b, d.occ_f, d.occ_b};
        const void* grads[6] = {d.grad_first, d.grad_last, d.grad_flow_f, d.grad_flow_b, d.grad_metric_f, d.grad_metric_b};
        for (int i = 0; i < 6; ++i) {
            if (N * C * H * W > 0 && !saved[i]) return set_error(DCB_E_NULL, "%s: level %d: saved forward output %d is required", fn, l, i);
            if ((uintptr_t)saved[i] % (uintptr_t)((i == 2 || i == 3) ? 4 : elem_size(dt)) || (uintptr_t)grads[i] % (uintptr_t)elem_size(dt))
                return set_error(DCB_E_ALIGN, "%s: level %d: a pointer is not aligned to its element size", fn, l);
        }
    }
    const long long need = pyramid_bwd_workspace(levels, n_levels);
    if (need > 0 && (!ws || ws_bytes < need || ((uintptr_t)ws & 255)))
        return set_error(DCB_E_WORKSPACE, "%s: workspace of %lld bytes (256 B aligned) required, got %lld", fn, need, (long long)ws_bytes);
    return bidir_pyramid_bwd_impl(levels, n_levels, ws, !(flags & DCB_PYRAMID_NO_HOLES), (cudaStream_t)stream);
}

int dcb_resample_batch(const DcbResampleJob* jobs, int32_t n_jobs, void* stream) {
    const char* fn = "dcb_resample_batch";
    if (n_jobs < 0) return set_error(DCB_E_SHAPE, "%s: n_jobs = %d", fn, n_jobs);
    if (n_jobs > 0 && !jobs) return set_error(DCB_E_NULL, "%s: jobs is required", fn);
    for (int j = 0; j < n_jobs; ++j) {
        const DcbTensor* s = jobs[j].src; const DcbTensor* d = jobs[j].dst;
        TRY(check_tensor(fn, "src", s, true));
        TRY(check_tensor(fn, "dst", d, true));
        if ((s->dtype != DCB_F32 && !is_half_storage(s->dtype)) || (d->dtype != DCB_F32 && !is_half_storage(d->dtype)))
            return set_error(DCB_E_DTYPE, "%s: job %d: F32, BF16 or F16 only", fn, j);
        if (s->size[0] != d->size[0] || s->size[1] != d->size[1])
            return set_error(DCB_E_SHAPE, "%s: job %d: src [N,C,H,W] -> dst [N,C,th,tw] expected", fn, j);
        if (s->size[2] * s->size[3] == 0 && d->size[0] * d->size[1] * d->size[2] * d->size[3] > 0)
            return set_error(DCB_E_SHAPE, "%s: job %d: empty source", fn, j);
        TRY(check_limits(fn, s));
        TRY(check_limits(fn, d));
        TRY(check_out(fn, "dst", d, d->dtype, elem_size(d->dtype)));
        if (jobs[j].op < DCB_RESAMPLE_NONE || jobs[j].op > DCB_RESAMPLE_DIV) return set_error(DCB_E_MODE, "%s: job %d: unknown op %d", fn, j, jobs[j].op);
    }
    return resample_batch_impl(jobs, n_jobs, (cudaStream_t)stream);
}

int dcb_flow_resize(const DcbTensor* flow, const DcbTensor* out, int32_t convention, void* stream) {
    const char* fn = "dcb_flow_resize";
    TRY(refuse_f16(fn, {flow, out}));
    TRY(check_tensor(fn, "flow", flow, true));
    TRY(check_tensor(fn, "out", out, true));
    if (convention < DCB_FLOW_BILINEAR_RESCALE || convention > DCB_FLOW_BILINEAR_NORMALIZE) return set_error(DCB_E_MODE, "%s: unknown convention %d", fn, convention);
    if (flow->size[1] != 2 || out->size[1] != 2 || out->size[0] != flow->size[0])
        return set_error(DCB_E_SHAPE, "%s: flow [N,2,H,W] -> out [N,2,th,tw] expected", fn);
    if (flow->size[0] * flow->size[2] * flow->size[3] == 0 && out->size[0] * out->size[2] * out->size[3] > 0)
        return set_error(DCB_E_SHAPE, "%s: empty source", fn);
    TRY(check_limits(fn, flow));
    TRY(check_limits(fn, out));
    if (out->dtype != DCB_F32 && out->dtype != DCB_BF16) return set_error(DCB_E_DTYPE, "%s: out must be F32 or BF16", fn);
    TRY(check_out(fn, "out", out, out->dtype, elem_size(out->dtype)));
    return flow_ingest_impl(flow, out, convention, (cudaStream_t)stream);
}

int dcb_convert(const void* src, int32_t src_dtype, void* dst, int32_t dst_dtype, int64_t n, float scale, void* stream) {
    const char* fn = "dcb_convert";
    if (n < 0) return set_error(DCB_E_SHAPE, "%s: n = %lld", fn, (long long)n);
    if (n > 0 && (!src || !dst)) return set_error(DCB_E_NULL, "%s: src and dst are required", fn);
    const int ss = src_dtype == DCB_U8 ? 1 : (src_dtype == DCB_F32 ? 4 : 2), ds = dst_dtype == DCB_F32 ? 4 : 2;
    if ((uintptr_t)src % (uintptr_t)ss || (uintptr_t)dst % (uintptr_t)ds) return set_error(DCB_E_ALIGN, "%s: pointer not aligned to its element size", fn);
    return convert_impl(src, src_dtype, dst, dst_dtype, n, scale, (cudaStream_t)stream);
}

}  // extern "C"
