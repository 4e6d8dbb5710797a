// extern "C" surface of libgfla_warp.so (declared in include/gfla_warp.h):
// argument validation + dispatch; no state, no allocation.
#include "common.cuh"

namespace gfla {
int block_extract_fwd(const void*, const void*, void*, int, int, int, int, int, int, int, int, int, cudaStream_t);
int block_extract_bwd(const void*, const void*, const void*, void*, void*, int, int, int, int, int, int, int, int, int, int, int, cudaStream_t);
int convert(const void*, int, void*, int, long long, cudaStream_t);
int attn_reshape_fwd(const void*, void*, int, int, int, int, int, cudaStream_t);
int attn_reshape_bwd(const void*, void*, int, int, int, int, int, int, cudaStream_t);
int resample2d_fwd(const void*, const void*, void*, int, int, int, int, int, int, int, int, int, cudaStream_t);
int resample2d_bwd(const void*, const void*, const void*, void*, void*, int, int, int, int, int, int, int, int, int, int, cudaStream_t);
int resample2d_cos_fwd(const void*, const void*, const void*, void*, void*, int, int, int, int, int, int, int, int, double, int, cudaStream_t);
int resample2d_cos_bwd(const void*, const void*, const void*, const void*, const void*, void*, void*, void*, void*, int, int, int, int, int,
                       int, int, int, double, int, int, cudaStream_t);
int resample2d_nhwc_fwd(const void*, const void*, void*, int, int, int, int, int, int, int, int, int, cudaStream_t);
int resample2d_nhwc_bwd(const void*, const void*, const void*, void*, void*, int, int, int, int, int, int, int, int, int, int, int, cudaStream_t);
int resample2d_nhwc_cos_fwd(const void*, const void*, const void*, void*, void*, int, int, int, int, int, int, int, int, double, int, cudaStream_t);
int resample2d_nhwc_cos_bwd(const void*, const void*, const void*, const void*, const void*, void*, void*, void*, void*, int, int, int, int,
                            int, int, int, int, double, int, int, int, cudaStream_t);
int local_attn_fwd_gather(const void*, const void*, const void*, void*, void*, const void*, const void*, int, int, int, int, int, int, int, int, int, int, cudaStream_t);
int local_attn_bwd_gather(const void*, const void*, const void*, const void*, void*, void*, void*, int, int, int, int, int, int, int, int, int, int, int, int, cudaStream_t);
bool local_attn_bwd_tc_supported(int C, int k, int dtype, int flow_dtype, int layout, const void* gout, const void* gsrc);
bool local_attn_bwd_q_tc_supported(int C, int k);
int local_attn_bwd_q_tc(const void* src, const void* flow, const void* logits, const void* gout, void* gflow, void* glogits, int B, int C, int Hs, int Ws, int H, int W, int k, int accumulate, cudaStream_t);
bool local_attn_bwd_fused_supported(int C, int k, const void* src);
int local_attn_bwd_fused_tc(const void* src, const void* flow, const void* logits, const void* gout, void* gsrc, void* gflow, void* glogits, int B, int C, int Hs, int Ws, int H, int W, int k, int accumulate, void* workspace, long long workspace_bytes, cudaStream_t);
int local_attn_bwd_gs_tc(const void* flow, const void* logits, const void* gout, void* gsrc, int B, int C, int Hs, int Ws, int H, int W, int k, cudaStream_t);
int local_attn_fwd_tc(const void*, const void*, const void*, void*, void*, const void*, const void*, int, int, int, int, int, int, int, int, int, int, cudaStream_t);
int relayout(const void*, void*, int, int, int, int, int, int, cudaStream_t);
int tc_debug_set_buffer(void*);
int tc_debug_set_buffer_bwd(void*);
int tc_wait_profile_fwd(int, unsigned long long*);
int tc_wait_profile_strip(int, unsigned long long*);
int tc_wait_profile_bwd_fused(int, unsigned long long*);
bool local_attn_fwd_tc_supported(int B, int C, int Hs, int Ws, int H, int W, int k, int dtype, int flow_dtype, int layout, const void* src, const void* out);
}  // namespace gfla

#include <atomic>
#include <cstdlib>

namespace gfla {
static std::atomic<unsigned long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
}  // namespace gfla

using namespace gfla;

// which backward the automatic path takes where both can serve the call (GFLA_BWD_FUSED=0/1 overrides)
constexpr bool kBwdFusedDefault = true;

#define REQ_PTR(p) do { if ((p) == nullptr) return GFLA_E_NULL; } while (0)
#define REQ_ALIGN(p, dt) do { if (!aligned((p), elem_size(dt))) return GFLA_E_ALIGN; } while (0)

static inline bool pos(int a) { return a > 0; }
static inline bool dtype_known(int d) { return elem_size(d) != 0; }
static inline bool dtype_16bit(int d) { return d == GFLA_BF16 || d == GFLA_F16; }
// grad_in1 of the channels-last 16-bit resample2d entries: the feature dtype, or fp32 (narrowed by the caller)
static inline bool grad_in1_dtype_ok(int dtype, int gdtype) { return gdtype == dtype || gdtype == GFLA_F32; }

extern "C" {

int gfla_abi_version(void) { return GFLA_ABI_VERSION; }

const char* gfla_error_string(int code) {
    switch (code) {
        case GFLA_OK: return "ok";
        case GFLA_E_NULL: return "gfla: required pointer is NULL";
        case GFLA_E_SHAPE: return "gfla: bad shape / kernel_size";
        case GFLA_E_DTYPE: return "gfla: unsupported dtype combination";
        case GFLA_E_ALIGN: return "gfla: misaligned pointer";
        case GFLA_E_NOTSUP: return "gfla: requested algorithm cannot serve this call";
        default: return code > 0 ? cudaGetErrorString(static_cast<cudaError_t>(code)) : "gfla: unknown error";
    }
}

int gfla_device_check(void) {
    int dev = 0, major = 0, minor = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return static_cast<int>(e);
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
    return (major == 10 && minor == 0) ? GFLA_OK : static_cast<int>(cudaErrorNoKernelImageForDevice);
}

int gfla_debug_wait_profile(int which, int enable, unsigned long long* out_u64x64) {
    if (which < 0 || which > 2) return GFLA_E_SHAPE;
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return static_cast<int>(e);
    if (which == 2) return tc_wait_profile_bwd_fused(enable, out_u64x64);
    return which == 0 ? tc_wait_profile_fwd(enable, out_u64x64) : tc_wait_profile_strip(enable, out_u64x64);
}

unsigned long long gfla_debug_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int gfla_debug_set_buffer(void* host_mapped_u64x8) {
    const int e = tc_debug_set_buffer(host_mapped_u64x8);
    return e ? e : tc_debug_set_buffer_bwd(host_mapped_u64x8);
}

int gfla_relayout(const void* src, void* dst, int B, int C, int H, int W, int dtype, int to_nhwc, gfla_stream_t stream) {
    REQ_PTR(src); REQ_PTR(dst);
    if (!pos(B) || !pos(C) || !pos(H) || !pos(W)) return GFLA_E_SHAPE;
    if (!dtype_known(dtype)) return GFLA_E_DTYPE;
    if (src == dst) return GFLA_E_NOTSUP;
    REQ_ALIGN(src, dtype); REQ_ALIGN(dst, dtype);
    return relayout(src, dst, B, C, H, W, dtype, to_nhwc, (cudaStream_t)stream);
}

int gfla_block_extract_fwd(const void* source, const void* flow, void* out, int B, int C, int Hs, int Ws, int Hf,
                           int Wf, int k, int dtype, int flow_dtype, gfla_stream_t stream) {
    REQ_PTR(source); REQ_PTR(flow); REQ_PTR(out);
    if (!pos(B) || !pos(C) || !pos(Hs) || !pos(Ws) || !pos(Hf) || !pos(Wf) || k < 1 || k > 9) return GFLA_E_SHAPE;
    if (!dtype_known(dtype) || !flow_dtype_ok(dtype, flow_dtype)) return GFLA_E_DTYPE;
    REQ_ALIGN(source, dtype); REQ_ALIGN(out, dtype); REQ_ALIGN(flow, flow_dtype);
    return block_extract_fwd(source, flow, out, B, C, Hs, Ws, Hf, Wf, k, dtype, flow_dtype, (cudaStream_t)stream);
}

int gfla_block_extract_bwd(const void* source, const void* flow, const void* grad_out, void* grad_source,
                           void* grad_flow, int B, int C, int Hs, int Ws, int Hf, int Wf, int k, int dtype,
                           int flow_dtype, int grad_source_dtype, int accumulate, gfla_stream_t stream) {
    REQ_PTR(source); REQ_PTR(flow); REQ_PTR(grad_out); REQ_PTR(grad_source); REQ_PTR(grad_flow);
    if (!pos(B) || !pos(C) || !pos(Hs) || !pos(Ws) || !pos(Hf) || !pos(Wf) || k < 1 || k > 9) return GFLA_E_SHAPE;
    if (!dtype_known(dtype) || !flow_dtype_ok(dtype, flow_dtype)) return GFLA_E_DTYPE;
    // grad_source is stored in `dtype`, or in fp32 when `dtype` is a 16-bit type
    if (grad_source_dtype != dtype && !((dtype == GFLA_BF16 || dtype == GFLA_F16) && grad_source_dtype == GFLA_F32)) return GFLA_E_DTYPE;
    REQ_ALIGN(source, dtype); REQ_ALIGN(grad_out, dtype); REQ_ALIGN(grad_source, grad_source_dtype);
    REQ_ALIGN(flow, flow_dtype); REQ_ALIGN(grad_flow, flow_dtype);
    return block_extract_bwd(source, flow, grad_out, grad_source, grad_flow, B, C, Hs, Ws, Hf, Wf, k, dtype, flow_dtype,
                             grad_source_dtype, accumulate, (cudaStream_t)stream);
}

int gfla_convert(const void* src, int src_dtype, void* dst, int dst_dtype, long long n, gfla_stream_t stream) {
    REQ_PTR(src); REQ_PTR(dst);
    if (n <= 0) return GFLA_E_SHAPE;
    if (!dtype_known(src_dtype) || !dtype_known(dst_dtype)) return GFLA_E_DTYPE;
    REQ_ALIGN(src, src_dtype); REQ_ALIGN(dst, dst_dtype);
    return convert(src, src_dtype, dst, dst_dtype, n, (cudaStream_t)stream);
}

int gfla_attn_reshape_fwd(const void* in, void* out, int B, int H, int W, int k, int dtype, gfla_stream_t stream) {
    REQ_PTR(in); REQ_PTR(out);
    if (!pos(B) || !pos(H) || !pos(W) || k < 1 || k > 9) return GFLA_E_SHAPE;
    if (!dtype_known(dtype)) return GFLA_E_DTYPE;
    REQ_ALIGN(in, dtype); REQ_ALIGN(out, dtype);
    return attn_reshape_fwd(in, out, B, H, W, k, dtype, (cudaStream_t)stream);
}

int gfla_attn_reshape_bwd(const void* grad_out, void* grad_in, int B, int H, int W, int k, int dtype, int accumulate,
                          gfla_stream_t stream) {
    REQ_PTR(grad_out); REQ_PTR(grad_in);
    if (!pos(B) || !pos(H) || !pos(W) || k < 1 || k > 9) return GFLA_E_SHAPE;
    if (!dtype_known(dtype)) return GFLA_E_DTYPE;
    REQ_ALIGN(grad_out, dtype); REQ_ALIGN(grad_in, dtype);
    return attn_reshape_bwd(grad_out, grad_in, B, H, W, k, dtype, accumulate, (cudaStream_t)stream);
}

int gfla_resample2d_fwd(const void* in1, const void* in2, void* out, int B, int C, int Hi, int Wi, int H, int W, int ks,
                        int dilation, int dtype, gfla_stream_t stream) {
    REQ_PTR(in1); REQ_PTR(in2); REQ_PTR(out);
    if (!pos(B) || !pos(C) || !pos(Hi) || !pos(Wi) || !pos(H) || !pos(W) || ks < 2 || ks > 9 || dilation < 1) return GFLA_E_SHAPE;
    if (dtype != GFLA_F32 && dtype != GFLA_F64) return GFLA_E_DTYPE;
    REQ_ALIGN(in1, dtype); REQ_ALIGN(in2, dtype); REQ_ALIGN(out, dtype);
    return resample2d_fwd(in1, in2, out, B, C, Hi, Wi, H, W, ks, dilation, dtype, (cudaStream_t)stream);
}

int gfla_resample2d_bwd(const void* in1, const void* in2, const void* grad_out, void* grad_in1, void* grad_in2, int B,
                        int C, int Hi, int Wi, int H, int W, int ks, int dilation, int dtype, int accumulate,
                        gfla_stream_t stream) {
    REQ_PTR(in1); REQ_PTR(in2); REQ_PTR(grad_out); REQ_PTR(grad_in1); REQ_PTR(grad_in2);
    if (!pos(B) || !pos(C) || !pos(Hi) || !pos(Wi) || !pos(H) || !pos(W) || ks < 2 || ks > 9 || dilation < 1) return GFLA_E_SHAPE;
    if (dtype != GFLA_F32 && dtype != GFLA_F64) return GFLA_E_DTYPE;
    REQ_ALIGN(in1, dtype); REQ_ALIGN(in2, dtype); REQ_ALIGN(grad_out, dtype); REQ_ALIGN(grad_in1, dtype); REQ_ALIGN(grad_in2, dtype);
    return resample2d_bwd(in1, in2, grad_out, grad_in1, grad_in2, B, C, Hi, Wi, H, W, ks, dilation, dtype, accumulate,
                          (cudaStream_t)stream);
}

int gfla_resample2d_cosine_fwd(const void* in1, const void* in2, const void* target, void* cos_out, void* stats, int B, int C, int Hi,
                               int Wi, int H, int W, int ks, int dilation, double eps, int dtype, gfla_stream_t stream) {
    REQ_PTR(in1); REQ_PTR(in2); REQ_PTR(target); REQ_PTR(cos_out); REQ_PTR(stats);
    if (!pos(B) || !pos(C) || !pos(Hi) || !pos(Wi) || !pos(H) || !pos(W) || ks < 2 || ks > 9 || dilation < 1 || !(eps >= 0)) return GFLA_E_SHAPE;
    if (dtype != GFLA_F32 && dtype != GFLA_F64) return GFLA_E_DTYPE;
    REQ_ALIGN(in1, dtype); REQ_ALIGN(in2, dtype); REQ_ALIGN(target, dtype); REQ_ALIGN(cos_out, dtype); REQ_ALIGN(stats, dtype);
    return resample2d_cos_fwd(in1, in2, target, cos_out, stats, B, C, Hi, Wi, H, W, ks, dilation, eps, dtype, (cudaStream_t)stream);
}

int gfla_resample2d_cosine_bwd(const void* in1, const void* in2, const void* target, const void* stats, const void* grad_cos,
                               void* grad_in1, void* grad_in2, void* grad_val, void* grad_target, int B, int C, int Hi, int Wi, int H,
                               int W, int ks, int dilation, double eps, int dtype, int accumulate, gfla_stream_t stream) {
    REQ_PTR(in1); REQ_PTR(in2); REQ_PTR(target); REQ_PTR(stats); REQ_PTR(grad_cos); REQ_PTR(grad_in2);
    if (grad_in1 != nullptr && grad_val == nullptr) return GFLA_E_NULL;      // the scatter runs on the materialised d/d(warped)
    if (!pos(B) || !pos(C) || !pos(Hi) || !pos(Wi) || !pos(H) || !pos(W) || ks < 2 || ks > 9 || dilation < 1 || !(eps >= 0)) return GFLA_E_SHAPE;
    if (dtype != GFLA_F32 && dtype != GFLA_F64) return GFLA_E_DTYPE;
    REQ_ALIGN(in1, dtype); REQ_ALIGN(in2, dtype); REQ_ALIGN(target, dtype); REQ_ALIGN(stats, dtype); REQ_ALIGN(grad_cos, dtype);
    REQ_ALIGN(grad_in2, dtype);
    if (grad_in1 != nullptr) { REQ_ALIGN(grad_in1, dtype); }
    if (grad_val != nullptr) { REQ_ALIGN(grad_val, dtype); }
    if (grad_target != nullptr) { REQ_ALIGN(grad_target, dtype); }
    return resample2d_cos_bwd(in1, in2, target, stats, grad_cos, grad_in1, grad_in2, grad_val, grad_target, B, C, Hi, Wi, H, W, ks, dilation,
                              eps, dtype, accumulate, (cudaStream_t)stream);
}

int gfla_resample2d_fwd_nhwc(const void* in1, const void* in2, void* out, int B, int C, int Hi, int Wi, int H, int W, int ks,
                             int dilation, int dtype, gfla_stream_t stream) {
    REQ_PTR(in1); REQ_PTR(in2); REQ_PTR(out);
    if (!pos(B) || !pos(C) || !pos(Hi) || !pos(Wi) || !pos(H) || !pos(W) || ks < 2 || ks > 9 || dilation < 1) return GFLA_E_SHAPE;
    if (!dtype_16bit(dtype)) return GFLA_E_DTYPE;
    REQ_ALIGN(in1, dtype); REQ_ALIGN(in2, GFLA_F32); REQ_ALIGN(out, dtype);
    return resample2d_nhwc_fwd(in1, in2, out, B, C, Hi, Wi, H, W, ks, dilation, dtype, (cudaStream_t)stream);
}

int gfla_resample2d_bwd_nhwc(const void* in1, const void* in2, const void* grad_out, void* grad_in1, void* grad_in2, int B, int C,
                             int Hi, int Wi, int H, int W, int ks, int dilation, int dtype, int grad_in1_dtype, int accumulate,
                             gfla_stream_t stream) {
    REQ_PTR(in1); REQ_PTR(in2); REQ_PTR(grad_out); REQ_PTR(grad_in1); REQ_PTR(grad_in2);
    if (!pos(B) || !pos(C) || !pos(Hi) || !pos(Wi) || !pos(H) || !pos(W) || ks < 2 || ks > 9 || dilation < 1) return GFLA_E_SHAPE;
    if (!dtype_16bit(dtype) || !grad_in1_dtype_ok(dtype, grad_in1_dtype)) return GFLA_E_DTYPE;
    REQ_ALIGN(in1, dtype); REQ_ALIGN(in2, GFLA_F32); REQ_ALIGN(grad_out, dtype); REQ_ALIGN(grad_in1, grad_in1_dtype);
    REQ_ALIGN(grad_in2, GFLA_F32);
    return resample2d_nhwc_bwd(in1, in2, grad_out, grad_in1, grad_in2, B, C, Hi, Wi, H, W, ks, dilation, dtype, grad_in1_dtype,
                               accumulate, (cudaStream_t)stream);
}

int gfla_resample2d_cosine_fwd_nhwc(const void* in1, const void* in2, const void* target, void* cos_out, void* stats, int B, int C,
                                    int Hi, int Wi, int H, int W, int ks, int dilation, double eps, int dtype, gfla_stream_t stream) {
    REQ_PTR(in1); REQ_PTR(in2); REQ_PTR(target); REQ_PTR(cos_out); REQ_PTR(stats);
    if (!pos(B) || !pos(C) || !pos(Hi) || !pos(Wi) || !pos(H) || !pos(W) || ks < 2 || ks > 9 || dilation < 1 || !(eps >= 0)) return GFLA_E_SHAPE;
    if (!dtype_16bit(dtype)) return GFLA_E_DTYPE;
    REQ_ALIGN(in1, dtype); REQ_ALIGN(target, dtype); REQ_ALIGN(in2, GFLA_F32); REQ_ALIGN(cos_out, GFLA_F32); REQ_ALIGN(stats, GFLA_F32);
    return resample2d_nhwc_cos_fwd(in1, in2, target, cos_out, stats, B, C, Hi, Wi, H, W, ks, dilation, eps, dtype, (cudaStream_t)stream);
}

int gfla_resample2d_cosine_bwd_nhwc(const void* in1, const void* in2, const void* target, const void* stats, const void* grad_cos,
                                    void* grad_in1, void* grad_in2, void* grad_val, void* grad_target, int B, int C, int Hi, int Wi,
                                    int H, int W, int ks, int dilation, double eps, int dtype, int grad_in1_dtype, int accumulate,
                                    gfla_stream_t stream) {
    REQ_PTR(in1); REQ_PTR(in2); REQ_PTR(target); REQ_PTR(stats); REQ_PTR(grad_cos); REQ_PTR(grad_in2);
    if (grad_in1 != nullptr && grad_val == nullptr) return GFLA_E_NULL;      // the scatter runs on the materialised d/d(warped)
    if (!pos(B) || !pos(C) || !pos(Hi) || !pos(Wi) || !pos(H) || !pos(W) || ks < 2 || ks > 9 || dilation < 1 || !(eps >= 0)) return GFLA_E_SHAPE;
    if (!dtype_16bit(dtype) || !grad_in1_dtype_ok(dtype, grad_in1_dtype)) return GFLA_E_DTYPE;
    REQ_ALIGN(in1, dtype); REQ_ALIGN(target, dtype); REQ_ALIGN(in2, GFLA_F32); REQ_ALIGN(stats, GFLA_F32); REQ_ALIGN(grad_cos, GFLA_F32);
    REQ_ALIGN(grad_in2, GFLA_F32);
    if (grad_in1 != nullptr) { REQ_ALIGN(grad_in1, grad_in1_dtype); }
    if (grad_val != nullptr) { REQ_ALIGN(grad_val, dtype); }
    if (grad_target != nullptr) { REQ_ALIGN(grad_target, dtype); }
    return resample2d_nhwc_cos_bwd(in1, in2, target, stats, grad_cos, grad_in1, grad_in2, grad_val, grad_target, B, C, Hi, Wi, H, W, ks,
                                   dilation, eps, dtype, grad_in1_dtype, accumulate, (cudaStream_t)stream);
}

static int local_attn_fwd_any(const void* source, const void* flow, const void* logits, void* out, void* probs,
                              const void* prev, const void* mask, int B, int C, int Hs, int Ws, int H, int W, int k, int dtype,
                              int flow_dtype, int layout, int algo, gfla_stream_t stream) {
    REQ_PTR(source); REQ_PTR(flow); REQ_PTR(logits); REQ_PTR(out);
    if (layout != GFLA_NCHW && layout != GFLA_NHWC) return GFLA_E_SHAPE;
    if (!pos(B) || !pos(C) || !pos(Hs) || !pos(Ws) || !pos(H) || !pos(W) || k < 1 || k > 9) return GFLA_E_SHAPE;
    if (!dtype_known(dtype) || !flow_dtype_ok(dtype, flow_dtype)) return GFLA_E_DTYPE;
    if (algo < 0 || algo > 2) return GFLA_E_NOTSUP;
    REQ_ALIGN(source, dtype); REQ_ALIGN(logits, dtype); REQ_ALIGN(out, dtype); REQ_ALIGN(flow, flow_dtype);
    if (probs) REQ_ALIGN(probs, dtype);
    if (prev) { REQ_ALIGN(prev, dtype); REQ_ALIGN(mask, dtype); }
    const bool tc_ok = local_attn_fwd_tc_supported(B, C, Hs, Ws, H, W, k, dtype, flow_dtype, layout, source, out) &&
                       (prev == nullptr || layout == GFLA_NCHW || aligned(prev, 16));
    if (algo == 2 && !tc_ok) return GFLA_E_NOTSUP;
    if (algo == 2 || (algo == 0 && tc_ok))
        return local_attn_fwd_tc(source, flow, logits, out, probs, prev, mask, B, C, Hs, Ws, H, W, k, dtype, flow_dtype, layout, (cudaStream_t)stream);
    return local_attn_fwd_gather(source, flow, logits, out, probs, prev, mask, B, C, Hs, Ws, H, W, k, dtype, flow_dtype, layout, (cudaStream_t)stream);
}

int gfla_local_attn_fwd(const void* source, const void* flow, const void* logits, void* out, void* probs, int B, int C,
                        int Hs, int Ws, int H, int W, int k, int dtype, int flow_dtype, int layout, int algo,
                        gfla_stream_t stream) {
    return local_attn_fwd_any(source, flow, logits, out, probs, nullptr, nullptr, B, C, Hs, Ws, H, W, k, dtype, flow_dtype,
                              layout, algo, stream);
}

int gfla_local_attn_blend_fwd(const void* source, const void* flow, const void* logits, const void* prev, const void* mask,
                              void* out, int B, int C, int Hs, int Ws, int H, int W, int k, int dtype, int flow_dtype,
                              int layout, int algo, gfla_stream_t stream) {
    REQ_PTR(prev); REQ_PTR(mask);
    return local_attn_fwd_any(source, flow, logits, out, nullptr, prev, mask, B, C, Hs, Ws, H, W, k, dtype, flow_dtype, layout,
                              algo, stream);
}

static int local_attn_bwd_any(const void* source, const void* flow, const void* logits, const void* grad_out,
                              void* grad_source, void* grad_flow, void* grad_logits, int B, int C, int Hs, int Ws, int H, int W,
                              int k, int dtype, int flow_dtype, int layout, int accumulate, int algo, void* workspace,
                              long long workspace_bytes, gfla_stream_t stream) {
    if (layout != GFLA_NCHW && layout != GFLA_NHWC) return GFLA_E_SHAPE;
    REQ_PTR(source); REQ_PTR(flow); REQ_PTR(logits); REQ_PTR(grad_out); REQ_PTR(grad_source); REQ_PTR(grad_flow); REQ_PTR(grad_logits);
    if (!pos(B) || !pos(C) || !pos(Hs) || !pos(Ws) || !pos(H) || !pos(W) || k < 1 || k > 9) return GFLA_E_SHAPE;
    if (!dtype_known(dtype) || !flow_dtype_ok(dtype, flow_dtype)) return GFLA_E_DTYPE;
    if (algo < 0 || algo > 2) return GFLA_E_NOTSUP;
    REQ_ALIGN(source, dtype); REQ_ALIGN(logits, dtype); REQ_ALIGN(grad_out, dtype); REQ_ALIGN(grad_source, dtype);
    REQ_ALIGN(grad_logits, dtype); REQ_ALIGN(flow, flow_dtype); REQ_ALIGN(grad_flow, flow_dtype);
    const bool tc_ok = local_attn_bwd_tc_supported(C, k, dtype, flow_dtype, layout, grad_out, grad_source);
    if (algo == 2 && !tc_ok) return GFLA_E_NOTSUP;
    if (algo == 2 || (algo == 0 && tc_ok)) {
        // grad_source: tile kernel (GEMM + TMA reduce-add); grad_flow / grad_logits: per-pixel dot products.
        // The batch is walked in chunks of `cb` samples (zero-fill, grad_source kernel, grad_flow/logits kernel per chunk):
        // with a chunk's grad_source + grad_out + source (3 * C*H*W*2 bytes per sample) inside the 126 MB L2, the zero-fill
        // never reaches HBM before the reduce-adds land on it, and the second kernel finds grad_out still in L2.
        const size_t per_s = (size_t)C * Hs * Ws * elem_size(dtype), per_o = (size_t)C * H * W * elem_size(dtype);
        const size_t per_f = (size_t)2 * H * W * elem_size(flow_dtype), per_l = (size_t)k * k * H * W * elem_size(dtype);
        int cb = B;
        {
            const char* v = getenv("GFLA_BWD_CHUNK");
            if (v) cb = atoi(v) > 0 ? atoi(v) : B;
        }
        const bool q_tc = local_attn_bwd_q_tc_supported(C, k);
        // one fused kernel (grad_out tile read once) where it can serve the shape; GFLA_BWD_FUSED=0 keeps the two-kernel path
        bool fused = kBwdFusedDefault && local_attn_bwd_fused_supported(C, k, source);
        {
            const char* v = getenv("GFLA_BWD_FUSED");
            if (v) fused = atoi(v) != 0 && local_attn_bwd_fused_supported(C, k, source);
        }
        for (int b0 = 0; b0 < B; b0 += cb) {
            const int nb = (B - b0 < cb) ? (B - b0) : cb;
            const char* s_ = (const char*)source + b0 * per_s;
            const char* f_ = (const char*)flow + b0 * per_f;
            const char* l_ = (const char*)logits + b0 * per_l;
            const char* g_ = (const char*)grad_out + b0 * per_o;
            char* gs_ = (char*)grad_source + b0 * per_s;
            char* gf_ = (char*)grad_flow + b0 * per_f;
            char* gl_ = (char*)grad_logits + b0 * per_l;
            int e = GFLA_OK;
            if (fused) {
                e = local_attn_bwd_fused_tc(s_, f_, l_, g_, gs_, gf_, gl_, nb, C, Hs, Ws, H, W, k, accumulate, workspace, workspace_bytes,
                                            (cudaStream_t)stream);
                if (e != GFLA_OK) return e;
                continue;
            }
            if (!accumulate) e = zero_async(gs_, nb * per_s, (cudaStream_t)stream);
            if (e == GFLA_OK) e = local_attn_bwd_gs_tc(f_, l_, g_, gs_, nb, C, Hs, Ws, H, W, k, (cudaStream_t)stream);
            if (e != GFLA_OK) return e;
            if (q_tc)
                e = local_attn_bwd_q_tc(s_, f_, l_, g_, gf_, gl_, nb, C, Hs, Ws, H, W, k, accumulate, (cudaStream_t)stream);
            else
                e = local_attn_bwd_gather(s_, f_, l_, g_, gs_, gf_, gl_, nb, C, Hs, Ws, H, W, k, dtype, flow_dtype, accumulate,
                                          layout, /*do_gs=*/0, (cudaStream_t)stream);
            if (e != GFLA_OK) return e;
        }
        return GFLA_OK;
    }
    return local_attn_bwd_gather(source, flow, logits, grad_out, grad_source, grad_flow, grad_logits, B, C, Hs, Ws, H, W,
                                 k, dtype, flow_dtype, accumulate, layout, /*do_gs=*/1, (cudaStream_t)stream);
}

int gfla_local_attn_bwd(const void* source, const void* flow, const void* logits, const void* grad_out,
                        void* grad_source, void* grad_flow, void* grad_logits, int B, int C, int Hs, int Ws, int H, int W,
                        int k, int dtype, int flow_dtype, int layout, int accumulate, int algo, gfla_stream_t stream) {
    return local_attn_bwd_any(source, flow, logits, grad_out, grad_source, grad_flow, grad_logits, B, C, Hs, Ws, H, W, k, dtype,
                              flow_dtype, layout, accumulate, algo, nullptr, 0, stream);
}

long long gfla_local_attn_bwd_workspace_bytes(int B) { return B > 0 ? 4LL * B + 4LL * 4096 : 0; }   // counters per sample + a progress word per CTA (<= SM count)

int gfla_local_attn_bwd_ws(const void* source, const void* flow, const void* logits, const void* grad_out,
                           void* grad_source, void* grad_flow, void* grad_logits, int B, int C, int Hs, int Ws, int H, int W,
                           int k, int dtype, int flow_dtype, int layout, int accumulate, int algo, void* workspace,
                           long long workspace_bytes, gfla_stream_t stream) {
    if (workspace != nullptr && workspace_bytes < 0) return GFLA_E_SHAPE;
    return local_attn_bwd_any(source, flow, logits, grad_out, grad_source, grad_flow, grad_logits, B, C, Hs, Ws, H, W, k, dtype,
                              flow_dtype, layout, accumulate, algo, workspace, workspace_bytes, stream);
}

}  // extern "C"
