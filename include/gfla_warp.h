/*
 * gfla_warp.h -- C ABI of the B200-native (sm_100a) GFLA warping library.
 *
 * This is the drop-in boundary for the warping hot path of
 * RenYurui/Global-Flow-Local-Attention: the three custom extensions under
 * model/networks/ (block_extractor, local_attn_reshape, resample2d_package)
 * and the local-attention softmax-weighted gather they feed (ExtractorAttn,
 * model/networks/base_function.py:790-818).  Each entry point names the
 * reference interface (pybind function, file:line) it replaces.
 *
 * Conventions (all entry points)
 *   - plain pointers + sizes only: no torch / ATen types cross this boundary.
 *     Pointers are DEVICE pointers to contiguous NCHW tensors on the device
 *     that owns `stream` (the caller's current device).
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).
 *     The reference launches on at::cuda::getCurrentCUDAStream()
 *     (block_extractor_kernel.cu:197); callers pass that same stream.
 *   - nothing is allocated, retained or synchronised inside the library; there
 *     is no global mutable state (safe under one host thread per GPU).
 *   - return value: 0 on success; a negative GFLA_E_* code for argument
 *     errors (nothing was launched); a positive cudaError_t if a launch
 *     failed.  (The reference returns the constant 1 and checks nothing,
 *     block_extractor_cuda.cc:12; see INTEGRATION.md for the shim that maps
 *     this back to the legacy `int` return.)
 *   - dtype codes describe the element type of source / output / logits /
 *     gradient tensors; `flow_dtype` that of the flow field and its gradient.
 *     F32 and F64 mirror the reference's AT_DISPATCH_FLOATING_TYPES
 *     (float, double only).  BF16 / F16 storage is an extension: arithmetic
 *     is fp32, and the flow may stay fp32 (`flow_dtype` = GFLA_F32) so the tap
 *     indices are bit-identical to the fp32 reference.
 *   - every size is an `int` like in the reference, but products are formed
 *     in 64 bits (the reference overflows `int n` above 2^31 elements,
 *     block_extractor_kernel.cu:33,180).
 *   - `accumulate` (backward entry points): 1 = reference semantics -- the
 *     gradients are ADDED into caller-provided (normally zero-filled) buffers
 *     (block_extractor.py:35-36, resample2d.py:32-33); 0 = the library
 *     overwrites them (zero-filling internally where it scatters), so the
 *     caller may pass uninitialised memory.
 */
#ifndef GFLA_WARP_H_
#define GFLA_WARP_H_

#ifdef __cplusplus
extern "C" {
#endif

#define GFLA_ABI_VERSION 1

typedef void* gfla_stream_t; /* cudaStream_t */

enum gfla_dtype { GFLA_F32 = 0, GFLA_F64 = 1, GFLA_BF16 = 2, GFLA_F16 = 3 };

/* storage order of the [B,C,H,W] feature tensors of the fused op (source, out and their gradients);
 * flow / logits / probs are always planar (NCHW).  NHWC = torch.channels_last. */
enum gfla_layout { GFLA_NCHW = 0, GFLA_NHWC = 1 };

enum gfla_error {
    GFLA_OK = 0,
    GFLA_E_NULL = -1,     /* a required pointer is NULL                          */
    GFLA_E_SHAPE = -2,    /* non-positive size, or kernel_size outside [1, 9]    */
    GFLA_E_DTYPE = -3,    /* unknown dtype code / unsupported dtype combination  */
    GFLA_E_ALIGN = -4,    /* pointer not aligned to its element size             */
    GFLA_E_NOTSUP = -5    /* requested fast path cannot serve this call          */
};

int gfla_abi_version(void);
/* static string for any code returned by this library (GFLA_E_* or cudaError_t) */
const char* gfla_error_string(int code);
/* compute capability the library was built for (100) and whether the running
 * device can execute it; returns 0 when usable. */
int gfla_device_check(void);

/* Debug aid for the tile kernels: `host_mapped_u64x8` is a DEVICE-visible pointer to 8
 * zero-initialised uint64 in pinned host memory (or NULL to disable).  If a pipeline
 * barrier inside a tile kernel ever times out, the kernel records which one there and
 * traps instead of hanging the GPU.  Not used on the normal path. */
int gfla_debug_set_buffer(void* host_mapped_u64x8);

/* Statistics: number of kernels this library has launched in this process so far (all entry points, all
 * threads; a relaxed counter that nothing inside the library reads).  bench.py reports the difference across
 * its timed region as `gpu_launches`. */
unsigned long long gfla_debug_launch_count(void);

/* Debug aid for tuning the tile kernels: cycles their warps spent blocked on the pipeline barriers.
 * Only in profile builds of the library (GFLA_BUILD_PROFILE=1 at build time, -DGFLA_TC_PROFILE); a normal build
 * carries no timing code and returns GFLA_E_NOTSUP.  `which`: 0 = per-tile forward kernel, 1 = strip forward kernel,
 * 2 = fused backward kernel.  Copies the 64 counters collected since the last call into `out_u64x64` (HOST memory, may
 * be NULL), clears them and switches collection on (enable = 1) or off (0).  Index = role * 8 + kind (roles and kinds per
 * kernel: tools/wait_profile.py); [7] = kernel cycles summed over the CTAs.  Synchronises the device. */
int gfla_debug_wait_profile(int which, int enable, unsigned long long* out_u64x64);

/* Re-layout of a [B,C,H,W] feature tensor between planar NCHW and channels-last NHWC storage
 * (out of place; to_nhwc = 1: NCHW -> NHWC, 0: NHWC -> NCHW).  Not part of the reference's API: the
 * Python layer uses it to serve planar bf16 callers with the channels-last tile kernels. */
int gfla_relayout(const void* src, void* dst, int B, int C, int H, int W, int dtype, int to_nhwc,
                  gfla_stream_t stream);

/* ------------------------------------------------------------------------ *
 * block_extractor
 *   replaces block_extractor_cuda.forward(source, flow_field, output, k)
 *            block_extractor_cuda.backward(source, flow_field, grad_output,
 *                                          grad_source, grad_flow_field, k)
 *   (block_extractor/block_extractor_cuda.cc:5-33, kernels
 *    block_extractor_kernel.cu:20-85 and :89-170)
 *   source [B,C,Hs,Ws], flow [B,2,Hf,Wf] (ch0 = x, ch1 = y, in pixels)
 *   out / grad_out [B,C,k*Hf,k*Wf]; Hs,Ws may differ from Hf,Wf
 *   (external_function.py:61-66).
 * ------------------------------------------------------------------------ */
int gfla_block_extract_fwd(const void* source, const void* flow, void* out,
                           int B, int C, int Hs, int Ws, int Hf, int Wf, int k,
                           int dtype, int flow_dtype, gfla_stream_t stream);
/* grad_source_dtype: == dtype (reference contract), or GFLA_F32 when dtype is a 16-bit type: the scatter then
 * uses native fp32 red.global instead of 16-bit compare-and-swap atomics; narrow with gfla_convert(). */
int gfla_block_extract_bwd(const void* source, const void* flow, const void* grad_out,
                           void* grad_source, void* grad_flow,
                           int B, int C, int Hs, int Ws, int Hf, int Wf, int k,
                           int dtype, int flow_dtype, int grad_source_dtype, int accumulate,
                           gfla_stream_t stream);
/* element-wise dtype conversion between fp32 and bf16 / f16 (n elements, contiguous) */
int gfla_convert(const void* src, int src_dtype, void* dst, int dst_dtype, long long n, gfla_stream_t stream);

/* ------------------------------------------------------------------------ *
 * local_attn_reshape  ([B,k*k,H,W] -> [B,1,k*H,k*W], depth-to-space)
 *   replaces local_attn_reshape_cuda.forward(inputs, output, k)
 *            local_attn_reshape_cuda.backward(inputs, grad_output, grad_inputs, k)
 *   (local_attn_reshape/local_attn_reshape_cuda.cc:5-29, kernels
 *    local_attn_reshape_kernel.cu:20-61 and :65-108; `inputs` is unused by
 *    the reference backward and is not part of this signature)
 * ------------------------------------------------------------------------ */
int gfla_attn_reshape_fwd(const void* in, void* out, int B, int H, int W, int k,
                          int dtype, gfla_stream_t stream);
int gfla_attn_reshape_bwd(const void* grad_out, void* grad_in, int B, int H, int W, int k,
                          int dtype, int accumulate, gfla_stream_t stream);

/* ------------------------------------------------------------------------ *
 * resample2d  (Gaussian-weighted ks x ks warp with dilation)
 *   replaces resample2d_cuda.forward(input1, input2, output, ks, dilation)
 *            resample2d_cuda.backward(input1, input2, gradOutput,
 *                                     gradInput1, gradInput2, ks, dilation)
 *   (resample2d_package/resample2d_cuda.cc:6-33, kernels
 *    resample2d_kernel.cu:20-95, :98-202, :204-330)
 *   in1 [B,C,Hi,Wi]; in2 [B,3,H,W] = (dx, dy, sigma) -- the sigma plane is
 *   appended by the Python module (resample2d.py:51-52); out [B,C,H,W];
 *   grad_in2 [B,3,H,W] (all three planes are written, like :328).
 *   in2 / grad_in2 have the same dtype as in1 (F32 or F64 only here; BF16 / F16
 *   feature maps take the *_nhwc entries below).
 * ------------------------------------------------------------------------ */
int gfla_resample2d_fwd(const void* in1, const void* in2, void* out,
                        int B, int C, int Hi, int Wi, int H, int W, int ks, int dilation,
                        int dtype, gfla_stream_t stream);
int gfla_resample2d_bwd(const void* in1, const void* in2, const void* grad_out,
                        void* grad_in1, void* grad_in2,
                        int B, int C, int Hi, int Wi, int H, int W, int ks, int dilation,
                        int dtype, int accumulate, gfla_stream_t stream);

/* ------------------------------------------------------------------------ *
 * resample2d -> cosine similarity, fused  (SURVEY row f4)
 *   replaces, in PerceptualCorrectness.calculate_loss
 *   (model/networks/external_function.py:275-279),
 *       input_sample      = Resample2d(4, 1, sigma=2)(source_vgg, flow)   # resample2d_cuda.forward
 *       correction_sample = F.cosine_similarity(input_sample, target_all) # over the channel axis
 *   and their backward (resample2d_cuda.backward + ATen) by one kernel each
 *   way; the warped feature tensor [B,C,H,W] is never written.
 *   in1 = source features [B,C,Hi,Wi]; in2 [B,3,H,W] as for resample2d;
 *   target [B,C,H,W]; cos_out [B,H,W];
 *   cos = sum_c (v_c / max(|v|,eps)) * (t_c / max(|t|,eps))   (ATen, eps = 1e-8 in the reference call);
 *   stats [B,3,H,W] = (v.t, |v|, |t|), written by the forward and read by the backward.
 *   Backward: grad_cos [B,H,W] -> grad_in2 [B,3,H,W] (always);
 *   grad_target [B,C,H,W] optional (NULL = not wanted);
 *   grad_in1 [B,C,Hi,Wi] optional -- it needs grad_val, a caller-provided
 *   [B,C,H,W] scratch tensor that receives d/d(warped) before the scatter.
 *   accumulate applies to grad_in1 / grad_in2 / grad_target.  F32 or F64 here;
 *   BF16 / F16 feature maps take the *_nhwc entries below.
 * ------------------------------------------------------------------------ */
int gfla_resample2d_cosine_fwd(const void* in1, const void* in2, const void* target,
                               void* cos_out, void* stats,
                               int B, int C, int Hi, int Wi, int H, int W, int ks, int dilation,
                               double eps, int dtype, gfla_stream_t stream);
int gfla_resample2d_cosine_bwd(const void* in1, const void* in2, const void* target,
                               const void* stats, const void* grad_cos,
                               void* grad_in1, void* grad_in2, void* grad_val, void* grad_target,
                               int B, int C, int Hi, int Wi, int H, int W, int ks, int dilation,
                               double eps, int dtype, int accumulate, gfla_stream_t stream);

/* ------------------------------------------------------------------------ *
 * resample2d and resample2d -> cosine on channels-last 16-bit feature maps
 *   the same four operations as gfla_resample2d_{fwd,bwd} (resample2d_cuda.cc:6-33,
 *   resample2d_kernel.cu:20-95, :98-202, :204-330) and gfla_resample2d_cosine_{fwd,bwd}
 *   (external_function.py:275-279), for BF16 / F16 feature storage (`dtype`) in
 *   NHWC = torch.channels_last order: in1 [B,Hi,Wi,C]; out, grad_out, target,
 *   grad_val, grad_target [B,H,W,C]; grad_in1 [B,Hi,Wi,C].
 *   in2 / grad_in2 [B,3,H,W], cos_out / grad_cos [B,H,W] and stats [B,3,H,W] are
 *   planar F32.  Arithmetic is fp32: a pixel's taps and weights are those of the
 *   F32 entries; sums over channels are fp32 in another order.
 *   grad_in1_dtype: == dtype (16-bit reductions, each add rounded), or GFLA_F32
 *   (fp32 reductions; narrow with gfla_convert()).  grad_val has `dtype`.
 * ------------------------------------------------------------------------ */
int gfla_resample2d_fwd_nhwc(const void* in1, const void* in2, void* out,
                             int B, int C, int Hi, int Wi, int H, int W, int ks, int dilation,
                             int dtype, gfla_stream_t stream);
int gfla_resample2d_bwd_nhwc(const void* in1, const void* in2, const void* grad_out,
                             void* grad_in1, void* grad_in2,
                             int B, int C, int Hi, int Wi, int H, int W, int ks, int dilation,
                             int dtype, int grad_in1_dtype, int accumulate, gfla_stream_t stream);
int gfla_resample2d_cosine_fwd_nhwc(const void* in1, const void* in2, const void* target,
                                    void* cos_out, void* stats,
                                    int B, int C, int Hi, int Wi, int H, int W, int ks, int dilation,
                                    double eps, int dtype, gfla_stream_t stream);
int gfla_resample2d_cosine_bwd_nhwc(const void* in1, const void* in2, const void* target,
                                    const void* stats, const void* grad_cos,
                                    void* grad_in1, void* grad_in2, void* grad_val, void* grad_target,
                                    int B, int C, int Hi, int Wi, int H, int W, int ks, int dilation,
                                    double eps, int dtype, int grad_in1_dtype, int accumulate,
                                    gfla_stream_t stream);

/* ------------------------------------------------------------------------ *
 * fused local attention = the tail of ExtractorAttn.forward
 *   (base_function.py:804-810 with softmax=True, generator.py:112):
 *     out = avg_pool2d( LocalAttnReshape(Softmax_dim1(logits)) *
 *                       BlockExtractor(k)(source, flow), k, k )
 *   computed without materialising the [B,C,k*H,k*W] block tensor.
 *   source [B,C,Hs,Ws]; flow [B,2,H,W]; logits [B,k*k,H,W] (pre-softmax);
 *   out [B,C,H,W]; probs (optional, may be NULL) [B,k*k,H,W] receives the
 *   softmax, i.e. what hook_attn_param returns (base_function.py:812-818).
 *   Backward: grad_source follows `accumulate`; grad_flow [B,2,H,W] and
 *   grad_logits [B,k*k,H,W] likewise.
 *   `layout`: GFLA_NCHW (the reference's contiguous layout) or GFLA_NHWC (channels-last: every
 *           source position is 2*C contiguous bytes -- the layout the tile kernels are fastest on).
 *   `algo`: 0 = automatic choice, 1 = CUDA-core gather kernel,
 *           2 = tcgen05 tile kernel (GFLA_E_NOTSUP if it cannot serve the call).
 * ------------------------------------------------------------------------ */
int gfla_local_attn_fwd(const void* source, const void* flow, const void* logits,
                        void* out, void* probs,
                        int B, int C, int Hs, int Ws, int H, int W, int k,
                        int dtype, int flow_dtype, int layout, int algo, gfla_stream_t stream);
/* Same forward with the caller's mask blend fused into the store (SURVEY 8(f2); generator.py:130,
 * `out = out*(1-mask) + out_attn*mask`, and the two-branch sum at generator.py:496-498):
 *     out = prev * (1 - mask) + local_attention(source, flow, logits) * mask
 * prev [B,C,H,W] (same dtype/layout as out; may alias nothing), mask [B,1,H,W] planar, same dtype.
 * Forward only (inference): training code keeps the unfused blend so autograd sees it. */
int gfla_local_attn_blend_fwd(const void* source, const void* flow, const void* logits,
                              const void* prev, const void* mask, void* out,
                              int B, int C, int Hs, int Ws, int H, int W, int k,
                              int dtype, int flow_dtype, int layout, int algo, gfla_stream_t stream);
int gfla_local_attn_bwd(const void* source, const void* flow, const void* logits,
                        const void* grad_out,
                        void* grad_source, void* grad_flow, void* grad_logits,
                        int B, int C, int Hs, int Ws, int H, int W, int k,
                        int dtype, int flow_dtype, int layout, int accumulate, int algo,
                        gfla_stream_t stream);
/* The same backward with a caller-provided scratch buffer (DEVICE memory, >= gfla_local_attn_bwd_workspace_bytes(B) bytes,
 * 4-byte aligned, contents irrelevant, may be reused by the next call on the same stream).  With it -- and accumulate = 0 --
 * the fused tcgen05 backward zero-fills grad_source INSIDE the kernel, sample by sample just ahead of its own reduce-adds
 * (per-sample completion counters live in the workspace), instead of a separate memset pass in front of it: one pass less
 * over the 2*C*Hs*Ws*B bytes, and the zeros are still in L2 when the adds land on them.  workspace = NULL behaves exactly
 * like gfla_local_attn_bwd.  The library itself never allocates. */
long long gfla_local_attn_bwd_workspace_bytes(int B);
int gfla_local_attn_bwd_ws(const void* source, const void* flow, const void* logits,
                           const void* grad_out,
                           void* grad_source, void* grad_flow, void* grad_logits,
                           int B, int C, int Hs, int Ws, int H, int W, int k,
                           int dtype, int flow_dtype, int layout, int accumulate, int algo,
                           void* workspace, long long workspace_bytes, gfla_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GFLA_WARP_H_ */
