// resample2d family on channels-last (NHWC) bf16 / fp16 feature maps, fp32 arithmetic, for sm_100a.
//
// The same five operations as resample2d.cu (forward, grad input1, grad input2, and the fused cosine forward / backward),
// for the feature tensors a network cast with `.bfloat16().to(memory_format=torch.channels_last)` produces.  The flow
// (in2 = dx, dy, sigma) and everything per pixel (grad_in2, cos, stats, grad_cos) stay planar fp32.
//
// Arithmetic contract: a pixel's taps and weights come from rs_setup<float, NT> / rs_weight_sum, the functions the fp32
// planar kernels use, in a translation unit also built with -fmad=false -- so they are the fp32 path's bits, including
// the reference quirks documented in resample2d.cu (fp64 SAFE_DIV / exp once per pixel, the int() fraction of grad
// input1).  Sums over channels are fp32.  Against the fp32 path run on the widened inputs, the only differences are the
// order of the sums over channels and the rounding at the 16-bit stores: the forward output is the fp32 path's output
// rounded once.
//
// Layout on the machine: a CTA is a 32 x 4 pixel tile (rs_pixel<4>, as in resample2d.cu), one warp per 32-pixel row
// segment, in two phases per warp:
//   1. lane = pixel: rs_setup once per pixel; the NQ = 4*(ks/2)^2 weights and clamped tap offsets go to shared memory
//      ([q][pixel], conflict-free both ways);
//   2. lanes = channels: a group of G lanes (G = the power of two that covers C / VEC, at most 32) walks one pixel's
//      channels, VEC = 8 channels (one 16-byte load) per lane and step, 32 / G pixels at a time.  In NHWC a tap is one
//      contiguous run of C channels, so a group's loads are whole 16-byte sectors instead of the planar layout's
//      one-element-per-plane gather.  C % 8 != 0 or an unaligned pointer selects VEC = 1 (scalar channels).
//   Per-pixel channel sums (grad input2's corner dot products, the cosine's three sums) are reduced across the group with
//   shuffles; grad input2's combine then runs once more with lane = pixel (phase 3), re-deriving the taps (rs_setup) rather
//   than holding them in registers through phase 2.
// grad input1 is a scatter: into an fp32 NHWC buffer with 16-byte red.global.add.v4.f32 (the caller narrows it with
// gfla_convert), or straight into 16-bit storage with 16-bit reductions (every add rounded to 16 bits: less accurate).
#include <type_traits>

#include "resample2d_common.cuh"

namespace gfla {

template <typename T> __device__ __forceinline__ float2 unpack2(unsigned u);
template <> __device__ __forceinline__ float2 unpack2<__nv_bfloat16>(unsigned u) {
    return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u));
}
template <> __device__ __forceinline__ float2 unpack2<__half>(unsigned u) { return __half22float2(*reinterpret_cast<const __half2*>(&u)); }
template <typename T> __device__ __forceinline__ unsigned pack2(float a, float b);
template <> __device__ __forceinline__ unsigned pack2<__nv_bfloat16>(float a, float b) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const unsigned*>(&h);
}
template <> __device__ __forceinline__ unsigned pack2<__half>(float a, float b) {
    const __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<const unsigned*>(&h);
}

// VEC consecutive channels as fp32 (VEC = 8: one 16-byte access)
template <typename T, int VEC>
__device__ __forceinline__ void ld_vec(const T* p, float (&v)[VEC]) {
    if constexpr (VEC == 8) {
        const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
        const float2 a = unpack2<T>(u.x), b = unpack2<T>(u.y), c = unpack2<T>(u.z), d = unpack2<T>(u.w);
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = d.x; v[7] = d.y;
    } else {
        v[0] = ld(p);
    }
}
template <typename T, int VEC>
__device__ __forceinline__ void st_vec(T* p, const float (&v)[VEC]) {
    if constexpr (VEC == 8) {
        *reinterpret_cast<uint4*>(p) = make_uint4(pack2<T>(v[0], v[1]), pack2<T>(v[2], v[3]), pack2<T>(v[4], v[5]), pack2<T>(v[6], v[7]));
    } else {
        st(p, v[0]);
    }
}
// read-modify-write of caller memory (grad_target with accumulate = 1): a plain load, not the read-only path
template <typename T, int VEC>
__device__ __forceinline__ void ld_vec_rw(const T* p, float (&v)[VEC]) {
    if constexpr (VEC == 8) {
        const uint4 u = *reinterpret_cast<const uint4*>(p);
        const float2 a = unpack2<T>(u.x), b = unpack2<T>(u.y), c = unpack2<T>(u.z), d = unpack2<T>(u.w);
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = d.x; v[7] = d.y;
    } else {
        v[0] = ld(p);
    }
}

__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
// 16-bit reductions in L2 (sm_90+): packed pairs, eight channels per instruction
__device__ __forceinline__ void red_add_v4x2(__nv_bfloat16* p, unsigned a, unsigned b, unsigned c, unsigned d) {
    asm volatile("red.global.add.noftz.v4.bf16x2 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void red_add_v4x2(__half* p, unsigned a, unsigned b, unsigned c, unsigned d) {
    asm volatile("red.global.add.noftz.v4.f16x2 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void red_add_1(__nv_bfloat16* p, float v) {
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    asm volatile("red.global.add.noftz.bf16 [%0], %1;" ::"l"(p), "h"(*reinterpret_cast<const unsigned short*>(&h)) : "memory");
}
__device__ __forceinline__ void red_add_1(__half* p, float v) {
    const __half h = __float2half_rn(v);
    asm volatile("red.global.add.noftz.f16 [%0], %1;" ::"l"(p), "h"(*reinterpret_cast<const unsigned short*>(&h)) : "memory");
}
__device__ __forceinline__ void red_add_1(float* p, float v) { atomicAdd(p, v); }
// scatter-add of VEC channels into grad_in1 (TG = float: fp32 reductions; TG = 16-bit: 16-bit reductions, each add rounded)
template <typename TG, int VEC>
__device__ __forceinline__ void red_vec(TG* p, const float (&v)[VEC]) {
    if constexpr (VEC == 8 && std::is_same<TG, float>::value) {
        red_add_v4(p, v[0], v[1], v[2], v[3]);
        red_add_v4(p + 4, v[4], v[5], v[6], v[7]);
    } else if constexpr (VEC == 8) {
        red_add_v4x2(p, pack2<TG>(v[0], v[1]), pack2<TG>(v[2], v[3]), pack2<TG>(v[4], v[5]), pack2<TG>(v[6], v[7]));
    } else {
        red_add_1(p, v[0]);
    }
}

// tap offset q of pixel p, re-read from shared memory at each use: a hoisted copy would hold 4*NT*NT 64-bit addresses
// in registers across the channel loop
__device__ __forceinline__ int tap_off(const int* so, int q, int p) { return *(static_cast<const volatile int*>(so) + q * 32 + p); }

__device__ __forceinline__ float group_sum(float v, int G) {
    for (int o = G >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// phase 1, lane = pixel: the forward weights (the fp32 path's w[q]), tap offsets and weight sum of the warp's 32 pixels
template <int NT>
__device__ __forceinline__ void rs16_stage(const float* __restrict__ in2, const RsPixel& px, int H, int W, int Hi, int Wi, int dil,
                                           float* sw, int* so, float* ssum, int lane) {
    if (px.active) {
        RsTaps<float, NT> t;
        rs_setup<float, NT>(t, in2, px.b, px.y, px.x, H, W, Hi, Wi, dil, false);
#pragma unroll
        for (int fy = 0; fy < NT; ++fy)
#pragma unroll
            for (int fx = 0; fx < NT; ++fx) {
                const int q = (fy * NT + fx) * 4;
                sw[(q + 0) * 32 + lane] = t.yT_P[fy] * t.xL_P[fx]; sw[(q + 1) * 32 + lane] = t.yT_P[fy] * t.xR_P[fx];
                sw[(q + 2) * 32 + lane] = t.yB_P[fy] * t.xL_P[fx]; sw[(q + 3) * 32 + lane] = t.yB_P[fy] * t.xR_P[fx];
            }
#pragma unroll
        for (int q = 0; q < NT * NT * 4; ++q) so[q * 32 + lane] = t.off[q];
        ssum[lane] = rs_weight_sum<float, NT>(t);
    }
    __syncwarp();
}

// the warped value of VEC channels of one pixel: exactly k_resample2d_fwd<float>'s output elements
template <typename T, int NT, int VEC>
__device__ __forceinline__ void rs16_warp(const T* __restrict__ src, const float* sw, const int* so, int p, int C, int c, float sum,
                                          float (&v)[VEC]) {
    float acc[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
#pragma unroll
    for (int q = 0; q < NT * NT * 4; ++q) {
        const float wq = sw[q * 32 + p];
        float s[VEC];
        ld_vec<T, VEC>(src + (long long)tap_off(so, q, p) * C + c, s);
#pragma unroll
        for (int j = 0; j < VEC; ++j) acc[j] += wq * s[j];
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j) v[j] = static_cast<float>(safe_div<float>(acc[j], sum));
}

template <int NT> struct Rs16Smem {           // bytes of dynamic shared memory per warp
    static constexpr int NQ = NT * NT * 4;
    static constexpr int fwd = NQ * 32 * 8 + 32 * 4;                 // weights, offsets, sum
    static constexpr int in1 = NQ * 32 * 12;                         // double weights, offsets
    static constexpr int in2 = NQ * 32 * 8;                          // offsets, corner dot products
    static constexpr int cos_bwd = NQ * 32 * 12 + 32 * 4 * 4;        // weights, offsets, dot products, sum, k1 / k2v / k2t
};

template <typename T, int NT, int VEC>
__global__ void __launch_bounds__(128)
k_resample2d_nhwc_fwd(const T* __restrict__ in1, const float* __restrict__ in2, T* __restrict__ out, int C, int Hi, int Wi, int H,
                      int W, int dil, int lg) {
    constexpr int NQ = NT * NT * 4;
    extern __shared__ __align__(16) unsigned char rs16_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* sw = reinterpret_cast<float*>(rs16_smem + warp * Rs16Smem<NT>::fwd);
    int* so = reinterpret_cast<int*>(sw + NQ * 32);
    float* ssum = sw + 2 * NQ * 32;
    const RsPixel px = rs_pixel<4>(H, W);
    if (px.y >= H) return;                                            // warp-uniform
    rs16_stage<NT>(in2, px, H, W, Hi, Wi, dil, sw, so, ssum, lane);
    const int G = 1 << lg, x0 = px.x - lane;
    const T* src = in1 + (long long)px.b * Hi * Wi * C;
    T* row = out + ((long long)px.b * H + px.y) * W * C;
    for (int p = lane >> lg; p < 32 && x0 + p < W; p += 32 >> lg) {
        const float sum = ssum[p];
        T* o = row + (long long)(x0 + p) * C;
        for (int c = (lane & (G - 1)) * VEC; c < C; c += G * VEC) {
            float v[VEC];
            rs16_warp<T, NT, VEC>(src, sw, so, p, C, c, sum, v);
            st_vec<T, VEC>(o + c, v);
        }
    }
}

// grad input1: grad_out's channels of a pixel scattered to its 4*NT*NT taps with the fp32 path's weights
// SAFE_DIV(w, sum) (fp64, from the truncating fraction) -- each contribution is float(wn * g), the fp32 path's value
template <typename T, typename TG, int NT, int VEC>
__global__ void __launch_bounds__(128)
k_resample2d_nhwc_bwd_in1(const float* __restrict__ in2, const T* __restrict__ gout, TG* __restrict__ gin1, int C, int Hi, int Wi,
                          int H, int W, int dil, int lg) {
    constexpr int NQ = NT * NT * 4;
    extern __shared__ __align__(16) unsigned char rs16_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* swn = reinterpret_cast<double*>(rs16_smem + warp * Rs16Smem<NT>::in1);
    int* so = reinterpret_cast<int*>(swn + NQ * 32);
    const RsPixel px = rs_pixel<4>(H, W);
    if (px.y >= H) return;
    if (px.active) {
        RsTaps<float, NT> t;
        rs_setup<float, NT>(t, in2, px.b, px.y, px.x, H, W, Hi, Wi, dil, true);   // truncating fraction for the weights
        const float sum = rs_weight_sum<float, NT>(t);
#pragma unroll
        for (int fy = 0; fy < NT; ++fy)
#pragma unroll
            for (int fx = 0; fx < NT; ++fx) {
                const int q = (fy * NT + fx) * 4;
                swn[(q + 0) * 32 + lane] = safe_div<float>(t.yT_P[fy] * t.xL_P[fx], sum);
                swn[(q + 1) * 32 + lane] = safe_div<float>(t.yT_P[fy] * t.xR_P[fx], sum);
                swn[(q + 2) * 32 + lane] = safe_div<float>(t.yB_P[fy] * t.xL_P[fx], sum);
                swn[(q + 3) * 32 + lane] = safe_div<float>(t.yB_P[fy] * t.xR_P[fx], sum);
            }
#pragma unroll
        for (int q = 0; q < NQ; ++q) so[q * 32 + lane] = t.off[q];
    }
    __syncwarp();
    const int G = 1 << lg, x0 = px.x - lane;
    TG* dst = gin1 + (long long)px.b * Hi * Wi * C;
    const T* row = gout + ((long long)px.b * H + px.y) * W * C;
    for (int p = lane >> lg; p < 32 && x0 + p < W; p += 32 >> lg) {
        const T* go = row + (long long)(x0 + p) * C;
        for (int c = (lane & (G - 1)) * VEC; c < C; c += G * VEC) {
            float g[VEC];
            ld_vec<T, VEC>(go + c, g);
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                const double wq = swn[q * 32 + p];
                float v[VEC];
#pragma unroll
                for (int j = 0; j < VEC; ++j) v[j] = static_cast<float>(wq * static_cast<double>(g[j]));
                red_vec<TG, VEC>(dst + (long long)tap_off(so, q, p) * C + c, v);
            }
        }
    }
}

// phase 3 of the kernels that produce grad input2: lane = pixel, the corner dot products D of its pixel are in sD
template <int NT>
__device__ __forceinline__ void rs16_in2_store(const float* __restrict__ in2, const RsPixel& px, int H, int W, int Hi, int Wi, int dil,
                                               const float* sD, float* __restrict__ gin2, int accumulate, int lane) {
    if (!px.active) return;
    RsTaps<float, NT> t;
    rs_setup<float, NT>(t, in2, px.b, px.y, px.x, H, W, Hi, Wi, dil, false);
    const float sum = rs_weight_sum<float, NT>(t);
    float D[NT * NT * 4];
#pragma unroll
    for (int q = 0; q < NT * NT * 4; ++q) D[q] = sD[q * 32 + lane];
    const long long opl = (long long)H * W;
    rs_in2_store<float, NT>(t, sum, D, gin2 + (long long)px.b * 3 * opl + (long long)px.y * W + px.x, opl, accumulate);
}

template <typename T, int NT, int VEC>
__global__ void __launch_bounds__(128)
k_resample2d_nhwc_bwd_in2(const T* __restrict__ in1, const float* __restrict__ in2, const T* __restrict__ gout, float* __restrict__ gin2,
                          int C, int Hi, int Wi, int H, int W, int dil, int lg, int accumulate) {
    constexpr int NQ = NT * NT * 4;
    extern __shared__ __align__(16) unsigned char rs16_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int* so = reinterpret_cast<int*>(rs16_smem + warp * Rs16Smem<NT>::in2);
    float* sD = reinterpret_cast<float*>(so + NQ * 32);
    const RsPixel px = rs_pixel<4>(H, W);
    if (px.y >= H) return;
    if (px.active) {
        RsTaps<float, NT> t;
        rs_setup<float, NT>(t, in2, px.b, px.y, px.x, H, W, Hi, Wi, dil, false);
#pragma unroll
        for (int q = 0; q < NQ; ++q) so[q * 32 + lane] = t.off[q];
    }
    __syncwarp();
    const int G = 1 << lg, sub = lane & (G - 1), x0 = px.x - lane;
    const T* src = in1 + (long long)px.b * Hi * Wi * C;
    const T* row = gout + ((long long)px.b * H + px.y) * W * C;
    for (int p0 = 0; p0 < 32; p0 += 32 >> lg) {                       // every lane runs every step: the group reduction shuffles
        const int p = p0 + (lane >> lg);
        const bool live = x0 + p < W;
        float D[NQ];
#pragma unroll
        for (int q = 0; q < NQ; ++q) D[q] = 0.f;
        if (live) {
            const T* go = row + (long long)(x0 + p) * C;
            for (int c = sub * VEC; c < C; c += G * VEC) {
                float g[VEC];
                ld_vec<T, VEC>(go + c, g);
#pragma unroll
                for (int q = 0; q < NQ; ++q) {
                    float s[VEC];
                    ld_vec<T, VEC>(src + (long long)tap_off(so, q, p) * C + c, s);
#pragma unroll
                    for (int j = 0; j < VEC; ++j) D[q] += g[j] * s[j];
                }
            }
        }
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            const float d = group_sum(D[q], G);
            if (live && sub == 0) sD[q * 32 + p] = d;
        }
    }
    __syncwarp();
    rs16_in2_store<NT>(in2, px, H, W, Hi, Wi, dil, sD, gin2, accumulate, lane);
}

// resample2d -> cosine similarity with the target (NHWC, same dtype), fused: the DESIGN 3.6 op on 16-bit channels-last maps.
// cos [B,H,W] and stats [B,3,H,W] = (v.t, |v|, |t|) are fp32.
template <typename T, int NT, int VEC>
__global__ void __launch_bounds__(128)
k_resample2d_nhwc_cos_fwd(const T* __restrict__ in1, const float* __restrict__ in2, const T* __restrict__ target,
                          float* __restrict__ cos_out, float* __restrict__ stats, int C, int Hi, int Wi, int H, int W, int dil, int lg,
                          float eps) {
    constexpr int NQ = NT * NT * 4;
    extern __shared__ __align__(16) unsigned char rs16_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* sw = reinterpret_cast<float*>(rs16_smem + warp * Rs16Smem<NT>::fwd);
    int* so = reinterpret_cast<int*>(sw + NQ * 32);
    float* ssum = sw + 2 * NQ * 32;
    const RsPixel px = rs_pixel<4>(H, W);
    if (px.y >= H) return;
    rs16_stage<NT>(in2, px, H, W, Hi, Wi, dil, sw, so, ssum, lane);
    const int G = 1 << lg, sub = lane & (G - 1), x0 = px.x - lane;
    const long long opl = (long long)H * W;
    const T* src = in1 + (long long)px.b * Hi * Wi * C;
    const T* row = target + ((long long)px.b * H + px.y) * W * C;
    for (int p0 = 0; p0 < 32; p0 += 32 >> lg) {
        const int p = p0 + (lane >> lg);
        const bool live = x0 + p < W;
        float dot = 0.f, vv = 0.f, tt = 0.f;
        if (live) {
            const float sum = ssum[p];
            const T* tg = row + (long long)(x0 + p) * C;
            for (int c = sub * VEC; c < C; c += G * VEC) {
                float v[VEC], tc[VEC];
                rs16_warp<T, NT, VEC>(src, sw, so, p, C, c, sum, v);
                ld_vec<T, VEC>(tg + c, tc);
#pragma unroll
                for (int j = 0; j < VEC; ++j) { dot += v[j] * tc[j]; vv += v[j] * v[j]; tt += tc[j] * tc[j]; }
            }
        }
        dot = group_sum(dot, G); vv = group_sum(vv, G); tt = group_sum(tt, G);
        if (live && sub == 0) {
            const long long pix = (long long)px.y * W + x0 + p;
            const float nv = sqrtf(vv), nt = sqrtf(tt);
            cos_out[(long long)px.b * opl + pix] = dot / (max(nv, eps) * max(nt, eps));
            float* st = stats + (long long)px.b * 3 * opl + pix;
            st[0] = dot; st[opl] = nv; st[2 * opl] = nt;
        }
    }
}

// Backward of the fused op: g_c = dcos/dv_c * grad_cos from the saved sums (k_resample2d_cos_bwd's expressions), the corner dot
// products of grad input2, and optionally grad_val (NHWC 16-bit, for the grad input1 scatter) and grad_target (NHWC 16-bit).
template <typename T, int NT, int VEC>
__global__ void __launch_bounds__(128)
k_resample2d_nhwc_cos_bwd(const T* __restrict__ in1, const float* __restrict__ in2, const T* __restrict__ target,
                          const float* __restrict__ stats, const float* __restrict__ gcos, float* __restrict__ gin2, T* __restrict__ gval,
                          T* __restrict__ gtarget, int C, int Hi, int Wi, int H, int W, int dil, int lg, float eps, int accumulate) {
    constexpr int NQ = NT * NT * 4;
    extern __shared__ __align__(16) unsigned char rs16_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* sw = reinterpret_cast<float*>(rs16_smem + warp * Rs16Smem<NT>::cos_bwd);
    int* so = reinterpret_cast<int*>(sw + NQ * 32);
    float* sD = reinterpret_cast<float*>(so + NQ * 32);
    float* ssum = sD + NQ * 32;
    float* sk = ssum + 32;                                            // k1, k2v, k2t per pixel
    const RsPixel px = rs_pixel<4>(H, W);
    if (px.y >= H) return;
    rs16_stage<NT>(in2, px, H, W, Hi, Wi, dil, sw, so, ssum, lane);
    const long long opl = (long long)H * W;
    if (px.active) {
        const long long pix = (long long)px.y * W + px.x;
        const float* st = stats + (long long)px.b * 3 * opl + pix;
        const float dot = st[0], nv = st[opl], nt = st[2 * opl];
        const float a = max(nv, eps), bb = max(nt, eps), g = gcos[(long long)px.b * opl + pix];
        sk[lane] = g / (a * bb);
        sk[32 + lane] = nv > eps ? g * dot / (a * a * bb * nv) : 0.f;
        sk[64 + lane] = nt > eps ? g * dot / (a * bb * bb * nt) : 0.f;
    }
    __syncwarp();
    const int G = 1 << lg, sub = lane & (G - 1), x0 = px.x - lane;
    const T* src = in1 + (long long)px.b * Hi * Wi * C;
    const long long row = ((long long)px.b * H + px.y) * W * C;
    for (int p0 = 0; p0 < 32; p0 += 32 >> lg) {
        const int p = p0 + (lane >> lg);
        const bool live = x0 + p < W;
        float D[NQ];
#pragma unroll
        for (int q = 0; q < NQ; ++q) D[q] = 0.f;
        if (live) {
            const float sum = ssum[p], k1 = sk[p], k2v = sk[32 + p], k2t = sk[64 + p];
            const long long o = row + (long long)(x0 + p) * C;
            for (int c = sub * VEC; c < C; c += G * VEC) {
                float v[VEC], tc[VEC], gc[VEC];
                rs16_warp<T, NT, VEC>(src, sw, so, p, C, c, sum, v);
                ld_vec<T, VEC>(target + o + c, tc);
#pragma unroll
                for (int j = 0; j < VEC; ++j) gc[j] = k1 * tc[j] - k2v * v[j];
#pragma unroll
                for (int q = 0; q < NQ; ++q) {                        // the taps again: L1 hits after rs16_warp's loads
                    float s[VEC];
                    ld_vec<T, VEC>(src + (long long)tap_off(so, q, p) * C + c, s);
#pragma unroll
                    for (int j = 0; j < VEC; ++j) D[q] += gc[j] * s[j];
                }
                if (gval != nullptr) st_vec<T, VEC>(gval + o + c, gc);
                if (gtarget != nullptr) {
                    float d[VEC];
#pragma unroll
                    for (int j = 0; j < VEC; ++j) d[j] = k1 * v[j] - k2t * tc[j];
                    if (accumulate) {
                        float old[VEC];
                        ld_vec_rw<T, VEC>(gtarget + o + c, old);
#pragma unroll
                        for (int j = 0; j < VEC; ++j) d[j] = old[j] + d[j];
                    }
                    st_vec<T, VEC>(gtarget + o + c, d);
                }
            }
        }
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            const float d = group_sum(D[q], G);
            if (live && sub == 0) sD[q * 32 + p] = d;
        }
    }
    __syncwarp();
    rs16_in2_store<NT>(in2, px, H, W, Hi, Wi, dil, sD, gin2, accumulate, lane);
}

// ------------------------------------------------------------------------------------------------------------------- host side
template <typename T> struct TypeTag { using type = T; };
template <int V> using IntC = std::integral_constant<int, V>;

// f(TypeTag<T>, IntC<NT>, IntC<VEC>) for the storage dtype, ks / 2 and the channel vector width
template <typename F>
static int rs16_dispatch(int dtype, int ks, bool vec, F&& f) {
    auto by_nt = [&](auto tt) -> int {
        switch (ks / 2) {
            case 1: return vec ? f(tt, IntC<1>{}, IntC<8>{}) : f(tt, IntC<1>{}, IntC<1>{});
            case 2: return vec ? f(tt, IntC<2>{}, IntC<8>{}) : f(tt, IntC<2>{}, IntC<1>{});
            case 3: return vec ? f(tt, IntC<3>{}, IntC<8>{}) : f(tt, IntC<3>{}, IntC<1>{});
            case 4: return vec ? f(tt, IntC<4>{}, IntC<8>{}) : f(tt, IntC<4>{}, IntC<1>{});
            default: return GFLA_E_SHAPE;
        }
    };
    if (dtype == GFLA_BF16) return by_nt(TypeTag<__nv_bfloat16>{});
    if (dtype == GFLA_F16) return by_nt(TypeTag<__half>{});
    return GFLA_E_DTYPE;
}

// log2 of the lanes that share one pixel's channels
static inline int rs16_lanes_log2(int C, int vec) {
    const int n = (C + vec - 1) / vec;
    int lg = 0;
    while ((1 << lg) < n && lg < 5) ++lg;
    return lg;
}

// 16-byte channel vectors need C % 8 == 0 and every channels-last pointer on a 16-byte boundary
static inline bool rs16_vec_ok(int C, std::initializer_list<const void*> ps) {
    if (C % 8 != 0) return false;
    for (const void* p : ps)
        if (p != nullptr && !aligned(p, 16)) return false;
    return true;
}

// dynamic shared memory above the default 48 KB limit (NT >= 3) needs a per-kernel opt-in
template <typename K>
static int rs16_smem_optin(K kernel, size_t smem) {
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return static_cast<int>(e);
    }
    return GFLA_OK;
}

#define RS16_TYPES                                   \
    using T = typename decltype(tt)::type;           \
    constexpr int NT = decltype(nt)::value;          \
    constexpr int VEC = decltype(vc)::value;         \
    (void)sizeof(T);

int resample2d_nhwc_fwd(const void* in1, const void* in2, void* out, int B, int C, int Hi, int Wi, int H, int W, int ks, int dil,
                        int dtype, cudaStream_t st_) {
    const bool vec = rs16_vec_ok(C, {in1, out});
    const int lg = rs16_lanes_log2(C, vec ? 8 : 1);
    const dim3 grid((unsigned)rs_tiles<4>(B, H, W));
    return rs16_dispatch(dtype, ks, vec, [&](auto tt, auto nt, auto vc) -> int {
        RS16_TYPES
        const size_t smem = 4 * Rs16Smem<NT>::fwd;
        int e = rs16_smem_optin(k_resample2d_nhwc_fwd<T, NT, VEC>, smem);
        if (e) return e;
        k_resample2d_nhwc_fwd<T, NT, VEC><<<grid, 128, smem, st_>>>((const T*)in1, (const float*)in2, (T*)out, C, Hi, Wi, H, W, dil, lg);
        return launch_status();
    });
}

// the grad input1 scatter (grad_in1 already zero-filled or holding what it accumulates into)
template <typename T, int NT, int VEC>
static int rs16_launch_in1(const void* in2, const void* gout, void* gin1, int gdtype, int B, int C, int Hi, int Wi, int H, int W,
                           int dil, int lg, cudaStream_t st_) {
    const dim3 grid((unsigned)rs_tiles<4>(B, H, W));
    const size_t smem = 4 * Rs16Smem<NT>::in1;
    if (gdtype == GFLA_F32) {
        int e = rs16_smem_optin(k_resample2d_nhwc_bwd_in1<T, float, NT, VEC>, smem);
        if (e) return e;
        k_resample2d_nhwc_bwd_in1<T, float, NT, VEC><<<grid, 128, smem, st_>>>((const float*)in2, (const T*)gout, (float*)gin1, C, Hi, Wi,
                                                                               H, W, dil, lg);
    } else {
        int e = rs16_smem_optin(k_resample2d_nhwc_bwd_in1<T, T, NT, VEC>, smem);
        if (e) return e;
        k_resample2d_nhwc_bwd_in1<T, T, NT, VEC><<<grid, 128, smem, st_>>>((const float*)in2, (const T*)gout, (T*)gin1, C, Hi, Wi, H, W,
                                                                           dil, lg);
    }
    return launch_status();
}

int resample2d_nhwc_bwd(const void* in1, const void* in2, const void* gout, void* gin1, void* gin2, int B, int C, int Hi, int Wi, int H,
                        int W, int ks, int dil, int dtype, int gdtype, int accumulate, cudaStream_t st_) {
    if (!accumulate) {
        const int e = zero_async(gin1, (size_t)B * C * Hi * Wi * elem_size(gdtype), st_);
        if (e != GFLA_OK) return e;
    }
    const bool vec = rs16_vec_ok(C, {in1, gout, gin1});
    const int lg = rs16_lanes_log2(C, vec ? 8 : 1);
    return rs16_dispatch(dtype, ks, vec, [&](auto tt, auto nt, auto vc) -> int {
        RS16_TYPES
        int e = rs16_launch_in1<T, NT, VEC>(in2, gout, gin1, gdtype, B, C, Hi, Wi, H, W, dil, lg, st_);
        if (e) return e;
        const dim3 grid((unsigned)rs_tiles<4>(B, H, W));
        const size_t smem = 4 * Rs16Smem<NT>::in2;
        e = rs16_smem_optin(k_resample2d_nhwc_bwd_in2<T, NT, VEC>, smem);
        if (e) return e;
        k_resample2d_nhwc_bwd_in2<T, NT, VEC><<<grid, 128, smem, st_>>>((const T*)in1, (const float*)in2, (const T*)gout, (float*)gin2, C,
                                                                        Hi, Wi, H, W, dil, lg, accumulate);
        return launch_status();
    });
}

int resample2d_nhwc_cos_fwd(const void* in1, const void* in2, const void* target, void* cos_out, void* stats, int B, int C, int Hi,
                            int Wi, int H, int W, int ks, int dil, double eps, int dtype, cudaStream_t st_) {
    const bool vec = rs16_vec_ok(C, {in1, target});
    const int lg = rs16_lanes_log2(C, vec ? 8 : 1);
    const dim3 grid((unsigned)rs_tiles<4>(B, H, W));
    return rs16_dispatch(dtype, ks, vec, [&](auto tt, auto nt, auto vc) -> int {
        RS16_TYPES
        const size_t smem = 4 * Rs16Smem<NT>::fwd;
        int e = rs16_smem_optin(k_resample2d_nhwc_cos_fwd<T, NT, VEC>, smem);
        if (e) return e;
        k_resample2d_nhwc_cos_fwd<T, NT, VEC><<<grid, 128, smem, st_>>>((const T*)in1, (const float*)in2, (const T*)target, (float*)cos_out,
                                                                        (float*)stats, C, Hi, Wi, H, W, dil, lg, static_cast<float>(eps));
        return launch_status();
    });
}

// grad_in1 != nullptr needs grad_val (a [B,H,W,C] 16-bit scratch tensor of the caller); accumulate = 0 zero-fills grad_in1 first
int resample2d_nhwc_cos_bwd(const void* in1, const void* in2, const void* target, const void* stats, const void* gcos, void* gin1,
                            void* gin2, void* gval, void* gtarget, int B, int C, int Hi, int Wi, int H, int W, int ks, int dil, double eps,
                            int dtype, int gdtype, int accumulate, cudaStream_t st_) {
    if (gin1 != nullptr && !accumulate) {
        const int e = zero_async(gin1, (size_t)B * C * Hi * Wi * elem_size(gdtype), st_);
        if (e != GFLA_OK) return e;
    }
    const bool vec = rs16_vec_ok(C, {in1, target, gval, gtarget, gin1});
    const int lg = rs16_lanes_log2(C, vec ? 8 : 1);
    return rs16_dispatch(dtype, ks, vec, [&](auto tt, auto nt, auto vc) -> int {
        RS16_TYPES
        const dim3 grid((unsigned)rs_tiles<4>(B, H, W));
        const size_t smem = 4 * Rs16Smem<NT>::cos_bwd;
        int e = rs16_smem_optin(k_resample2d_nhwc_cos_bwd<T, NT, VEC>, smem);
        if (e) return e;
        k_resample2d_nhwc_cos_bwd<T, NT, VEC><<<grid, 128, smem, st_>>>(
            (const T*)in1, (const float*)in2, (const T*)target, (const float*)stats, (const float*)gcos, (float*)gin2, (T*)gval, (T*)gtarget,
            C, Hi, Wi, H, W, dil, lg, static_cast<float>(eps), accumulate);
        e = launch_status();
        if (e || gin1 == nullptr) return e;
        return rs16_launch_in1<T, NT, VEC>(in2, gval, gin1, gdtype, B, C, Hi, Wi, H, W, dil, lg, st_);
    });
}

}  // namespace gfla
