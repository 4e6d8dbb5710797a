// resample2d (Gaussian-weighted ks x ks warp, FlowNet2-derived) for sm_100a.
//
// Arithmetic contract: resample2d_package/resample2d_kernel.cu:20-95 (forward),
// :98-202 (grad input1), :204-330 (grad input2 = d/d(dx, dy, sigma)).
// Reference quirks that are reproduced on purpose:
//   * SAFE_DIV(a,b) = b==0 ? a/1e-8 : a/b with a *double* 1e-8 (:14-15): for
//     float tensors the quotient is formed in float, widened, and exp() runs in
//     double before being narrowed -- done here the same way, but ONCE PER
//     PIXEL instead of once per (pixel, channel);
//   * grad_input1 takes its Gaussian weights from alpha = xf - int(xf)
//     (truncation, :137-138) while the tap indices use floor(xf);
//   * all three planes of grad_input2 (including d/dsigma) are produced.
// Layout on the machine (not the reference's):
//   * one thread per output PIXEL (b,y,x); the 4*(ks/2)^2 weights and clamped
//     tap offsets live in registers and are reused for every channel;
//     a CTA owns a 32 x 4 pixel tile: a warp is a 128-byte
//     row segment, and the ks rows a pixel row reads are shared with the rows
//     above / below through L1 (one-row CTAs pulled every source row ks times
//     over the L2 -> L1 fabric: 6.4x the tensor, profiles/r2_resample2d.md);
//     channel slices in grid.y for small images;
//   * grad_input1: warps whose taps are one integer shift of their pixel run merge the scatter through shuffles.
//     (Measured and dropped, profiles/r2_resample2d.md: accumulating the CTA's scatter in a shared-memory box and
//     flushing the box -- fp32 shared-memory atomics are ATOMS.CAST.SPIN loops, 2.6 tries and 7 wavefronts per
//     add on a stretching flow, no faster than the L2's native fp32 RED.)
//   * grad_input2: the reference runs 3*H*W threads that each stride twice
//     through all C channel planes; here one thread per pixel accumulates the
//     4*(ks/2)^2 corner dot products sum_c g[c]*v[c,corner] in ONE pass and
//     derives the three gradients from them.
// Compiled with -fmad=false: the fp32/fp64 forward is bit-identical to the
// (uncontracted) CPU oracle up to the last-ulp behaviour of exp().
#include "resample2d_common.cuh"

namespace gfla {

template <typename A, int NT>
__global__ void __launch_bounds__(128)
k_resample2d_fwd(const A* __restrict__ in1, const A* __restrict__ in2, A* __restrict__ out, int B, int C, int Hi, int Wi,
                 int H, int W, int dil, int c_per_slice) {
    const RsPixel px = rs_pixel<4>(H, W);
    if (!px.active) return;
    const int x = px.x, y = px.y, b = px.b;
    RsTaps<A, NT> t;
    rs_setup<A, NT>(t, in2, b, y, x, H, W, Hi, Wi, dil, false);
    A w[NT * NT * 4];
#pragma unroll
    for (int fy = 0; fy < NT; ++fy)
#pragma unroll
        for (int fx = 0; fx < NT; ++fx) {
            A* q = w + (fy * NT + fx) * 4;
            q[0] = t.yT_P[fy] * t.xL_P[fx]; q[1] = t.yT_P[fy] * t.xR_P[fx];
            q[2] = t.yB_P[fy] * t.xL_P[fx]; q[3] = t.yB_P[fy] * t.xR_P[fx];
        }
    const A sum = rs_weight_sum<A, NT>(t);
    const long long ipl = (long long)Hi * Wi, opl = (long long)H * W;
    const int c0 = blockIdx.y * c_per_slice, c1 = min(C, c0 + c_per_slice);
    const A* s = in1 + ((long long)b * C + c0) * ipl;
    A* o = out + ((long long)b * C + c0) * opl + (long long)y * W + x;
#pragma unroll 4
    for (int c = c0; c < c1; ++c, s += ipl, o += opl) {   // unrolled: 4 channels x taps of independent loads in flight
        A val = static_cast<A>(0);
#pragma unroll
        for (int q = 0; q < NT * NT * 4; ++q) val += w[q] * s[t.off[q]];
        *o = static_cast<A>(safe_div<A>(val, sum));
    }
}

// grad_input1: a scatter of 4*(ks/2)^2 weighted copies of grad_out per (pixel, channel).  A warp is a 32-pixel run of one
// image row (rs_pixel).  When its taps are the same integer shift (the usual case for a smooth flow) and no
// tap is clamped, lane L's contribution to column (x_L + shift + co) is exactly what lane L+co accumulates for its
// own centre column: the (2*ks/2)^2 scalar atomics per element collapse to one red.global per tap ROW per lane
// (plus the few taps that leave the warp's 32 columns) after a register-level exchange with __shfl_sync.
template <typename A, int NT>
__global__ void __launch_bounds__(128)
k_resample2d_bwd_in1(const A* __restrict__ in2, const A* __restrict__ gout, A* __restrict__ gin1, int B, int C, int Hi,
                     int Wi, int H, int W, int dil, int c_per_slice) {
    const RsPixel px = rs_pixel<4>(H, W);
    const bool active = px.active;
    const int x = min(px.x, W - 1), y = min(px.y, H - 1), b = px.b;   // inactive lanes stay alive for the warp shuffles
    RsTaps<A, NT> t;
    rs_setup<A, NT>(t, in2, b, y, x, H, W, Hi, Wi, dil, true);  // truncating fraction for the weights
    const A sum = rs_weight_sum<A, NT>(t);
    double wn[NT * NT * 4];  // SAFE_DIV(w, sum), kept in double like the reference expression (:195-198)
#pragma unroll
    for (int fy = 0; fy < NT; ++fy)
#pragma unroll
        for (int fx = 0; fx < NT; ++fx) {
            double* q = wn + (fy * NT + fx) * 4;
            q[0] = safe_div<A>(t.yT_P[fy] * t.xL_P[fx], sum); q[1] = safe_div<A>(t.yT_P[fy] * t.xR_P[fx], sum);
            q[2] = safe_div<A>(t.yB_P[fy] * t.xL_P[fx], sum); q[3] = safe_div<A>(t.yB_P[fy] * t.xR_P[fx], sum);
        }
    const long long ipl = (long long)Hi * Wi, opl = (long long)H * W;
    const int c0 = blockIdx.y * c_per_slice, c1 = min(C, c0 + c_per_slice);
    A* gi = gin1 + ((long long)b * C + c0) * ipl;
    const A* go = gout + ((long long)b * C + c0) * opl + (long long)y * W + x;

    bool fast = false;
    if (NT <= 2) {
        const unsigned full = 0xffffffffu;
        bool ok = active && dil == 1 && t.flx - (NT - 1) >= 0 && t.flx + NT <= Wi - 1 &&
                  t.fly - (NT - 1) >= 0 && t.fly + NT <= Hi - 1;
        const int shift = t.flx - x;
        // warp-collective: every lane executes the shuffles (no short-circuit in front of them)
        const int shift0 = __shfl_sync(full, shift, 0);
        const int fly0 = __shfl_sync(full, t.fly, 0);
        ok = ok && (shift == shift0) && (t.fly == fly0);
        fast = __all_sync(full, ok);
    }
    if (fast) {
        constexpr int N2 = 2 * NT;   // taps per axis: offsets -(NT-1) .. NT around (fly, flx)
        const unsigned full = 0xffffffffu;
        const int lane = threadIdx.x & 31;
        double wg[N2 * N2];          // weight of (row offset ri-(NT-1), column offset ci-(NT-1))
#pragma unroll
        for (int fy = 0; fy < NT; ++fy)
#pragma unroll
            for (int fx = 0; fx < NT; ++fx) {
                const double* q = wn + (fy * NT + fx) * 4;
                wg[(NT - 1 - fy) * N2 + (NT - 1 - fx)] = q[0];   // yT, xL
                wg[(NT - 1 - fy) * N2 + (NT + fx)] = q[1];       // yT, xR
                wg[(NT + fy) * N2 + (NT - 1 - fx)] = q[2];       // yB, xL
                wg[(NT + fy) * N2 + (NT + fx)] = q[3];           // yB, xR
            }
        const int centre = (t.fly - (NT - 1)) * Wi + t.flx;      // first tap row, this lane's centre column
        for (int c = c0; c < c1; ++c, gi += ipl, go += opl) {
            const double g = static_cast<double>(*go);
#pragma unroll
            for (int ri = 0; ri < N2; ++ri) {
                A acc = static_cast<A>(0);
#pragma unroll
                for (int ci = 0; ci < N2; ++ci) {
                    const int co = ci - (NT - 1);
                    const A v = static_cast<A>(wg[ri * N2 + ci] * g);
                    const A recv = __shfl_sync(full, v, (lane - co) & 31);   // what lane - co sends to column offset co = me
                    if (lane - co >= 0 && lane - co < 32) acc += recv;
                    if (lane + co < 0 || lane + co > 31) atomicAdd(gi + centre + ri * Wi + co, v);   // leaves the warp's span
                }
                atomicAdd(gi + centre + ri * Wi, acc);
            }
        }
        return;
    }
    if (!active) return;
#pragma unroll 4
    for (int c = c0; c < c1; ++c, gi += ipl, go += opl) {
        const double g = static_cast<double>(*go);
#pragma unroll
        for (int q = 0; q < NT * NT * 4; ++q) atomicAdd(gi + t.off[q], static_cast<A>(wn[q] * g));
    }
}

template <typename A, int NT>
__global__ void __launch_bounds__(128)
k_resample2d_bwd_in2(const A* __restrict__ in1, const A* __restrict__ in2, const A* __restrict__ gout,
                     A* __restrict__ gin2, int B, int C, int Hi, int Wi, int H, int W, int dil, int accumulate) {
    const RsPixel px = rs_pixel<4>(H, W);
    if (!px.active) return;
    const int x = px.x, y = px.y, b = px.b;
    RsTaps<A, NT> t;
    rs_setup<A, NT>(t, in2, b, y, x, H, W, Hi, Wi, dil, false);
    const A sum = rs_weight_sum<A, NT>(t);
    // corner dot products over the channels: D[q] = sum_c g[c] * in1[c, tap q]
    A D[NT * NT * 4];
#pragma unroll
    for (int q = 0; q < NT * NT * 4; ++q) D[q] = static_cast<A>(0);
    const long long ipl = (long long)Hi * Wi, opl = (long long)H * W;
    const A* s = in1 + (long long)b * C * ipl;
    const A* go = gout + (long long)b * C * opl + (long long)y * W + x;
#pragma unroll 4
    for (int c = 0; c < C; ++c, s += ipl, go += opl) {
        const A g = *go;
#pragma unroll
        for (int q = 0; q < NT * NT * 4; ++q) D[q] += g * s[t.off[q]];
    }
    rs_in2_store<A, NT>(t, sum, D, gin2 + (long long)b * 3 * opl + (long long)y * W + x, opl, accumulate);
}

// ---------------------------------------------------------------------------------------------------------------------
// resample2d -> cosine similarity with a target feature map, fused (SURVEY row f4).
// PerceptualCorrectness.calculate_loss (external_function.py:275-279) warps the source VGG features with Resample2d, writes
// them out, and reads them back once for F.cosine_similarity(input_sample, target_all) over the channel axis.  Here a pixel's
// thread warps one channel at a time in registers and folds it straight into the three sums the cosine needs; the warped
// tensor never exists.  cos = sum_c (v_c / max(|v|, eps)) * (t_c / max(|t|, eps))  (ATen's cosine_similarity: each norm clamped).
// stats[b, 0..2, y, x] = (v.t, |v|, |t|) are kept for the backward.
// TS > 1: the 4 warps of a CTA are TS channel slices of ONE 32-pixel row segment (feature maps of a loss are small: a thread per
// pixel alone leaves the SMs with a handful of warps each, walking C channels one after the other); the partial sums meet in shared memory.
template <typename A, int NT, int TS>
__global__ void __launch_bounds__(128)
k_resample2d_cos_fwd(const A* __restrict__ in1, const A* __restrict__ in2, const A* __restrict__ target, A* __restrict__ cos_out,
                     A* __restrict__ stats, int B, int C, int Hi, int Wi, int H, int W, int dil, A eps) {
    constexpr int TH = 4 / TS;                                   // pixel rows per CTA
    __shared__ A part[TS > 1 ? 3 * TS * 32 * TH : 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slice = TS > 1 ? warp % TS : 0, row = TS > 1 ? warp / TS : warp;
    const RsPixel px = rs_pixel<TH>(H, W, row);
    if (TS == 1 && !px.active) return;
    const int x = min(px.x, W - 1), y = min(px.y, H - 1), b = px.b;
    RsTaps<A, NT> t;
    rs_setup<A, NT>(t, in2, b, y, x, H, W, Hi, Wi, dil, false);
    A w[NT * NT * 4];
#pragma unroll
    for (int fy = 0; fy < NT; ++fy)
#pragma unroll
        for (int fx = 0; fx < NT; ++fx) {
            A* q = w + (fy * NT + fx) * 4;
            q[0] = t.yT_P[fy] * t.xL_P[fx]; q[1] = t.yT_P[fy] * t.xR_P[fx];
            q[2] = t.yB_P[fy] * t.xL_P[fx]; q[3] = t.yB_P[fy] * t.xR_P[fx];
        }
    const A sum = rs_weight_sum<A, NT>(t);
    const long long ipl = (long long)Hi * Wi, opl = (long long)H * W, pix = (long long)y * W + x;
    const int cs = (C + TS - 1) / TS, c0 = slice * cs, c1 = min(C, c0 + cs);
    const A* s = in1 + ((long long)b * C + c0) * ipl;
    const A* tg = target + ((long long)b * C + c0) * opl + pix;
    A dot = static_cast<A>(0), vv = static_cast<A>(0), tt = static_cast<A>(0);
#pragma unroll 4
    for (int c = c0; c < c1; ++c, s += ipl, tg += opl) {
        A val = static_cast<A>(0);
#pragma unroll
        for (int q = 0; q < NT * NT * 4; ++q) val += w[q] * s[t.off[q]];
        const A v = static_cast<A>(safe_div<A>(val, sum));        // exactly k_resample2d_fwd's output element
        const A tc = *tg;
        dot += v * tc; vv += v * v; tt += tc * tc;
    }
    if (TS > 1) {
        A* mine = part + ((row * TS + slice) * 3) * 32 + lane;
        mine[0] = dot; mine[32] = vv; mine[64] = tt;
        __syncthreads();
        if (slice != 0 || !px.active) return;
        dot = vv = tt = static_cast<A>(0);
#pragma unroll
        for (int sl = 0; sl < TS; ++sl) {                         // fixed order: deterministic
            const A* o = part + ((row * TS + sl) * 3) * 32 + lane;
            dot += o[0]; vv += o[32]; tt += o[64];
        }
    }
    const A nv = sqrt(vv), nt = sqrt(tt);
    cos_out[(long long)b * opl + pix] = dot / (max(nv, eps) * max(nt, eps));
    A* st = stats + (long long)b * 3 * opl + pix;
    st[0] = dot; st[opl] = nv; st[2 * opl] = nt;
}

// Backward of the fused op for one pixel, one pass over the channels: the warped value v_c is rebuilt from the taps that are in
// registers anyway, g_c = dcos/dv_c * grad_cos follows from the saved sums, and the corner dot products of grad_input2 accumulate
// g_c * tap -- so the flow gradient (the one PerceptualCorrectness trains through) costs one read of the source and the
// target and writes 3 floats per pixel.  grad_val (optional) receives g_c for the grad_input1 scatter (k_resample2d_bwd_in1 runs on
// it afterwards; VGG features of data carry no gradient in the reference's use), grad_target (optional) dcos/dt_c * grad_cos.
template <typename A, int NT, int TS>
__global__ void __launch_bounds__(128)
k_resample2d_cos_bwd(const A* __restrict__ in1, const A* __restrict__ in2, const A* __restrict__ target, const A* __restrict__ stats,
                     const A* __restrict__ gcos, A* __restrict__ gin2, A* __restrict__ gval, A* __restrict__ gtarget, int B, int C,
                     int Hi, int Wi, int H, int W, int dil, A eps, int accumulate) {
    constexpr int TH = 4 / TS, NQ = NT * NT * 4;
    __shared__ A part[TS > 1 ? NQ * TS * 32 * TH : 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slice = TS > 1 ? warp % TS : 0, row = TS > 1 ? warp / TS : warp;
    const RsPixel px = rs_pixel<TH>(H, W, row);
    if (TS == 1 && !px.active) return;
    const int x = min(px.x, W - 1), y = min(px.y, H - 1), b = px.b;
    RsTaps<A, NT> t;
    rs_setup<A, NT>(t, in2, b, y, x, H, W, Hi, Wi, dil, false);
    A w[NQ], D[NQ];
#pragma unroll
    for (int fy = 0; fy < NT; ++fy)
#pragma unroll
        for (int fx = 0; fx < NT; ++fx) {
            A* q = w + (fy * NT + fx) * 4;
            q[0] = t.yT_P[fy] * t.xL_P[fx]; q[1] = t.yT_P[fy] * t.xR_P[fx];
            q[2] = t.yB_P[fy] * t.xL_P[fx]; q[3] = t.yB_P[fy] * t.xR_P[fx];
        }
#pragma unroll
    for (int q = 0; q < NQ; ++q) D[q] = static_cast<A>(0);
    const A sum = rs_weight_sum<A, NT>(t);
    const long long ipl = (long long)Hi * Wi, opl = (long long)H * W, pix = (long long)y * W + x;
    const A* st = stats + (long long)b * 3 * opl + pix;
    const A dot = st[0], nv = st[opl], nt = st[2 * opl];
    const A a = max(nv, eps), bb = max(nt, eps), g = gcos[(long long)b * opl + pix];
    // cos = dot / (a * bb);  da/dv_c = v_c / |v| above the clamp, 0 below it
    const A k1 = g / (a * bb);
    const A k2v = nv > eps ? g * dot / (a * a * bb * nv) : static_cast<A>(0);
    const A k2t = nt > eps ? g * dot / (a * bb * bb * nt) : static_cast<A>(0);
    const int cs = (C + TS - 1) / TS, c0 = slice * cs, c1 = min(C, c0 + cs);
    const A* s = in1 + ((long long)b * C + c0) * ipl;
    const long long o0 = ((long long)b * C + c0) * opl + pix;
    const A* tg = target + o0;
    const bool live = px.active;                                  // inactive lanes only keep the CTA barrier company
    A* gv = gval != nullptr && live ? gval + o0 : nullptr;
    A* gt = gtarget != nullptr && live ? gtarget + o0 : nullptr;
#pragma unroll 2
    for (int c = c0; c < c1; ++c, s += ipl, tg += opl) {
        A tap[NQ];
        A val = static_cast<A>(0);
#pragma unroll
        for (int q = 0; q < NQ; ++q) { tap[q] = s[t.off[q]]; val += w[q] * tap[q]; }
        const A v = static_cast<A>(safe_div<A>(val, sum));
        const A tc = *tg;
        const A gc = k1 * tc - k2v * v;
#pragma unroll
        for (int q = 0; q < NQ; ++q) D[q] += gc * tap[q];
        if (gv != nullptr) gv[(long long)(c - c0) * opl] = gc;
        if (gt != nullptr) {
            const A d = k1 * v - k2t * tc;
            gt[(long long)(c - c0) * opl] = accumulate ? gt[(long long)(c - c0) * opl] + d : d;
        }
    }
    if (TS > 1) {
        A* mine = part + ((row * TS + slice) * NQ) * 32 + lane;
#pragma unroll
        for (int q = 0; q < NQ; ++q) mine[q * 32] = D[q];
        __syncthreads();
        if (slice != 0 || !live) return;
#pragma unroll
        for (int q = 0; q < NQ; ++q) D[q] = static_cast<A>(0);
#pragma unroll
        for (int sl = 0; sl < TS; ++sl) {
            const A* o = part + ((row * TS + sl) * NQ) * 32 + lane;
#pragma unroll
            for (int q = 0; q < NQ; ++q) D[q] += o[q * 32];
        }
    }
    rs_in2_store<A, NT>(t, sum, D, gin2 + (long long)b * 3 * opl + pix, opl, accumulate);
}

template <typename A, int NT>
static int rs_launch_fwd(const void* in1, const void* in2, void* out, int B, int C, int Hi, int Wi, int H, int W, int dil,
                         cudaStream_t st_) {
    const long long total = (long long)B * H * W;
    const int threads = 128, slices0 = channel_splits(total, C, threads), cps = (C + slices0 - 1) / slices0;
    dim3 grid((unsigned)rs_tiles<4>(B, H, W), (unsigned)((C + cps - 1) / cps));
    k_resample2d_fwd<A, NT><<<grid, threads, 0, st_>>>((const A*)in1, (const A*)in2, (A*)out, B, C, Hi, Wi, H, W, dil, cps);
    return launch_status();
}

template <typename A, int NT>
static int rs_launch_bwd(const void* in1, const void* in2, const void* gout, void* gin1, void* gin2, int B, int C, int Hi,
                         int Wi, int H, int W, int dil, int accumulate, cudaStream_t st_) {
    const long long total = (long long)B * H * W;
    const int threads = 128, slices0 = channel_splits(total, C, threads), cps = (C + slices0 - 1) / slices0;
    dim3 grid((unsigned)rs_tiles<4>(B, H, W), (unsigned)((C + cps - 1) / cps));
    k_resample2d_bwd_in1<A, NT><<<grid, threads, 0, st_>>>((const A*)in2, (const A*)gout, (A*)gin1, B, C, Hi, Wi, H, W, dil, cps);
    int e = launch_status();
    if (e) return e;
    k_resample2d_bwd_in2<A, NT><<<(unsigned)rs_tiles<4>(B, H, W), 128, 0, st_>>>(
        (const A*)in1, (const A*)in2, (const A*)gout, (A*)gin2, B, C, Hi, Wi, H, W, dil, accumulate);
    return launch_status();
}

// channel slices per pixel: 4 when the map is too small to fill the machine with one thread per pixel (and C is worth splitting)
static inline int rs_cos_slices(int B, int C, int H, int W) {
    // measured (bench.py f4_resample_cosine, fwd+bwd): 65 k pixels x 256 channels 0.92 -> 0.76 ms with slices, 262 k pixels x 128 channels 1.17 -> 1.56 ms
    return (C >= 64 && (long long)B * H * W < (long long)sm_count() * 1024) ? 4 : 1;
}

template <typename A, int NT>
static int rs_launch_cos_fwd(const void* in1, const void* in2, const void* target, void* cos_out, void* stats, int B, int C, int Hi,
                             int Wi, int H, int W, int dil, double eps, cudaStream_t st_) {
    bool sliced = false;
    if constexpr (NT <= 2) sliced = rs_cos_slices(B, C, H, W) == 4;      // (larger windows: the partial sums would not fit static shared memory)
    if constexpr (NT <= 2) if (sliced)
        k_resample2d_cos_fwd<A, NT, 4><<<(unsigned)rs_tiles<1>(B, H, W), 128, 0, st_>>>((const A*)in1, (const A*)in2, (const A*)target, (A*)cos_out,
                                                                                        (A*)stats, B, C, Hi, Wi, H, W, dil, static_cast<A>(eps));
    if (!sliced)
        k_resample2d_cos_fwd<A, NT, 1><<<(unsigned)rs_tiles<4>(B, H, W), 128, 0, st_>>>((const A*)in1, (const A*)in2, (const A*)target, (A*)cos_out,
                                                                                        (A*)stats, B, C, Hi, Wi, H, W, dil, static_cast<A>(eps));
    return launch_status();
}

template <typename A, int NT>
static int rs_launch_cos_bwd(const void* in1, const void* in2, const void* target, const void* stats, const void* gcos, void* gin1,
                             void* gin2, void* gval, void* gtarget, int B, int C, int Hi, int Wi, int H, int W, int dil, double eps,
                             int accumulate, cudaStream_t st_) {
    bool sliced = false;
    if constexpr (NT <= 2) sliced = rs_cos_slices(B, C, H, W) == 4;
    if constexpr (NT <= 2) if (sliced)
        k_resample2d_cos_bwd<A, NT, 4><<<(unsigned)rs_tiles<1>(B, H, W), 128, 0, st_>>>(
            (const A*)in1, (const A*)in2, (const A*)target, (const A*)stats, (const A*)gcos, (A*)gin2, (A*)gval, (A*)gtarget, B, C, Hi, Wi,
            H, W, dil, static_cast<A>(eps), accumulate);
    if (!sliced)
        k_resample2d_cos_bwd<A, NT, 1><<<(unsigned)rs_tiles<4>(B, H, W), 128, 0, st_>>>(
            (const A*)in1, (const A*)in2, (const A*)target, (const A*)stats, (const A*)gcos, (A*)gin2, (A*)gval, (A*)gtarget, B, C, Hi, Wi,
            H, W, dil, static_cast<A>(eps), accumulate);
    int e = launch_status();
    if (e || gin1 == nullptr) return e;
    const long long total = (long long)B * H * W;
    const int threads = 128, slices0 = channel_splits(total, C, threads), cps = (C + slices0 - 1) / slices0;
    dim3 grid((unsigned)rs_tiles<4>(B, H, W), (unsigned)((C + cps - 1) / cps));
    k_resample2d_bwd_in1<A, NT><<<grid, threads, 0, st_>>>((const A*)in2, (const A*)gval, (A*)gin1, B, C, Hi, Wi, H, W, dil, cps);
    return launch_status();
}

#define GFLA_RS_DISPATCH(A_, fn, ...)                          \
    switch (ks / 2) {                                          \
        case 1: return fn<A_, 1>(__VA_ARGS__);                 \
        case 2: return fn<A_, 2>(__VA_ARGS__);                 \
        case 3: return fn<A_, 3>(__VA_ARGS__);                 \
        case 4: return fn<A_, 4>(__VA_ARGS__);                 \
        default: return GFLA_E_SHAPE;                          \
    }

int resample2d_fwd(const void* in1, const void* in2, void* out, int B, int C, int Hi, int Wi, int H, int W, int ks,
                   int dil, int dtype, cudaStream_t st_) {
    if (dtype == GFLA_F32) { GFLA_RS_DISPATCH(float, rs_launch_fwd, in1, in2, out, B, C, Hi, Wi, H, W, dil, st_) }
    if (dtype == GFLA_F64) { GFLA_RS_DISPATCH(double, rs_launch_fwd, in1, in2, out, B, C, Hi, Wi, H, W, dil, st_) }
    return GFLA_E_DTYPE;
}

int resample2d_bwd(const void* in1, const void* in2, const void* gout, void* gin1, void* gin2, int B, int C, int Hi,
                   int Wi, int H, int W, int ks, int dil, int dtype, int accumulate, cudaStream_t st_) {
    if (!accumulate) {
        const int e = zero_async(gin1, (size_t)B * C * Hi * Wi * elem_size(dtype), st_);
        if (e != GFLA_OK) return e;
    }
    if (dtype == GFLA_F32) { GFLA_RS_DISPATCH(float, rs_launch_bwd, in1, in2, gout, gin1, gin2, B, C, Hi, Wi, H, W, dil, accumulate, st_) }
    if (dtype == GFLA_F64) { GFLA_RS_DISPATCH(double, rs_launch_bwd, in1, in2, gout, gin1, gin2, B, C, Hi, Wi, H, W, dil, accumulate, st_) }
    return GFLA_E_DTYPE;
}

int resample2d_cos_fwd(const void* in1, const void* in2, const void* target, void* cos_out, void* stats, int B, int C, int Hi, int Wi,
                       int H, int W, int ks, int dil, double eps, int dtype, cudaStream_t st_) {
    if (dtype == GFLA_F32) { GFLA_RS_DISPATCH(float, rs_launch_cos_fwd, in1, in2, target, cos_out, stats, B, C, Hi, Wi, H, W, dil, eps, st_) }
    if (dtype == GFLA_F64) { GFLA_RS_DISPATCH(double, rs_launch_cos_fwd, in1, in2, target, cos_out, stats, B, C, Hi, Wi, H, W, dil, eps, st_) }
    return GFLA_E_DTYPE;
}

// grad_in1 != nullptr needs grad_val (a [B,C,H,W] scratch tensor of the caller); accumulate = 0 zero-fills grad_in1 first
int resample2d_cos_bwd(const void* in1, const void* in2, const void* target, const void* stats, const void* gcos, void* gin1, void* gin2,
                       void* gval, void* gtarget, int B, int C, int Hi, int Wi, int H, int W, int ks, int dil, double eps, int dtype,
                       int accumulate, cudaStream_t st_) {
    if (gin1 != nullptr && !accumulate) {
        const int e = zero_async(gin1, (size_t)B * C * Hi * Wi * elem_size(dtype), st_);
        if (e != GFLA_OK) return e;
    }
    if (dtype == GFLA_F32) { GFLA_RS_DISPATCH(float, rs_launch_cos_bwd, in1, in2, target, stats, gcos, gin1, gin2, gval, gtarget, B, C, Hi, Wi, H, W, dil, eps, accumulate, st_) }
    if (dtype == GFLA_F64) { GFLA_RS_DISPATCH(double, rs_launch_cos_bwd, in1, in2, target, stats, gcos, gin1, gin2, gval, gtarget, B, C, Hi, Wi, H, W, dil, eps, accumulate, st_) }
    return GFLA_E_DTYPE;
}

}  // namespace gfla
