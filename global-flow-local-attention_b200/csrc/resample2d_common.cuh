// Per-pixel arithmetic of the resample2d family, shared by the planar fp32/fp64 kernels (resample2d.cu) and the
// channels-last 16-bit kernels (resample2d_nhwc.cu): the taps, the Gaussian weights and the grad_input2 combine.
// Both translation units are compiled with -fmad=false, so a pixel's taps and weights are the same bits in either.
#pragma once
#include "common.cuh"

namespace gfla {

template <typename A>
__device__ __forceinline__ double safe_div(A a, A b) {  // the reference macro, same typing
    return (b == static_cast<A>(0)) ? (static_cast<double>(a) / 1e-8) : static_cast<double>(a / b);
}

// per-pixel quantities shared by the kernels
template <typename A, int NT>
struct RsTaps {
    int off[NT * NT * 4];   // clamped tap offsets y*Wi+x, order per (fy,fx): TL, TR, BL, BR
    A xL_[NT], xR_[NT], yT_[NT], yB_[NT];          // distances
    A xL_P[NT], xR_P[NT], yT_P[NT], yB_P[NT];      // Gaussian factors (depend on fx resp. fy only)
    A sigma;
    int flx, fly;           // floor(x + dx), floor(y + dy)
};

// CTA = 32 x TH pixel tile of one sample; blockIdx.x enumerates (sample, tile row, tile column)
struct RsPixel { int x, y, b; bool active; };
template <int TH>
__device__ __forceinline__ RsPixel rs_pixel(int H, int W, int row = -1) {
    const int tiles_x = (W + 31) >> 5, tiles_y = (H + TH - 1) / TH;
    unsigned t = blockIdx.x;
    const int tx = (int)(t % (unsigned)tiles_x); t /= (unsigned)tiles_x;
    const int ty = (int)(t % (unsigned)tiles_y);
    RsPixel p;
    p.b = (int)(t / (unsigned)tiles_y);
    p.x = tx * 32 + (int)(threadIdx.x & 31);
    p.y = ty * TH + (row >= 0 ? row : (int)(threadIdx.x >> 5));
    p.active = p.x < W && p.y < H;
    return p;
}
template <int TH>
static inline long long rs_tiles(int B, int H, int W) { return (long long)B * ((H + TH - 1) / TH) * ((W + 31) >> 5); }

template <typename A, int NT>
__device__ __forceinline__ void rs_setup(RsTaps<A, NT>& t, const A* __restrict__ in2, int b, int y, int x, int H, int W,
                                         int Hi, int Wi, int dil, bool trunc_frac) {
    const long long hw = (long long)H * W;
    const A* p = in2 + (long long)b * 3 * hw + (long long)y * W + x;
    const A dx = p[0], dy = p[hw];
    t.sigma = p[2 * hw];
    const A xf = static_cast<A>(x) + dx, yf = static_cast<A>(y) + dy;
    const A alpha = trunc_frac ? xf - static_cast<A>(static_cast<int>(xf)) : xf - flr(xf);
    const A beta = trunc_frac ? yf - static_cast<A>(static_cast<int>(yf)) : yf - flr(yf);
    t.flx = static_cast<int>(flr(xf));
    t.fly = static_cast<int>(flr(yf));
    const A two_s2 = 2 * t.sigma * t.sigma;
#pragma unroll
    for (int f = 0; f < NT; ++f) {
        t.xL_[f] = static_cast<A>(f * dil) + alpha;
        t.xR_[f] = static_cast<A>((1. + f) * dil) - alpha;
        t.yT_[f] = static_cast<A>(f * dil) + beta;
        t.yB_[f] = static_cast<A>((1. + f) * dil) - beta;
        t.xL_P[f] = static_cast<A>(exp(safe_div<A>(-t.xL_[f] * t.xL_[f], two_s2)));
        t.xR_P[f] = static_cast<A>(exp(safe_div<A>(-t.xR_[f] * t.xR_[f], two_s2)));
        t.yT_P[f] = static_cast<A>(exp(safe_div<A>(-t.yT_[f] * t.yT_[f], two_s2)));
        t.yB_P[f] = static_cast<A>(exp(safe_div<A>(-t.yB_[f] * t.yB_[f], two_s2)));
    }
#pragma unroll
    for (int fy = 0; fy < NT; ++fy) {
        const int yT = clampi(static_cast<int>(flr(yf) - fy * dil), Hi - 1);
        const int yB = clampi(static_cast<int>(flr(yf) + (fy + 1) * dil), Hi - 1);
#pragma unroll
        for (int fx = 0; fx < NT; ++fx) {
            const int xL = clampi(static_cast<int>(flr(xf) - fx * dil), Wi - 1);
            const int xR = clampi(static_cast<int>(flr(xf) + (fx + 1) * dil), Wi - 1);
            int* o = t.off + (fy * NT + fx) * 4;
            o[0] = yT * Wi + xL; o[1] = yT * Wi + xR; o[2] = yB * Wi + xL; o[3] = yB * Wi + xR;
        }
    }
}

// sum of the 4*NT*NT weights in the reference's order (:80-92)
template <typename A, int NT>
__device__ __forceinline__ A rs_weight_sum(const RsTaps<A, NT>& t) {
    A sum = static_cast<A>(0);
#pragma unroll
    for (int fy = 0; fy < NT; ++fy)
#pragma unroll
        for (int fx = 0; fx < NT; ++fx)
            sum += (t.yT_P[fy] * t.xL_P[fx] + t.yT_P[fy] * t.xR_P[fx] + t.yB_P[fy] * t.xL_P[fx] + t.yB_P[fy] * t.xR_P[fx]);
    return sum;
}

// d/d(dx, dy, sigma) of one pixel from its corner dot products D[q] = sum_c g[c] * in1[c, tap q]
template <typename A, int NT>
__device__ __forceinline__ void rs_in2_store(const RsTaps<A, NT>& t, A sum, const A* D, A* gp, long long opl, int accumulate) {
    // combine (per pixel, in double): reference :271-296 (grad1, sumgrad), :304-326 (grad2), :328
    const double sg = static_cast<double>(t.sigma);
    const bool s0 = (t.sigma == static_cast<A>(0));
    const double den_xy = s0 ? 1e-8 : -(sg * sg);          // SAFE_DIV(., -sigma*sigma)
    const double den_s = s0 ? 1e-8 : sg * sg * sg;         // SAFE_DIV(., sigma^3)
    double g1[3] = {0, 0, 0}, sgrad[3] = {0, 0, 0}, wd = 0;
#pragma unroll
    for (int fy = 0; fy < NT; ++fy)
#pragma unroll
        for (int fx = 0; fx < NT; ++fx) {
            const A* d = D + (fy * NT + fx) * 4;
            const double xL = t.xL_[fx], xR = t.xR_[fx], yT = t.yT_[fy], yB = t.yB_[fy];
            const double wTL = (double)t.yT_P[fy] * t.xL_P[fx], wTR = (double)t.yT_P[fy] * t.xR_P[fx];
            const double wBL = (double)t.yB_P[fy] * t.xL_P[fx], wBR = (double)t.yB_P[fy] * t.xR_P[fx];
            g1[0] += (xL * wTL * d[0] - xR * wTR * d[1] + xL * wBL * d[2] - xR * wBR * d[3]) / den_xy;
            sgrad[0] += (xL * wTL - xR * wTR + xL * wBL - xR * wBR) / den_xy;
            g1[1] += (yT * wTL * d[0] + yT * wTR * d[1] - yB * wBL * d[2] - yB * wBR * d[3]) / den_xy;
            sgrad[1] += (yT * wTL + yT * wTR - yB * wBL - yB * wBR) / den_xy;
            const double rTL = yT * yT + xL * xL, rTR = yT * yT + xR * xR, rBL = yB * yB + xL * xL, rBR = yB * yB + xR * xR;
            g1[2] += (rTL * wTL * d[0] + rTR * wTR * d[1] + rBL * wBL * d[2] + rBR * wBR * d[3]) / den_s;
            sgrad[2] += (rTL * wTL + rTR * wTR + rBL * wBL + rBR * wBR) / den_s;
            wd += wTL * d[0] + wTR * d[1] + wBL * d[2] + wBR * d[3];
        }
    const double S = static_cast<double>(sum);
    const double inv1 = (sum == static_cast<A>(0)) ? 1e8 : 1.0 / S;
    const double S2 = static_cast<double>(sum * sum);
    const double inv2 = (sum * sum == static_cast<A>(0)) ? 1e8 : 1.0 / S2;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const A v = static_cast<A>(g1[c] * inv1 - (sgrad[c] * wd) * inv2);
        gp[c * opl] = accumulate ? gp[c * opl] + v : v;
    }
}

}  // namespace gfla
