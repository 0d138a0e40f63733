// augment.cuh — auto-augmented decode: the 14 ops of torchvision's AutoAugment / RandAugment / TrivialAugmentWide
// (_apply_op on the PIL path) applied to each decoded entry right after its op, byte-identical to Pillow 12
// (include/xpng_b200.h, xpngb_decode_augment).
//
// An entry's program is up to XPNGB_AUG_STEPS_MAX steps; step k of every entry of the chunk that has one runs in stage k,
// and each stage is a handful of launches, batched by kind, never one per entry:
//   k_aug_pix        steps that read one buffer and write another (the warps AFFINE / TRANSPOSE, and SHARPNESS): one
//                    thread per pixel of the destination, coalesced along x; the buffers are the entry's pixels and its
//                    slice of the lane's bscr scratch, ping-ponged;
//   k_color_mean, k_color   BRIGHTNESS, COLOR and CONTRAST, which are colour decode's blends (color.cuh) with one step on;
//   k_aug_hist       256-bin histograms per entry and RGB channel, privatised in shared memory (EQUALIZE, AUTOCONTRAST);
//   k_aug_lut_build  one CTA per entry: its 3 x 256-byte LUT from the histograms (Python's integer and double rules);
//   k_aug_lut        the LUT applied in place (also POSTERIZE, SOLARIZE and INVERT, whose LUT the host builds).
// A CTA finds its descriptor by binary search over first CTAs, as k_orient does.
//
// Geometry.  Pillow's ImagingTransformAffine picks one of four code paths, restated operation for operation, every double
// operation with its own rounding (Pillow's x86-64 build contracts nothing into FMA):
//   NEAREST, a1 == a3 == 0 (ImagingScaleAffine): x = a2 + a0 / 2, then x += a0 once per column; y likewise per row;
//   NEAREST, four corners within +-32768 (affine_fixed): 16.16 fixed point, xx = a2' + y a1 + x a0 in wrapping int32;
//   NEAREST otherwise: running double sums, across each row from a start that itself runs down the image;
//   BILINEAR / BICUBIC (ImagingGenericTransform): the source point a0 (x + .5) + a1 (y + .5) + a2, Pillow's filters.
// The running sums are what Pillow computes, so a thread recomputes its pixel's sums (x + y additions at most): the closed
// form a0 * x would differ from them in the last bits.  The host refuses coefficients of 2^64 or more, so no sum reaches
// infinity or NaN, and a coordinate is inside exactly when 0 <= v < side.  Pixels whose source is outside keep the fill.
//
// Orientation.  A tensor entry sits in tsrc in its pre-op layout (k_to_tensor applies the op), a uint8 one as written.  A
// warp acts on the output image's axes, so a thread maps its staged pixel to output coordinates through the entry's op,
// finds the source there and maps that back.  SMOOTH, the blends and the LUTs do not depend on pixel order or commute with
// every op (SMOOTH's kernel and its border rule are symmetric), so they run on the staged pixels as they sit.
#pragma once
#include "../../include/xpng_b200.h"
#include "common.cuh"
#include "color.cuh"
#include "orient.cuh"

namespace xpb {

constexpr uint32_t AP_THREADS = 256;   // k_aug_pix: destination pixels per CTA
constexpr uint32_t AH_PX = 8192;       // k_aug_hist: pixels per CTA

enum { AP_TRANSPOSE = 0, AP_FIXED, AP_SEQ, AP_BILINEAR, AP_BICUBIC, AP_SHARP };

struct AugPix {
    uint64_t src, dst;     // the entry's packed staged pixels, and the buffer this step writes (w x h, pxsz bytes each)
    double a[6];           // AP_SEQ: x start, x per row, x per column, then the same for y; AP_BILINEAR / BICUBIC: the matrix
    int32_t fx[6];         // AP_FIXED: Pillow's 16.16 a0, a1, a2 + a0 / 2 + a1 / 2, a3, a4, a5 + a3 / 2 + a4 / 2
    uint32_t w, h, pxsz;   // staged dimensions
    uint32_t eop;          // the entry's op: staged pixel -> output pixel (OP_TL for uint8 entries, staged as written)
    uint32_t mode, top;    // AP_*; AP_TRANSPOSE: the op it applies to the output image
    uint8_t fill[4];
    float fac;             // AP_SHARP: Image.blend's factor
    uint32_t first_cta;
};

struct AugLut {
    uint64_t px, npx;      // the entry's packed pixels, changed in place
    uint64_t hist;         // 0, or 3 x 256 uint64 bins: the LUT is built from them (EQUALIZE, AUTOCONTRAST)
    uint32_t pxsz, kind;   // XPNGB_AUG_*
    uint32_t first_cta, hfirst_cta;   // this entry's first CTA in k_aug_lut and in k_aug_hist (no CTAs there without hist)
    uint8_t lut[3 * 256];
};

__device__ __forceinline__ bool aug_quarter(uint32_t op) { return op == OP_R90 || op == OP_R270; }

// pixel (x, y) of a w x h image -> its position in op(image); aug_op_inv is the way back (tensor.cuh's index map)
__device__ __forceinline__ void aug_op_fwd(uint32_t op, uint32_t w, uint32_t h, uint32_t x, uint32_t y, uint32_t& X, uint32_t& Y) {
    if (op == OP_R90) { X = h - 1 - y; Y = x; }
    else if (op == OP_R270) { X = y; Y = w - 1 - x; }
    else { X = (op == OP_MH || op == OP_MVH) ? w - 1 - x : x; Y = (op == OP_MV || op == OP_MVH) ? h - 1 - y : y; }
}
__device__ __forceinline__ void aug_op_inv(uint32_t op, uint32_t w, uint32_t h, uint32_t X, uint32_t Y, uint32_t& x, uint32_t& y) {
    if (op == OP_R90) { x = Y; y = h - 1 - X; }
    else if (op == OP_R270) { x = w - 1 - Y; y = X; }
    else { x = (op == OP_MH || op == OP_MVH) ? w - 1 - X : X; y = (op == OP_MV || op == OP_MVH) ? h - 1 - Y : Y; }
}

// Pillow's FLOOR for doubles well inside int range (the generic filters only see in-range coordinates)
__device__ __forceinline__ int aug_floor(double v) { return v < 0.0 ? (int)floor(v) : (int)v; }

// BICUBIC of Geometry.c: p1 = v2, p2 = -v1 + v3, p3 = 2 (v1 - v2) + v3 - v4, p4 = -v1 + v2 - v3 + v4, v = p1 + d (p2 + d (p3 + d p4))
__device__ __forceinline__ double aug_cubic(double v1, double v2, double v3, double v4, double d) {
    const double p2 = __dadd_rn(-v1, v3);
    const double p3 = __dsub_rn(__dadd_rn(__dmul_rn(2.0, __dsub_rn(v1, v2)), v3), v4);
    const double p4 = __dadd_rn(__dsub_rn(__dadd_rn(-v1, v2), v3), v4);
    return __dadd_rn(v2, __dmul_rn(d, __dadd_rn(p2, __dmul_rn(d, __dadd_rn(p3, __dmul_rn(d, p4))))));
}
__device__ __forceinline__ double aug_lin(double a, double b, double d) { return __dadd_rn(a, __dmul_rn(__dsub_rn(b, a), d)); }

__global__ void __launch_bounds__(AP_THREADS) k_aug_pix(const AugPix* __restrict__ descs, uint32_t n) {
    uint32_t lo = 0, hi = n - 1;
    while (lo < hi) { const uint32_t mid = (lo + hi + 1) >> 1; if (descs[mid].first_cta <= blockIdx.x) lo = mid; else hi = mid - 1; }
    const AugPix& D = descs[lo];
    const uint64_t j = (uint64_t)(blockIdx.x - D.first_cta) * AP_THREADS + threadIdx.x;
    const uint32_t w = D.w, h = D.h, pxsz = D.pxsz, mode = D.mode, eop = D.eop;
    if (j >= (uint64_t)w * h) return;
    const uint32_t sx = (uint32_t)(j % w), sy = (uint32_t)(j / w);
    const uint8_t* __restrict__ src = reinterpret_cast<const uint8_t*>(D.src);
    uint8_t* __restrict__ dst = reinterpret_cast<uint8_t*>(D.dst) + j * pxsz;
    const uint8_t* self = src + j * pxsz;
    if (mode == AP_SHARP) {   // Image.blend(SMOOTH(img), img, f); SMOOTH copies the border and images with a side below 3
        for (uint32_t c = 0; c < pxsz; c++) {
            const uint32_t p = self[c];
            uint32_t v = p;
            if (c < 3 && sx > 0 && sy > 0 && sx + 1 < w && sy + 1 < h) {
                // Pillow sums the nine float products of (1 1 1 / 1 5 1 / 1 1 1) / 13 plus 0.5 and truncates.  The exact mean
                // S / 13 is never within 1/26 of a half and the float error is below 0.004, so that is (S + 6) / 13.
                uint32_t S = 4 * p;
                for (int dy = -1; dy <= 1; dy++)
                    for (int dx = -1; dx <= 1; dx++) S += src[((uint64_t)(sy + dy) * w + (sx + dx)) * pxsz + c];
                v = color_blend((S + 6) / 13, p, D.fac);
            }
            dst[c] = (uint8_t)v;
        }
        return;
    }
    const bool q = aug_quarter(eop);
    const uint32_t W = q ? h : w, H = q ? w : h;   // the output image
    uint32_t X, Y;
    aug_op_fwd(eop, w, h, sx, sy, X, Y);
    auto at = [&](uint32_t u, uint32_t v) -> const uint8_t* {   // output pixel (u, v) in the staged buffer
        uint32_t x, y;
        aug_op_inv(eop, w, h, u, v, x, y);
        return src + ((uint64_t)y * w + x) * pxsz;
    };
    if (mode == AP_TRANSPOSE) {   // only square outputs are turned a quarter, so the output keeps its size
        uint32_t u, v;
        aug_op_inv(D.top, W, H, X, Y, u, v);
        const uint8_t* s = at(u, v);
        for (uint32_t c = 0; c < pxsz; c++) dst[c] = s[c];
        return;
    }
    if (mode == AP_FIXED || mode == AP_SEQ) {   // NEAREST
        int64_t xi, yi;
        if (mode == AP_FIXED) {
            xi = (int32_t)((uint32_t)D.fx[2] + (uint32_t)Y * (uint32_t)D.fx[1] + (uint32_t)X * (uint32_t)D.fx[0]) >> 16;
            yi = (int32_t)((uint32_t)D.fx[5] + (uint32_t)Y * (uint32_t)D.fx[4] + (uint32_t)X * (uint32_t)D.fx[3]) >> 16;
        } else {
            double xv = D.a[0], yv = D.a[3];
            if (D.a[1] != 0.0 || D.a[4] != 0.0)
                for (uint32_t k = 0; k < Y; k++) { xv = __dadd_rn(xv, D.a[1]); yv = __dadd_rn(yv, D.a[4]); }
            if (D.a[2] != 0.0 || D.a[5] != 0.0)
                for (uint32_t k = 0; k < X; k++) { xv = __dadd_rn(xv, D.a[2]); yv = __dadd_rn(yv, D.a[5]); }
            xi = (xv >= 0.0 && xv < (double)W) ? (int64_t)xv : -1;
            yi = (yv >= 0.0 && yv < (double)H) ? (int64_t)yv : -1;
        }
        if (xi >= 0 && xi < W && yi >= 0 && yi < H) {
            const uint8_t* s = at((uint32_t)xi, (uint32_t)yi);
            for (uint32_t c = 0; c < pxsz; c++) dst[c] = s[c];
        } else for (uint32_t c = 0; c < pxsz; c++) dst[c] = D.fill[c];
        return;
    }
    // BILINEAR / BICUBIC: affine_transform, then Pillow's bilinear_filter32RGB / bicubic_filter32RGB
    const double xo = (double)X + 0.5, yo = (double)Y + 0.5;
    double xin = __dadd_rn(__dadd_rn(__dmul_rn(D.a[0], xo), __dmul_rn(D.a[1], yo)), D.a[2]);
    double yin = __dadd_rn(__dadd_rn(__dmul_rn(D.a[3], xo), __dmul_rn(D.a[4], yo)), D.a[5]);
    if (!(xin >= 0.0 && xin < (double)W && yin >= 0.0 && yin < (double)H)) {
        for (uint32_t c = 0; c < pxsz; c++) dst[c] = D.fill[c];
        return;
    }
    xin = __dsub_rn(xin, 0.5); yin = __dsub_rn(yin, 0.5);
    const int xf = aug_floor(xin), yf = aug_floor(yin);
    const double dx = __dsub_rn(xin, (double)xf), dy = __dsub_rn(yin, (double)yf);
    auto clipx = [&](int x) -> uint32_t { return x < 0 ? 0u : x < (int)W ? (uint32_t)x : W - 1; };
    auto clipy = [&](int y) -> uint32_t { return y < 0 ? 0u : y < (int)H ? (uint32_t)y : H - 1; };
    auto inside = [&](int y) { return y >= 0 && y < (int)H; };
    for (uint32_t c = 0; c < 3; c++) {
        double v;
        if (mode == AP_BILINEAR) {
            const uint32_t y0 = clipy(yf), x0 = clipx(xf), x1 = clipx(xf + 1);
            const double v1 = aug_lin(at(x0, y0)[c], at(x1, y0)[c], dx);
            const double v2 = inside(yf + 1) ? aug_lin(at(x0, (uint32_t)(yf + 1))[c], at(x1, (uint32_t)(yf + 1))[c], dx) : v1;
            v = aug_lin(v1, v2, dy);
            dst[c] = (uint8_t)(int)v;   // between two bytes: truncation, no clipping
        } else {
            const int xm = xf - 1, ym = yf - 1;
            const uint32_t xs[4] = { clipx(xm), clipx(xm + 1), clipx(xm + 2), clipx(xm + 3) };
            auto rowv = [&](uint32_t y) { return aug_cubic(at(xs[0], y)[c], at(xs[1], y)[c], at(xs[2], y)[c], at(xs[3], y)[c], dx); };
            const double v1 = rowv(clipy(ym));
            const double v2 = inside(ym + 1) ? rowv((uint32_t)(ym + 1)) : v1;
            const double v3 = inside(ym + 2) ? rowv((uint32_t)(ym + 2)) : v2;
            const double v4 = inside(ym + 3) ? rowv((uint32_t)(ym + 3)) : v3;
            v = aug_cubic(v1, v2, v3, v4, dy);
            dst[c] = v <= 0.0 ? 0 : v >= 255.0 ? 255 : (uint8_t)(int)v;
        }
    }
    if (pxsz == 4) dst[3] = self[3];
}

__device__ __forceinline__ uint32_t aug_find(const AugLut* descs, uint32_t n, bool hist) {
    uint32_t lo = 0, hi = n - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if ((hist ? descs[mid].hfirst_cta : descs[mid].first_cta) <= blockIdx.x) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__global__ void __launch_bounds__(256) k_aug_hist(const AugLut* __restrict__ descs, uint32_t n) {
    __shared__ uint32_t bins[3 * 256];
    const AugLut& D = descs[aug_find(descs, n, true)];
    for (uint32_t b = threadIdx.x; b < 3 * 256; b += blockDim.x) bins[b] = 0;
    __syncthreads();
    const uint64_t p0 = (uint64_t)(blockIdx.x - D.hfirst_cta) * AH_PX, p1 = min(p0 + AH_PX, D.npx);
    const uint8_t* px = reinterpret_cast<const uint8_t*>(D.px);
    for (uint64_t p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
        const uint8_t* q = px + p * D.pxsz;
        atomicAdd(&bins[q[0]], 1u); atomicAdd(&bins[256 + q[1]], 1u); atomicAdd(&bins[512 + q[2]], 1u);
    }
    __syncthreads();
    unsigned long long* g = reinterpret_cast<unsigned long long*>(D.hist);
    for (uint32_t b = threadIdx.x; b < 3 * 256; b += blockDim.x)
        if (bins[b]) atomicAdd(g + b, (unsigned long long)bins[b]);
}

// One CTA of 256 threads per descriptor, thread i owning bin i of each channel.
//   equalize:     with the non-empty bins h, step = (sum h - last h) // 255; fewer than two of them or step 0: identity;
//                 else lut[i] = (step // 2 + sum of bins below i) // step, clipped to 255 by Image.point.
//   autocontrast: lo, hi = first and last non-empty bins; hi <= lo: identity; else scale = 255.0 / (hi - lo),
//                 offset = -lo * scale, lut[i] = clamp(int(i * scale + offset), 0, 255), all in double.
__global__ void __launch_bounds__(256) k_aug_lut_build(AugLut* __restrict__ descs) {
    __shared__ unsigned long long scan[256];
    __shared__ int lo_s, hi_s;
    AugLut& D = descs[blockIdx.x];
    if (!D.hist) return;
    const uint32_t i = threadIdx.x;
    const unsigned long long* g = reinterpret_cast<const unsigned long long*>(D.hist);
    for (uint32_t c = 0; c < 3; c++) {
        const unsigned long long h = g[c * 256 + i];
        if (i == 0) { lo_s = 256; hi_s = -1; }
        __syncthreads();
        if (h) { atomicMin(&lo_s, (int)i); atomicMax(&hi_s, (int)i); }
        const int nz = __syncthreads_count(h != 0);
        scan[i] = h;
        __syncthreads();
        for (uint32_t o = 1; o < 256; o <<= 1) {   // inclusive prefix sums
            const unsigned long long v = i >= o ? scan[i - o] : 0ull;
            __syncthreads();
            scan[i] += v;
            __syncthreads();
        }
        const int lo = lo_s, hi = hi_s;
        uint32_t v = i;
        if (D.kind == XPNGB_AUG_EQUALIZE) {
            const unsigned long long total = scan[255], last = g[c * 256 + hi];
            const unsigned long long step = (total - last) / 255;
            if (nz > 1 && step) {
                const unsigned long long m = (step / 2 + scan[i] - h) / step;
                v = m > 255 ? 255u : (uint32_t)m;
            }
        } else if (hi > lo) {
            const double scale = __ddiv_rn(255.0, (double)(hi - lo)), offset = __dmul_rn((double)-lo, scale);
            const int t = __double2int_rz(__dadd_rn(__dmul_rn((double)i, scale), offset));
            v = t < 0 ? 0u : t > 255 ? 255u : (uint32_t)t;
        }
        D.lut[c * 256 + i] = (uint8_t)v;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) k_aug_lut(const AugLut* __restrict__ descs, uint32_t n) {
    __shared__ uint8_t lut[3 * 256];
    const AugLut& D = descs[aug_find(descs, n, false)];
    for (uint32_t b = threadIdx.x; b < 3 * 256; b += blockDim.x) lut[b] = D.lut[b];
    __syncthreads();
    const uint64_t p0 = (uint64_t)(blockIdx.x - D.first_cta) * CL_PX, p1 = min(p0 + CL_PX, D.npx);
    uint8_t* px = reinterpret_cast<uint8_t*>(D.px);
    for (uint64_t p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
        uint8_t* q = px + p * D.pxsz;
        q[0] = lut[q[0]]; q[1] = lut[256 + q[1]]; q[2] = lut[512 + q[2]];
    }
}

}  // namespace xpb
