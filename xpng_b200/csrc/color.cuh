// color.cuh — colour decode: torchvision's ColorJitter (brightness, contrast, saturation, hue in a per-entry order) and
// RandomGrayscale applied to each decoded entry, byte-identical to their PIL path (include/xpng_b200.h, xpngb_decode_color).
//
// Every step maps bytes to bytes, as Pillow, where each step returns a new 8-bit image.  Brightness, contrast and saturation
// are Image.blend(degenerate, img, factor) (Blend.c): t = d + a * (p - d) in float, truncated and clipped to a byte, with d
// 0, the entry's rounded mean luma, or the pixel's own luma.  Hue goes through Pillow's rgb2hsv / hsv2rgb (Convert.c) and
// shifts H by a byte.  Grayscale is Pillow's L24 luma in every colour channel.  Every float and double operation is written
// with an _rn intrinsic, so that no build flag can contract or approximate one: each is rounded on its own, as on the host.
//
// The chain is per pixel and contrast's mean does not depend on pixel order, so it runs on the entry's pixels as they are
// written (after the op) or, for tensor output, on its uint8 source before k_to_tensor.  Two launches per chunk:
//   k_color_mean  for each entry with contrast on, the 64-bit sum of the luma of its pixels after the steps that precede
//                 contrast in its order (integer sums: deterministic, and an 8K entry's sum exceeds 2^32);
//   k_color       the whole chain, in place on the entry's packed pixels.
// A CTA takes CL_PX consecutive pixels of one entry and finds its entry by binary search over the first CTAs, as k_orient.
#pragma once
#include "../../include/xpng_b200.h"
#include "common.cuh"

namespace xpb {

constexpr uint32_t CL_PX = 2048;   // pixels per CTA (256 threads, 8 pixels each)

struct ColorDesc {
    uint64_t px, npx;               // device address of the entry's packed pixels (modified in place), their count
    float fac[4];                   // brightness, contrast, saturation factors narrowed to float as Pillow does; [3] unused
    uint32_t hue;                   // hue shift of H, 0..255
    uint32_t pxsz, on, gray;        // bytes per pixel, xpngb_color::on and ::gray
    uint8_t order[4];               // xpngb_color::order
    uint32_t pre;                   // steps of `order` that precede contrast (k_color_mean applies these)
    uint32_t first_cta, mfirst_cta; // this entry's first CTA in k_color and in k_color_mean (zero CTAs there without contrast)
};

__device__ __forceinline__ uint32_t color_luma(uint32_t r, uint32_t g, uint32_t b) {   // Pillow's L24
    return (19595u * r + 38470u * g + 7471u * b + 0x8000u) >> 16;
}

// One channel of Image.blend(deg, img, a).  For 0 <= a <= 1 Pillow truncates t without clipping, but t then lies between d
// and p, so the clipped form is the same function for every a.
__device__ __forceinline__ uint32_t color_blend(uint32_t d, uint32_t p, float a) {
    const float t = __fadd_rn((float)d, __fmul_rn(a, (float)((int)p - (int)d)));
    return t <= 0.f ? 0u : t >= 255.f ? 255u : (uint32_t)__float2int_rz(t);
}

__device__ __forceinline__ uint32_t color_clip8(int v) { return v <= 0 ? 0u : v >= 255 ? 255u : (uint32_t)v; }

// torchvision's adjust_hue on PIL: rgb2hsv, H + k mod 256, hsv2rgb (Pillow's Convert.c, operation for operation).
__device__ __forceinline__ void color_hue(uint32_t& r, uint32_t& g, uint32_t& b, uint32_t k) {
    const uint32_t mx = max(r, max(g, b)), mn = min(r, min(g, b));
    if (mx == mn) return;   // H = S = 0, and hsv2rgb of S == 0 is (V, V, V): the pixel itself
    const float cr = (float)(mx - mn), s = __fdiv_rn(cr, (float)mx);
    const float rc = __fdiv_rn((float)(mx - r), cr), gc = __fdiv_rn((float)(mx - g), cr), bc = __fdiv_rn((float)(mx - b), cr);
    float h;
    if (r == mx) h = __fsub_rn(bc, gc);
    else if (g == mx) h = __double2float_rn(__dsub_rn(__dadd_rn(2.0, (double)rc), (double)bc));
    else h = __double2float_rn(__dsub_rn(__dadd_rn(4.0, (double)gc), (double)rc));
    // fmod(h / 6.0 + 1.0, 1.0): h lies in [-1, 5], so the sum lies in [5/6, 11/6] and the remainder is one exact subtraction
    double x = __dadd_rn(__ddiv_rn((double)h, 6.0), 1.0);
    if (x >= 1.0) x = __dsub_rn(x, 1.0);
    h = __double2float_rn(x);
    const uint32_t H = (color_clip8(__double2int_rz(__dmul_rn((double)h, 255.0))) + k) & 255u;
    const uint32_t S = color_clip8(__double2int_rz(__dmul_rn((double)s, 255.0))), V = mx;
    if (S == 0) { r = g = b = V; return; }
    const double hx = __ddiv_rn(__dmul_rn((double)H, 6.0), 255.0);
    const int i = (int)floor(hx);
    const float f = __double2float_rn(__dsub_rn(hx, (double)i));
    const float fs = __double2float_rn(__ddiv_rn((double)S, 255.0));
    const double v = (double)V;
    const uint32_t p = color_clip8((int)round(__dmul_rn(v, __dsub_rn(1.0, (double)fs))));
    const uint32_t q = color_clip8((int)round(__dmul_rn(v, __dsub_rn(1.0, (double)__fmul_rn(fs, f)))));
    const uint32_t t = color_clip8((int)round(__dmul_rn(v, __dsub_rn(1.0, __dmul_rn((double)fs, __dsub_rn(1.0, (double)f))))));
    switch (i % 6) {
        case 0: r = V; g = t; b = p; break;
        case 1: r = q; g = V; b = p; break;
        case 2: r = p; g = V; b = t; break;
        case 3: r = p; g = q; b = V; break;
        case 4: r = t; g = p; b = V; break;
        default: r = V; g = p; b = q; break;
    }
}

// The first `nsteps` steps of the entry's order, each only when its bit of `on` is set; m is the entry's contrast mean.
// Alpha is each blend's own degenerate, so it is unchanged there; hue leaves it 255, as torchvision's adjust_hue does.
__device__ __forceinline__ void color_steps(uint32_t& r, uint32_t& g, uint32_t& b, uint32_t& a, const ColorDesc& D,
                                            uint32_t nsteps, uint32_t m) {
#pragma unroll
    for (uint32_t s = 0; s < 4; s++) {   // unrolled, so that the descriptor stays in registers
        const uint32_t step = D.order[s];
        if (s >= nsteps || !((D.on >> step) & 1u)) continue;
        if (step == XPNGB_CJ_HUE) { color_hue(r, g, b, D.hue); a = 255; continue; }
        const uint32_t d = step == XPNGB_CJ_BRIGHTNESS ? 0u : step == XPNGB_CJ_CONTRAST ? m : color_luma(r, g, b);
        const float f = step == XPNGB_CJ_BRIGHTNESS ? D.fac[0] : step == XPNGB_CJ_CONTRAST ? D.fac[1] : D.fac[2];
        r = color_blend(d, r, f); g = color_blend(d, g, f); b = color_blend(d, b, f);
    }
}

__device__ __forceinline__ uint32_t color_find(const ColorDesc* descs, uint32_t n, bool mean) {
    uint32_t lo = 0, hi = n - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if ((mean ? descs[mid].mfirst_cta : descs[mid].first_cta) <= blockIdx.x) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__global__ void __launch_bounds__(256) k_color_mean(const ColorDesc* __restrict__ descs, uint32_t n, unsigned long long* sums) {
    __shared__ uint32_t part[8];
    const uint32_t e = color_find(descs, n, true);
    const ColorDesc D = descs[e];
    const uint64_t p0 = (uint64_t)(blockIdx.x - D.mfirst_cta) * CL_PX, p1 = min(p0 + CL_PX, D.npx);
    const uint8_t* px = reinterpret_cast<const uint8_t*>(D.px);
    uint32_t acc = 0;   // at most 8 pixels of 255
    for (uint64_t p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
        const uint8_t* q = px + p * D.pxsz;
        uint32_t r = q[0], g = q[1], b = q[2], a = 255;
        color_steps(r, g, b, a, D, D.pre, 0);
        acc += color_luma(r, g, b);
    }
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (uint32_t w = 0; w < (blockDim.x >> 5); w++) t += part[w];
        atomicAdd(sums + e, (unsigned long long)t);
    }
}

__global__ void __launch_bounds__(256) k_color(const ColorDesc* __restrict__ descs, uint32_t n, const unsigned long long* __restrict__ sums) {
    const uint32_t e = color_find(descs, n, false);
    const ColorDesc D = descs[e];
    // ImageStat's mean (a double quotient of exact integers: sums below 2^53) rounded as int(mean + 0.5)
    const uint32_t m = (D.on >> XPNGB_CJ_CONTRAST) & 1u
                           ? (uint32_t)__double2int_rz(__dadd_rn(__ddiv_rn(__ull2double_rn(sums[e]), __ull2double_rn(D.npx)), 0.5))
                           : 0u;
    const uint64_t p0 = (uint64_t)(blockIdx.x - D.first_cta) * CL_PX, p1 = min(p0 + CL_PX, D.npx);
    uint8_t* px = reinterpret_cast<uint8_t*>(D.px);
    for (uint64_t p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
        uint8_t* q = px + p * D.pxsz;
        uint32_t r = q[0], g = q[1], b = q[2], a = D.pxsz == 4 ? q[3] : 255u;
        color_steps(r, g, b, a, D, 4, m);
        if (D.gray) r = g = b = color_luma(r, g, b);
        q[0] = (uint8_t)r; q[1] = (uint8_t)g; q[2] = (uint8_t)b;
        if (D.pxsz == 4) q[3] = (uint8_t)a;
    }
}

}  // namespace xpb
