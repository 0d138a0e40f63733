// blur.cuh — blurred and solarized decode: Pillow's ImageFilter.GaussianBlur and ImageOps.solarize applied to each decoded
// entry after its colour step, byte-identical to Pillow (include/xpng_b200.h, xpngb_decode_blur).
//
// Pillow's GaussianBlur is three box blurs along x, then three along y (BoxBlur.c).  Each box pass is integer arithmetic on
// one line of one channel, edges clamped to the nearest pixel, and rounds to a byte before the next pass reads it:
//   acc  = sum of p[clamp(x + k)] for k = -ri .. ri
//   bulk = acc * ww + (p[clamp(x - ri - 1)] + p[clamp(x + ri + 1)]) * fw
//   out  = (bulk + 2^23) >> 24
// The host computes (ri, ww, fw) per axis in float exactly as Pillow does; the device gets integers only.
//
// Why uint32 is enough.  The host refuses radii whose (ri, ww, fw) could wrap.  For every accepted radius (2 ri + 1) * ww
// <= 2^24, so fw = (2^24 - (2 ri + 1) * ww) / 2 does not wrap and (2 ri + 1) * ww + 2 fw <= 2^24.  With bytes of at most 255,
// acc <= 255 (2 ri + 1) and far = p[..] + p[..] <= 2 * 255, so
//   acc * ww + far * fw + 2^23 <= 255 * ((2 ri + 1) * ww + 2 fw) + 2^23 <= 255 * 2^24 + 2^23 < 2^32,
// and acc itself is at most 255 * (2^24 - 1) < 2^32 since ri < 2^23.  The running sum below adds and subtracts bytes in
// uint32: intermediate wraps cancel, and every value it is read at is the true sum.
//
// One launch per pass stage and chunk, every entry with a pass at that stage in it.  A pass reads one packed buffer and
// writes another (the entry's pixels and its scratch, ping-ponged); a CTA takes 256 lines of one pass and finds it by binary
// search over first_cta, as k_orient does.  A thread walks one line with a running sum, so the work per pixel does not
// depend on the radius:
//   vertical passes   one thread per byte column: a warp reads and writes 32 consecutive bytes of a row per step;
//   horizontal passes one thread per row and channel.
// Solarize is a byte LUT (v < t ? v : 255 - v) on the stored value of an entry's last pass; an entry with nothing else to
// do gets one identity pass (ri = 0, ww = 2^24, fw = 0) that carries it.
#pragma once
#include "common.cuh"

namespace xpb {

constexpr uint32_t BL_THREADS = 256;   // lines per CTA
constexpr uint32_t BLUR_STAGES = 6;    // passes of one entry at most: three per axis (an odd count gets one more)

struct BlurPass {
    uint64_t src, dst;      // device addresses of the packed source and destination pixels (different buffers)
    uint64_t pitch;         // bytes per row (w * pxsz)
    uint32_t w, h, pxsz;
    uint32_t vert;          // 1: along columns (one line per byte column), 0: along rows (one line per row and channel)
    uint32_t ri, ww, fw;    // Pillow's box radius and weights for this axis
    uint32_t t;             // solarize: bytes v < t are kept, others become 255 - v; 256 keeps every byte
    uint32_t first_cta;     // this pass's first CTA in the launch
};

__global__ void __launch_bounds__(BL_THREADS) k_blur(const BlurPass* __restrict__ descs, uint32_t n) {
    uint32_t lo = 0, hi = n - 1;
    while (lo < hi) { const uint32_t mid = (lo + hi + 1) >> 1; if (descs[mid].first_cta <= blockIdx.x) lo = mid; else hi = mid - 1; }
    const BlurPass D = descs[lo];
    const uint64_t j = (uint64_t)(blockIdx.x - D.first_cta) * BL_THREADS + threadIdx.x;
    uint64_t base, es;   // the line's first byte and the bytes between its elements
    uint32_t len;
    if (D.vert) {
        if (j >= (uint64_t)D.w * D.pxsz) return;
        base = j; es = D.pitch; len = D.h;
    } else {
        if (j >= (uint64_t)D.h * D.pxsz) return;
        base = (j / D.pxsz) * D.pitch + j % D.pxsz; es = D.pxsz; len = D.w;
    }
    const uint8_t* __restrict__ s = reinterpret_cast<const uint8_t*>(D.src) + base;
    uint8_t* __restrict__ d = reinterpret_cast<uint8_t*>(D.dst) + base;
    const uint32_t ri = D.ri, ww = D.ww, fw = D.fw, t = D.t, last = len - 1;
    // the window of x = 0: p[0] ri + 1 times, then p[1 .. ri], the ones past the end clamped to p[last]
    const uint32_t m = min(ri, last);
    uint32_t acc = (ri + 1) * s[0];
    for (uint32_t k = 1; k <= m; k++) acc += s[k * es];
    acc += (ri - m) * s[(uint64_t)last * es];
    uint32_t lo_px = s[0];   // p[clamp(x - ri - 1)]
#pragma unroll 4
    for (uint32_t x = 0; x < len; x++) {
        const uint32_t lead = s[(uint64_t)(ri < last - x ? x + ri + 1 : last) * es];   // p[clamp(x + ri + 1)], no overflow
        const uint32_t trail = s[(uint64_t)(x > ri ? x - ri : 0) * es];                // p[clamp(x - ri)]
        uint32_t v = (acc * ww + (lo_px + lead) * fw + (1u << 23)) >> 24;
        v = v < t ? v : 255u - v;
        d[(uint64_t)x * es] = (uint8_t)v;
        acc += lead - trail;
        lo_px = trail;
    }
}

}  // namespace xpb
