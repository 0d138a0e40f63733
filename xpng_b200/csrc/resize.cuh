// resize.cuh — resized decode: each decoded crop resampled to a requested size, byte-identical to Pillow's
// Image.resize(size, filter) of the crop (Resample.c, 8-bit path) for its five convolution filters, with every channel
// (alpha included) resampled on its own, then a window of the resized image written as its op leaves it.
//
// Pillow resamples one axis at a time.  Per axis (input length `in`, output length `out`) it precomputes, for every
// output coordinate o, a window [xmin, xmin + n) of input coordinates and 22-bit fixed-point weights k[0..n) (its
// precompute_coeffs + normalize_coeffs_8bpc); a pass then computes clamp((2^21 + sum src[xmin + t] * k[t]) >> 22, 0, 255).
// The horizontal pass runs first and its results are rounded to bytes; the vertical pass reads those.  Pillow 12 runs the
// vertical pass first instead for crops more than 100 times taller than wide that shrink vertically (resize_vfirst).
// A pass with in == out is the identity and is skipped.  The filters differ only in f, its support and, for the two with
// negative lobes (bicubic, lanczos), in weights below zero, which Pillow rounds half away from zero.
//
// A window of the resized image is the same computation restricted to some output coordinates: table entry o is resized
// coordinate window origin + o, and its xmin is stored relative to the first decoded source pixel of that axis (`base`),
// so that only the source span the window's support reaches is decoded, and the first pass runs only over the rows (or,
// vertical first, the columns) the second pass reads.
//
// Three launches per chunk, every resized entry of the chunk in each; a CTA or thread finds its entry by binary search
// over the entry's first index, as k_orient does:
//   k_resize_coeffs  one thread per output coordinate per resampled axis: the windows and weights (tables in scratch)
//   k_resize_h       horizontal pass: RH_ROWS source rows x RH_X output pixels per CTA, source row segments staged in
//                    shared memory by aligned 32-bit words (any source alignment and pitch)
//   k_resize_v       vertical pass: RV_ROWS output rows x RV_X bytes per CTA, one byte per thread along x (coalesced)
// The last pass of an entry writes its output through the op's index map, so the op costs no pass of its own.
#pragma once
#include "common.cuh"
#include "orient.cuh"

namespace xpb {

constexpr int RS_BITS = 22;                    // Pillow's PRECISION_BITS for 8-bit images (32 - 8 - 2)
constexpr int RH_X = 256, RH_ROWS = 4;         // horizontal pass: output pixels x crop rows per CTA
constexpr int RH_SMEM = 24 * 1024;             // bytes of one staged source row segment
constexpr int RV_X = 256, RV_ROWS = 8;         // vertical pass: output bytes x output rows per CTA
// Pillow's Image.Resampling numbers (XPNGB_LANCZOS .. XPNGB_HAMMING); NEAREST (0) is not a convolution filter
enum : uint32_t { RF_LANCZOS = 1, RF_BILINEAR = 2, RF_BICUBIC = 3, RF_BOX = 4, RF_HAMMING = 5 };

// One resized entry: an in_w x in_h crop resampled to full_w x full_h pixels, of which the out_w x out_h window at (wx, wy)
// is written packed through op.  The passes read from the first decoded source pixel (bx, by) of the crop on: each reads
// rows `pitch` bytes apart at any byte alignment (the decoded span, or the first pass's packed rows in scratch) and writes
// packed rows, the last pass through op.  Tables at coef: for each resampled axis (x first), out int2 windows (xmin - base,
// n), then out * ksize int32 weights.
struct ResizePass {
    uint64_t src, pitch, dst;
    uint32_t n;                                // rows of the horizontal pass, pixels per row of the vertical pass
    uint32_t last;                             // 1: writes the output through op
};
struct ResizeDesc {
    ResizePass h, v;
    uint64_t coef;
    uint32_t in_w, in_h, out_w, out_h;
    uint32_t full_w, full_h, wx, wy, bx, by;
    uint32_t filter, pxsz, op, kx, ky;         // ksize per axis (0: the axis is not resampled)
    uint32_t first_coef, first_h, first_v;     // this entry's first thread / CTA in each launch
    uint32_t h_tiles_x;                        // horizontal-pass CTAs per group of RH_ROWS rows
};

// Pillow's pass order (Resample.c of Pillow 12): vertical first for a crop more than 100 times taller than wide that
// shrinks vertically and is resampled on both axes.
__host__ __device__ inline bool resize_vfirst(uint64_t in_w, uint64_t in_h, uint64_t out_w, uint64_t out_h) {
    return in_w != out_w && out_h < in_h && in_h > 100 * in_w;
}

// Bytes of one axis's tables, rounded up to 8 so that the next axis's int2 windows stay aligned (ksize is odd).
__host__ __device__ inline uint64_t resize_table_bytes(uint32_t out, uint32_t ksize) {
    return ksize ? ((uint64_t)out * (2 + ksize) * 4 + 7) & ~7ull : 0;
}

// Pillow's support of each filter (Resample.c); 0 for a number that is not one of them.
__host__ __device__ inline double resize_support(uint32_t filter) {
    switch (filter) {
        case RF_BOX: return 0.5;
        case RF_BILINEAR: case RF_HAMMING: return 1.0;
        case RF_BICUBIC: return 2.0;
        case RF_LANCZOS: return 3.0;
        default: return 0.0;
    }
}

// The last entry whose first index (member `first`) is at most idx: entries with nothing to do in a launch are skipped.
__device__ __forceinline__ uint32_t resize_find(const ResizeDesc* __restrict__ d, uint32_t n, uint32_t idx, uint32_t ResizeDesc::*first) {
    uint32_t lo = 0, hi = n - 1;
    while (lo < hi) { const uint32_t mid = (lo + hi + 1) >> 1; if (d[mid].*first <= idx) lo = mid; else hi = mid - 1; }
    return lo;
}

__device__ __forceinline__ double tri(double x) {
    if (x < 0.0) x = -x;
    return x < 1.0 ? __dsub_rn(1.0, x) : 0.0;
}

// sin(x) / x of Pillow's sinc_filter, x already multiplied by pi
__device__ __forceinline__ double sinc_pi(double x) {
    if (x == 0.0) return 1.0;
    x = __dmul_rn(x, M_PI);
    return __ddiv_rn(sin(x), x);
}

// Pillow's filter functions, operation by operation (bicubic with a = -0.5).  sin and cos are CUDA's double ones; the
// weight tables they give are compared with the host C library's in the tests (xpngb_resize_coeffs).
__device__ double resize_filter(uint32_t filter, double x) {
    switch (filter) {
        case RF_BOX: return x > -0.5 && x <= 0.5 ? 1.0 : 0.0;
        case RF_HAMMING:
            if (x < 0.0) x = -x;
            if (x == 0.0) return 1.0;
            if (x >= 1.0) return 0.0;
            x = __dmul_rn(x, M_PI);
            return __dmul_rn(__ddiv_rn(sin(x), x), __dadd_rn((double)0.54f, __dmul_rn((double)0.46f, cos(x))));   // float literals in Pillow
        case RF_BICUBIC:
            if (x < 0.0) x = -x;
            if (x < 1.0) return __dadd_rn(__dmul_rn(__dmul_rn(__dsub_rn(__dmul_rn(1.5, x), 2.5), x), x), 1.0);
            if (x < 2.0) return __dmul_rn(__dsub_rn(__dmul_rn(__dadd_rn(__dmul_rn(__dsub_rn(x, 5.0), x), 8.0), x), 4.0), -0.5);
            return 0.0;
        case RF_LANCZOS: return -3.0 <= x && x < 3.0 ? __dmul_rn(sinc_pi(x), sinc_pi(__ddiv_rn(x, 3.0))) : 0.0;
        default: return tri(x);
    }
}

// Window and weights of output coordinate o0 + o (stored at o), every double operation rounded on its own as in Pillow's
// C (no FMA contraction).  The weights are computed twice (sum, then each divided by it) so that nothing is kept per tap.
// xmin is stored relative to base, the first source coordinate the pass reads (at most the smallest xmin of the table).
__device__ void resize_axis(uint32_t filter, uint32_t in, uint32_t out, uint32_t ksize, uint32_t o0, uint32_t base, uint32_t o,
                            int2* bounds, int32_t* k) {
    const double scale = __ddiv_rn((double)in, (double)out);
    const double fs = scale < 1.0 ? 1.0 : scale, support = __dmul_rn(resize_support(filter), fs), ss = __ddiv_rn(1.0, fs);
    const double center = __dmul_rn((double)(o0 + o) + 0.5, scale);
    int xmin = __double2int_rz(__dadd_rn(__dsub_rn(center, support), 0.5));
    int xmax = __double2int_rz(__dadd_rn(__dadd_rn(center, support), 0.5));
    if (xmin < 0) xmin = 0;
    if (xmax > (int)in) xmax = (int)in;
    const int n = xmax - xmin;
    double ww = 0.0;
    for (int t = 0; t < n; t++)
        ww = __dadd_rn(ww, resize_filter(filter, __dmul_rn(__dadd_rn(__dsub_rn((double)(t + xmin), center), 0.5), ss)));
    int32_t* kk = k + (uint64_t)o * ksize;
    for (int t = 0; t < n; t++) {
        double w = resize_filter(filter, __dmul_rn(__dadd_rn(__dsub_rn((double)(t + xmin), center), 0.5), ss));
        if (ww != 0.0) w = __ddiv_rn(w, ww);
        kk[t] = __double2int_rz(__dadd_rn(w < 0.0 ? -0.5 : 0.5, __dmul_rn(w, (double)(1 << RS_BITS))));
    }
    bounds[o] = make_int2(xmin - (int)base, n);
}

__global__ void __launch_bounds__(256) k_resize_coeffs(const ResizeDesc* __restrict__ descs, uint32_t n, uint32_t total) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const ResizeDesc& D = descs[resize_find(descs, n, idx, &ResizeDesc::first_coef)];
    uint32_t o = idx - D.first_coef;
    uint8_t* tab = reinterpret_cast<uint8_t*>(D.coef);
    if (D.kx) {
        if (o < D.out_w) {
            resize_axis(D.filter, D.in_w, D.full_w, D.kx, D.wx, D.bx, o, reinterpret_cast<int2*>(tab), reinterpret_cast<int32_t*>(tab + (uint64_t)D.out_w * 8));
            return;
        }
        o -= D.out_w;
        tab += resize_table_bytes(D.out_w, D.kx);
    }
    resize_axis(D.filter, D.in_h, D.full_h, D.ky, D.wy, D.by, o, reinterpret_cast<int2*>(tab), reinterpret_cast<int32_t*>(tab + (uint64_t)D.out_h * 8));
}

// Byte offset of output pixel (x, y) of a w x h image after op (the index maps of k_orient).
__device__ __forceinline__ uint64_t op_pixel(uint32_t op, uint32_t x, uint32_t y, uint32_t w, uint32_t h) {
    switch (op) {
        case OP_R90: return (uint64_t)x * h + (h - 1 - y);
        case OP_R270: return (uint64_t)(w - 1 - x) * h + y;
        case OP_MV: return (uint64_t)(h - 1 - y) * w + x;
        case OP_MH: return (uint64_t)y * w + (w - 1 - x);
        case OP_MVH: return (uint64_t)(h - 1 - y) * w + (w - 1 - x);
        default: return (uint64_t)y * w + x;
    }
}

__device__ __forceinline__ uint8_t clip8(int32_t acc) { return (uint8_t)min(max(acc >> RS_BITS, 0), 255); }

// Horizontal pass.  A CTA takes RH_X output pixels of RH_ROWS source rows, one thread per output pixel (all channels).  The
// source span the CTA's windows cover is staged row by row in shared memory, in pieces of RH_SMEM bytes when it is
// longer (extreme downscales), each thread adding the taps of its window that fall in the piece.
__global__ void __launch_bounds__(RH_X, 4) k_resize_h(const ResizeDesc* __restrict__ descs, uint32_t n) {
    __shared__ uint32_t sm[RH_SMEM / 4 + 1];
    const ResizeDesc D = descs[resize_find(descs, n, blockIdx.x, &ResizeDesc::first_h)];
    const uint32_t cta = blockIdx.x - D.first_h;
    const uint32_t X0 = (cta % D.h_tiles_x) * RH_X, Y0 = (cta / D.h_tiles_x) * RH_ROWS;
    const uint32_t X1 = min(X0 + RH_X, D.out_w), Y1 = min(Y0 + RH_ROWS, D.h.n), pxsz = D.pxsz;
    const int2* bounds = reinterpret_cast<const int2*>(D.coef);
    const uint32_t o = X0 + threadIdx.x;
    const bool act = o < X1;
    const int2 b = act ? bounds[o] : make_int2(0, 0);
    const int32_t* k = reinterpret_cast<const int32_t*>(D.coef + (uint64_t)D.out_w * 8) + (uint64_t)o * D.kx;
    const uint32_t lo = bounds[X0].x, hi = bounds[X1 - 1].x + bounds[X1 - 1].y;   // the CTA's source pixels
    const uint32_t piece = (RH_SMEM - 4) / pxsz;
    const uint8_t* smb = reinterpret_cast<const uint8_t*>(sm);
    for (uint32_t y = Y0; y < Y1; y++) {
        const uint64_t row = D.h.src + (uint64_t)y * D.h.pitch;
        int32_t a0 = 1 << (RS_BITS - 1), a1 = a0, a2 = a0, a3 = a0;
        for (uint32_t p0 = lo; p0 < hi; p0 += piece) {
            const uint32_t p1 = min(p0 + piece, hi);
            const uint64_t a = row + (uint64_t)p0 * pxsz, aw = a & ~3ull;
            const uint32_t sh = (uint32_t)(a - aw), nw = (sh + (p1 - p0) * pxsz + 3) >> 2;
            __syncthreads();   // the previous piece has been read
            for (uint32_t j = threadIdx.x; j < nw; j += RH_X) sm[j] = __ldg(reinterpret_cast<const uint32_t*>(aw) + j);
            __syncthreads();
            if (act) {
                const int t0 = max(b.x, (int)p0) - b.x, t1 = min(b.x + b.y, (int)p1) - b.x;
                const uint8_t* s = smb + sh + (b.x - (int)p0) * (int)pxsz;
                if (pxsz == 3) {
                    for (int t = t0; t < t1; t++) {
                        const int32_t w = __ldg(k + t);
                        a0 += s[3 * t] * w; a1 += s[3 * t + 1] * w; a2 += s[3 * t + 2] * w;
                    }
                } else {
                    for (int t = t0; t < t1; t++) {
                        const int32_t w = __ldg(k + t);
                        a0 += s[4 * t] * w; a1 += s[4 * t + 1] * w; a2 += s[4 * t + 2] * w; a3 += s[4 * t + 3] * w;
                    }
                }
            }
        }
        if (act) {
            uint8_t* q = reinterpret_cast<uint8_t*>(D.h.dst) + (D.h.last ? op_pixel(D.op, o, y, D.out_w, D.out_h) : (uint64_t)y * D.out_w + o) * pxsz;
            q[0] = clip8(a0); q[1] = clip8(a1); q[2] = clip8(a2);
            if (pxsz == 4) q[3] = clip8(a3);
        }
    }
}

// Vertical pass.  A CTA takes RV_X bytes of RV_ROWS output rows, one byte per thread.  which: bit 0 the entries whose
// vertical pass comes first, bit 1 those whose vertical pass is the last.
__global__ void __launch_bounds__(RV_X) k_resize_v(const ResizeDesc* __restrict__ descs, uint32_t n, uint32_t which) {
    const ResizeDesc D = descs[resize_find(descs, n, blockIdx.x, &ResizeDesc::first_v)];
    if (!((D.v.last ? 2u : 1u) & which)) return;
    const uint32_t cta = blockIdx.x - D.first_v, pxsz = D.pxsz;
    const uint32_t row_bytes = D.v.n * pxsz, tiles_x = (row_bytes + RV_X - 1) / RV_X;
    const uint32_t bx = (cta % tiles_x) * RV_X + threadIdx.x, Y0 = (cta / tiles_x) * RV_ROWS;
    if (bx >= row_bytes) return;
    const uint8_t* src = reinterpret_cast<const uint8_t*>(D.v.src) + bx;
    const uint64_t pitch = D.v.pitch;
    const uint8_t* tab = reinterpret_cast<const uint8_t*>(D.coef) + resize_table_bytes(D.out_w, D.kx);
    const int2* bounds = reinterpret_cast<const int2*>(tab);
    const int32_t* ky = reinterpret_cast<const int32_t*>(tab + (uint64_t)D.out_h * 8);
    const uint32_t x = bx / pxsz, c = bx - x * pxsz;
    uint8_t* dst = reinterpret_cast<uint8_t*>(D.v.dst) + c;
    for (uint32_t y = Y0; y < min(Y0 + RV_ROWS, D.out_h); y++) {
        const int2 b = bounds[y];
        const int32_t* k = ky + (uint64_t)y * D.ky;
        const uint8_t* s = src + (uint64_t)b.x * pitch;
        int32_t acc = 1 << (RS_BITS - 1);
        for (int t = 0; t < b.y; t++) acc += __ldg(s + (uint64_t)t * pitch) * __ldg(k + t);
        dst[(D.v.last ? op_pixel(D.op, x, y, D.out_w, D.out_h) : (uint64_t)y * D.v.n + x) * pxsz] = clip8(acc);
    }
}

}  // namespace xpb
