// tensor.cuh — tensor decode: each decoded (cropped, resized) entry written through its op as a (C, H, W) or (H, W, C)
// tensor of uint8, float32, float16 or bfloat16, bit-identical to torchvision's to_tensor / ToDtype(scale=True) followed
// by Normalize (include/xpng_b200.h, xpngb_decode_tensor).
//
// One launch per chunk, every entry of the chunk in it.  A CTA takes one TT x TT patch of an entry's SOURCE pixels (its crop
// in a decode window or a stored file, or its resized pixels in scratch): it stages the patch's bytes in shared memory as
// aligned 32-bit words (any source alignment and pitch), then writes the patch's image under the op, coalesced along the
// destination's x: per channel plane for CHW, rows of C * width contiguous elements for HWC.  The CTA finds its entry by
// binary search over first_cta, as k_orient does.
//
// The arithmetic is one function, tensor_value, written with __fdiv_rn / __fmul_rn / __fsub_rn so that no build flag can
// contract b * (1/255) - mean into one FMA or approximate a division: each operation is rounded on its own, as torch does.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include "../../include/xpng_b200.h"
#include "common.cuh"
#include "orient.cuh"

namespace xpb {

constexpr int TT = 64;                          // patch edge in source pixels
constexpr int TT_PITCH = 67;                    // words per staged row: 64 RGBA pixels + 3 bytes of misalignment; odd, so that
                                                // reading down a column (quarter turns) hits 32 different banks

struct TensorDesc {
    uint64_t src, src_pitch, dst;   // device addresses: source rectangle (rows src_pitch bytes apart), the entry's tensor
    uint32_t w, h;                  // SOURCE dimensions (before the op)
    uint32_t pxsz, c, op;           // source bytes per pixel, output channels (3, or pxsz), XPNGB_OP_*
    uint32_t tiles_x, first_cta;    // patches per source row; index of this entry's first CTA in the launch
};

// Element of channel c for byte b: xpngb_decode_tensor's arithmetic contract, every float operation rounded on its own.
__device__ __forceinline__ float tensor_value(uint32_t b, const xpngb_tensor& f, uint32_t c) {
    const float mean = c == 0 ? f.mean[0] : c == 1 ? f.mean[1] : c == 2 ? f.mean[2] : f.mean[3];
    const float std = c == 0 ? f.std[0] : c == 1 ? f.std[1] : c == 2 ? f.std[2] : f.std[3];
    const float v = f.scale == XPNGB_SCALE_DIV ? __fdiv_rn((float)b, 255.0f) : __fmul_rn((float)b, (float)(1.0 / 255));
    return __fdiv_rn(__fsub_rn(v, mean), std);
}
template <typename T> __device__ __forceinline__ T tensor_elem(uint32_t b, const xpngb_tensor& f, uint32_t c);
template <> __device__ __forceinline__ uint8_t tensor_elem<uint8_t>(uint32_t b, const xpngb_tensor&, uint32_t) { return (uint8_t)b; }
template <> __device__ __forceinline__ float tensor_elem<float>(uint32_t b, const xpngb_tensor& f, uint32_t c) { return tensor_value(b, f, c); }
template <> __device__ __forceinline__ __half tensor_elem<__half>(uint32_t b, const xpngb_tensor& f, uint32_t c) {
    return __float2half_rn(tensor_value(b, f, c));
}
template <> __device__ __forceinline__ __nv_bfloat16 tensor_elem<__nv_bfloat16>(uint32_t b, const xpngb_tensor& f, uint32_t c) {
    return __float2bfloat16_rn(tensor_value(b, f, c));
}

// Writes the staged patch (source origin x0, y0; tw x th pixels; byte (lx, ly, c) at smb[ly * TT_PITCH * 4 + sh + lx * pxsz + c])
// into the entry's tensor under the op.  The destination patch is dw x dh at (DX0, DY0) of the W2 x H2 output.
template <typename T>
__device__ __forceinline__ void tensor_write(const TensorDesc& D, const xpngb_tensor& f, const uint8_t* smb, uint32_t sh,
                                             uint32_t x0, uint32_t y0, uint32_t tw, uint32_t th) {
    const uint32_t op = D.op, pxsz = D.pxsz, C = D.c;
    const bool quarter = op == XPNGB_OP_R90 || op == XPNGB_OP_R270;
    const uint32_t W2 = quarter ? D.h : D.w, H2 = quarter ? D.w : D.h;
    const uint32_t dw = quarter ? th : tw, dh = quarter ? tw : th;
    const bool fy = op == XPNGB_OP_MV || op == XPNGB_OP_MVH, fx = op == XPNGB_OP_MH || op == XPNGB_OP_MVH;
    uint32_t DX0, DY0;
    if (op == XPNGB_OP_R90) { DX0 = D.h - (y0 + th); DY0 = x0; }
    else if (op == XPNGB_OP_R270) { DX0 = y0; DY0 = D.w - (x0 + tw); }
    else { DX0 = fx ? D.w - (x0 + tw) : x0; DY0 = fy ? D.h - (y0 + th) : y0; }
    // source byte of destination-patch pixel (dx, dy), channel 0
    auto at = [&](uint32_t dx, uint32_t dy) -> uint32_t {
        uint32_t lx, ly;
        if (op == XPNGB_OP_R90) { lx = dy; ly = th - 1 - dx; }
        else if (op == XPNGB_OP_R270) { lx = tw - 1 - dy; ly = dx; }
        else { lx = fx ? tw - 1 - dx : dx; ly = fy ? th - 1 - dy : dy; }
        return ly * (TT_PITCH * 4) + sh + lx * pxsz;
    };
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
    T* dst = reinterpret_cast<T*>(D.dst);
    if (f.layout == XPNGB_CHW) {   // one destination row of one channel plane per warp, lanes along x
        const uint64_t plane = (uint64_t)W2 * H2;
        for (uint32_t row = warp; row < C * dh; row += nwarp) {
            const uint32_t c = row / dh, dy = row - c * dh;
            T* out = dst + c * plane + (uint64_t)(DY0 + dy) * W2 + DX0;
            for (uint32_t dx = lane; dx < dw; dx += 32) out[dx] = tensor_elem<T>(smb[at(dx, dy) + c], f, c);
        }
    } else {                       // one destination row per warp: C * dw contiguous elements
        for (uint32_t dy = warp; dy < dh; dy += nwarp) {
            T* out = dst + ((uint64_t)(DY0 + dy) * W2 + DX0) * C;
            for (uint32_t e = lane; e < C * dw; e += 32) {
                const uint32_t dx = e / C, c = e - dx * C;
                out[e] = tensor_elem<T>(smb[at(dx, dy) + c], f, c);
            }
        }
    }
}

__global__ void __launch_bounds__(256) k_to_tensor(const TensorDesc* __restrict__ descs, uint32_t n, const xpngb_tensor f) {
    __shared__ uint32_t sm[TT * TT_PITCH];
    uint32_t lo = 0, hi = n - 1;
    while (lo < hi) { const uint32_t mid = (lo + hi + 1) >> 1; if (descs[mid].first_cta <= blockIdx.x) lo = mid; else hi = mid - 1; }
    const TensorDesc D = descs[lo];
    const uint32_t patch = blockIdx.x - D.first_cta;
    const uint32_t x0 = (patch % D.tiles_x) * TT, y0 = (patch / D.tiles_x) * TT;
    const uint32_t tw = min((uint32_t)TT, D.w - x0), th = min((uint32_t)TT, D.h - y0);
    // Every staged row starts at byte sh0 of its shared-memory row.  A source row whose first byte has that alignment too
    // (every row when the pitch is a multiple of 4) is staged by aligned words, any other (stored files with odd pitches)
    // byte by byte.
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
    const uint64_t a0 = D.src + (uint64_t)y0 * D.src_pitch + (uint64_t)x0 * D.pxsz;
    const uint32_t sh0 = (uint32_t)(a0 & 3);
    for (uint32_t r = warp; r < th; r += nwarp) {
        const uint64_t a = a0 + (uint64_t)r * D.src_pitch, aw = a & ~3ull;
        const uint32_t sh = (uint32_t)(a - aw), nw = (sh + tw * D.pxsz + 3) >> 2;
        const uint32_t* s = reinterpret_cast<const uint32_t*>(aw);
        uint8_t* row = reinterpret_cast<uint8_t*>(sm + r * TT_PITCH);
        if (sh == sh0) { for (uint32_t j = lane; j < nw; j += 32) sm[r * TT_PITCH + j] = __ldg(s + j); }
        else {
            const uint8_t* sb = reinterpret_cast<const uint8_t*>(a);
            for (uint32_t j = lane; j < tw * D.pxsz; j += 32) row[sh0 + j] = __ldg(sb + j);
        }
    }
    __syncthreads();
    const uint8_t* smb = reinterpret_cast<const uint8_t*>(sm);
    switch (f.dtype) {
        case XPNGB_DT_U8: tensor_write<uint8_t>(D, f, smb, sh0, x0, y0, tw, th); break;
        case XPNGB_DT_F32: tensor_write<float>(D, f, smb, sh0, x0, y0, tw, th); break;
        case XPNGB_DT_F16: tensor_write<__half>(D, f, smb, sh0, x0, y0, tw, th); break;
        default: tensor_write<__nv_bfloat16>(D, f, smb, sh0, x0, y0, tw, th); break;
    }
}

}  // namespace xpb
