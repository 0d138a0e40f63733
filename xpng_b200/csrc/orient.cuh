// orient.cuh — traversal-order operations of the exchange scheme (reference Mirroring_and_Rotating/tool.c:3-125):
// mirror vertical / horizontal / both, rotate by 90 and 270 degrees.  The reference rewrites the pixmap on the CPU
// (op_r90 is a cache-hostile scatter, tool.c:92-112); here every op is the same kernel: a 64x64-pixel patch of the
// SOURCE is read row by row (coalesced), parked in shared memory, and written row by row of the DESTINATION
// (coalesced again) through the op's index map, so a quarter turn costs the same as a mirror: one read and one write
// of the raw bytes.  `tl` and `tr` are empty functions in the reference (tool.c:121-127) and are plain copies here.
// The source is a rectangle with a row pitch of its own (a whole pixmap, a crop inside a decode window, or the rows of a
// stored file at any byte alignment); the destination is always packed.
#pragma once
#include "common.cuh"

enum { OP_R90 = 0, OP_R270 = 1, OP_MV = 2, OP_MH = 3, OP_MVH = 4, OP_TL = 5, OP_TR = 6 };   // order of tool.c:133
constexpr int ORI_T = 64;                      // patch edge in pixels

struct OrientDesc {
    uint64_t src, dst;      // device addresses: source rectangle, packed destination
    uint64_t src_pitch;     // bytes from one source row to the next (w * pxsz for a packed pixmap)
    uint32_t w, h;          // SOURCE dimensions
    uint32_t pxsz, op;
    uint32_t tiles_x, first_cta;   // patches per source row; index of this image's first CTA in the launch
};

// E = element type moved per access (u32 for RGBA when source, pitch and destination are word-aligned, else u8),
// EPP = elements per pixel
template <typename E, int EPP>
__device__ __forceinline__ void orient_patch(const OrientDesc& D, uint32_t patch, E* sm) {
    constexpr int PITCH = ORI_T * EPP + (EPP == 1 ? 1 : 4);   // bytes/4 odd in both cases: column reads hit 32 different banks
    const uint32_t x0 = (patch % D.tiles_x) * ORI_T, y0 = (patch / D.tiles_x) * ORI_T;
    const uint32_t tw = min((uint32_t)ORI_T, D.w - x0), th = min((uint32_t)ORI_T, D.h - y0);
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
    E* dst = reinterpret_cast<E*>(D.dst);
    for (uint32_t r = warp; r < th; r += nwarp) {
        const E* row = reinterpret_cast<const E*>(D.src + (uint64_t)(y0 + r) * D.src_pitch) + (uint64_t)x0 * EPP;
        for (uint32_t b = lane; b < tw * EPP; b += 32) sm[r * PITCH + b] = __ldg(row + b);
    }
    __syncthreads();
    const uint32_t op = D.op;
    if (op == OP_R90 || op == OP_R270) {
        // destination is h wide; one destination row per source column
        const uint64_t W2 = D.h;
        for (uint32_t c = warp; c < tw; c += nwarp) {
            const uint64_t Y = op == OP_R90 ? x0 + c : D.w - 1 - (x0 + c);
            const uint64_t X0 = op == OP_R90 ? D.h - (y0 + th) : y0;
            E* row = dst + (Y * W2 + X0) * EPP;
            for (uint32_t b = lane; b < th * EPP; b += 32) {
                const uint32_t dx = b / EPP, e = b - dx * EPP;
                const uint32_t ly = op == OP_R90 ? th - 1 - dx : dx;
                row[b] = sm[ly * PITCH + c * EPP + e];
            }
        }
    } else {
        const bool fy = op == OP_MV || op == OP_MVH, fx = op == OP_MH || op == OP_MVH;
        for (uint32_t r = warp; r < th; r += nwarp) {
            const uint64_t Y = fy ? D.h - 1 - (y0 + r) : y0 + r;
            const uint64_t X0 = fx ? D.w - (x0 + tw) : x0;
            E* row = dst + (Y * D.w + X0) * EPP;
            for (uint32_t b = lane; b < tw * EPP; b += 32) {
                const uint32_t dx = b / EPP, e = b - dx * EPP;
                const uint32_t lx = fx ? tw - 1 - dx : dx;
                row[b] = sm[r * PITCH + lx * EPP + e];
            }
        }
    }
}

// One CTA per 64x64 source patch; the CTA finds its image by binary search over first_cta.
__global__ void __launch_bounds__(256) k_orient(const OrientDesc* __restrict__ descs, uint32_t n) {
    __shared__ __align__(16) uint8_t sm[ORI_T * (ORI_T * 4 + 4)];
    uint32_t lo = 0, hi = n - 1;
    while (lo < hi) { const uint32_t mid = (lo + hi + 1) >> 1; if (descs[mid].first_cta <= blockIdx.x) lo = mid; else hi = mid - 1; }
    const OrientDesc D = descs[lo];
    const uint32_t patch = blockIdx.x - D.first_cta;
    if (D.pxsz == 3) orient_patch<uint8_t, 3>(D, patch, sm);
    else if (((D.src | D.src_pitch | D.dst) & 3) == 0) orient_patch<uint32_t, 1>(D, patch, reinterpret_cast<uint32_t*>(sm));
    else orient_patch<uint8_t, 4>(D, patch, sm);   // stored RGBA files at offsets that are not a multiple of 4
}
