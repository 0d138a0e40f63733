// region.cuh — region decode: the rectangle of each image is copied out of the tiles that hold it (or, for stored level-7
// files, straight out of the file) into a packed crop.  The tile chains themselves are the unchanged decode kernels,
// driven by a plan that lists only the selected tiles (api.cu, xpngb_decode_region).
#pragma once
#include "common.cuh"

namespace xpb {

// One crop: `rows` rows of `row_bytes` bytes, row k read at src + k * pitch and written packed at dst + k * row_bytes.
// Neither the source column offset nor the destination row starts are aligned; dst itself is 16-byte aligned.
struct CropDesc {
    uint64_t src, dst;   // absolute device addresses
    uint64_t pitch;
    uint32_t row_bytes, rows;
};

// grid = (row blocks, crops), 256 threads: one warp per row.  Each lane writes whole 16-byte words of the destination row,
// built by funnel shifts from the aligned 32-bit source words that hold their bytes (as ld_rgb4); the unaligned head and
// tail bytes of the row (at most 15 each) go byte by byte.  Only source words that hold a byte of the row are read.
__global__ void __launch_bounds__(256) k_crop_rows(const CropDesc* __restrict__ crops) {
    const CropDesc c = crops[blockIdx.y];
    const uint32_t lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    for (uint32_t k = blockIdx.x * wpb + (threadIdx.x >> 5); k < c.rows; k += gridDim.x * wpb) {
        const uint8_t* src = reinterpret_cast<const uint8_t*>(c.src + (uint64_t)k * c.pitch);
        uint8_t* dst = reinterpret_cast<uint8_t*>(c.dst + (uint64_t)k * c.row_bytes);
        const uint32_t head = min((uint32_t)(-reinterpret_cast<uintptr_t>(dst) & 15u), c.row_bytes);
        const uint32_t nbody = (c.row_bytes - head) >> 4, tail0 = head + (nbody << 4);
        if (lane < head) dst[lane] = __ldg(src + lane);
        if (tail0 + lane < c.row_bytes) dst[tail0 + lane] = __ldg(src + tail0 + lane);
        for (uint32_t j = lane; j < nbody; j += 32) {
            const uintptr_t a = reinterpret_cast<uintptr_t>(src + head + (j << 4));
            const uint32_t* q = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
            const uint32_t sh = (uint32_t)(a & 3u) * 8u;
            const uint32_t a0 = __ldg(q), a1 = __ldg(q + 1), a2 = __ldg(q + 2), a3 = __ldg(q + 3), a4 = sh ? __ldg(q + 4) : 0u;
            uint4 v;
            v.x = __funnelshift_r(a0, a1, sh); v.y = __funnelshift_r(a1, a2, sh);
            v.z = __funnelshift_r(a2, a3, sh); v.w = __funnelshift_r(a3, a4, sh);
            *reinterpret_cast<uint4*>(dst + head + (j << 4)) = v;
        }
    }
}

}  // namespace xpb
