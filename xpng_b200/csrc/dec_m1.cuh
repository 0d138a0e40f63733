// dec_m1.cuh — level-1 decode: tile offsets, block parsing, v2 rANS decode (libxpng.c:429-493),
// alpha plane, context walk (nl = *cx[nl]++, libxpng.c:803), row prefix tables and the wavefront
// un-predict (libxpng.c:796-830).  Also the stored (level 7) and raw-tile copies.
#pragma once
#include "common.cuh"

namespace xpb {

enum DecErr { DEC_OK = 0, DEC_BAD_TILE_CHAIN = 1, DEC_BAD_BLOCK = 2, DEC_BAD_COUNTS = 3, DEC_BAD_HEADER = 4 };

struct DecImage {
    uint64_t file_off, file_size;   // inside the input buffer
    uint64_t px_off;                // output pixel offset
    uint32_t w, h, pxsz, mode;      // mode: 1, 2, 7; 0x100 = whole-image single colour
    uint32_t tile0, ntiles;         // planned (selected) tiles: DecTile tile0 + (row - r0) * ncols + (col - c0)
    uint32_t gcols;                 // tile columns of the image's grid
    uint32_t r0, c0, nrows, ncols;  // selected tile rows [r0, r0 + nrows) and columns [c0, c0 + ncols): the whole grid for a full decode
    uint32_t pad;
};

struct DecBlock { uint32_t off; uint32_t n; uint32_t type; uint32_t soff; };   // off: from blob start; soff: in stream slice

struct DecTile {
    uint64_t blob_off;       // inside the input buffer
    uint32_t size, m;        // blob size, tile type byte
    uint32_t bsz;            // side/residual bit stream bytes incl. its size word
    uint32_t nsym;           // total context symbols (coded pixels - 1 + ... ) = sum n[0..8]
    DecBlock blk[MAX_STREAMS];
    uint32_t bitpos[MAX_STREAMS];   // mode 2: bit offset of each block's table / raw symbols in the shared stream
    uint32_t pad[2];
};

__device__ __forceinline__ void dec_fail(int* err, int code) { atomicCAS(err, 0, code); }
__host__ __device__ __forceinline__ uint32_t align16u_dec(uint32_t v) { return (v + 15u) & ~15u; }

// ------------------------------------------------------------------------------------------------
// Tile offsets: serial chain over the 24-bit tile sizes of one image (libxpng.c:982).  The chain is walked from the
// first tile with the same checks for every tile; only the selected tiles get a DecTile, and the walk ends after the
// last selected row (a region decode reads nothing of the tiles it skips but their size words).
// ------------------------------------------------------------------------------------------------
__global__ void k_dec_tile_offsets(const DecImage* imgs, const uint8_t* in, DecTile* dt, uint32_t nimg, int* err) {
    const uint32_t im = blockIdx.x * blockDim.x + threadIdx.x;
    if (im >= nimg) return;
    const DecImage I = imgs[im];
    if ((I.mode & 0xFF) == 7 || (I.mode & 0x100)) return;
    uint64_t off = 8;
    const uint32_t rend = I.r0 + I.nrows;
    for (uint32_t row = 0, col = 0; row < rend;) {
        DecTile* d = (row >= I.r0 && col - I.c0 < I.ncols) ? dt + I.tile0 + (row - I.r0) * I.ncols + (col - I.c0) : nullptr;
        if (++col == I.gcols) { col = 0; row++; }
        if (off + 4 > I.file_size) { dec_fail(err, DEC_BAD_TILE_CHAIN); if (d) { d->size = 0; d->m = 0xFE; d->blob_off = I.file_off; } continue; }
        const uint32_t w0 = ld32u(in + I.file_off + off);
        const uint32_t size = w0 & 0xFFFFFFu;
        const bool bad = size < 4 || off + size > I.file_size;
        if (bad) dec_fail(err, DEC_BAD_TILE_CHAIN);
        if (d) { d->blob_off = I.file_off + off; d->size = size; d->m = bad ? 0xFE : w0 >> 24; }
        off += size < 4 ? 4 : size;
    }
}

// ------------------------------------------------------------------------------------------------
// Level-1 tile parse: bit-stream size, the 9 (10) v2 block headers, stream offsets.
// ------------------------------------------------------------------------------------------------
__global__ void k_dec_parse_m1(const TileDesc* tiles, const DecImage* imgs, const uint8_t* in, DecTile* dt, uint32_t ntiles, int* err) {
    const uint32_t tile = blockIdx.x * blockDim.x + threadIdx.x;
    if (tile >= ntiles) return;
    const TileDesc t = tiles[tile];
    const DecImage I = imgs[t.img];
    if (I.mode != 1) return;
    DecTile* d = dt + tile;
    if (d->m == 0xFE) return;
    if (d->m == 0) { if (d->size != t.npx * t.pxsz + 4) { dec_fail(err, DEC_BAD_TILE_CHAIN); d->m = 0xFE; } return; }
    const uint8_t* blob = in + d->blob_off;
    const int nblk = t.pxsz == 4 ? 10 : 9;
    bool bad = d->size < 8 || (d->m >> 4) != 1 || (((d->m >> 2) & 1) != (t.pxsz == 4));
    uint32_t bsz = bad ? 4 : ld32u(blob + 4);
    if (bsz < 4 || (uint64_t)4 + bsz > d->size) bad = true;
    uint32_t off = 4 + bsz, soff = 0, nsym = 0;
    for (int c = 0; c < nblk && !bad; c++) {
        if (off + 4 > d->size) { bad = true; break; }
        const uint32_t w0 = ld32u(blob + off), type = w0 >> 24;
        uint32_t csz = w0 & 0xFFFFFFu, n = 0;
        if (type == 0) csz = 4;
        else {
            if (type > 4 || csz < 8 || off + csz > d->size) { bad = true; break; }
            n = ld32u(blob + off + 4) & 0xFFFFFFu;
            if (type >= 3 && csz < 28) { bad = true; break; }
        }
        if (c < 9) { nsym += n; if (nsym > t.npx) { bad = true; break; } }
        else if (n != t.npx - 1) { bad = true; break; }
        d->blk[c] = DecBlock{ off, n, type, c < 9 ? soff : 0u };
        if (c < 9) soff += align16u_dec(n);
        off += csz;
    }
    if (!bad && t.pxsz == 3 && nsym != t.npx - 1) bad = true;
    if (bad) { dec_fail(err, DEC_BAD_BLOCK); d->m = 0xFE; return; }
    d->bsz = bsz; d->nsym = nsym;
}

// ------------------------------------------------------------------------------------------------
// Entropy blocks: the bit reader of block headers and frequency tables, and the argument block of
// the level-1 rANS decoder (k_dec_rans_v2_lat, dec_rans_lat.cuh).
// ------------------------------------------------------------------------------------------------
struct BitR {   // MSB-first reader over unaligned LE words; zero past `end` (libxpng.c:12)
    const uint8_t* base; const uint8_t* end; uint32_t pos;
    __device__ __forceinline__ uint32_t get(uint32_t c) {
        uint32_t v = 0;
        while (c) {
            const uint32_t off = pos & 31u; uint32_t take = 32u - off; if (take > c) take = c;
            const uint8_t* p = base + 4ull * (pos >> 5);
            const uint32_t word = (p + 4 <= end) ? ld32u(p) : 0u;
            const uint32_t bits = (word >> (32u - off - take)) & (take == 32u ? 0xFFFFFFFFu : ((1u << take) - 1u));
            v = take == 32u ? bits : ((v << take) | bits);
            pos += take; c -= take;
        }
        return v;
    }
};

struct RansDecArgs {
    const TileDesc* tiles;
    const DecImage* imgs;
    const DecTile* dt;
    const uint8_t* in;
    uint8_t* streams;     // ctx streams at stream_slice
    uint8_t* alpha;       // alpha symbols at px_off
    uint32_t ntiles;
    uint32_t c0, nc;
    int* err;
};

// ------------------------------------------------------------------------------------------------
// Context walk: nl_{i+1} = next unread symbol of stream nl_i.  Inherently serial per tile; the kernels
// (k_dec_walk_smem, k_dec_walk_ring in dec_rans_lat.cuh, k_dec_walk3 in dec_walk3.cuh) take this argument block.
// ------------------------------------------------------------------------------------------------
struct WalkArgs {
    const TileDesc* tiles;
    const DecImage* imgs;
    const DecTile* dt;
    const uint8_t* streams;
    uint8_t* nlseq;          // per tile at px_off: nl of every coded pixel in raster order
    uint32_t ntiles;
    uint32_t mode;
};

// ------------------------------------------------------------------------------------------------
// Alpha plane (RGBA): un-zig-zag + prefix sums (column 0 down, then along each row), per-row counts
// of coded (alpha != 0) pixels.  One CTA per tile.
// ------------------------------------------------------------------------------------------------
struct RowInfo { uint32_t idx; uint32_t bit; };   // per tile row: index into nlseq and bit offset of its first coded pixel

struct AlphaArgs {
    const TileDesc* tiles;
    const DecImage* imgs;
    const DecTile* dt;
    const uint8_t* in;
    uint8_t* alpha;        // in: symbols (index raster-1) ; out: alpha plane values (index raster), in place via plane
    uint8_t* plane;        // alpha plane per tile at px_off (index raster)
    uint32_t* rowcnt;      // per tile row (at row_off): coded pixels in the row
};

__global__ void __launch_bounds__(256) k_dec_alpha(AlphaArgs A) {
    __shared__ uint32_t wsum[8];
    __shared__ uint32_t carry_s;
    const uint32_t tile = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const TileDesc t = A.tiles[tile];
    if (A.imgs[t.img].mode != 1 || t.pxsz != 4) return;
    const DecTile* d = A.dt + tile;
    if (d->m == 0 || d->m == 0xFE) return;
    const uint8_t* sym = A.alpha + t.px_off;     // symbol of raster r at sym[r-1]
    uint8_t* pl = A.plane + t.px_off;
    // The first pixel is stored as 32 bits MSB-first: R,G,B,A -> LE word bytes are A,B,G,R.
    const uint32_t fp = ld32u(A.in + d->blob_off + 8);
    const uint32_t alpha0 = fp & 0xFFu;
    // column 0: alpha(0,y) = alpha0 + sum_{yy<=y} unzz(sym[yy*w - 1])  (mod 256), block scan over rows
    if (tid == 0) carry_s = alpha0;
    __syncthreads();
    for (uint32_t y0 = 0; y0 < t.h; y0 += 256) {
        const uint32_t y = y0 + tid;
        int v = (y < t.h && y > 0) ? unzz(sym[(uint64_t)y * t.w - 1]) : 0;
        int inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int n = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += n; }
        if (lane == 31) wsum[wid] = (uint32_t)inc;
        __syncthreads();
        int pre = (int)carry_s;
        for (uint32_t k = 0; k < wid; k++) pre += (int)wsum[k];
        if (y < t.h) pl[(uint64_t)y * t.w] = (uint8_t)(pre + inc);
        __syncthreads();
        if (tid == 255) carry_s = (uint32_t)(pre + inc);
        __syncthreads();
    }
    // rows: warp per row, scan along x in chunks of 32
    for (uint32_t y = wid; y < t.h; y += 8) {
        int run = pl[(uint64_t)y * t.w];
        uint32_t cnt = 0;
        if (lane == 0 && run != 0 && y > 0) cnt = 1;   // (0,0) is never counted as a coded symbol
        for (uint32_t x0 = 1; x0 < t.w; x0 += 32) {
            const uint32_t x = x0 + lane;
            int v = x < t.w ? unzz(sym[(uint64_t)y * t.w + x - 1]) : 0;
            int inc = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int n = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += n; }
            const uint8_t a = (uint8_t)(run + inc);
            if (x < t.w) { pl[(uint64_t)y * t.w + x] = a; cnt += a != 0; }
            run += __shfl_sync(0xffffffffu, inc, 31);
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        if (lane == 0) A.rowcnt[t.row_off + y] = cnt;
    }
}

// ------------------------------------------------------------------------------------------------
// Copies: stored images (level 7), raw tiles (m = 0) and whole-image single colour.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_dec_copy(const TileDesc* tiles, const DecImage* imgs, const DecTile* dt, const uint8_t* in, uint8_t* px) {
    const uint32_t tile = blockIdx.x;
    const TileDesc t = tiles[tile];
    const DecImage I = imgs[t.img];
    uint8_t* dst = px + t.src_off;
    const uint32_t rowb = t.w * t.pxsz;
    if ((I.mode & 0xFF) == 7) return;   // stored images are copied by k_load7
    if (I.mode & 0x100) {   // libxpng.c:976-980
        const uint8_t* col = in + I.file_off + 8;
        for (uint32_t y = threadIdx.x >> 5; y < t.h; y += 8)
            for (uint32_t k = threadIdx.x & 31; k < rowb; k += 32) dst[(uint64_t)y * t.bpr + k] = col[k % t.pxsz];
        return;
    }
    const DecTile* d = dt + tile;
    if (d->m == 0) {        // libxpng.c:846
        const uint8_t* src = in + d->blob_off + 4;
        for (uint32_t y = threadIdx.x >> 5; y < t.h; y += 8)
            for (uint32_t k = threadIdx.x & 31; k < rowb; k += 32) dst[(uint64_t)y * t.bpr + k] = src[(uint64_t)y * rowb + k];
    } else if (d->m == 0xFF) {   // single-colour tile (level 2, libxpng.c:916-927)
        const uint8_t* col = in + d->blob_off + 4;
        for (uint32_t y = threadIdx.x >> 5; y < t.h; y += 8)
            for (uint32_t k = threadIdx.x & 31; k < rowb; k += 32) dst[(uint64_t)y * t.bpr + k] = col[k % 3];
    }
}

}  // namespace xpb
