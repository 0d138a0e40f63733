// enc_m2.cuh — level-2 encode specifics: tile classification (single colour / grey / RGB,
// libxpng.c:628-643, :583-626), grey candidate planes, backward 2-state rANS with v1 blocks
// (libxpng.c:160-260), the shared side bit stream, size decisions and assembly (libxpng.c:645-686).
#pragma once
#include "common.cuh"
#include "enc_front.cuh"
#include "enc_back.cuh"

namespace xpb {

// ------------------------------------------------------------------------------------------------
// Tile classification.  One CTA per tile.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_m2_classify(const TileDesc* __restrict__ tiles, const ImageDesc* __restrict__ imgs,
                                                     uint8_t* __restrict__ tclass) {
    const uint32_t tile = blockIdx.x;
    const TileDesc t = tiles[tile];
    if (imgs[t.img].mode != 2) { if (threadIdx.x == 0) tclass[tile] = TC_NONE; return; }
    const uint8_t* src = reinterpret_cast<const uint8_t*>(t.src_off);
    const uint32_t f0 = src[0], f1 = src[1], f2 = src[2];
    int single = 1, grey = 1;
    const uint32_t first = f0 | (f1 << 8) | (f2 << 16), wq = 3 * t.w >= 16 ? (3 * t.w - 16) / 12 + 1 : 0;   // 16-byte windows inside the row
    for (uint32_t y = threadIdx.x >> 5; y < t.h; y += 8) {
        if (!__any_sync(0xffffffffu, single | grey)) break;              // this warp has seen a pixel that rules out both classes: the tile is RGB
        const uint8_t* row = src + (uint64_t)y * t.bpr;
        for (uint32_t g = threadIdx.x & 31; g < wq; g += 32) {           // four pixels per lane and iteration (ld_rgb4)
            uint32_t v[4]; ld_rgb4(row + 12 * g, v);
#pragma unroll
            for (int k = 0; k < 4; k++) { single &= v[k] == first; grey &= v[k] == (v[k] & 0xFFu) * 0x010101u; }
        }
        for (uint32_t x = (wq << 2) + (threadIdx.x & 31); x < t.w; x += 32) {
            const uint32_t a = row[3 * x], b = row[3 * x + 1], c = row[3 * x + 2];
            single &= (a == f0) & (b == f1) & (c == f2);
            grey &= (a == b) & (b == c);
        }
    }
    single = __syncthreads_and(single);
    grey = __syncthreads_and(grey);
    if (threadIdx.x == 0) tclass[tile] = single ? TC_SINGLE : (grey ? TC_GREY : TC_RGB);
}

// tile_skip[tile] = 1 unless the tile takes the RGB path
__global__ void k_m2_skipmask(const uint8_t* __restrict__ tclass, uint8_t* __restrict__ skip, uint32_t ntiles) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < ntiles) skip[i] = tclass[i] != TC_RGB;
}

// ------------------------------------------------------------------------------------------------
// Grey tiles: four candidate residual planes (left, up, avg2, grad3; row 0 left, column 0 up) and
// their 256-bin histograms (libxpng.c:597-604).  One CTA per segment.
// ------------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t grey_plane_pitch(uint32_t npx) { return (npx + 15u) & ~15u; }

__global__ void __launch_bounds__(256) k_m2_grey_front(const TileDesc* __restrict__ tiles, const uint32_t* __restrict__ seg_tile,
                                                       const uint8_t* __restrict__ tclass, uint8_t* __restrict__ streams,
                                                       uint32_t* __restrict__ hist) {
    __shared__ uint32_t sh[4 * 256];
    const uint32_t gseg = blockIdx.x, tile = seg_tile[gseg], tid = threadIdx.x;
    if (tclass[tile] != TC_GREY) return;
    const TileDesc t = tiles[tile];
    for (int k = tid; k < 1024; k += 256) sh[k] = 0;
    __syncthreads();
    const uint32_t r0 = (gseg - t.seg0) * SEG, r1 = min(r0 + (uint32_t)SEG, t.npx);
    const uint8_t* src = reinterpret_cast<const uint8_t*>(t.src_off);
    uint8_t* planes = streams + t.str_off;
    const uint32_t pitch = grey_plane_pitch(t.npx);
    for (uint32_t i = r0 + tid; i < r1; i += 256) {
        if (i == 0) continue;
        const uint32_t y = i / t.w, x = i - y * t.w;
        const uint8_t* p = src + (uint64_t)y * t.bpr + 3ull * x;
        const int v = p[0];
        int c[4];
        if (y == 0) c[0] = c[1] = c[2] = c[3] = v - p[-3];
        else if (x == 0) c[0] = c[1] = c[2] = c[3] = v - p[-(int64_t)t.bpr];
        else {
            const int L = p[-3], U = p[-(int64_t)t.bpr], UL = p[-(int64_t)t.bpr - 3];
            c[0] = v - L; c[1] = v - U; c[2] = v - pred_avg2(L, U); c[3] = v - pred_grad3(L, U, UL);
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t u = zz8(c[k]);
            planes[(uint64_t)k * pitch + i - 1] = (uint8_t)u;
            atomicAdd(&sh[k * 256 + u], 1u);
        }
    }
    __syncthreads();
    for (int k = tid; k < 1024; k += 256) { const uint32_t v = sh[k]; if (v) atomicAdd(hist + (uint64_t)tile * HIST_STRIDE_M2 + k, v); }
}

// ------------------------------------------------------------------------------------------------
// v1 blocks (libxpng.c:160-260; encoder k_rans_v1_pair, enc_rans_lat.cuh): symbols are consumed from the
// END of the stream, the renormalisation words are stored at descending addresses, so the finished block
// [hdr][n][state0][state1][words] sits at the end of the stream's scratch region.  The frequency
// table (or the raw symbols of a type-2 block) is a separate bit-string "piece" that k_assemble_m2
// splices into the tile's shared side stream.
// Stream numbering: RGB tile c = 0..8 contexts (9 symbols), 9..16 values of nl = 1..8; grey tile
// c = 0..3 candidate planes (256 symbols, PB 15).
// ------------------------------------------------------------------------------------------------
constexpr int TAB_WORDS = 136;   // 256 symbols x 16 bits = 128 words (+ slack)

struct RansV1Args {
    const TileDesc* tiles;
    TileState* state;
    const uint32_t* hist;
    const uint8_t* tclass;
    const uint8_t* streams;
    uint8_t* blocks;
    uint32_t* tabs;            // [ntiles][17][TAB_WORDS]
    uint32_t ntiles;
    uint32_t c0, nc;
    uint32_t grey;             // 1: grey candidates, 0: RGB streams
    uint32_t nmin;             // skip alphabets of <= nmin symbols (done by the launch with the smaller table)
    const uint32_t* order = nullptr; const uint32_t* total = nullptr;   // pair encoders: sorted work list instead of the id range
};

__device__ __constant__ const uint16_t M2_NSYM[17] = { 9, 9, 9, 9, 9, 9, 9, 9, 9, 8, 64, 8, 16, 32, 64, 128, 256 };

// ------------------------------------------------------------------------------------------------
// Per-tile size decisions (libxpng.c:606-626, :672-678).  One thread per tile.
// ------------------------------------------------------------------------------------------------
__global__ void k_m2_finish(const TileDesc* __restrict__ tiles, const uint8_t* __restrict__ tclass, TileState* __restrict__ state,
                            uint32_t ntiles) {
    const uint32_t tile = blockIdx.x * blockDim.x + threadIdx.x;
    if (tile >= ntiles) return;
    const TileDesc t = tiles[tile];
    TileState* st = state + tile;
    const uint8_t cls = tclass[tile];
    if (cls == TC_NONE) return;
    if (cls == TC_SINGLE) { st->kind = 3; st->size = 8; return; }
    if (cls == TC_GREY) {
        uint32_t best = 0, bb = 0, br = 0;
        for (uint32_t i = 0; i < 4; i++) {
            const uint32_t bsz = 4 + ((8 + st->pbits[i] + 31) / 32) * 4, rsz = st->bsize[i];
            if (i == 0 || bsz + rsz < bb + br) { best = i; bb = bsz; br = rsz; }          // strict <, ties to the lowest
        }
        if (bb + br >= t.npx) { st->kind = 5; st->size = t.npx + 4; }
        else { st->kind = 4; st->size = bb + br + 4; st->grey_pick = best; }
        return;
    }
    uint32_t bit = 24, rsz = 0;
    for (int c = 0; c < 17; c++) { st->pbo[c] = bit; bit += st->pbits[c]; rsz += st->bsize[c]; }
    st->kbits_lo = bit; st->kbits_hi = 0;
    const uint32_t bsz = 4 + ((bit + 31) / 32) * 4;
    if ((uint64_t)bsz + rsz >= 3ull * t.npx) { st->kind = 0; st->size = 3 * t.npx + 4; }
    else { st->kind = 2; st->size = bsz + rsz + 4; }
}

// ------------------------------------------------------------------------------------------------
// Assembly, level 2.  One CTA per tile.
// ------------------------------------------------------------------------------------------------
struct AssembleM2Args {
    AssembleArgs a;
    const uint8_t* tclass;
    const uint32_t* tabs;
    const uint8_t* streams;
};

__global__ void __launch_bounds__(256) k_assemble_m2(AssembleM2Args M) {
    __shared__ uint64_t sbit[18];
    __shared__ uint32_t snb[18];
    __shared__ const uint32_t* sptr[18];
    __shared__ uint32_t fpw;
    const AssembleArgs& A = M.a;
    const uint32_t tile = blockIdx.x, tid = threadIdx.x;
    const TileDesc t = A.tiles[tile];
    const ImageDesc I = A.imgs[t.img];
    const ImageOut O = A.outs[t.img];
    const TileState* st = A.state + tile;
    uint8_t* file = A.out + O.off;
    const uint8_t* src = A.px + t.src_off;
    const uint32_t part = blockIdx.y, nparts = gridDim.y;        // RGB tiles: the side-stream gather and the 17 block copies are sliced over gridDim.y CTAs
    if (part && ((O.mode & 0x100) || (O.mode & 0xFF) == 7 || st->kind != 2)) return;
    if (assemble_common(t, I, O, file, src)) return;
    uint8_t* blob = file + st->out_off;
    const uint8_t* bsrc = A.blocks + t.blk_off;
    switch (st->kind) {
    case 0:   // raw tile (libxpng.c:675-677)
        if (tid == 0) st32u(blob, st->size);
        copy_tile_rows(blob + 4, (uint64_t)t.w * 3, src, t);
        return;
    case 3:   // single colour (libxpng.c:637-640)
        if (tid == 0) { st32u(blob, (255u << 24) | 8u); blob[4] = src[0]; blob[5] = src[1]; blob[6] = src[2]; blob[7] = 0; }
        return;
    case 5:   // raw grey plane (libxpng.c:615-619)
        if (tid == 0) st32u(blob, st->size + (5u << 27));
        for (uint32_t y = tid >> 5; y < t.h; y += 8)
            for (uint32_t x = tid & 31; x < t.w; x += 32) blob[4 + (uint64_t)y * t.w + x] = src[(uint64_t)y * t.bpr + 3ull * x];
        return;
    case 4: { // grey, one v1 block (libxpng.c:622-624)
        const uint32_t g = st->grey_pick;
        const uint32_t bits = 8 + st->pbits[g], words = (bits + 31) / 32;
        if (tid == 0) {
            st32u(blob, st->size + (2u << 28) + (g << 24)); st32u(blob + 4, 4 + 4 * words);
            fpw = (uint32_t)src[0] << 24;
            sbit[0] = 0; snb[0] = 8; sptr[0] = &fpw;
            sbit[1] = 8; snb[1] = st->pbits[g];
            sptr[1] = st->btype[g] == 2 ? reinterpret_cast<const uint32_t*>(bsrc + st->breg[g]) : M.tabs + ((uint64_t)tile * 17 + g) * TAB_WORDS;
        }
        __syncthreads();
        for (uint32_t wi = tid; wi < words; wi += 256) st32u(blob + 8 + 4ull * wi, gather_word(wi, 2, sbit, snb, sptr));
        copy_bytes(blob + 8 + 4ull * words, bsrc + st->boff[g], st->bsize[g]);
        return;
    }
    default: break;
    }
    // RGB: [hdr][bsz][shared side stream][9 context blocks][8 value blocks]   (libxpng.c:680-683)
    const uint32_t bits = st->kbits_lo, words = (bits + 31) / 32;
    if (tid == 0) {
        if (part == 0) { st32u(blob, st->size + (1u << 28) + (st->pr << 24)); st32u(blob + 4, 4 + 4 * words); }
        fpw = ((uint32_t)src[0] << 24) | ((uint32_t)src[1] << 16) | ((uint32_t)src[2] << 8);
        sbit[0] = 0; snb[0] = 24; sptr[0] = &fpw;
    }
    if (tid < 17) {
        sbit[tid + 1] = st->pbo[tid]; snb[tid + 1] = st->pbits[tid];
        sptr[tid + 1] = st->btype[tid] == 2 ? reinterpret_cast<const uint32_t*>(bsrc + st->breg[tid]) : M.tabs + ((uint64_t)tile * 17 + tid) * TAB_WORDS;
    }
    __syncthreads();
    for (uint32_t wi = part * 256 + tid; wi < words; wi += 256 * nparts) st32u(blob + 8 + 4ull * wi, gather_word(wi, 18, sbit, snb, sptr));
    uint8_t* dst = blob + 8 + 4ull * words;
    for (int c = 0; c < 17; c++) { copy_bytes_part(dst, bsrc + st->boff[c], st->bsize[c], part, nparts); dst += st->bsize[c]; }
}

}  // namespace xpb
