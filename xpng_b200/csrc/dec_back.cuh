// dec_back.cuh — decode back end shared by levels 1 and 2, plus the level-2 tile parse (libxpng.c:868-961;
// the v1 rANS decoders, libxpng.c:262-301, are in dec_rans_lat.cuh and dec_rans_pair.cuh).
//   nl sequence  ->  per-chunk counts  ->  per-tile scan (bit / value offsets)  ->  residual plane
//   (one packed zig-zag triple per coded pixel)  ->  wavefront un-predict.
// Everything except the per-tile chunk scan and the wavefront itself is data-parallel.
#pragma once
#include "common.cuh"
#include "enc_front.cuh"   // Cnt9 helpers
#include "dec_m1.cuh"

namespace xpb {

// Level-2 alphabets (libxpng.c:951): contexts 9, then nl = 1..8 -> 8,64,8,16,32,64,128,256.
__device__ __constant__ const uint16_t DEC_M2_NSYM[17] = { 9, 9, 9, 9, 9, 9, 9, 9, 9, 8, 64, 8, 16, 32, 64, 128, 256 };

// ------------------------------------------------------------------------------------------------
// Level-2 tile parse: tile kind, the 17 (or 1) v1 block headers and where each block's frequency
// table / raw symbols start in the tile's shared side bit stream (type-4 tables are variable
// length, so the offsets form a short serial chain).  One thread per tile.
// ------------------------------------------------------------------------------------------------
__global__ void k_dec_parse_m2(const TileDesc* tiles, const DecImage* imgs, const uint8_t* in, DecTile* dt, uint32_t ntiles, int* err) {
    const uint32_t tile = blockIdx.x * blockDim.x + threadIdx.x;
    if (tile >= ntiles) return;
    const TileDesc t = tiles[tile];
    if (imgs[t.img].mode != 2) return;
    DecTile* d = dt + tile;
    if (d->m == 0xFE) return;
    const uint8_t* blob = in + d->blob_off;
    bool bad = false;
    if (d->m == 0) bad = d->size != t.npx * 3 + 4;
    else if (d->m == 0xFF) bad = d->size != 8;
    else if ((d->m >> 4) == 2 && (d->m & 8)) bad = d->size != t.npx + 4;
    else if ((d->m >> 4) == 2 || (d->m >> 4) == 1) {
        const bool grey = (d->m >> 4) == 2;
        const int nblk = grey ? 1 : 17, pb = grey ? 15 : 14;
        bad = d->size < 12;
        uint32_t bsz = bad ? 4 : ld32u(blob + 4);
        if (bsz < 4 || (uint64_t)4 + bsz > d->size) bad = true;
        const uint8_t* kend = blob + 4 + bsz;
        uint32_t off = 4 + bsz, bit = grey ? 8 : 24, soff = 0, nsym = 0, nval = 0;
        for (int c = 0; c < nblk && !bad; c++) {
            if (off + 4 > d->size) { bad = true; break; }
            const uint32_t N = grey ? 256u : (uint32_t)DEC_M2_NSYM[c], nbit = bitlen32(N - 1);
            const uint32_t w0 = ld32u(blob + off), type = w0 >> 24, bsize = w0 & 0xFFFFFFu;
            uint32_t n = 0;
            if (type > 4 || bsize < 4 || off + bsize > d->size || (type && bsize < 8) || (type >= 3 && bsize < 24)) { bad = true; break; }
            if (type) { n = ld32u(blob + off + 4); if (type == 1) n &= 0xFFFFFFu; }
            if (n > 3 * t.npx) { bad = true; break; }
            d->blk[c] = DecBlock{ off, n, type, soff };
            d->bitpos[c] = bit;
            if (type == 2) bit += nbit * n;
            else if (type == 3) bit += N * (uint32_t)pb;
            else if (type == 4) {
                BitR r{ blob + 8, kend, bit };
                for (uint32_t k = 0; k < N; k++) if (r.get(1)) r.pos += (uint32_t)pb;
                bit = r.pos;
            }
            soff += align16u_dec(n);
            if (c < 9) nsym += n;
            // the value blocks together hold at most three bytes per coded pixel: anything above that would run past the
            // tile's slice of the stream scratch ((align16(npx) + 256) * 4 bytes), so it is refused before any rANS kernel runs
            else { nval += n; if (nval > 3 * (t.npx - 1)) { bad = true; break; } }
            off += bsize;
        }
        if (!bad && nsym != t.npx - 1 && !grey) bad = true;
        if (!bad && grey && d->blk[0].n != t.npx - 1) bad = true;
        if (!bad && (uint64_t)bit > 8ull * (bsz - 4)) bad = true;
        if (!bad && (uint64_t)soff > ((uint64_t)align16u_dec(t.npx) + 256) * 4) bad = true;
        d->bsz = bsz; d->nsym = grey ? t.npx - 1 : nsym;
    } else bad = true;
    if (bad) { dec_fail(err, DEC_BAD_BLOCK); d->m = 0xFE; }
}

// ------------------------------------------------------------------------------------------------
// Chunk counts: how many coded pixels of each nl a 4096-entry chunk of the nl sequence holds.
// ------------------------------------------------------------------------------------------------
struct ChunkArgs {
    const TileDesc* tiles;
    const uint32_t* seg_tile;
    const DecImage* imgs;
    const DecTile* dt;
    const uint8_t* nlseq;
    const uint8_t* streams;
    const uint8_t* in;
    uint32_t* ccnt;      // [nseg][9] counts, then (after the scan) exclusive prefixes per nl
    uint32_t* cbit;      // [nseg] bit offset of the chunk's first residual (level 1)
    uint32_t* resv;      // residual plane per tile (resv_base): u0 | u1 << 8 | u2 << 16 per coded pixel
    uint32_t ntiles;
    int* err;
    uint32_t pitched;    // 1: RGB tiles that k_dec_unpredict_rgb takes get the row-pitched layout (tile_pitched)
};

// Residual plane of a tile.  Linear layout: entry k = k-th coded pixel (raster index k + 1 for RGB).  Row-pitched layout
// (batches, RGB tiles with word-aligned rows): pixel (x, y) at y * pitch + x, pitch = w rounded up to 4 words, so that a
// row starts 16-byte aligned and k_dec_unpredict_rgb fetches four residuals per load.  The base leaves 4 words per row
// of every earlier tile for the padding (px_off and row_off are running sums over the chunk's tiles).
__device__ __forceinline__ uint64_t resv_base(const TileDesc& t) { return t.px_off + 4ull * t.row_off; }
__host__ __device__ __forceinline__ bool tile_pitched(const TileDesc& t) {
    return t.pxsz == 3 && t.w <= 672u && ((t.src_off | t.bpr) & 3u) == 0;   // 672 = UNR_MAXW
}

__device__ __forceinline__ bool coded_tile(const DecTile* d) { return d->m != 0 && d->m < 0x20; }   // RGB entropy-coded tile

__global__ void __launch_bounds__(256) k_dec_chunk_hist(ChunkArgs A) {
    __shared__ Cnt9 wc[8];
    const uint32_t gseg = blockIdx.x, tile = A.seg_tile[gseg], tid = threadIdx.x;
    const TileDesc t = A.tiles[tile];
    const DecTile* d = A.dt + tile;
    if (A.imgs[t.img].mode == 7 || (A.imgs[t.img].mode & 0x100) || !coded_tile(d)) return;
    const uint32_t c0 = (gseg - t.seg0) * SEG;
    if (c0 >= d->nsym) return;
    const uint32_t c1 = min(c0 + (uint32_t)SEG, d->nsym);
    const uint8_t* seq = A.nlseq + t.px_off;
    Cnt9 cc{ 0, 0, 0 };
    const uint32_t e0 = c0 + tid * 16;
    if (e0 < c1) {
        const uint4 q = *reinterpret_cast<const uint4*>(seq + e0);
        const uint32_t w[4] = { q.x, q.y, q.z, q.w };
#pragma unroll
        for (int e = 0; e < 16; e++) if (e0 + e < c1) cnt9_inc(cc, (w[e >> 2] >> (8 * (e & 3))) & 0xFu);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        cc.a += __shfl_xor_sync(0xffffffffu, cc.a, o); cc.b += __shfl_xor_sync(0xffffffffu, cc.b, o); cc.c += __shfl_xor_sync(0xffffffffu, cc.c, o);
    }
    if ((tid & 31) == 0) wc[tid >> 5] = cc;
    __syncthreads();
    if (tid < 9) {
        uint32_t s = 0;
        for (int k = 0; k < 8; k++) s += cnt9_get(wc[k], tid);
        A.ccnt[(uint64_t)gseg * 9 + tid] = s;
    }
}

// Per-tile exclusive scan of the chunk counts (warp per tile, lane c = nl value).  Also checks the
// totals against what the bit stream / value streams actually hold.
__global__ void __launch_bounds__(128) k_dec_chunk_scan(ChunkArgs A) {
    const uint32_t tile = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (tile >= A.ntiles) return;
    const TileDesc t = A.tiles[tile];
    const DecTile* d = A.dt + tile;
    const uint32_t mode = A.imgs[t.img].mode;
    if (mode == 7 || (mode & 0x100) || !coded_tile(d)) return;
    const uint32_t nchunk = (d->nsym + SEG - 1) / SEG;
    uint32_t run = 0, bit = (mode == 1 ? t.pxsz : 3u) * 8u;
    for (uint32_t j = 0; j < nchunk; j++) {
        const uint32_t v = lane < 9 ? A.ccnt[(uint64_t)(t.seg0 + j) * 9 + lane] : 0;
        if (lane < 9) A.ccnt[(uint64_t)(t.seg0 + j) * 9 + lane] = run;
        run += v;
        uint32_t b = 3 * lane * v;
#pragma unroll
        for (int o = 16; o; o >>= 1) b += __shfl_xor_sync(0xffffffffu, b, o);
        if (lane == 0) A.cbit[t.seg0 + j] = bit;
        bit += b;
    }
    bool bad = false;
    if (mode == 1) bad = (uint64_t)bit > 8ull * (d->bsz - 4);
    else if (lane >= 1 && lane < 9) bad = run * (lane < 3 ? 1u : 3u) != d->blk[8 + lane].n;
    if (__any_sync(0xffffffffu, bad) && lane == 0) dec_fail(A.err, DEC_BAD_COUNTS);
}

// Residual plane: level 1 reads 3*nl bits per coded pixel at its bit offset; level 2 reads 1 or 3
// bytes from value stream nl at its rank.  CTA per chunk, 16 consecutive entries per thread.
template <int MODE>
__global__ void __launch_bounds__(256) k_dec_residuals(ChunkArgs A) {
    __shared__ uint32_t wsum[8];
    __shared__ Cnt9 wc[8];
    const uint32_t gseg = blockIdx.x, tile = A.seg_tile[gseg], tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const TileDesc t = A.tiles[tile];
    const DecTile* d = A.dt + tile;
    if (A.imgs[t.img].mode != MODE || !coded_tile(d)) return;
    const uint32_t c0 = (gseg - t.seg0) * SEG;
    if (c0 >= d->nsym) return;
    const uint32_t c1 = min(c0 + (uint32_t)SEG, d->nsym);
    const uint8_t* seq = A.nlseq + t.px_off;
    uint32_t* res = A.resv + resv_base(t);
    const uint8_t* blob = A.in + d->blob_off;
    const uint32_t e0 = c0 + tid * 16;
    // a thread produces 16 consecutive entries; written straight from here they would be 16 word stores 64 bytes apart per
    // lane (32 sectors per request).  They are staged in shared memory (pitch 17: conflict-free) and leave below with
    // consecutive lanes on consecutive words.
    __shared__ uint32_t sres[256 * 17];
    uint32_t se = tid * 17;
    auto put = [&](uint32_t v) { sres[se++] = v; };
    uint32_t w[4] = { 0, 0, 0, 0 };
    if (e0 < c1) { const uint4 q = *reinterpret_cast<const uint4*>(seq + e0); w[0] = q.x; w[1] = q.y; w[2] = q.z; w[3] = q.w; }
    if (MODE == 1) {
        uint32_t mine = 0;
#pragma unroll
        for (int e = 0; e < 16; e++) if (e0 + e < c1) mine += 3 * ((w[e >> 2] >> (8 * (e & 3))) & 0xFu);
        uint32_t inc = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t n = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += n; }
        if (lane == 31) wsum[wid] = inc;
        __syncthreads();
        uint32_t bit = A.cbit[gseg] + inc - mine;
        for (uint32_t k = 0; k < wid; k++) bit += wsum[k];
        const uint8_t* kb = blob + 8; const uint8_t* kend = blob + 4 + d->bsz;
#pragma unroll
        for (int e = 0; e < 16; e++) {
            if (e0 + e >= c1) break;
            const uint32_t nl = (w[e >> 2] >> (8 * (e & 3))) & 0xFu;
            uint32_t v = 0;
            if (nl) {
                const uint8_t* p = kb + 4ull * (bit >> 5);
                const uint32_t w0 = (p + 4 <= kend) ? ld32u(p) : 0u, sh = bit & 31u;
                const uint32_t w1 = (sh + 3 * nl > 32 && p + 8 <= kend) ? ld32u(p + 4) : 0u;
                const uint32_t f = (sh ? ((w0 << sh) | (w1 >> (32u - sh))) : w0) >> (32u - 3 * nl), mk = (1u << nl) - 1u;
                v = (f >> (2 * nl)) | (((f >> nl) & mk) << 8) | ((f & mk) << 16);
                bit += 3 * nl;
            }
            put(v);
        }
    } else {
        Cnt9 cc{ 0, 0, 0 };
#pragma unroll
        for (int e = 0; e < 16; e++) if (e0 + e < c1) cnt9_inc(cc, (w[e >> 2] >> (8 * (e & 3))) & 0xFu);
        Cnt9 tot;
        Cnt9 pos = block_scan_cnt9(cc, wc, tot);
        uint32_t base[9], pp[9];
#pragma unroll
        for (int k = 0; k < 9; k++) { base[k] = A.ccnt[(uint64_t)gseg * 9 + k] + cnt9_get(pos, k); pp[k] = d->blk[k < 1 ? 0 : 8 + k].soff; }
        const uint8_t* sbase = A.streams + t.str_off;
#pragma unroll
        for (int e = 0; e < 16; e++) {
            if (e0 + e >= c1) break;
            const uint32_t nl = (w[e >> 2] >> (8 * (e & 3))) & 0xFu;
            uint32_t v = 0;
            if (nl) {
                uint32_t rank = 0, so = 0;
#pragma unroll
                for (int k = 1; k < 9; k++) if (nl == (uint32_t)k) { rank = base[k]; base[k]++; so = pp[k]; }
                if (nl == 1) { const uint32_t b = sbase[so + rank]; v = (b >> 2) | (((b >> 1) & 1u) << 8) | ((b & 1u) << 16); }
                else if (nl == 2) { const uint32_t b = sbase[so + rank]; v = (b >> 4) | (((b >> 2) & 3u) << 8) | ((b & 3u) << 16); }
                else { const uint8_t* q = sbase + so + 3ull * rank; v = (uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16); }
            }
            put(v);
        }
    }
    __syncthreads();
    const uint32_t cnt = c1 - c0;
    if (!(A.pitched && tile_pitched(t))) {
        for (uint32_t k = tid; k < cnt; k += 256) res[c0 + k] = sres[(k >> 4) * 17 + (k & 15u)];
    } else {   // row-pitched plane: entry k is pixel k + 1 of the raster
        const uint32_t w = t.w, pitch = (w + 3u) & ~3u, magic = 0xFFFFFFFFu / w + 1u;   // (p * magic) >> 32 == p / w for p < 2^20
        for (uint32_t k = tid; k < cnt; k += 256) {
            const uint32_t p = c0 + k + 1;
            uint32_t y = w > 1u ? __umulhi(p, magic) : p;
            if (y * w > p) y--;
            res[y * pitch + (p - y * w)] = sres[(k >> 4) * 17 + (k & 15u)];
        }
    }
}

// Grey tiles: the single decoded plane becomes (u,u,u) residual triples.
__global__ void __launch_bounds__(256) k_dec_residuals_grey(ChunkArgs A) {
    const uint32_t gseg = blockIdx.x, tile = A.seg_tile[gseg];
    const TileDesc t = A.tiles[tile];
    const DecTile* d = A.dt + tile;
    if (A.imgs[t.img].mode != 2 || (d->m >> 4) != 2 || (d->m & 8) || d->m == 0xFE || d->m == 0xFF) return;
    const uint32_t c0 = (gseg - t.seg0) * SEG, c1 = min(c0 + (uint32_t)SEG, t.npx - 1);
    const uint8_t* s = A.streams + t.str_off + d->blk[0].soff;
    uint32_t* res = A.resv + resv_base(t);
    if (A.pitched && tile_pitched(t)) {
        const uint32_t pitch = (t.w + 3u) & ~3u;
        for (uint32_t k = c0 + threadIdx.x; k < c1; k += 256) { const uint32_t y = (k + 1) / t.w, x = (k + 1) - y * t.w; res[y * pitch + x] = (uint32_t)s[k] * 0x010101u; }
    } else
    for (uint32_t k = c0 + threadIdx.x; k < c1; k += 256) res[k] = (uint32_t)s[k] * 0x010101u;
}

// Row index table for RGBA tiles: rows[y].idx = coded pixels before row y (from k_dec_alpha's counts).
__global__ void __launch_bounds__(32) k_dec_rows_rgba(const TileDesc* tiles, const DecImage* imgs, const DecTile* dt, const uint32_t* rowcnt,
                                                      RowInfo* rows) {
    const uint32_t tile = blockIdx.x, lane = threadIdx.x;
    const TileDesc t = tiles[tile];
    if (imgs[t.img].mode != 1 || t.pxsz != 4) return;
    const DecTile* d = dt + tile;
    if (!coded_tile(d)) return;
    uint32_t run = 0;
    for (uint32_t y0 = 0; y0 < t.h; y0 += 32) {
        const uint32_t y = y0 + lane, v = y < t.h ? rowcnt[t.row_off + y] : 0;
        uint32_t inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t n = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += n; }
        if (y < t.h) rows[t.row_off + y].idx = run + inc - v;
        run += __shfl_sync(0xffffffffu, inc, 31);
    }
}

// ------------------------------------------------------------------------------------------------
// Wavefront un-predict (libxpng.c:811-814, :866-897, :911-914).  Thread x owns column x of a strip;
// at step s it reconstructs pixel (x, s - x).  L comes from thread x-1's slot of the previous step,
// UL is that neighbour's value one step earlier, U is the thread's own previous pixel.  The index of
// the pixel's residual travels along the row with the pixel (RGBA skips transparent pixels).
// ------------------------------------------------------------------------------------------------
constexpr int UNP_THREADS = 704;

struct UnpredArgs {
    const TileDesc* tiles;
    const DecImage* imgs;
    const DecTile* dt;
    const uint8_t* in;
    const uint32_t* resv;
    const uint8_t* plane;     // alpha plane (RGBA)
    const RowInfo* rows;      // RGBA: first residual index of each row
    uint4* edge;              // strip hand-over scratch per tile row (tiles wider than UNP_THREADS)
    uint32_t min_w;           // k_dec_unpredict only: skip tiles up to this width (they go to k_dec_unpredict_rows)
    uint32_t pitched;         // 1: tiles with tile_pitched() belong to k_dec_unpredict_rgb (row-pitched residual plane)
};

template <int PXSZ>
__device__ __forceinline__ void unpredict_tile(const UnpredArgs& A, const TileDesc& t, const DecTile* d, uint2 (*slots)[UNP_THREADS + 1]) {
    const uint32_t tid = threadIdx.x;
    const uint8_t* blob = A.in + d->blob_off;
    const uint32_t* res = A.resv + resv_base(t);
    const uint8_t* pl = A.plane + t.px_off;
    const RowInfo* rows = A.rows + t.row_off;
    uint8_t* dst = reinterpret_cast<uint8_t*>(t.src_off);
    const bool grey = (d->m >> 4) == 2;
    const uint32_t pm = grey ? (d->m & 3u) : (((d->m >> 1) & 1u) ? 3u : 2u);   // interior predictor: 0 left 1 up 2 avg2 3 grad3
    const bool G = !grey && (d->m & 1u);
    const uint32_t fp = ld32u(blob + 8);   // first pixel, MSB-first bits
    uint32_t first;
    if (grey) first = (fp >> 24) * 0x010101u;
    else if (PXSZ == 4) first = ((fp >> 24) & 255u) | (((fp >> 16) & 255u) << 8) | (((fp >> 8) & 255u) << 16) | ((fp & 255u) << 24);
    else first = ((fp >> 24) & 255u) | (((fp >> 16) & 255u) << 8) | (((fp >> 8) & 255u) << 16);
    for (uint32_t xs = 0; xs < t.w; xs += UNP_THREADS) {
        const uint32_t sw = min((uint32_t)UNP_THREADS, t.w - xs), x = xs + tid;
        uint32_t own = 0, ownprev = 0, lprev = 0;
        const uint32_t steps = t.h + sw - 1;
        uint32_t rnext = 0;   // RGB: residual of my next pixel, loaded one step ahead
        if (PXSZ == 3 && tid < sw && x) rnext = res[x - 1];
        for (uint32_t s = 0; s < steps; s++) {
            const uint32_t y = s - tid;
            const bool act = tid < sw && tid <= s && y < t.h;
            uint2 me = make_uint2(0, 0);
            if (act) {
                uint2 lf;
                if (tid) lf = slots[(s + 1) & 1][tid - 1];
                else if (xs) { const uint4 e = A.edge[t.row_off + y]; lf = make_uint2(e.x, e.y); lprev = e.z; }
                else lf = make_uint2(0u, PXSZ == 4 ? rows[y].idx : 0u);
                const uint32_t L = lf.x, U = own, UL = lprev;
                uint32_t idx = lf.y, pix;
                uint32_t rv = rnext;
                if (PXSZ == 3 && y + 1 < t.h) rnext = res[(uint64_t)(y + 1) * t.w + x - 1];
                if (x == 0 && y == 0) pix = first;
                else {
                    uint32_t a = 255;
                    if (PXSZ == 4) a = pl[(uint64_t)y * t.w + x];
                    if (a == 0) pix = 0;
                    else {
                        if (PXSZ == 4) { rv = res[idx]; idx++; }
                        int r0 = unzz(rv & 255u), r1 = unzz((rv >> 8) & 255u), r2 = unzz((rv >> 16) & 255u);
                        if (G && x && y) { r0 += r1; r2 += r1; }
                        const int r[3] = { r0, r1, r2 };
                        pix = PXSZ == 4 ? (a << 24) : 0u;
#pragma unroll
                        for (int c = 0; c < 3; c++) {
                            const int l = (L >> (8 * c)) & 255, u = (U >> (8 * c)) & 255, ul = (UL >> (8 * c)) & 255;
                            int pd;
                            if (y == 0) pd = l; else if (x == 0) pd = u;
                            else pd = pm == 0 ? l : (pm == 1 ? u : (pm == 2 ? pred_avg2(l, u) : pred_grad3(l, u, ul)));
                            pix |= (uint32_t)((r[c] + pd) & 255) << (8 * c);
                        }
                    }
                }
                uint8_t* o = dst + (uint64_t)y * t.bpr + (uint64_t)x * PXSZ;
                if (PXSZ == 4) *reinterpret_cast<uint32_t*>(o) = pix;
                else { o[0] = (uint8_t)pix; o[1] = (uint8_t)(pix >> 8); o[2] = (uint8_t)(pix >> 16); }
                me = make_uint2(pix, idx);
                lprev = L; ownprev = own; own = pix;
                if (tid == sw - 1 && xs + sw < t.w) A.edge[t.row_off + y] = make_uint4(pix, idx, ownprev, 0);
            }
            slots[s & 1][tid] = me;
            __syncthreads();
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(UNP_THREADS) k_dec_unpredict(UnpredArgs A) {
    __shared__ uint2 slots[2][UNP_THREADS + 1];
    const uint32_t tile = blockIdx.x;
    const TileDesc t = A.tiles[tile];
    const uint32_t mode = A.imgs[t.img].mode;
    if (mode == 7 || (mode & 0x100)) return;
    const DecTile* d = A.dt + tile;
    if (d->m == 0 || d->m == 0xFE || d->m == 0xFF || ((d->m >> 4) == 2 && (d->m & 8))) return;
    if (t.w <= A.min_w) return;   // (wider than UNR_MAXW: never a pitched tile)
    if (t.pxsz == 4) unpredict_tile<4>(A, t, d, slots);
    else unpredict_tile<3>(A, t, d, slots);
}

// ------------------------------------------------------------------------------------------------
// Un-predict, row-band pipeline (libxpng.c:811-814, :866-897, :911-914).
// A pixel needs L, U, UL.  Lane r of a warp owns ROW y0 + r of a 32-row band and walks it left to
// right one pixel per step, one step behind the lane above: at step s lane r is at x = s - r.  Then
//   L  = the lane's own previous pixel (register),
//   U  = the pixel lane r-1 produced in the previous step (one shfl_up),
//   UL = the U of the lane's own previous step (register),
// so a step is a shuffle plus ALU work: no block barrier and no shared-memory slots per step, and
// every lane streams through its own row (sector-friendly loads, word-sized stores).  Bands are
// pipelined over the warps of the CTA: warp b % NW owns band b, lane 0 takes U from the last row of
// the band above, which that band's last lane leaves in a shared boundary row together with a
// monotonic progress counter (published every 32 columns; the lower band waits on it).
// ------------------------------------------------------------------------------------------------
constexpr int UNR_WARPS = 16;       // warps per CTA of the single-frame variant; batches use 8 (two CTAs per SM)
constexpr int UNR_MAXW = 672;        // widest tile (666) rounded up
constexpr int UNR_PITCH = 32 * 4 + 4;   // bytes per staged row chunk (32 pixels of up to 4 bytes, padded)

// Output staging: a lane's pixels would be 32 scattered sub-word stores per step; instead each warp stages
// two 32-column chunks of its band in shared memory and writes a finished chunk row by row (contiguous bytes).
template <int PXSZ>
__device__ __forceinline__ void unr_flush(const uint8_t* sb, uint8_t* dst, const TileDesc& t, uint32_t y0, uint32_t chunk, uint32_t lane) {
    const uint32_t ncols = min(32u, t.w - 32u * chunk), nbytes = ncols * PXSZ, nw = nbytes >> 2;
    const uint8_t* src = sb + (chunk & 1u) * (32 * UNR_PITCH);
    const uint32_t nrows = min(32u, t.h - y0);
    uint8_t* o = dst + (uint64_t)y0 * t.bpr + (uint64_t)PXSZ * 32u * chunk;
#pragma unroll 4
    for (uint32_t r = 0; r < nrows; r++, o += t.bpr, src += UNR_PITCH) {
        if ((reinterpret_cast<uintptr_t>(o) & 3u) == 0) {          // warp-uniform; a staged row starts word-aligned (UNR_PITCH = 132)
            if (lane < nw) reinterpret_cast<uint32_t*>(o)[lane] = reinterpret_cast<const uint32_t*>(src)[lane];
            const uint32_t k = (nw << 2) + lane;                    // a narrow last chunk may end inside a word
            if (k < nbytes) o[k] = src[k];
        } else for (uint32_t k = lane; k < nbytes; k += 32) o[k] = src[k];
    }
}

// Byte-parallel arithmetic on the three colour channels packed in one word (0x00BBGGRR): every operation below is
// exact modulo 256 per byte, which is all the reconstruction needs (libxpng.c:21, :27-30, :813).
__device__ __forceinline__ uint32_t swar_add(uint32_t a, uint32_t b) {        // per-byte a + b (mod 256)
    return ((a & 0x7F7F7F7Fu) + (b & 0x7F7F7F7Fu)) ^ ((a ^ b) & 0x80808080u);
}
__device__ __forceinline__ uint32_t swar_unzz(uint32_t u) {                   // per-byte (u >> 1) ^ -(u & 1)
    return ((u >> 1) & 0x7F7F7F7Fu) ^ ((u & 0x01010101u) * 0xFFu);
}
__device__ __forceinline__ uint32_t swar_avg2(uint32_t l, uint32_t u) {       // per-byte (l + u + 1) >> 1
    return (l | u) - (((l ^ u) >> 1) & 0x7F7F7F7Fu);
}
__device__ __forceinline__ uint32_t swar_grad3(uint32_t l, uint32_t u, uint32_t ul) {   // per-byte ((3l + 3u - 2ul + 2) >> 2) mod 256
    // 16-bit lanes with a +512 bias keep every lane non-negative (range 4 .. 2044); 512 >> 2 = 128 is removed mod 256
    const uint32_t l01 = (l & 0xFFu) | ((l & 0xFF00u) << 8), u01 = (u & 0xFFu) | ((u & 0xFF00u) << 8), q01 = (ul & 0xFFu) | ((ul & 0xFF00u) << 8);
    const uint32_t l2 = (l >> 16) & 0xFFu, u2 = (u >> 16) & 0xFFu, q2 = (ul >> 16) & 0xFFu;
    const uint32_t t01 = 3u * (l01 + u01) + 0x02020202u - 2u * q01;            // + 514 per lane = 2 + 512
    const uint32_t t2 = 3u * (l2 + u2) + 514u - 2u * q2;
    const uint32_t p01 = ((t01 >> 2) + 0x00800080u) & 0x00FF00FFu, p2 = ((t2 >> 2) + 128u) & 0xFFu;   // +128 == -128 (mod 256), no borrow
    return (p01 & 0xFFu) | ((p01 >> 8) & 0xFF00u) | (p2 << 16);
}

// PM: interior predictor 0 left, 1 up, 2 avg2, 3 grad3; GSUB: residual green added back to red and blue.
template <int PXSZ, int PM, bool GSUB, int NW>
__device__ __forceinline__ void unpredict_rows(const UnpredArgs& A, const TileDesc& t, const DecTile* d, uint32_t (*brow)[UNR_MAXW],
                                               volatile uint32_t* prog, uint8_t* stage) {
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint8_t* blob = A.in + d->blob_off;
    const uint32_t* res = A.resv + resv_base(t);
    const uint8_t* pl = A.plane + t.px_off;
    const RowInfo* rows = A.rows + t.row_off;
    uint8_t* dst = reinterpret_cast<uint8_t*>(t.src_off);
    const bool grey = (d->m >> 4) == 2;
    const uint32_t fp = ld32u(blob + 8);   // first pixel, MSB-first bits
    uint32_t first;
    if (grey) first = (fp >> 24) * 0x010101u;
    else if (PXSZ == 4) first = ((fp >> 24) & 255u) | (((fp >> 16) & 255u) << 8) | (((fp >> 8) & 255u) << 16) | ((fp & 255u) << 24);
    else first = ((fp >> 24) & 255u) | (((fp >> 16) & 255u) << 8) | (((fp >> 8) & 255u) << 16);
    const uint32_t w = t.w, nbands = (t.h + 31) / 32;
    const uint32_t stride = w + 1;                         // progress units per band: columns done (0..w)
    uint8_t* sb = stage + wid * (2 * 32 * UNR_PITCH);
    for (uint32_t b = wid, seq = 0; b < nbands; b += NW, seq++) {
        const uint32_t y = b * 32 + lane;
        const bool rowok = y < t.h;
        const uint32_t lastlane = min(31u, t.h - 1 - b * 32);   // lane holding the band's last row
        uint32_t* mybrow = brow[wid];
        const uint32_t upidx = (wid + NW - 1) % NW;
        const uint32_t* upbrow = brow[upidx];
        const uint32_t upbase = (wid == 0 ? seq - 1 : seq) * stride;     // progress value of the band above when it has done 0 columns
        uint32_t left = 0, uprev = 0, prevout = 0;           // L, previous U (= UL), my pixel of the previous step (handed down)
        uint32_t idx = (PXSZ == 4 && rowok) ? rows[y].idx : 0u;
        const uint8_t* prow = pl + (uint64_t)y * w;
        const uint32_t* rrow = res + (uint64_t)y * w - 1;    // RGB: residual of (x, y) at rrow[x]
        // RGB: the lane's residuals are consecutive words of its row; they are fetched RING steps ahead into a
        // register ring (static indices: the step loop is unrolled by RING), so no load ever sits on the
        // L -> pixel -> L chain.  RGBA residuals are indexed by the running count of coded pixels: one step ahead.
        constexpr int RING = 8;
        uint32_t rn[RING];
        uint32_t rnext = 0, anext = 255;
#pragma unroll
        for (int k = 0; k < RING; k++) rn[k] = 0;
        if (rowok) {
            if (PXSZ == 3) {   // slot j is consumed at steps s == j (mod RING); the lane's column c is consumed at step c + lane
#pragma unroll
                for (int c = 0; c < RING; c++) {
                    const uint32_t v = ((uint32_t)c < w && (y || c)) ? rrow[c] : 0u;
                    const uint32_t slot = (lane + (uint32_t)c) % RING;
#pragma unroll
                    for (int k = 0; k < RING; k++) rn[k] = slot == (uint32_t)k ? v : rn[k];
                }
            } else { anext = prow[0]; rnext = res[idx]; }
        }
        const uint32_t steps = (w + 31 + RING - 1) / RING * RING;   // whole rings: the extra steps find every lane past its row
        uint32_t flushed = 0;                                // chunks written out so far
        const bool row0 = y == 0;
        const uint32_t stage_lane = lane * UNR_PITCH;
        for (uint32_t s0 = 0; s0 < steps; s0 += RING) {
#pragma unroll
            for (int j = 0; j < RING; j++) {
                const uint32_t s = s0 + j;
                if (NW > 1 && b && j == 0) {                 // lane 0 will need columns s .. s + 7 of the band above
                    const uint32_t need = upbase + min(s + 8u, w);
                    while (prog[upidx] < need) { }
                    __syncwarp();
                }
                const uint32_t x = s - lane;                 // lanes that have not started yet wrap around: x >= w
                const bool act = rowok && x < w;
                // U: the pixel the lane above produced in the previous step; lane 0 takes it from the boundary row of the band
                // above (band 0 has none, and never uses it: its lane 0 is image row 0, predicted from the left)
                const uint32_t ub = upbrow[min(s, w - 1)];
                uint32_t U = __shfl_up_sync(0xffffffffu, prevout, 1);
                U = lane == 0 ? ub : U;
                uint32_t pix = 0;
                const uint32_t rv3 = rn[j];                  // static ring index: slot j <-> steps s == j (mod RING)
                if (PXSZ == 3) {
                    // refill slot j for the step RING steps from now.  A predicated load straight INTO the ring register: written
                    // as `rn[j] = __ldg(..)` inside the branch below, the compiler loads into a temporary and moves it at once,
                    // which waits for the whole memory latency on every step (ncu: 40 % of the kernel's stall samples sat on that move).
                    // The index is clamped into the row (row 0 has no residual at x = 0: rrow[0] would be the word before the slice).
                    const uint32_t xi = max(min(x + RING, w - 1), row0 ? 1u : 0u);
                    asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %2, 0;\n @q ld.global.nc.u32 %0, [%1];\n}"
                                 : "+r"(rn[j]) : "l"(rrow + xi), "r"((uint32_t)act));
                }
                if (act) {
                    const bool origin = (x | y) == 0;
                    bool coded = !origin;
                    const uint32_t a = anext, rv = PXSZ == 3 ? rv3 : rnext;
                    if (PXSZ == 4) {
                        if (a == 0) coded = false;
                        if (coded) idx++;
                        if (x + 1 < w) anext = prow[x + 1];
                        rnext = res[idx];                    // the slice has slack behind its last residual
                    }
                    // all three channels at once (byte 3 of every operand is zero for RGB; RGBA keeps alpha there and masks it)
                    uint32_t r = swar_unzz(PXSZ == 3 ? rv : (rv & 0x00FFFFFFu));
                    if (GSUB) { const uint32_t rg = swar_add(r, ((r >> 8) & 0xFFu) * 0x00010001u); r = (x && !row0) ? rg : r; }
                    const uint32_t l3 = PXSZ == 3 ? left : (left & 0x00FFFFFFu), u3 = PXSZ == 3 ? U : (U & 0x00FFFFFFu),
                                   q3 = PXSZ == 3 ? uprev : (uprev & 0x00FFFFFFu);
                    uint32_t pd = PM == 0 ? l3 : (PM == 1 ? u3 : (PM == 2 ? swar_avg2(l3, u3) : swar_grad3(l3, u3, q3)));
                    pd = row0 ? l3 : (x == 0 ? u3 : pd);
                    const uint32_t val = (swar_add(r, pd) & 0x00FFFFFFu) | (PXSZ == 4 ? (a << 24) : 0u);
                    pix = origin ? first : (coded ? val : 0u);
                    uint8_t* o = sb + stage_lane + (x & 32u) * UNR_PITCH + PXSZ * (x & 31u);
                    if (PXSZ == 4) *reinterpret_cast<uint32_t*>(o) = pix;
                    else { o[0] = (uint8_t)pix; o[1] = (uint8_t)(pix >> 8); o[2] = (uint8_t)(pix >> 16); }
                    left = pix;
                    if (lane == lastlane) mybrow[x] = pix;
                }
                uprev = U;
                prevout = pix;
                if (NW > 1 && lane == lastlane && act && ((x & 7u) == 7u || x == w - 1)) {   // publish progress of the band's last row
                    __threadfence_block();
                    prog[wid] = seq * stride + x + 1;
                }
                if (j == RING - 2 && (s & 31u) == 30u && s >= 62) {   // every lane has finished chunk (s - 62) / 32
                    __syncwarp();
                    unr_flush<PXSZ>(sb, dst, t, b * 32, flushed, lane);
                    flushed++;
                    __syncwarp();
                }
            }
        }
        __syncwarp();
        for (; flushed * 32 < w; flushed++) unr_flush<PXSZ>(sb, dst, t, b * 32, flushed, lane);
        __syncwarp();
    }
}

template <int NW>
__global__ void __launch_bounds__(NW * 32) k_dec_unpredict_rows(UnpredArgs A) {
    extern __shared__ __align__(16) uint8_t unr_stage[];   // [NW][2][32][UNR_PITCH]
    __shared__ uint32_t brow[NW][UNR_MAXW];
    __shared__ uint32_t prog_s[NW];
    const uint32_t tile = blockIdx.x;
    const TileDesc t = A.tiles[tile];
    const uint32_t mode = A.imgs[t.img].mode;
    if (mode == 7 || (mode & 0x100)) return;
    const DecTile* d = A.dt + tile;
    if (d->m == 0 || d->m == 0xFE || d->m == 0xFF || ((d->m >> 4) == 2 && (d->m & 8))) return;
    if (t.w > UNR_MAXW) return;                       // very wide, flat tiles (thin images): k_dec_unpredict
    if (A.pitched && tile_pitched(t)) return;         // k_dec_unpredict_rgb
    if (threadIdx.x < NW) prog_s[threadIdx.x] = 0;
    __syncthreads();
    // specialise the inner loop on the tile's predictor (grey tiles: m & 3; colour tiles: avg2 / grad3, optional G)
    const bool grey = (d->m >> 4) == 2;
    const uint32_t pm = grey ? (d->m & 3u) : (((d->m >> 1) & 1u) ? 3u : 2u);
    const bool G = !grey && (d->m & 1u);
    if (t.pxsz == 4) {
        if (pm == 3) { if (G) unpredict_rows<4, 3, true, NW>(A, t, d, brow, prog_s, unr_stage); else unpredict_rows<4, 3, false, NW>(A, t, d, brow, prog_s, unr_stage); }
        else { if (G) unpredict_rows<4, 2, true, NW>(A, t, d, brow, prog_s, unr_stage); else unpredict_rows<4, 2, false, NW>(A, t, d, brow, prog_s, unr_stage); }
    } else if (pm == 3) { if (G) unpredict_rows<3, 3, true, NW>(A, t, d, brow, prog_s, unr_stage); else unpredict_rows<3, 3, false, NW>(A, t, d, brow, prog_s, unr_stage); }
    else if (pm == 2) { if (G) unpredict_rows<3, 2, true, NW>(A, t, d, brow, prog_s, unr_stage); else unpredict_rows<3, 2, false, NW>(A, t, d, brow, prog_s, unr_stage); }
    else if (pm == 1) unpredict_rows<3, 1, false, NW>(A, t, d, brow, prog_s, unr_stage);
    else unpredict_rows<3, 0, false, NW>(A, t, d, brow, prog_s, unr_stage);
}

// ------------------------------------------------------------------------------------------------
// Un-predict for batches: one warp per RGB tile, the row-band wavefront of unpredict_rows with the memory side rebuilt
// for thousands of resident warps (ncu on 4000 tiles: the older kernel issued one instruction per 25 cycles and warp,
// 58 % of it waiting for shared memory, L1 hit rate 24 % on its word-sized residual loads, 19 warps per SM for its
// 8.4 KB stage):
//   * residuals come from the row-pitched plane, FOUR per 128-bit cp.async, twelve steps ahead, into a four-slot ring per lane
//     in shared memory (2 KB per warp).  Loads into a register ring were tracked by ONE hardware scoreboard (SASS control
//     bits: every LDG with write barrier 5), so the first use of any slot waited for the load issued a moment before it:
//     43 % of the kernel's stall samples (ncu r03k); cp.async groups count completions per group instead;
//   * finished pixels are packed in a 96-bit shift register and leave as three aligned words per four pixels, straight
//     to global memory (each lane writes its own row; L2 merges the sectors): no staging buffer, no flush loop;
//   * shared memory per warp is the 2.7 KB boundary row only, so registers (64) bound the residency at 32 warps per SM.
// Requires word-aligned rows (tile_pitched).  libxpng.c:811-814, :866-897, :911-914.
// ------------------------------------------------------------------------------------------------
template <int PM, bool GSUB>
__device__ __forceinline__ void unpredict_rgb(const UnpredArgs& A, const TileDesc& t, const DecTile* d, uint32_t* brow, uint4* ring_base) {
    const uint32_t lane = threadIdx.x & 31;
    uint4* ring = ring_base + lane;                                   // [slot][lane]
    const uint32_t ring_s = (uint32_t)__cvta_generic_to_shared(ring);
    const uint8_t* blob = A.in + d->blob_off;
    const uint32_t w = t.w, pitch = (w + 3u) & ~3u;
    const uint32_t* res = A.resv + resv_base(t);
    uint8_t* dst = reinterpret_cast<uint8_t*>(t.src_off);
    const uint32_t fp = ld32u(blob + 8);   // first pixel, MSB-first bits
    const uint32_t first = (d->m >> 4) == 2 ? (fp >> 24) * 0x010101u : (((fp >> 24) & 255u) | (((fp >> 16) & 255u) << 8) | (((fp >> 8) & 255u) << 16));
    const uint32_t nbands = (t.h + 31) / 32;
    // Lane r runs FOUR columns behind lane r - 1 (x = s - 4r): every lane is at the same column phase, so the 128-bit
    // residual load (x = 0 mod 4) and the three-word pixel store (x = 3 mod 4) sit at fixed places of the unrolled loop,
    // are executed by all lanes at once, and consecutive loads never share a destination register (with a skew of
    // one column some lanes load at every step, each load waits for the previous one: 13 of 17 cycles per instruction
    // were long-scoreboard stalls).  U is the upper lane's pixel of four steps ago (static 4-entry history).
    constexpr int RING = 16, AHEAD = 12, SKEW = 4;
    const bool tailw = (w & 3u) != 0;
    for (uint32_t b = 0; b < nbands; b++) {
        const uint32_t y = b * 32 + lane;
        const bool rowok = y < t.h, row0 = y == 0;
        const uint32_t lastlane = min(31u, t.h - 1 - b * 32);
        const uint32_t* rrow = res + (uint64_t)y * pitch;            // 16-byte aligned
        uint8_t* orow = dst + (uint64_t)y * t.bpr;                    // word aligned
        uint32_t left = 0, uprev = 0, a0 = 0, a1 = 0, a2 = 0;
        uint32_t hist[SKEW] = { 0, 0, 0, 0 };
        // the lane's column group cg (columns 4cg .. 4cg + 3) lives in slot (cg + lane) % 4, i.e. slot (j / 4) % 4 at step j of the
        // unrolled loop for every lane; one cp.async group per four steps, three groups in flight
        asm volatile("cp.async.wait_all;" ::: "memory");
#pragma unroll
        for (int g = 0; g < AHEAD / 4; g++) {   // columns 0 .. 11
            const uint32_t go = (rowok && 4u * g < pitch) ? 1u : 0u;
            asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %2, 0;\n @q cp.async.cg.shared.global [%0], [%1], 16;\n}"
                         :: "r"(ring_s + (((uint32_t)g + lane) & 3u) * 512u), "l"(rrow + 4 * g), "r"(go) : "memory");
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
        uint4 r4 = make_uint4(0, 0, 0, 0);
        const uint32_t steps = (w + SKEW * 31 + RING - 1) / RING * RING;
        for (uint32_t s0 = 0; s0 < steps; s0 += RING) {
#pragma unroll
            for (int j = 0; j < RING; j++) {
                const uint32_t s = s0 + j;
                const uint32_t x = s - SKEW * lane;                   // lanes that have not started yet wrap around: x >= w
                const bool act = rowok && x < w;
                const uint32_t ub = brow[min(s, w - 1)];              // row above the band (band 0 never uses it)
                uint32_t U = __shfl_up_sync(0xffffffffu, hist[j % SKEW], 1);   // the upper lane's pixel of four steps ago: column x
                U = lane == 0 ? ub : U;
                if (j % 4 == 0) {   // my four residuals of columns x .. x + 3 have landed; request columns x + 12 .. x + 15
                    asm volatile("cp.async.wait_group 2;" ::: "memory");
                    r4 = ring[((j / 4) % 4) * 32];
                    const uint32_t go = (act && x + AHEAD < pitch) ? 1u : 0u;
                    asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %2, 0;\n @q cp.async.cg.shared.global [%0], [%1], 16;\n}"
                                 :: "r"(ring_s + ((j / 4 + 3) % 4) * 512u), "l"(rrow + x + AHEAD), "r"(go) : "memory");
                    asm volatile("cp.async.commit_group;" ::: "memory");
                }
                const uint32_t rv = j % 4 == 0 ? r4.x : (j % 4 == 1 ? r4.y : (j % 4 == 2 ? r4.z : r4.w));
                uint32_t pix = 0;
                if (act) {
                    uint32_t r = swar_unzz(rv);
                    if (GSUB) { const uint32_t rg = swar_add(r, ((r >> 8) & 0xFFu) * 0x00010001u); r = (x && !row0) ? rg : r; }
                    uint32_t pd = PM == 0 ? left : (PM == 1 ? U : (PM == 2 ? swar_avg2(left, U) : swar_grad3(left, U, uprev)));
                    pd = row0 ? left : (x == 0 ? U : pd);
                    const uint32_t val = swar_add(r, pd) & 0x00FFFFFFu;
                    pix = (x | y) == 0 ? first : val;
                    left = pix;
                    // 96-bit shift register: after pixels 4k .. 4k + 3 it holds their twelve bytes in memory order
                    a0 = __funnelshift_r(a0, a1, 24); a1 = __funnelshift_r(a1, a2, 24); a2 = __funnelshift_r(a2, pix, 24);
                    if (lane == lastlane) brow[x] = pix;
                    if (j % 4 == 3) {                                 // x = 3 (mod 4) for every lane
                        uint32_t* o = reinterpret_cast<uint32_t*>(orow + 3u * (x - 3u));
                        o[0] = a0; o[1] = a1; o[2] = a2;
                    } else if (tailw && x == w - 1) {                 // 1 .. 3 pixels left over at the row end: byte stores
                        const uint32_t np = (x & 3u) + 1u, sh = 24u * (4u - np);   // bring them down to bit 0 (sh = 24, 48, 72)
                        uint32_t t0 = a0, t1 = a1, t2 = a2;
                        if (sh >= 64) { t0 = t2; t1 = 0; t2 = 0; } else if (sh >= 32) { t0 = t1; t1 = t2; t2 = 0; }
                        const uint32_t rs = sh & 31u;
                        const uint32_t b0 = __funnelshift_r(t0, t1, rs), b1 = __funnelshift_r(t1, t2, rs), b2 = t2 >> rs;
                        uint8_t* o = orow + 3u * (x + 1u - np);
                        for (uint32_t k = 0; k < 3u * np; k++) { const uint32_t wv = k < 4u ? b0 : (k < 8u ? b1 : b2); o[k] = (uint8_t)(wv >> (8u * (k & 3u))); }
                    }
                }
                uprev = U;
                hist[j % SKEW] = pix;
            }
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(32) k_dec_unpredict_rgb(UnpredArgs A) {
    __shared__ uint32_t brow[UNR_MAXW];
    __shared__ uint4 rring[4][32];                     // residual ring: four column groups per lane
    const uint32_t tile = blockIdx.x;
    const TileDesc t = A.tiles[tile];
    const uint32_t mode = A.imgs[t.img].mode;
    if (mode == 7 || (mode & 0x100)) return;
    const DecTile* d = A.dt + tile;
    if (d->m == 0 || d->m == 0xFE || d->m == 0xFF || ((d->m >> 4) == 2 && (d->m & 8))) return;
    if (!tile_pitched(t)) return;                      // RGBA, very wide or unaligned tiles: the older kernels
    const bool grey = (d->m >> 4) == 2;
    const uint32_t pm = grey ? (d->m & 3u) : (((d->m >> 1) & 1u) ? 3u : 2u);
    const bool G = !grey && (d->m & 1u);
    if (pm == 3) { if (G) unpredict_rgb<3, true>(A, t, d, brow, &rring[0][0]); else unpredict_rgb<3, false>(A, t, d, brow, &rring[0][0]); }
    else if (pm == 2) { if (G) unpredict_rgb<2, true>(A, t, d, brow, &rring[0][0]); else unpredict_rgb<2, false>(A, t, d, brow, &rring[0][0]); }
    else if (pm == 1) unpredict_rgb<1, false>(A, t, d, brow, &rring[0][0]);
    else unpredict_rgb<0, false>(A, t, d, brow, &rring[0][0]);
}

// Raw grey plane (level 2, m = 0x28, libxpng.c:875-879)
__global__ void __launch_bounds__(256) k_dec_grey_raw(const TileDesc* tiles, const DecImage* imgs, const DecTile* dt, const uint8_t* in) {
    const uint32_t tile = blockIdx.x;
    const TileDesc t = tiles[tile];
    if (imgs[t.img].mode != 2) return;
    const DecTile* d = dt + tile;
    if ((d->m >> 4) != 2 || !(d->m & 8) || d->m == 0xFE || d->m == 0xFF) return;
    const uint8_t* src = in + d->blob_off + 4;
    uint8_t* dst = reinterpret_cast<uint8_t*>(t.src_off);
    for (uint32_t y = threadIdx.x >> 5; y < t.h; y += 8)
        for (uint32_t x = threadIdx.x & 31; x < t.w; x += 32) {
            const uint8_t v = src[(uint64_t)y * t.w + x];
            uint8_t* o = dst + (uint64_t)y * t.bpr + 3ull * x;
            o[0] = v; o[1] = v; o[2] = v;
        }
}

}  // namespace xpb
