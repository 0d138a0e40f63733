// enc_back.cuh — encode back end for level 1: per-tile segment scan, stream compaction, frequency
// normalisation and rANS encoder symbols (the v2 block encoder, libxpng.c:307-427, is k_rans_v2_pair in
// enc_rans_lat.cuh), size decisions and final assembly (libxpng.c:534-571, :723-789).
#pragma once
#include "common.cuh"
#include "enc_front.cuh"

namespace xpb {

// Scratch geometry: the host lays out per-tile slices (TileDesc::str_off / blk_off).
__host__ __device__ __forceinline__ uint64_t stream_slice(const TileDesc& t) { return t.str_off; }
__host__ __device__ __forceinline__ uint64_t block_slice(const TileDesc& t, uint32_t) { return t.blk_off; }
__host__ __device__ __forceinline__ uint32_t align16u(uint32_t v) { return (v + 15u) & ~15u; }

// ------------------------------------------------------------------------------------------------
// Per-tile scan over segments: chunk destinations, segment-first symbols, bit offsets, stream
// lengths / offsets.  One warp per tile; lane c < 9 owns context stream c.
// ------------------------------------------------------------------------------------------------
struct TileScanArgs {
    const TileDesc* tiles;
    const SegInfo* seginfo;
    const uint32_t* costs;
    const uint16_t* vcnt;     // mode 2
    SegPlace* place;
    SegPlace* vplace;         // mode 2: value chunk destinations (pos[nl], in bytes)
    uint32_t* hist;
    TileState* state;
    const uint8_t* tile_skip; // mode 2
    uint32_t ntiles;
};

template <int MODE>
__global__ void __launch_bounds__(128) k_tile_scan(TileScanArgs A) {
    const uint32_t tile = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (tile >= A.ntiles) return;
    if (MODE == 2 && A.tile_skip && A.tile_skip[tile]) return;
    const TileDesc t = A.tiles[tile];
    constexpr int HSTRIDE = MODE == 1 ? HIST_STRIDE_M1 : HIST_STRIDE_M2;
    uint32_t* F = A.hist + (uint64_t)tile * HSTRIDE;
    uint32_t run = 0, vrun = 0, carry = 0;
    uint64_t bit = (MODE == 1 ? t.pxsz : 3u) * 8u;
    for (uint32_t j = 0; j < t.nseg; j++) {
        const SegInfo si = A.seginfo[t.seg0 + j];
        uint32_t fpos = 0;
        if (si.has_valid) {
            fpos = __shfl_sync(0xffffffffu, run, carry);
            if (lane == carry) { run++; F[HIST_CTX + carry * 16 + si.first_nl]++; }
        }
        if (lane < 9) A.place[t.seg0 + j].pos[lane] = run;
        if (lane == 0) {
            SegPlace* p = A.place + t.seg0 + j;
            p->first_pos = fpos; p->first_ctx = carry; p->bit_off = bit;
        }
        if (lane < 9) run += si.cnt[lane];
        if (MODE == 2 && lane >= 1 && lane < 9) {
            A.vplace[t.seg0 + j].pos[lane] = vrun;
            vrun += (uint32_t)A.vcnt[(uint64_t)(t.seg0 + j) * 9 + lane] * (lane < 3 ? 1u : 3u);
        }
        if (si.has_valid) carry = si.last_nl;
        bit += si.nbits;
    }
    // stream lengths and 16-aligned offsets (exclusive scan across lanes)
    TileState* st = A.state + tile;
    const uint32_t len = lane < 9 ? run : 0, a = align16u(len);
    uint32_t inc = a;
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) { const uint32_t n = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += n; }
    const uint32_t ctx_total = __shfl_sync(0xffffffffu, inc, 8);
    if (lane < 9) {
        st->len[lane] = len; st->soff[lane] = inc - a;
        // block scratch: generous bound 2*len + 256 per stream (payload <= PB/8 bytes per symbol)
    }
    uint32_t bb = lane < 9 ? align16u(2 * len + 256) : 0, binc = bb;
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) { const uint32_t n = __shfl_up_sync(0xffffffffu, binc, o); if (lane >= o) binc += n; }
    if (lane < 9) { st->boff[lane] = binc - bb; st->breg[lane] = binc - bb; }
    const uint32_t blk_total = __shfl_sync(0xffffffffu, binc, 8);
    if (MODE == 1) {
        if (lane == 9) {   // alpha stream: raster order, lives in the alpha slice
            st->len[9] = t.pxsz == 4 ? t.npx - 1 : 0; st->soff[9] = 0;
            st->boff[9] = blk_total; st->breg[9] = blk_total;
        }
    } else {
        const uint32_t vlen = (lane >= 1 && lane < 9) ? vrun : 0, va = align16u(vlen);
        uint32_t vinc = va;
#pragma unroll
        for (int o = 1; o < 16; o <<= 1) { const uint32_t n = __shfl_up_sync(0xffffffffu, vinc, o); if (lane >= o) vinc += n; }
        uint32_t vb = (lane >= 1 && lane < 9) ? align16u(2 * vlen + 256) : 0, vbinc = vb;
#pragma unroll
        for (int o = 1; o < 16; o <<= 1) { const uint32_t n = __shfl_up_sync(0xffffffffu, vbinc, o); if (lane >= o) vbinc += n; }
        if (lane >= 1 && lane < 9) {
            st->len[8 + lane] = vlen; st->soff[8 + lane] = ctx_total + vinc - va;
            st->boff[8 + lane] = blk_total + vbinc - vb; st->breg[8 + lane] = blk_total + vbinc - vb;
        }
    }
    if (lane == 0) {
        st->pr = pick_predictor(A.costs + 4 * tile, t.w, t.h, MODE == 2 ? 3u : t.pxsz);
        st->kbits_lo = (uint32_t)bit; st->kbits_hi = (uint32_t)(bit >> 32);
    }
}

// ------------------------------------------------------------------------------------------------
// Compaction: move each segment's chunks to their place in the tile's contiguous streams.
// ------------------------------------------------------------------------------------------------
struct CompactArgs {
    const TileDesc* tiles;
    const uint32_t* seg_tile;
    const SegInfo* seginfo;
    const SegPlace* place;
    const SegPlace* vplace;
    const uint16_t* vcnt;
    const TileState* state;
    const uint8_t* sym_area;
    const uint8_t* bits_area;
    uint8_t* streams;
    const uint8_t* tile_skip;
};

// n bytes from src to dst, any alignment, by the 256 threads of a CTA: whole destination words are written as words (the
// source through two aligned words and a funnel shift; reads may touch up to 3 bytes past src + n: every scratch buffer has
// slack), the bytes around them one by one.  Neighbouring chunks of a stream are written by other CTAs: only bytes of
// [dst, dst + n) are touched.
__device__ __forceinline__ void cta_copy_bytes(uint8_t* dst, const uint8_t* src, uint32_t n, uint32_t tid) {
    const uint32_t head = min(n, (4u - (uint32_t)(reinterpret_cast<uintptr_t>(dst) & 3u)) & 3u);
    if (tid < head) dst[tid] = src[tid];
    dst += head; src += head; n -= head;
    const uint32_t nw = n >> 2, sh = (uint32_t)(reinterpret_cast<uintptr_t>(src) & 3u) * 8u;
    const uint32_t* s4 = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(src) & ~(uintptr_t)3);
    uint32_t* d4 = reinterpret_cast<uint32_t*>(dst);
    if (sh == 0) for (uint32_t k = tid; k < nw; k += 256) d4[k] = s4[k];
    else for (uint32_t k = tid; k < nw; k += 256) d4[k] = __funnelshift_r(s4[k], s4[k + 1], sh);
    const uint32_t tail = n & 3u;
    if (tid < tail) dst[4u * nw + tid] = src[4u * nw + tid];
}

template <int MODE>
__global__ void __launch_bounds__(256) k_compact(CompactArgs A) {
    const uint32_t gseg = blockIdx.x, tile = A.seg_tile[gseg], tid = threadIdx.x;
    if (MODE == 2 && A.tile_skip && A.tile_skip[tile]) return;
    const TileDesc t = A.tiles[tile];
    const TileState* st = A.state + tile;
    const SegInfo si = A.seginfo[gseg];
    const SegPlace pl = A.place[gseg];
    uint8_t* sbase = A.streams + stream_slice(t);
    const uint8_t* src = A.sym_area + (uint64_t)gseg * SEG;
    uint32_t so = 0;
#pragma unroll 1
    for (int c = 0; c < 9; c++) {
        uint8_t* dst = sbase + st->soff[c] + pl.pos[c];
        const uint32_t n = si.cnt[c];
        cta_copy_bytes(dst, src + so, n, tid);
        so += n;
    }
    if (tid == 0 && si.has_valid) sbase[st->soff[pl.first_ctx] + pl.first_pos] = si.first_nl;
    if (MODE == 2) {
        const SegPlace vp = A.vplace[gseg];
        const uint8_t* vsrc = A.bits_area + (uint64_t)gseg * SEG_BITS_BYTES;
        uint32_t vo = 0;
#pragma unroll 1
        for (int c = 1; c < 9; c++) {
            uint8_t* dst = sbase + st->soff[8 + c] + vp.pos[c];
            const uint32_t n = (uint32_t)A.vcnt[(uint64_t)gseg * 9 + c] * (c < 3 ? 1u : 3u);
            cta_copy_bytes(dst, vsrc + vo, n, tid);
            vo += n;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Frequency normalisation (libxpng.c:316-329 / :166-182).  cum has N+1 entries (local memory).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void normalise_freqs(const uint32_t* F, uint32_t* cum, uint32_t N, uint32_t total, int pb) {
    cum[0] = 0;
    for (uint32_t i = 0; i < N; i++) cum[i + 1] = cum[i] + F[i];
    for (uint32_t i = 1; i <= N; i++) cum[i] = (uint32_t)(((uint64_t)cum[i] << pb) / total);
    for (uint32_t i = 0; i < N; i++) {
        if (F[i] && cum[i + 1] == cum[i]) {
            uint32_t best = ~0u, donor = 0;
            for (uint32_t j = 0; j < N; j++) {
                const uint32_t wdt = cum[j + 1] - cum[j];
                if (wdt > 1 && wdt < best) { best = wdt; donor = j; }
            }
            if (donor < i) for (uint32_t j = donor + 1; j <= i; j++) cum[j]--;
            else for (uint32_t j = i + 1; j <= donor; j++) cum[j]++;
        }
    }
}

// Encoder symbol (ryg-rans Rans64EncSymbolInit, libxpng.c:331-360) packed into 16 bytes:
//   x = rcp_freq lo, y = rcp_freq hi, z = bias | cmpl_freq << 16, w = freq | rcp_shift << 16
__device__ __forceinline__ uint4 make_encsym(uint32_t freq, uint32_t start, int pb) {
    uint64_t rcp; uint32_t shift, bias;
    if (freq < 2) { rcp = ~0ull; shift = 0; bias = start + (1u << pb) - 1; }
    else {
        uint32_t sh = 0; while (freq > (1u << sh)) sh++;
        const uint64_t x1 = 1ull << (sh + 31);
        const uint64_t t1 = x1 / freq;
        const uint64_t x0 = (uint64_t)(freq - 1) + ((x1 % freq) << 32);
        const uint64_t t0 = x0 / freq;
        rcp = t0 + (t1 << 32); shift = sh - 1; bias = start;
    }
    const uint32_t cmpl = (1u << pb) - freq;
    return make_uint4((uint32_t)rcp, (uint32_t)(rcp >> 32), bias | (cmpl << 16), freq | (shift << 16));
}

// MSB-first bit writer over 32-bit words (libxpng.c:8-11).
struct BitW {
    uint64_t acc; uint32_t n; uint32_t* out;
    __device__ __forceinline__ void put(uint32_t c, uint32_t v) {
        acc = (acc << c) | v; n += c;
        if (n >= 32) { n -= 32; *out++ = (uint32_t)(acc >> n); }
    }
    __device__ __forceinline__ void end() { if (n) { *out++ = (uint32_t)(acc << (32 - n)); n = 0; } }
};

// ------------------------------------------------------------------------------------------------
// v2 block encoder arguments (k_rans_v2_pair, enc_rans_lat.cuh).
// ------------------------------------------------------------------------------------------------
struct RansV2Args {
    const TileDesc* tiles;
    TileState* state;
    uint32_t* hist;           // per tile HIST_STRIDE_M1
    const uint8_t* streams;   // ctx streams (stream_slice)
    const uint8_t* alpha;     // alpha streams (px_off)
    uint8_t* blocks;          // block scratch (block_slice)
    uint32_t ntiles;
    uint32_t c0, nc;          // stream index range handled by this launch [c0, c0+nc)
    const uint32_t* order = nullptr; const uint32_t* total = nullptr;   // pair encoders: sorted work list instead of the id range
};

// ------------------------------------------------------------------------------------------------
// Sizes: per image, serial over its tiles (tile blob sizes, raw-tile and whole-file fallbacks,
// libxpng.c:561-568, :771-777); then file offsets over images.
// ------------------------------------------------------------------------------------------------
struct ImageOut { uint64_t off; uint64_t size; uint32_t mode; uint32_t pad; };

__global__ void k_image_sizes(const ImageDesc* imgs, const TileDesc* tiles, TileState* state, ImageOut* outs, uint32_t nimg) {
    const uint32_t im = blockIdx.x * blockDim.x + threadIdx.x;
    if (im >= nimg) return;
    const ImageDesc I = imgs[im];
    uint32_t mode = I.mode & 0xFF;
    uint64_t total = 0;
    if (I.mode & 0x100) { outs[im].size = 8 + I.pxsz; outs[im].mode = 2 | 0x100; return; }   // whole-image single colour (:741-753)
    if (mode != 7) {
        for (uint32_t k = 0; k < I.ntiles; k++) {
            const TileDesc t = tiles[I.tile0 + k];
            TileState* st = state + I.tile0 + k;
            uint32_t size;
            if (mode == 1) {
                const uint64_t kbits = (uint64_t)st->kbits_lo | ((uint64_t)st->kbits_hi << 32);
                uint64_t coded = 8 + ((kbits + 31) / 32) * 4;
                for (int c = 0; c < (t.pxsz == 4 ? 10 : 9); c++) coded += st->bsize[c];
                const uint64_t raw = (uint64_t)t.npx * t.pxsz + 4;
                if (coded < raw) { size = (uint32_t)coded; st->kind = 1; } else { size = (uint32_t)raw; st->kind = 0; }
                st->size = size;
            } else size = st->size;   // mode 2: decided by k_m2_tile_size
            st->out_off = 8 + total;
            total += size;
        }
        if (total >= I.raw_size) mode = 7;
    }
    outs[im].size = mode == 7 ? 8 + I.raw_size : 8 + total;
    outs[im].mode = mode;
}

__global__ void k_image_offsets(ImageOut* outs, uint32_t nimg, uint64_t base) {   // single thread: tiny serial scan
    if (blockIdx.x || threadIdx.x) return;
    uint64_t off = base;
    for (uint32_t i = 0; i < nimg; i++) { outs[i].off = off; off += (outs[i].size + 15) & ~15ull; }
}

// ------------------------------------------------------------------------------------------------
// Assembly, level 1: header, residual bit stream gathered from the segments with a bit shift, blocks.
// One CTA per tile.
// ------------------------------------------------------------------------------------------------
struct AssembleArgs {
    const ImageDesc* imgs;
    const TileDesc* tiles;
    const TileState* state;
    const ImageOut* outs;
    const SegInfo* seginfo;
    const SegPlace* place;
    const uint8_t* px;
    const uint8_t* bits_area;
    const uint8_t* blocks;
    uint8_t* out;
};

__device__ __forceinline__ void copy_bytes(uint8_t* dst, const uint8_t* src, uint64_t n) {
    // block-cooperative copy; word path when both sides are 4-aligned
    if (((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) & 3u) == 0) {
        const uint64_t nw = n >> 2;
        for (uint64_t k = threadIdx.x; k < nw; k += blockDim.x) reinterpret_cast<uint32_t*>(dst)[k] = reinterpret_cast<const uint32_t*>(src)[k];
        for (uint64_t k = (nw << 2) + threadIdx.x; k < n; k += blockDim.x) dst[k] = src[k];
    } else for (uint64_t k = threadIdx.x; k < n; k += blockDim.x) dst[k] = src[k];
}

// Slice `part` of `nparts` of the same copy (a tile's assembly is spread over gridDim.y CTAs when tiles are few).
__device__ __forceinline__ void copy_bytes_part(uint8_t* dst, const uint8_t* src, uint64_t n, uint32_t part, uint32_t nparts) {
    if (nparts == 1) { copy_bytes(dst, src, n); return; }
    if (((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) & 3u) == 0) {
        const uint64_t nw = n >> 2, lo = nw * part / nparts, hi = nw * (part + 1) / nparts;
        for (uint64_t k = lo + threadIdx.x; k < hi; k += blockDim.x) reinterpret_cast<uint32_t*>(dst)[k] = reinterpret_cast<const uint32_t*>(src)[k];
        if (part == 0) for (uint64_t k = (nw << 2) + threadIdx.x; k < n; k += blockDim.x) dst[k] = src[k];
    } else {
        const uint64_t lo = n * part / nparts, hi = n * (part + 1) / nparts;
        for (uint64_t k = lo + threadIdx.x; k < hi; k += blockDim.x) dst[k] = src[k];
    }
}

__device__ __forceinline__ void copy_tile_rows(uint8_t* dst, uint64_t dst_pitch, const uint8_t* src, const TileDesc& t) {
    const uint32_t rowb = t.w * t.pxsz;
    for (uint32_t y = threadIdx.x >> 5; y < t.h; y += blockDim.x >> 5)
        for (uint32_t k = threadIdx.x & 31; k < rowb; k += 32) dst[(uint64_t)y * dst_pitch + k] = src[(uint64_t)y * t.bpr + k];
}

__device__ __forceinline__ void write_file_header(uint8_t* file, const ImageDesc& I, uint32_t mode) {
    st32u(file, (I.w - 1) | ((mode & 0xFF) << 24));
    st32u(file + 4, (I.h - 1) | ((I.pxsz - 3) << 24) | ((mode & 0x100) ? (2u << 24) : 0));
}

// Header, stored image and whole-image single colour are common to both levels.  Returns true when
// the tile needs nothing else.
__device__ __forceinline__ bool assemble_common(const TileDesc& t, const ImageDesc& I, const ImageOut& O, uint8_t* file, const uint8_t* src) {
    if (t.tix == 0 && threadIdx.x == 0) write_file_header(file, I, O.mode);
    if (O.mode & 0x100) {        // libxpng.c:746-751: header + one pixel
        if (t.tix == 0 && threadIdx.x < I.pxsz) file[8 + threadIdx.x] = src[threadIdx.x];
        return true;
    }
    if ((O.mode & 0xFF) == 7) {  // stored image: every tile copies its own rectangle
        copy_tile_rows(file + 8 + (uint64_t)t.y0 * t.bpr + (uint64_t)t.x0 * t.pxsz, t.bpr, src, t);
        return true;
    }
    return false;
}

// One 32-bit word of a bit string that is the concatenation of `nsrc` MSB-first bit strings (sources sorted
// by their destination bit offset sbit[]; source i contributes snb[i] bits read from the words at sptr[i]).
__device__ __forceinline__ uint32_t gather_word(uint32_t wi, uint32_t nsrc, const uint64_t* sbit, const uint32_t* snb,
                                                const uint32_t* const* sptr) {
    uint64_t B = (uint64_t)wi * 32; uint32_t need = 32, word = 0;
    uint32_t lo = 0, hi = nsrc;
    while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (sbit[mid] <= B) lo = mid; else hi = mid; }
    uint32_t j = lo;
    while (need && j < nsrc) {
        const uint64_t s0 = sbit[j]; const uint32_t nb = snb[j];
        if (B >= s0 + nb) { j++; continue; }
        const uint32_t loc = (uint32_t)(B - s0), avail = nb - loc, take = avail < need ? avail : need;
        const uint32_t* sw = sptr[j];
        const uint32_t w0 = sw[loc >> 5], sh = loc & 31;
        const uint32_t w1 = (sh && ((loc + take - 1) >> 5) != (loc >> 5)) ? sw[(loc >> 5) + 1] : 0u;
        const uint32_t bits32 = sh ? ((w0 << sh) | (w1 >> (32 - sh))) : w0;   // 32 bits starting at loc
        const uint32_t got = take == 32 ? bits32 : (bits32 >> (32 - take));
        word = take == 32 ? got : ((word << take) | got);
        need -= take; B += take;
    }
    if (need) word <<= need;   // final partial word: zero padding (libxpng.c:11)
    return word;
}

constexpr int MAX_SRC = 128;   // a tile has at most 109 segments (666 x 666 pixels / 4096) + the first pixel

__global__ void __launch_bounds__(256) k_assemble_m1(AssembleArgs A) {
    __shared__ uint64_t sbit[MAX_SRC];
    __shared__ uint32_t snb[MAX_SRC];
    __shared__ const uint32_t* sptr[MAX_SRC];
    __shared__ uint32_t fpw;
    const uint32_t tile = blockIdx.x, tid = threadIdx.x;
    const TileDesc t = A.tiles[tile];
    const ImageDesc I = A.imgs[t.img];
    const ImageOut O = A.outs[t.img];
    const TileState* st = A.state + tile;
    uint8_t* file = A.out + O.off;
    const uint8_t* src = A.px + t.src_off;
    const uint32_t part = blockIdx.y, nparts = gridDim.y;        // coded tiles: the bit gather and the block copies are sliced over gridDim.y CTAs
    if (part && ((O.mode & 0x100) || (O.mode & 0xFF) == 7 || st->kind == 0)) return;
    if (assemble_common(t, I, O, file, src)) return;
    uint8_t* blob = file + st->out_off;
    if (st->kind == 0) {          // raw tile (libxpng.c:566-567)
        if (tid == 0) st32u(blob, st->size);
        copy_tile_rows(blob + 4, (uint64_t)t.w * t.pxsz, src, t);
        return;
    }
    const uint64_t kbits = (uint64_t)st->kbits_lo | ((uint64_t)st->kbits_hi << 32);
    const uint32_t kwords = (uint32_t)((kbits + 31) / 32);
    if (tid == 0) {
        if (part == 0) { st32u(blob, (1u << 28) + (st->pr << 24) + st->size); st32u(blob + 4, 4 + 4 * kwords); }
        uint32_t fp = 0;            // first pixel, MSB first (libxpng.c:547), left-aligned in one word
        for (uint32_t c = 0; c < t.pxsz; c++) fp = (fp << 8) | src[c];
        fpw = fp << (32 - 8 * t.pxsz);
        sbit[0] = 0; snb[0] = 8 * t.pxsz; sptr[0] = &fpw;
    }
    for (uint32_t j = tid; j < t.nseg; j += 256) {
        sbit[j + 1] = A.place[t.seg0 + j].bit_off; snb[j + 1] = A.seginfo[t.seg0 + j].nbits;
        sptr[j + 1] = reinterpret_cast<const uint32_t*>(A.bits_area + (uint64_t)(t.seg0 + j) * SEG_BITS_BYTES);
    }
    __syncthreads();
    for (uint32_t wi = part * 256 + tid; wi < kwords; wi += 256 * nparts) st32u(blob + 8 + 4ull * wi, gather_word(wi, t.nseg + 1, sbit, snb, sptr));
    // entropy blocks
    uint8_t* dst = blob + 8 + 4ull * kwords;
    const uint8_t* bsrc = A.blocks + block_slice(t, tile);
    for (int c = 0; c < (t.pxsz == 4 ? 10 : 9); c++) {
        copy_bytes_part(dst, bsrc + st->boff[c], st->bsize[c], part, nparts);
        dst += st->bsize[c];
    }
}

}  // namespace xpb
