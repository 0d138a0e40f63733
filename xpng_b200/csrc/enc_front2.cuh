// enc_front2.cuh — encode front end for RGB tiles, second generation (libxpng.c:497-532 m1e_*, :33-44 ENC*).
//
// Same contract as front_segment<MODE, 3> of enc_front.cuh (same SegInfo / chunk / bit layout, so k_tile_scan,
// k_compact and the assembly are unchanged), about a third of its instructions:
//   stage    the tile rows that hold raster [r0 - w - 1, r1) are copied as aligned 16-byte vectors global -> shared by
//            cp.async, then repacked in shared memory as ONE packed byte run (rows back to back), so a pixel's L / U / UL
//            neighbours sit at fixed byte distances (3, 3w, 3w + 3) whatever the tile's alignment in the image;
//   phase 1  a thread owns 16 consecutive pixels (48 bytes: three 128-bit shared loads, the row above through fourteen
//            words and one funnel shift each); predictor, residual, zig-zag and bit length are computed on the three
//            channels at once (byte- or 16-bit-lane arithmetic), everything stays in registers;
//   phase 2  the context of a pixel is the nl of the pixel before it (RGB has no skipped pixels), so only the thread's
//            first pixel needs its neighbour's result; per-thread counters of the stable 9-way split live in shared
//            memory columns (one byte / halfword per thread and context), one block scan orders them;
//   phase 3  coalesced copy-out, as before.
// RGBA tiles (alpha plane, skipped pixels) keep the first-generation kernel.
#pragma once
#include "common.cuh"
#include "enc_front.cuh"

namespace xpb {

// CTAs per SM (64 registers) at both levels: the kernel waits on latency more than it issues, and at level 2 four CTAs with
// the spills that 64 registers cost beat two CTAs at 128 registers without them (1000 1080p frames: 25.0 -> 22.1 ms)
constexpr int F2_MINB = 4;
constexpr int F2_PADPX = 672;                       // pixels staged before the segment's first (>= FRONT2_MAXW + 2, multiple of 16)
static_assert(F2_PADPX >= (int)FRONT2_MAXW + 2 && F2_PADPX % 16 == 0, "staging pad");
constexpr int F2_PIXB = (F2_PADPX + SEG) * 3;       // 14304 bytes
static_assert(F2_PIXB >= SEG_BITS_BYTES, "the bit area reuses the staged pixels");

// The stage copies the rows of a segment global -> shared by cp.async, all at once when they span at most F2_MAXROWS tile
// rows (every segment of a tile at least 142 pixels wide), else row by row in each warp.
constexpr int F2_MAXROWS = 32;
constexpr int F2_RAWV = F2_PIXB / 16 + 2 * F2_MAXROWS;   // 16-byte slots: the packed run's, plus two per row (lead and tail)
constexpr int F2_WARPV = F2_RAWV / (FRONT_THREADS / 32); // a warp's slice of them for the rows of narrower tiles
static_assert(16 * F2_WARPV >= 3 * (SEG / (F2_MAXROWS - 2)) + 30, "a row of a narrow tile fits a warp's slice");

struct Front2Shared {
    union {
        uint32_t pix[F2_PIXB / 4 + 8];              // packed RGB bytes of raster [r0 - F2_PADPX, r0 + SEG)
        uint32_t bits[SEG_BITS_BYTES / 4];          // phase 2 (the pixels are in registers by then): residual bits / value bytes
    };
    union {
        uint4 raw[F2_RAWV];                         // stage only: the aligned source vectors of each row, as cp.async lands them
        struct {                                    // phases 1-3 (zeroed once the stage is done)
            uint8_t sym[SEG];                       // context chunks, concatenated
            uint8_t cnt[9][FRONT_THREADS];          // per-thread symbols per context
            uint16_t pos[9][FRONT_THREADS];         // per-thread write positions per context (then per value stream, mode 2)
            uint32_t hist[9 * 16];
            uint32_t hist2[576];                    // mode 2: value histograms (VAL_OFF)
        };
    };
    ScanA wa[FRONT_THREADS / 32];
    Cnt9 wc[FRONT_THREADS / 32];
    uint8_t lastnl[FRONT_THREADS];
    uint32_t chunk_start[9];
    uint32_t vchunk_start[9];
    uint32_t first_nl;
    uint32_t vbytes;
};

// 16 bytes global -> shared by cp.async (no register holds them); the bytes at and past `limit` (the end of the image)
// are not read and land as zero.  `a` is 16-aligned and below `limit`.
__device__ __forceinline__ void f2_cp16(uint4* dst, const uint8_t* a, const uint8_t* limit) {
    const uint32_t n = a + 16 <= limit ? 16u : (uint32_t)(limit - a);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;"
                 :: "r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(a), "r"(n) : "memory");
}

// Write the nb bytes of a row to shared byte offset d of `pixb` (any alignment) from the row's aligned source vectors
// src[0, nvec) that cp.async has put in shared memory (byte 0 of the row is byte `lead` of src[0]), one warp.  The carry
// between lanes moves vectors that have already landed.  Whole destination words are written as words; the (at most two)
// words a row shares with its neighbours byte by byte.
__device__ __forceinline__ void f2_pack_row(uint8_t* pixb, uint32_t d, const uint4* src, uint32_t lead, uint32_t nb, uint32_t lane) {
    const uint32_t nvec = (lead + nb + 15u) >> 4;
    const int32_t e0 = (int32_t)d - (int32_t)lead;             // destination of byte 0 of vector 0 (may be negative)
    const uint32_t b = (uint32_t)e0 & 3u, sh = 8u * b;
    uint32_t carry = 0;                                         // last word of the vector before this round's first
    for (uint32_t v0 = 0; v0 < nvec + 1; v0 += 32) {
        const uint32_t v = v0 + lane;
        const uint4 V = v < nvec ? src[v] : make_uint4(0, 0, 0, 0);
        uint32_t prev = __shfl_up_sync(0xffffffffu, V.w, 1);
        if (lane == 0) prev = carry;
        carry = __shfl_sync(0xffffffffu, V.w, 31);
        if (v <= nvec) {
            const uint32_t o[4] = { b ? __funnelshift_l(prev, V.x, sh) : V.x, b ? __funnelshift_l(V.x, V.y, sh) : V.y,
                                    b ? __funnelshift_l(V.y, V.z, sh) : V.z, b ? __funnelshift_l(V.z, V.w, sh) : V.w };
            const int32_t wb = e0 - (int32_t)b + 16 * (int32_t)v;   // byte offset of the first destination word of this vector
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int32_t p = wb + 4 * i;
                if (p >= (int32_t)d && p + 4 <= (int32_t)(d + nb)) *reinterpret_cast<uint32_t*>(pixb + p) = o[i];
                else if (p + 4 > (int32_t)d && p < (int32_t)(d + nb)) {
#pragma unroll
                    for (int k = 0; k < 4; k++) if (p + k >= (int32_t)d && p + k < (int32_t)(d + nb)) pixb[p + k] = (uint8_t)(o[i] >> (8 * k));
                }
            }
        }
    }
}

// per-byte a - b (mod 256)
__device__ __forceinline__ uint32_t f2_sub(uint32_t a, uint32_t b) {
    return ((a | 0x80808080u) - (b & 0x7F7F7F7Fu)) ^ ((a ^ ~b) & 0x80808080u);
}

template <int MODE, bool Y, bool G>
__device__ __forceinline__ void front2_segment(const FrontArgs& A, Front2Shared& S, const TileDesc& t, uint32_t tile, uint32_t gseg) {
    const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint32_t j = gseg - t.seg0, w = t.w;
    const uint32_t r0 = j * SEG, r1 = min(r0 + (uint32_t)SEG, t.npx);
    constexpr int HSTRIDE = MODE == 1 ? HIST_STRIDE_M1 : HIST_STRIDE_M2;
    uint8_t* pixb = reinterpret_cast<uint8_t*>(S.pix);

    // ---------------- stage: rows of raster [ps, r1), ps = max(0, r0 - w - 1)
    {
        const uint32_t ps = r0 > w + 1 ? r0 - w - 1 : 0u;
        const uint32_t ys = ps / w, ye = (r1 - 1) / w;
        const uint8_t* base = A.px + t.src_off;
        // end of the image: the tile's last row may be the image's last row, whose final vector must not read past it
        const uint8_t* limit = base + (uint64_t)(t.h - 1) * t.bpr + (uint64_t)w * 3 + ((uint64_t)t.bpr - (uint64_t)t.x0 * 3 - (uint64_t)w * 3);
        // row y: source bytes [src, src + nb) go to packed-run bytes [d, d + nb)
        auto row = [&](uint32_t y, uint32_t& d, uint32_t& nb) {
            const uint32_t xa = y == ys ? ps - ys * w : 0u, xb = y == ye ? r1 - ye * w : w;
            d = (y * w + xa + F2_PADPX - r0) * 3u; nb = (xb - xa) * 3u;
            return base + (uint64_t)y * t.bpr + (uint64_t)xa * 3;
        };
        if (ye - ys < (uint32_t)F2_MAXROWS) {
            // every load of the segment in flight at once: row y's aligned vectors go to raw slots from (d >> 4) + 2 (y - ys) on
            // (two slots per row more than the packed run: the lead and the tail vector)
            for (uint32_t y = ys + wid; y <= ye; y += FRONT_THREADS / 32) {
                uint32_t d, nb;
                const uint8_t* src = row(y, d, nb);
                const uint8_t* a0 = reinterpret_cast<const uint8_t*>(reinterpret_cast<uintptr_t>(src) & ~(uintptr_t)15);
                const uint32_t nvec = ((uint32_t)(reinterpret_cast<uintptr_t>(src) & 15u) + nb + 15u) >> 4;
                uint4* dst = S.raw + (d >> 4) + 2 * (y - ys);
                for (uint32_t v = lane; v < nvec; v += 32) f2_cp16(dst + v, a0 + 16ull * v, limit);
            }
            asm volatile("cp.async.wait_all;" ::: "memory");
            __syncthreads();
            for (uint32_t y = ys + wid; y <= ye; y += FRONT_THREADS / 32) {
                uint32_t d, nb;
                const uint8_t* src = row(y, d, nb);
                f2_pack_row(pixb, d, S.raw + (d >> 4) + 2 * (y - ys), (uint32_t)(reinterpret_cast<uintptr_t>(src) & 15u), nb, lane);
            }
        } else {
            // narrow tile (w <= SEG / (F2_MAXROWS - 2)): each warp stages its rows one at a time through its own slice of raw[]
            uint4* dst = S.raw + wid * F2_WARPV;
            for (uint32_t y = ys + wid; y <= ye; y += FRONT_THREADS / 32) {
                uint32_t d, nb;
                const uint8_t* src = row(y, d, nb);
                const uint8_t* a0 = reinterpret_cast<const uint8_t*>(reinterpret_cast<uintptr_t>(src) & ~(uintptr_t)15);
                const uint32_t lead = (uint32_t)(reinterpret_cast<uintptr_t>(src) & 15u), nvec = (lead + nb + 15u) >> 4;
                for (uint32_t v = lane; v < nvec; v += 32) f2_cp16(dst + v, a0 + 16ull * v, limit);
                asm volatile("cp.async.wait_all;" ::: "memory");
                __syncwarp();
                f2_pack_row(pixb, d, dst, lead, nb, lane);
                __syncwarp();                                   // the slice is free for the warp's next row
            }
        }
    }
    __syncthreads();                                            // the packed run is complete, raw[] is free
    if (tid < 144) S.hist[tid] = 0;
    if (MODE == 2) for (uint32_t k = tid; k < 576; k += FRONT_THREADS) S.hist2[k] = 0;
#pragma unroll
    for (int c = 0; c < 9; c++) S.cnt[c][tid] = 0;

    // ---------------- phase 1: 16 consecutive pixels per thread, all in registers
    uint32_t fld[16];             // mode 1: residual bit field; mode 2: zig-zagged residual bytes u0 | u1 << 8 | u2 << 16
    uint32_t nlp[2] = { 0, 0 };   // nl of the 16 pixels, one nibble each (15 = not coded)
    uint32_t nbits = 0, nvalid = 0, lastnl = 15;
    {
        const uint32_t B0 = F2_PADPX * 3 + 48 * tid;            // byte offset of my first pixel (16-aligned)
        uint32_t Cw[13];                                        // Cw[0]: the word before my pixels (left neighbour of the first)
        Cw[0] = S.pix[B0 / 4 - 1];
#pragma unroll
        for (int q = 0; q < 3; q++) {
            const uint4 v = *reinterpret_cast<const uint4*>(&S.pix[B0 / 4 + 4 * q]);
            Cw[1 + 4 * q] = v.x; Cw[2 + 4 * q] = v.y; Cw[3 + 4 * q] = v.z; Cw[4 + 4 * q] = v.w;
        }
        uint32_t Uw[13];                                        // the same 52 bytes one tile row up
        {
            // 14 words from word ui = (B0 - 3w - 4) >> 2: five aligned 128-bit loads (threads are 12 words apart: conflict-free,
            // where word loads at that stride collide four ways); ui & 3 is the same for every thread of the CTA
            const uint32_t ub = B0 - 3 * w - 4, ush = (ub & 3u) * 8u, ui = ub >> 2, ua = ui & 3u;
            uint32_t v20[20];
#pragma unroll
            for (int q = 0; q < 5; q++) {
                const uint4 v = *reinterpret_cast<const uint4*>(&S.pix[(ui & ~3u) + 4 * q]);
                v20[4 * q] = v.x; v20[4 * q + 1] = v.y; v20[4 * q + 2] = v.z; v20[4 * q + 3] = v.w;
            }
            uint32_t raw[14];
#pragma unroll
            for (int q = 0; q < 14; q++) raw[q] = ua == 0 ? v20[q] : (ua == 1 ? v20[q + 1] : (ua == 2 ? v20[q + 2] : v20[q + 3]));
#pragma unroll
            for (int q = 0; q < 13; q++) Uw[q] = __funnelshift_r(raw[q], raw[q + 1], ush);
        }
        const uint32_t gi = r0 + 16 * tid;
        uint32_t y = gi / w, x = gi - y * w;
        uint32_t Lp = Cw[0] >> 8, ULp = Uw[0] >> 8;             // packed 0x??BBGGRR, byte 3 is never used
#pragma unroll
        for (int k = 0; k < 16; k++) {
            const int q = 3 * (k >> 2) + 1;
            uint32_t cur, up;
            if ((k & 3) == 0) { cur = Cw[q]; up = Uw[q]; }
            else if ((k & 3) == 1) { cur = __byte_perm(Cw[q], Cw[q + 1], 0x6543); up = __byte_perm(Uw[q], Uw[q + 1], 0x6543); }
            else if ((k & 3) == 2) { cur = __byte_perm(Cw[q + 1], Cw[q + 2], 0x5432); up = __byte_perm(Uw[q + 1], Uw[q + 2], 0x5432); }
            else { cur = Cw[q + 2] >> 8; up = Uw[q + 2] >> 8; }
            const bool valid = gi + k < r1 && gi + k != 0;
            const bool row0 = y == 0, col0 = x == 0;
            uint32_t pint;
            if (Y) {   // ((3L + 3U - 2UL + 2) >> 2) mod 256 in 16-bit lanes; the +1024 bias keeps lanes positive and vanishes mod 256
                const uint32_t lrb = Lp & 0x00FF00FFu, urb = up & 0x00FF00FFu, qrb = ULp & 0x00FF00FFu;
                const uint32_t lg = (Lp >> 8) & 0xFFu, ug = (up >> 8) & 0xFFu, qg = (ULp >> 8) & 0xFFu;
                const uint32_t trb = 3u * (lrb + urb) + 0x04020402u - 2u * qrb, tg = 3u * (lg + ug) + 0x0402u - 2u * qg;
                pint = ((trb >> 2) & 0x00FF00FFu) | (((tg >> 2) & 0xFFu) << 8);
            } else pint = (Lp | up) - (((Lp ^ up) >> 1) & 0x7F7F7F7Fu);     // (L + U + 1) >> 1 per byte
            const uint32_t pd = row0 ? Lp : (col0 ? up : pint);
            uint32_t r = f2_sub(cur, pd);
            if (G) {   // interior pixels only: red and blue residuals minus the green one (libxpng.c:44, :513)
                const uint32_t rg = f2_sub(r, ((r >> 8) & 0xFFu) * 0x00010001u);
                r = (row0 || col0) ? r : rg;
            }
            const uint32_t z = (((r << 1) & 0x00FEFEFEu) ^ (((r >> 7) & 0x00010101u) * 0xFFu));   // zig-zag per byte
            const uint32_t m = (z | (z >> 8) | (z >> 16)) & 0xFFu;
            const uint32_t nl = 32u - (uint32_t)__clz((int)m);
            if (MODE == 1) fld[k] = ((z & 0xFFu) << (2 * nl)) | (((z >> 8) & 0xFFu) << nl) | (z >> 16);
            else fld[k] = z;
            const uint32_t nle = valid ? nl : 15u;
            nlp[k >> 3] |= nle << (4 * (k & 7));
            if (valid) { nbits += nl; nvalid++; lastnl = nl; }
            Lp = cur; ULp = up;
            x++; if (x == w) { x = 0; y++; }
        }
        nbits *= 3u;
    }
    S.lastnl[tid] = (uint8_t)lastnl;
    __syncthreads();                                            // every thread has read its pixels: the bit area may be written
    for (uint32_t k = tid; k < SEG_BITS_BYTES / 4; k += FRONT_THREADS) S.bits[k] = 0;

    // ---------------- phase 2
    const uint32_t pl_in = tid ? S.lastnl[tid - 1] : 15u;       // context of my first pixel (15: the segment's first coded pixel)
    Cnt9 vc{ 0, 0, 0 };
    {
        uint32_t pl = pl_in;
#pragma unroll
        for (int k = 0; k < 16; k++) {
            const uint32_t nl = (nlp[k >> 3] >> (4 * (k & 7))) & 15u;
            if (nl != 15u) {
                if (pl != 15u) S.cnt[pl][tid]++;
                pl = nl;
                if (MODE == 2) cnt9_inc(vc, nl);
            }
        }
    }
    ScanA totA;
    const ScanA preA = block_scan_A(ScanA{ nbits | (nvalid << 17), 0 }, S.wa, totA);
    Cnt9 cc{ 0, 0, 0 };
#pragma unroll
    for (int c = 0; c < 9; c++) {
        const unsigned long long v = S.cnt[c][tid];
        if (c < 4) cc.a |= v << (16 * c); else if (c < 8) cc.b |= v << (16 * (c - 4)); else cc.c |= v;
    }
    Cnt9 totC;
    const Cnt9 posC = block_scan_cnt9(cc, S.wc, totC);
    if (tid < 9) {
        uint32_t s = 0;
        for (uint32_t c = 0; c < tid; c++) s += cnt9_get(totC, c);
        S.chunk_start[tid] = s;
    }
    Cnt9 vposC{ 0, 0, 0 };
    if (MODE == 2) {
        Cnt9 totV;
        vposC = block_scan_cnt9(vc, S.wc, totV);
        if (tid < 9) {   // value chunks in bytes: nl 1,2 -> 1 byte per pixel, nl >= 3 -> 3 bytes
            uint32_t s = 0;
            for (uint32_t c = 1; c < tid; c++) s += cnt9_get(totV, c) * (c < 3 ? 1u : 3u);
            S.vchunk_start[tid] = s;
            A.vcnt[(uint64_t)gseg * 9 + tid] = (uint16_t)cnt9_get(totV, tid);
            if (tid == 8) S.vbytes = s + 3 * cnt9_get(totV, 8);
        }
    }
    __syncthreads();
#pragma unroll
    for (int c = 0; c < 9; c++) S.pos[c][tid] = (uint16_t)(S.chunk_start[c] + cnt9_get(posC, c));
    {
        uint32_t pl = pl_in;
        const uint32_t bit0 = preA.sum & 0x1FFFFu;
        unsigned long long acc = 0; uint32_t nacc = bit0 & 31u, widx = bit0 >> 5; bool first_word = true;
#pragma unroll
        for (int k = 0; k < 16; k++) {
            const uint32_t nl = (nlp[k >> 3] >> (4 * (k & 7))) & 15u;
            if (nl == 15u) continue;
            if (pl != 15u) {
                const uint32_t p = S.pos[pl][tid];
                S.pos[pl][tid] = (uint16_t)(p + 1);
                S.sym[p] = (uint8_t)nl;
                atomicAdd(&S.hist[pl * 16 + nl], 1u);
            } else S.first_nl = nl;
            pl = nl;
            if (MODE == 1 && nl) {
                acc = (acc << (3 * nl)) | fld[k]; nacc += 3 * nl;
                if (nacc >= 32) {
                    nacc -= 32;
                    const uint32_t wv = (uint32_t)(acc >> nacc);
                    if (first_word) { atomicOr(&S.bits[widx], wv); first_word = false; } else S.bits[widx] = wv;
                    widx++;
                }
            }
        }
        if (MODE == 1 && nacc && (nacc != (bit0 & 31u) || !first_word))
            atomicOr(&S.bits[widx], (uint32_t)(acc << (32 - nacc)));
    }
    if (MODE == 2) {   // value bytes: the same per-thread position columns, now per nl
        __syncthreads();
#pragma unroll
        for (int c = 1; c < 9; c++) S.pos[c][tid] = (uint16_t)(S.vchunk_start[c] + cnt9_get(vposC, c) * (c < 3 ? 1u : 3u));
        uint8_t* vbytes = reinterpret_cast<uint8_t*>(S.bits);
#pragma unroll
        for (int k = 0; k < 16; k++) {
            const uint32_t nl = (nlp[k >> 3] >> (4 * (k & 7))) & 15u;
            if (nl == 15u || nl == 0u) continue;
            const uint32_t u0 = fld[k] & 0xFFu, u1 = (fld[k] >> 8) & 0xFFu, u2 = (fld[k] >> 16) & 0xFFu;
            const uint32_t vp = S.pos[nl][tid];
            uint32_t* hv = S.hist2 + VAL_OFF[nl];
            if (nl == 1) { const uint32_t v = (u0 << 2) | (u1 << 1) | u2; vbytes[vp] = (uint8_t)v; atomicAdd(hv + v, 1u); S.pos[nl][tid] = (uint16_t)(vp + 1); }
            else if (nl == 2) { const uint32_t v = (u0 << 4) | (u1 << 2) | u2; vbytes[vp] = (uint8_t)v; atomicAdd(hv + v, 1u); S.pos[nl][tid] = (uint16_t)(vp + 1); }
            else {
                vbytes[vp] = (uint8_t)u0; vbytes[vp + 1] = (uint8_t)u1; vbytes[vp + 2] = (uint8_t)u2;
                atomicAdd(hv + u0, 1u); atomicAdd(hv + u1, 1u); atomicAdd(hv + u2, 1u);
                S.pos[nl][tid] = (uint16_t)(vp + 3);
            }
        }
    }
    __syncthreads();

    // ---------------- phase 3
    const uint32_t nv = totA.sum >> 17, nb = totA.sum & 0x1FFFFu;
    const uint32_t nsym = nv ? nv - 1 : 0;
    {
        uint4* dst = reinterpret_cast<uint4*>(A.sym_area + (uint64_t)gseg * SEG);
        const uint4* src = reinterpret_cast<const uint4*>(S.sym);
        for (uint32_t k = tid; k < (nsym + 15) / 16; k += FRONT_THREADS) dst[k] = src[k];
        uint32_t nbytes = MODE == 1 ? ((nb + 31) / 32) * 4 : S.vbytes;
        uint4* bd = reinterpret_cast<uint4*>(A.bits_area + (uint64_t)gseg * SEG_BITS_BYTES);
        const uint4* bs = reinterpret_cast<const uint4*>(S.bits);
        for (uint32_t k = tid; k < (nbytes + 15) / 16; k += FRONT_THREADS) bd[k] = bs[k];
    }
    if (tid < 144) { const uint32_t v = S.hist[tid]; if (v) atomicAdd(A.hist + (uint64_t)tile * HSTRIDE + HIST_CTX + tid, v); }
    if (MODE == 2) for (uint32_t k = tid; k < 576; k += FRONT_THREADS) { const uint32_t v = S.hist2[k]; if (v) atomicAdd(A.hist + (uint64_t)tile * HSTRIDE + HIST_VAL + k, v); }
    if (tid == 0) {
        SegInfo si;
#pragma unroll
        for (int c = 0; c < 9; c++) si.cnt[c] = (uint16_t)cnt9_get(totC, c);
        si.nvalid = (uint16_t)nv; si.nbits = nb;
        // the last coded pixel of the segment: the last in-range thread's last nl
        const uint32_t lt = (r1 - r0 - 1) >> 4;
        si.has_valid = nv != 0; si.first_nl = nv ? (uint8_t)S.first_nl : 0; si.last_nl = nv ? (uint8_t)(S.lastnl[lt] & 15u) : 0;
        si.pad = 0; si.pad2 = 0;
        A.seginfo[gseg] = si;
    }
}

template <int MODE>
__global__ void __launch_bounds__(FRONT_THREADS, F2_MINB) k_front2(FrontArgs A) {
    __shared__ __align__(16) Front2Shared S;
    const uint32_t gseg = blockIdx.x, tile = A.seg_tile[gseg];
    const TileDesc t = A.tiles[tile];
    if (t.pxsz != 3 || t.w > FRONT2_MAXW) return;               // RGBA tiles and very wide one-tile images: k_front
    if (MODE == 2 && A.tile_skip && A.tile_skip[tile]) return;
    const uint32_t pr = pick_predictor(A.costs + 4 * tile, t.w, t.h, 3u);
    switch (pr & 3u) {
    case 0: front2_segment<MODE, false, false>(A, S, t, tile, gseg); break;
    case 1: front2_segment<MODE, false, true>(A, S, t, tile, gseg); break;
    case 2: front2_segment<MODE, true, false>(A, S, t, tile, gseg); break;
    default: front2_segment<MODE, true, true>(A, S, t, tile, gseg); break;
    }
}

}  // namespace xpb
