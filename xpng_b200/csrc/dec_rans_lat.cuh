// dec_rans_lat.cuh — latency-optimised rANS block decoders (v2: libxpng.c:429-493, v1: :262-301).
//
// The two rANS states of a block share one word pointer, so a block is ONE serial chain; with few
// blocks in flight (a single frame has 45 tiles x 9..17 blocks) the GPU is latency-bound and the only
// thing that matters is the length of the dependent instruction chain per symbol.  These kernels give
// every block a whole warp and a direct slot -> (symbol, freq, slot - start) table in shared memory:
//     slot = x & mask                       LOP      4 cycles
//     e    = lut[slot]                      LDS     23 cycles
//     x    = f * (x >> pb) + bias           IMAD.WIDE + IMAD
//     x    = x < 2^31 ? x << 32 | w : x     SHF, ISETP, SEL (branch-free; the word pointer moves by the predicate)
// All 32 lanes execute the chain redundantly (warp-uniform, broadcast loads); lane 0 stores.  The lanes
// cooperate on everything that is parallel: table construction, run (type 1) and raw (type 2) blocks.
// Alphabets above 16 symbols (or PROB_BITS 15) use a byte table slot -> symbol plus a 256-entry
// (freq, start) table: two dependent shared loads per symbol.
// Large batches decode with the pair decoders of dec_rans_pair.cuh.
#pragma once
#include "common.cuh"
#include "dec_m1.cuh"
#include "dec_back.cuh"

namespace xpb {

// Renormalisation words are staged through a shared-memory ring by the whole warp (bulk, coalesced,
// misalignment removed with a funnel shift, zeros past the end: libxpng.c:295, :475), so that the
// chain reads them with fixed-latency shared loads.  The first LAT_TAIL slots are mirrored behind the ring, so the ring
// offset is wrapped once per group of 32 symbols and only grows inside it (two instructions less per symbol pair).
constexpr uint32_t LAT_RING = 512;               // words; refilled in halves (a group of 32 symbols consumes at most 32)
constexpr uint32_t LAT_HALF = LAT_RING / 2;
constexpr uint32_t LAT_TAIL = 36;                // slots 0 .. LAT_TAIL-1 are mirrored behind the ring: a group reads up to 33 words past its start without wrapping
constexpr uint32_t LAT_KEEP = LAT_RING + LAT_TAIL;   // 32 words behind the tail: the table entries of the current group of 32 symbols
constexpr uint32_t LAT_RING_WORDS = LAT_RING + LAT_TAIL + 32;

template <int DIR>
struct WordSrc {
    const uint32_t* base;   // 4-aligned address at or below word 0
    uint32_t sh;            // 8 * misalignment
    uint32_t nwords;        // words available
    uint32_t jmax;          // forward: highest aligned index that may be touched
    // first = address of word 0; DIR = +1: words at first + 4k; DIR = -1: words at first - 4k.
    // Backward sources are followed by the block's two states, so base - k + 1 is always inside the block.
    __device__ __forceinline__ void init(const uint8_t* first, uint32_t n) {
        const uintptr_t a = reinterpret_cast<uintptr_t>(first);
        base = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
        sh = (uint32_t)(a & 3u) * 8u;
        nwords = n;
        jmax = sh ? n : (n ? n - 1 : 0);
    }
    // Stage words [k0, k0 + LAT_HALF) into ring slots (k0 .. ) mod LAT_RING.  All lanes.
    __device__ __forceinline__ void stage(uint32_t* ring, uint32_t k0, uint32_t lane) const {
        // all loads first (clamped addresses, no branch), then the stores: one memory latency per call, not one per word
        uint32_t a0[LAT_HALF / 32], a1[LAT_HALF / 32];
        const uint32_t kmax = nwords ? nwords - 1 : 0;
#pragma unroll
        for (uint32_t i = 0; i < LAT_HALF / 32; i++) {
            const uint32_t k = min(k0 + lane + 32 * i, kmax);
            if (DIR > 0) { a0[i] = __ldg(base + k); a1[i] = __ldg(base + min(k + 1, jmax)); }
            else { a0[i] = __ldg(base - k); a1[i] = __ldg(base - k + 1); }
        }
#pragma unroll
        for (uint32_t i = 0; i < LAT_HALF / 32; i++) {
            const uint32_t k = k0 + lane + 32 * i;
            const uint32_t v = k < nwords ? __funnelshift_r(a0[i], a1[i], sh) : 0u;
            const uint32_t slot = k & (LAT_RING - 1);
            ring[slot] = v;
            if (slot < LAT_TAIL) ring[LAT_RING + slot] = v;
        }
    }
};

// Direct table for alphabets of at most 16 symbols and PROB_BITS <= 14:
//   entry = (slot - start) | sym << 14 | freq << 18.   clamp: symbols above 8 decode as 0 (context streams).
__device__ __forceinline__ void lat_build_lut1(uint32_t* lut, const uint32_t* cum, uint32_t N, int pb, uint32_t lane, bool clamp) {
    const uint32_t total = 1u << pb;
    for (uint32_t s = 0; s < N; s++) {
        const uint32_t c0 = min(cum[s], total), c1 = min(cum[s + 1], total), f = c1 - c0;
        const uint32_t hi = (f << 18) | ((clamp && s > 8u ? 0u : s) << 14);
        for (uint32_t i = c0 + lane; i < c1; i += 32) lut[i] = (i - c0) | hi;
    }
    for (uint32_t i = min(cum[N], total) + lane; i < total; i += 32) lut[i] = 0;   // corrupt table: uncovered slots
}
// Two-level tables: sym8[slot] and tab[sym] = start | freq << 16.
__device__ __forceinline__ void lat_build_lut2(uint8_t* sym8, uint32_t* tab, const uint32_t* cum, uint32_t N, int pb, uint32_t lane) {
    const uint32_t total = 1u << pb;
    for (uint32_t s = lane; s < 256; s += 32) {
        const uint32_t c0 = s < N ? min(cum[s], total) : total, c1 = s < N ? min(cum[s + 1], total) : total;
        tab[s] = (c0 & 0xFFFFu) | ((c1 - c0) << 16);
    }
    for (uint32_t s = 0; s < N; s++) {
        const uint32_t c0 = min(cum[s], total), c1 = min(cum[s + 1], total);
        for (uint32_t i = c0 + lane; i < c1; i += 32) sym8[i] = (uint8_t)s;
    }
    for (uint32_t i = min(cum[N], total) + lane; i < total; i += 32) sym8[i] = 0;
}

// The chain.  DIR = +1: symbols 0..n-1 in order (v1); DIR = -1: symbols n-1..0 (v2).  Symbol i uses
// state (i & 1).  Symbols are decoded in groups of 32 = 16 rounds of (state A, state B); the two cores of
// a round are independent instruction streams, the ring words ring[k], ring[k + 1] of a round are loaded
// at its start (k is known from the previous round), and lane j keeps symbol j of the group (one AND-OR
// with a per-lane mask), so a group ends with one coalesced 32-byte store.
template <int DIR, bool TWO>
__device__ __forceinline__ void lat_chain(const uint32_t* lut, const uint8_t* sym8, const uint32_t* tab, uint32_t* ring, const int pb, uint64_t x0,
                                          uint64_t x1, const WordSrc<DIR>& ws, uint8_t* out, const uint32_t n, const uint32_t lane) {
    const uint32_t mask = (1u << pb) - 1u;
    ws.stage(ring, 0, lane); ws.stage(ring, LAT_HALF, lane);
    __syncwarp();
    const char* ringb = reinterpret_cast<const char*>(ring);
    uint32_t kb = 0, kw = 0, loaded = LAT_RING;      // ring byte offset, words consumed, words staged
    uint32_t x0lo = (uint32_t)x0, x0hi = (uint32_t)(x0 >> 32), x1lo = (uint32_t)x1, x1hi = (uint32_t)(x1 >> 32);
    // one symbol, any state: used for the (at most 31) symbols outside full groups
    auto single = [&](uint32_t& lo, uint32_t& hi) -> uint32_t {
        const uint32_t slot = lo & mask;
        uint32_t f, bias, s;
        if (TWO) { s = sym8[slot]; const uint32_t e = tab[s]; f = e >> 16; bias = slot - (e & 0xFFFFu); }
        else { const uint32_t e = lut[slot]; f = e >> 18; bias = e & 0x3FFFu; s = (e >> 14) & 15u; }
        const uint64_t x = (uint64_t)f * ((((uint64_t)hi << 32) | lo) >> pb) + bias;
        lo = (uint32_t)x; hi = (uint32_t)(x >> 32);
        if ((hi | (lo & 0x80000000u)) == 0) { kb &= LAT_RING * 4 - 1; hi = lo; lo = *reinterpret_cast<const uint32_t*>(ringb + kb); kb += 4; kw++; }
        return s;
    };
    // Symbol j of a group is parked in shared memory (one store per symbol, on the load/store pipe) and lane j picks it up at
    // the end of the group: cheaper than masks in registers, which the compiler re-derives from lane compares (3 ALU ops).
    uint32_t* kslot = ring + LAT_KEEP;
    // group of 32 symbols; A decodes first.  Forward: A = x0 (even index); backward from an even top: A = x1.
    auto group = [&](uint32_t& alo, uint32_t& ahi, uint32_t& blo, uint32_t& bhi) -> uint32_t {
        kb &= LAT_RING * 4 - 1;                       // wrapped once per group; inside it the offset only grows (mirrored tail)
        const uint32_t kb0 = kb;
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
            const uint32_t c0 = *reinterpret_cast<const uint32_t*>(ringb + kb), c1 = *reinterpret_cast<const uint32_t*>(ringb + kb + 4);
            uint32_t ka, kbv;
            {   const uint32_t slot = alo & mask; uint32_t f, bias;
                if (TWO) { const uint32_t s = sym8[slot]; const uint32_t e = tab[s]; f = e >> 16; bias = slot - (e & 0xFFFFu); ka = s; }
                else { const uint32_t e = lut[slot]; f = e >> 18; bias = e & 0x3FFFu; ka = e; }
                const uint32_t qlo = __funnelshift_r(alo, ahi, pb), qhi = ahi >> pb;
                const uint64_t t = (uint64_t)f * qlo + bias; alo = (uint32_t)t; ahi = f * qhi + (uint32_t)(t >> 32); }
            {   const uint32_t slot = blo & mask; uint32_t f, bias;
                if (TWO) { const uint32_t s = sym8[slot]; const uint32_t e = tab[s]; f = e >> 16; bias = slot - (e & 0xFFFFu); kbv = s; }
                else { const uint32_t e = lut[slot]; f = e >> 18; bias = e & 0x3FFFu; kbv = e; }
                const uint32_t qlo = __funnelshift_r(blo, bhi, pb), qhi = bhi >> pb;
                const uint64_t t = (uint64_t)f * qlo + bias; blo = (uint32_t)t; bhi = f * qhi + (uint32_t)(t >> 32); }
            const bool pa = (ahi | (alo & 0x80000000u)) == 0, pq = (bhi | (blo & 0x80000000u)) == 0;
            const uint32_t wb = pa ? c1 : c0;
            ahi = pa ? alo : ahi; alo = pa ? c0 : alo;
            bhi = pq ? blo : bhi; blo = pq ? wb : blo;
            kb += (pa ? 4u : 0u) + (pq ? 4u : 0u);
            kslot[DIR > 0 ? j : 31 - j] = ka; kslot[DIR > 0 ? j + 1 : 30 - j] = kbv;
        }
        __syncwarp();
        const uint32_t keep = kslot[lane];
        __syncwarp();
        kw += (kb - kb0) >> 2;
        if (kw + LAT_HALF >= loaded) { __syncwarp(); ws.stage(ring, loaded, lane); loaded += LAT_HALF; __syncwarp(); }   // warp-uniform
        return TWO ? keep : ((keep >> 14) & 15u);
    };
    if (DIR > 0) {
        uint32_t i = 0;
        for (; i + 32 <= n; i += 32) { const uint32_t s = group(x0lo, x0hi, x1lo, x1hi); out[i + lane] = (uint8_t)s; }
        for (; i < n; i++) { const uint32_t s = (i & 1) ? single(x1lo, x1hi) : single(x0lo, x0hi); if (lane == 0) out[i] = (uint8_t)s; }
    } else {
        uint32_t i = n;                              // symbols left; next to decode is i - 1
        for (; i & 31u; i--) { const uint32_t s = ((i - 1) & 1) ? single(x1lo, x1hi) : single(x0lo, x0hi); if (lane == 0) out[i - 1] = (uint8_t)s; }
        for (; i >= 32; i -= 32) { const uint32_t s = group(x1lo, x1hi, x0lo, x0hi); out[i - 32 + lane] = (uint8_t)s; }
    }
}

// Parallel fills for the trivial block types.
__device__ __forceinline__ void lat_fill_run(uint8_t* out, uint32_t n, uint32_t sym, uint32_t lane) {
    const uint32_t v4 = sym * 0x01010101u;
    for (uint32_t k = lane; k < (n + 3) / 4; k += 32) reinterpret_cast<uint32_t*>(out)[k] = v4;
}
__device__ __forceinline__ void lat_fill_raw(uint8_t* out, uint32_t n, uint32_t nbit, const uint8_t* bits, const uint8_t* end, uint32_t bit0, uint32_t lane,
                                             bool clamp) {
    for (uint32_t k = lane; k < n; k += 32) {
        BitR r{ bits, end, bit0 + k * nbit };
        uint32_t v = r.get(nbit); if (clamp && v > 8u) v = 0;
        out[k] = (uint8_t)v;
    }
}

// Frequency table -> cum[0..N] in shared memory (lane 0; type 4 tables are a serial bit scan).
__device__ __forceinline__ void lat_read_table(uint32_t* cum, const uint8_t* bits, const uint8_t* end, uint32_t bit0, uint32_t N, int pb, bool sparse,
                                               uint32_t lane) {
    if (!sparse) {   // fixed-width entries: parallel read, then a serial prefix (N <= 256)
        for (uint32_t i = lane; i < N; i += 32) { BitR r{ bits, end, bit0 + i * (uint32_t)pb }; cum[i + 1] = r.get((uint32_t)pb); }
        __syncwarp();
        if (lane == 0) { cum[0] = 0; uint32_t acc = 0; for (uint32_t i = 0; i < N; i++) { acc += cum[i + 1]; cum[i + 1] = acc; } }
    } else if (lane == 0) {
        BitR r{ bits, end, bit0 };
        uint32_t acc = 0; cum[0] = 0;
        for (uint32_t i = 0; i < N; i++) { if (r.get(1)) acc += r.get((uint32_t)pb); cum[i + 1] = acc; }
    }
    __syncwarp();
}

constexpr uint32_t LAT_CUM_WORDS = 260;   // cum[257] + pad, at the start of dynamic shared memory

// ---------------------------------------------------------------------------------------------------
// v2 blocks (level 1).  One warp (= one CTA) per block; id = j * ntiles + tile with c = c0 + j.
// lut_bytes = dynamic shared memory behind cum[] available for tables.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) k_dec_rans_v2_lat(RansDecArgs A, uint32_t lut_bytes) {
    extern __shared__ __align__(16) uint32_t lat_smem[];
    uint32_t* cum = lat_smem;
    uint32_t* lut = lat_smem + LAT_CUM_WORDS;
    const uint32_t id = blockIdx.x, lane = threadIdx.x;
    const uint32_t c = A.c0 + id / A.ntiles, tile = id % A.ntiles;
    const TileDesc t = A.tiles[tile];
    if (A.imgs[t.img].mode != 1) return;
    if (c == 9 && t.pxsz != 4) return;
    const DecTile* d = A.dt + tile;
    if (d->m == 0 || d->m == 0xFE) return;
    const DecBlock b = d->blk[c];
    const uint8_t* blk = A.in + d->blob_off + b.off;
    uint8_t* out = c == 9 ? A.alpha + t.px_off : A.streams + t.str_off + b.soff;
    const uint32_t n = b.n;
    if (b.type == 0 || n == 0) return;
    const uint32_t w1 = ld32u(blk + 4), v2 = w1 >> 24, csz = ld32u(blk) & 0xFFFFFFu;
    const bool ctx = c < 9;
    if (b.type == 1) { lat_fill_run(out, n, ctx && v2 > 8u ? 0u : v2, lane); return; }
    if (b.type == 2) { lat_fill_raw(out, n, v2, blk + 8, blk + csz, 0, lane, ctx); return; }
    const uint32_t N = v2 + 2, w2 = ld32u(blk + 8); const int pb = (int)(w2 >> 24);
    const uint32_t tabw = w2 & 0xFFFFFFu;
    const bool two = N > 16 || (4u << pb) > lut_bytes;
    // a context stream never has more than 9 symbols: a table of more than 16 is corrupt data, and the block decodes as zeros
    if (N > 256 || (ctx && N > 16) || pb < 10 || pb > 15 || 8 + 4ull * tabw > csz || tabw < 5 || (two && (1u << pb) + 1024u > lut_bytes)) {
        for (uint32_t k = lane; k < n; k += 32) out[k] = 0;
        return;
    }
    const uint8_t* tab = blk + 8 + 4ull * tabw;
    lat_read_table(cum, tab, blk + csz, 0, N, pb, b.type == 4, lane);
    if (cum[N] != (1u << pb)) {   // a valid table sums to 2^PROB_BITS exactly (libxpng.c:316-329); any other sum fails the call
        if (lane == 0) dec_fail(A.err, DEC_BAD_BLOCK);
        for (uint32_t k = lane; k < n; k += 32) out[k] = 0;
        return;
    }
    uint32_t* tab2 = lut; uint8_t* sym8 = reinterpret_cast<uint8_t*>(lut + 256);
    if (two) lat_build_lut2(sym8, tab2, cum, N, pb, lane); else lat_build_lut1(lut, cum, N, pb, lane, ctx);
    __syncwarp();
    const uint8_t* sp = tab - 16;                       // state0, state1 (libxpng.c:467)
    const uint64_t x0 = ld64u(sp), x1 = ld64u(sp + 8);
    WordSrc<-1> ws; ws.init(sp - 4, (uint32_t)((sp - (blk + 12)) / 4));
    uint32_t* ring = lut + lut_bytes / 4;
    if (two) lat_chain<-1, true>(nullptr, sym8, tab2, ring, pb, x0, x1, ws, out, n, lane);
    else lat_chain<-1, false>(lut, nullptr, nullptr, ring, pb, x0, x1, ws, out, n, lane);
}

// ---------------------------------------------------------------------------------------------------
// v1 blocks (level 2; libxpng.c:262-301).  Block order: long value streams first, so that the longest
// chains start in the first wave of CTAs.
// ---------------------------------------------------------------------------------------------------
__device__ __constant__ const uint8_t LAT_M2_ORDER[18] = { 12, 11, 9, 13, 14, 15, 16, 10, 0, 1, 2, 3, 4, 5, 6, 7, 8, 0 };   // see the launches in api.cu

struct RansV1LatArgs {
    const TileDesc* tiles;
    const DecImage* imgs;
    const DecTile* dt;
    const uint8_t* in;
    uint8_t* streams;
    uint32_t ntiles;
    uint32_t j0, nj;        // range of LAT_M2_ORDER handled by this launch
    uint32_t lut_bytes;
    uint32_t n_lo, n_hi;    // only blocks with n_lo <= symbols < n_hi (long and short blocks get differently sized tables)
    int* err;
};

__global__ void __launch_bounds__(32) k_dec_rans_v1_lat(RansV1LatArgs A) {
    extern __shared__ __align__(16) uint32_t lat_smem[];
    uint32_t* cum = lat_smem;
    uint32_t* lut = lat_smem + LAT_CUM_WORDS;
    const uint32_t id = blockIdx.x, lane = threadIdx.x;
    const uint32_t c = LAT_M2_ORDER[A.j0 + id / A.ntiles], tile = id % A.ntiles;
    const TileDesc t = A.tiles[tile];
    if (A.imgs[t.img].mode != 2) return;
    const DecTile* d = A.dt + tile;
    const uint32_t kind = d->m >> 4;
    if (d->m == 0xFE || d->m == 0xFF || d->m == 0 || (kind == 2 && (d->m & 8))) return;
    const bool grey = kind == 2;
    if (grey != (A.j0 == 17)) return;                 // the grey plane (block 0 of a grey tile) has its own launch
    const uint32_t N = grey ? 256u : (uint32_t)DEC_M2_NSYM[c]; const int pb = grey ? 15 : 14;
    const DecBlock b = d->blk[c];
    const uint8_t* blob = A.in + d->blob_off; const uint8_t* blk = blob + b.off;
    uint8_t* out = A.streams + t.str_off + b.soff;
    const uint32_t n = b.n;
    if (b.type == 0 || n == 0) return;
    if (n < A.n_lo || n >= A.n_hi) return;
    const uint8_t* side = blob + 8; const uint8_t* side_end = blob + 4 + d->bsz;
    const uint32_t bitpos = d->bitpos[c];
    const bool ctx = !grey && c < 9;
    if (b.type == 1) { const uint32_t v = ld32u(blk + 4) >> 24; lat_fill_run(out, n, ctx && v > 8u ? 0u : v, lane); return; }
    if (b.type == 2) { lat_fill_raw(out, n, bitlen32(N - 1), side, side_end, bitpos, lane, ctx); return; }
    const uint32_t bsize = ld32u(blk) & 0xFFFFFFu;
    const bool two = N > 16 || (4u << pb) > A.lut_bytes;
    if (two && (1u << pb) + 1024u > A.lut_bytes) { for (uint32_t k = lane; k < n; k += 32) out[k] = 0; return; }
    lat_read_table(cum, side, side_end, bitpos, N, pb, b.type == 4, lane);
    if (cum[N] != (1u << pb)) {   // see k_dec_rans_v2_lat
        if (lane == 0) dec_fail(A.err, DEC_BAD_BLOCK);
        for (uint32_t k = lane; k < n; k += 32) out[k] = 0;
        return;
    }
    uint32_t* tab2 = lut; uint8_t* sym8 = reinterpret_cast<uint8_t*>(lut + 256);
    if (two) lat_build_lut2(sym8, tab2, cum, N, pb, lane); else lat_build_lut1(lut, cum, N, pb, lane, ctx);
    __syncwarp();
    const uint64_t x0 = ld64u(blk + 8), x1 = ld64u(blk + 16);
    WordSrc<1> ws; ws.init(blk + 24, bsize >= 24 ? (bsize - 24) / 4 : 0u);
    uint32_t* ring = lut + A.lut_bytes / 4;
    if (two) lat_chain<1, true>(nullptr, sym8, tab2, ring, pb, x0, x1, ws, out, n, lane);
    else lat_chain<1, false>(lut, nullptr, nullptr, ring, pb, x0, x1, ws, out, n, lane);
}

// ---------------------------------------------------------------------------------------------------
// Context walk (nl_{i+1} = next unread symbol of stream nl_i, libxpng.c:803).  One warp per tile, lane
// c < 9 owns stream c (64-bit register window of up to 16 nibble symbols, the next eight packed behind
// it).  Every lane publishes the head of its stream in `info`; the whole dependent chain is ONE shuffle
// per symbol: got = shfl(info, cur) with cur = the previous got.  The owner pops its window while the
// shuffle is in flight (the pop depends on cur only), so self-transitions cost nothing extra.  Lane j
// of each group of 32 steps keeps symbol j; one coalesced store per 32 symbols.  The walks below differ
// in where a window refill comes from; k_dec_walk3 (dec_walk3.cuh) walks three tiles per warp.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t walk_pack8(uint2 q) {   // eight byte symbols (<= 15) -> eight nibbles, first symbol lowest
    uint32_t a = (q.x | (q.x >> 4)) & 0x00FF00FFu; a = (a | (a >> 8)) & 0xFFFFu;
    uint32_t b = (q.y | (q.y >> 4)) & 0x00FF00FFu; b = (b | (b >> 8)) & 0xFFFFu;
    return a | (b << 16);
}

// Shared-memory variant (the tile's streams fit): the warp first packs the nine streams to nibbles in
// shared memory (coalesced), then walks; a window refill is one shared load of eight symbols, so no
// global-memory latency remains inside the walk.  ~31 cycles per symbol.
constexpr uint32_t WALK_SMEM_MAX_SYMS = 400000;   // 200 KB of nibbles (+ 9 pad words) per tile

template <int DUMMY>
__global__ void __launch_bounds__(32) k_dec_walk_smem(WalkArgs A) {
    extern __shared__ __align__(16) uint32_t walk_sm[];
    const uint32_t tile = blockIdx.x, lane = threadIdx.x;
    const TileDesc t = A.tiles[tile];
    if (A.imgs[t.img].mode != A.mode) return;
    const DecTile* d = A.dt + tile;
    if (d->m == 0 || d->m >= 0x20) return;   // raw / grey / single colour / failed
    uint8_t* out = A.nlseq + t.px_off;
    const uint32_t m = d->nsym;
    // pack (whole warp): stream k at word offset wo[k], one zero word behind each stream
    uint32_t myoff = 0, mynch = 0, acc = 0;
#pragma unroll 1
    for (uint32_t k = 0; k < 9; k++) {
        const uint32_t nw = (d->blk[k].n + 7) / 8;
        const uint2* s = reinterpret_cast<const uint2*>(A.streams + t.str_off + d->blk[k].soff);
        for (uint32_t i = lane; i < nw; i += 32) walk_sm[acc + i] = walk_pack8(__ldg(s + i));
        if (lane == 0) walk_sm[acc + nw] = 0;
        if (lane == k) { myoff = acc; mynch = nw; }
        acc += nw + 1;
    }
    __syncwarp();
    const uint32_t nch = mynch;
    const uint32_t* src = walk_sm + myoff;                       // lanes >= 9: nch = 0, src[0] is a valid word
    auto chunk = [&](uint32_t k) -> uint32_t { return k < nch ? src[k] : 0u; };
    uint32_t wlo = chunk(0), whi = chunk(1), cnt = 16, nbuf = chunk(2), ch = 3;
    uint32_t info = wlo & 0xFu, cur = 0, nm = 0, nx = 0;
    uint32_t mk[32];
#pragma unroll
    for (int j = 0; j < 32; j++) { mk[j] = lane == (uint32_t)j ? 0xFFFFFFFFu : 0u; asm volatile("" : "+r"(mk[j])); }
    for (uint32_t pos = 0; pos < m; pos += 32) {
        uint32_t keep = 0;
#pragma unroll
        for (int j = 0; j < 32; j++) {
            const uint32_t got = __shfl_sync(0xffffffffu, info, cur);   // the chain: one shuffle per symbol
            const bool own = lane == cur;                               // the owner pops while the shuffle is in flight
            const uint32_t plo = __funnelshift_r(wlo, whi, 4), phi = whi >> 4;
            wlo = own ? plo : wlo; whi = own ? phi : whi; cnt -= own ? 1u : 0u;
            info = wlo & 0xFu;
            keep |= got & mk[j];
            cur = got;
            if ((j & 7) == 1) {
                // every 8 steps, branch-free: windows at <= 8 symbols append the next 8.  cnt >= 1 holds at every
                // check (16 at start; a refilled window has >= 9, and at most 8 are popped until the next check),
                // so `info` is never stale.
                nm = cnt <= 8u ? 0xFFFFFFFFu : 0u;
                const unsigned long long add = (unsigned long long)(nbuf & nm) << (4u * min(cnt, 8u));
                wlo |= (uint32_t)add; whi |= (uint32_t)(add >> 32);
                cnt += nm & 8u;
                nx = src[min(ch, nch)];                                 // word nch is the zero pad; consumed four steps later
                ch += nm & 1u;
            }
            if ((j & 7) == 5) nbuf = (nx & nm) | (nbuf & ~nm);
        }
        if (pos + lane < m) out[pos + lane] = (uint8_t)keep;
    }
}


// ---------------------------------------------------------------------------------------------------
// Same walk for tiles whose streams do not all fit next to each other in shared memory (batches, tiles above
// WALK_SMEM_MAX_SYMS): every context stream gets a small RING of nibble-packed chunks in shared memory, and the warp
// keeps the rings topped up between groups of 32 steps — one coalesced 256-byte read per refill, loaded during one
// group and packed / stored at the start of the next, so its memory latency never meets the chain.  The 32 steps of a
// group are the loop of k_dec_walk_smem (fixed-latency shared loads only).
//   ring: WRING_CH chunks of 8 symbols per stream; lane k < 9 owns stream k: ch = next chunk it will pop into its
//   window, st = chunks staged.  One refill (32 chunks) per group at most, for the first stream with st - ch <=
//   WRING_LOW.  A stream pops at most 4 chunks per group, nine needy streams are served within 9 groups (+1 group of
//   load latency): 40 < WRING_LOW chunks, so a staged chunk is always ahead of ch; st - ch <= WRING_LOW + 32 <
//   WRING_CH, so a refill never overwrites an unread chunk.
// ---------------------------------------------------------------------------------------------------
constexpr uint32_t WRING_CH = 128, WRING_LOW = 64;
template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) k_dec_walk_ring(WalkArgs A) {
    __shared__ uint32_t wring[WARPS][9][WRING_CH];
    const uint32_t wid = threadIdx.x >> 5, tile = blockIdx.x * WARPS + wid, lane = threadIdx.x & 31;
    if (tile >= A.ntiles) return;
    const TileDesc t = A.tiles[tile];
    if (A.imgs[t.img].mode != A.mode) return;
    const DecTile* d = A.dt + tile;
    if (d->m == 0 || d->m >= 0x20) return;   // raw / grey / single colour / failed
    uint8_t* out = A.nlseq + t.px_off;
    const uint32_t m = d->nsym;
    const uint32_t c = lane < 9 ? lane : 0;
    const uint32_t nch = lane < 9 ? (d->blk[c].n + 7) / 8 : 0;   // 8-symbol chunks of my stream
    const uint2* gsrc = reinterpret_cast<const uint2*>(A.streams + t.str_off + d->blk[c].soff);
    uint32_t* myring = wring[wid][c];
    uint32_t st = 0, ch = 0;
    // one refill of stream p: 32 chunks from chunk index s0 (all lanes)
    auto fetch = [&](uint32_t p, uint2& r) {
        const uint2* base = reinterpret_cast<const uint2*>(__shfl_sync(0xffffffffu, (unsigned long long)gsrc, p));
        const uint32_t s0 = __shfl_sync(0xffffffffu, st, p), np = __shfl_sync(0xffffffffu, nch, p);
        const uint32_t k = s0 + lane;
        r = k < np ? __ldg(base + k) : make_uint2(0u, 0u);
    };
    auto store = [&](uint32_t p, const uint2 r) {
        const uint32_t s0 = __shfl_sync(0xffffffffu, st, p);
        wring[wid][p][(s0 + lane) & (WRING_CH - 1)] = walk_pack8(r);
        if (lane == p) st += 32;
    };
    auto needy = [&]() -> uint32_t { return __ballot_sync(0xffffffffu, lane < 9 && st < nch && st - ch <= WRING_LOW); };
    // initial fill: up to three refills per stream
    for (uint32_t nb = needy(); nb; nb = needy()) {
        const uint32_t p = __ffs(nb) - 1;
        uint2 r; fetch(p, r); store(p, r);
    }
    __syncwarp();
    auto chunk = [&](uint32_t k) -> uint32_t { const uint32_t v = myring[k & (WRING_CH - 1)]; return k < nch ? v : 0u; };
    uint32_t wlo = chunk(0), whi = chunk(1), cnt = 16, nbuf = chunk(2);
    ch = 3;
    uint32_t info = wlo & 0xFu, cur = 0, nm = 0, nx = 0;
    uint32_t mk[32];
#pragma unroll
    for (int j = 0; j < 32; j++) { mk[j] = lane == (uint32_t)j ? 0xFFFFFFFFu : 0u; asm volatile("" : "+r"(mk[j])); }
    uint32_t pend = 32;                                     // stream whose refill is in flight (32 = none)
    uint2 preg = make_uint2(0u, 0u);
    for (uint32_t pos = 0; pos < m; pos += 32) {
        // between groups (warp-uniform): land the refill loaded during the previous group, start the next one
        if (pend < 32) { store(pend, preg); __syncwarp(); }
        {
            const uint32_t nb = needy();
            pend = nb ? __ffs(nb) - 1 : 32u;
            if (nb) fetch(pend, preg);
        }
        uint32_t keep = 0;
#pragma unroll
        for (int j = 0; j < 32; j++) {
            const uint32_t got = __shfl_sync(0xffffffffu, info, cur);   // the chain: one shuffle per symbol
            const bool own = lane == cur;                               // the owner pops while the shuffle is in flight
            const uint32_t plo = __funnelshift_r(wlo, whi, 4), phi = whi >> 4;
            wlo = own ? plo : wlo; whi = own ? phi : whi; cnt -= own ? 1u : 0u;
            info = wlo & 0xFu;
            keep |= got & mk[j];
            cur = got;
            if ((j & 7) == 1) {                                         // see k_dec_walk_smem
                nm = cnt <= 8u ? 0xFFFFFFFFu : 0u;
                const unsigned long long add = (unsigned long long)(nbuf & nm) << (4u * min(cnt, 8u));
                wlo |= (uint32_t)add; whi |= (uint32_t)(add >> 32);
                cnt += nm & 8u;
                nx = chunk(ch);                                         // consumed four steps later
                ch += nm & 1u;
            }
            if ((j & 7) == 5) nbuf = (nx & nm) | (nbuf & ~nm);
        }
        if (pos + lane < m) out[pos + lane] = (uint8_t)keep;
    }
}

}  // namespace xpb
