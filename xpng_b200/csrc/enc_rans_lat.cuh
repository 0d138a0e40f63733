// enc_rans_lat.cuh — latency-optimised rANS block encoders (v2: libxpng.c:307-427, v1: :160-260).
//
// A block has two rANS states that never interact: state 0 codes the even symbols, state 1 the odd
// ones; only the ORDER of their renormalisation words in the output couples them.  Here a block is
// given to a PAIR of lanes (lane h owns state h), so both recurrences advance in the same instruction
// stream (half the instructions per symbol of a one-lane-two-states loop and no branch divergence).
// Per step each lane publishes "I renormalised" with one ballot; a word's position is the running word
// count plus the partner's bit when the partner emits first (v2: state 0 first, ascending addresses;
// v1: state 1 first, descending addresses).  The store of step t is issued in step t + 1, so the ballot
// latency never stalls the recurrence.  16 blocks per warp; everything that is not the recurrence
// (normalisation, tables, headers, raw fallback) is the even lane's job.
#pragma once
#include "common.cuh"
#include "enc_back.cuh"
#include "enc_m2.cuh"

namespace xpb {

constexpr int PAIR_BLK = 16;   // blocks per warp

// Encoder symbol split over two shared arrays so that the recurrence loads ready-to-use words:
//   EA[sym][PAIR_BLK] = { rcp_freq lo, rcp_freq hi, bias, cmpl_freq }      (ryg-rans Rans64EncSymbol, libxpng.c:331-360)
//   EB[sym][PAIR_BLK] = { x_max >> 32 = freq << (31 - PROB_BITS), rcp_shift }
// Row NSYM of both arrays is the identity symbol (rcp = 0, bias = 0, x_max = 2^32 - 1: never renormalises,
// x' = x), used for the positions past the end of a lane's stream, so the recurrence carries no validity test.
__device__ __forceinline__ void pair_put_sym(uint4* EA, uint2* EB, uint32_t row, uint32_t blk, uint32_t freq, uint32_t start, int pb) {
    const uint4 e = make_encsym(freq, start, pb);
    EA[row * PAIR_BLK + blk] = make_uint4(e.x, e.y, e.z & 0xFFFFu, e.z >> 16);
    EB[row * PAIR_BLK + blk] = make_uint2((e.w & 0xFFFFu) << (31 - pb), e.w >> 16);
}
__device__ __forceinline__ void pair_put_ident(uint4* EA, uint2* EB, uint32_t row, uint32_t blk) {
    EA[row * PAIR_BLK + blk] = make_uint4(0u, 0u, 0u, 0u);
    EB[row * PAIR_BLK + blk] = make_uint2(0xFFFFFFFFu, 0u);
}

// One warp: the 2-lane recurrences of up to 16 blocks.  `live`: this lane's block runs the recurrence.
// EA/EB point at the lane's block column.  Emission e (0-based) goes to wbase[e] (VER 2) or wbase[-1 - e]
// (VER 1).  Returns the block's word count; xlo/xhi hold the lane's final state.
template <int VER, int NSYM>
__device__ __forceinline__ uint32_t pair_chain(const uint4* EA, const uint2* EB, const uint8_t* in, const uint32_t n, const bool live, uint32_t* wbase,
                                               uint32_t& xlo, uint32_t& xhi) {
    const uint32_t lane = threadIdx.x & 31, h = lane & 1;
    const uint32_t my = 1u << lane, bsh = lane & 30u;
    const uint32_t firstm = (VER == 2 ? (1u << (lane & 30u)) : (1u << (lane | 1u))) & ~my;   // the partner's bit when it emits before me
    xlo = 0x80000000u; xhi = 0;                                   // RANS64_L = 2^31
    auto core = [&](const uint4 e, const uint32_t sh) {           // state update after the renormalisation decision
        const uint64_t x = ((uint64_t)xhi << 32) | xlo;
        const uint64_t q = __umul64hi(x, ((uint64_t)e.y << 32) | e.x) >> sh;
        const uint64_t y = q * e.w + (x + e.z);
        xlo = (uint32_t)y; xhi = (uint32_t)(y >> 32);
    };
    const uint32_t nn = VER == 2 ? n : (n & ~1u);                  // v1: the odd tail symbol is coded first, by state 0, without renormalisation
    if (VER == 1 && live && (n & 1u) && h == 0) { const uint32_t s = in[n - 1]; core(EA[s * PAIR_BLK], EB[s * PAIR_BLK].y); }   // :218-225
    const uint32_t G = live ? (nn + 15) / 16 : 0;                  // groups of 8 pairs
    uint32_t Gmax = G;
#pragma unroll
    for (int o = 16; o; o >>= 1) Gmax = max(Gmax, __shfl_xor_sync(0xffffffffu, Gmax, o));
    const uint4* in16 = reinterpret_cast<const uint4*>(in);
    const char* EAb = reinterpret_cast<const char*>(EA); const char* EBb = reinterpret_cast<const char*>(EB);
    uint32_t wcount = 0, pend_w = 0, pend_bal = 0;
    auto flush = [&]() {                                          // store of the previous step (its ballot is one step old)
        const uint32_t idx = wcount + ((pend_bal & firstm) ? 1u : 0u);
        uint32_t* dst = VER == 2 ? wbase + idx : wbase - 1 - (int64_t)idx;
        // predicated store, never a branch: a divergent branch per step would cost more than the whole recurrence
        asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %2, 0;\n @q st.global.u32 [%0], %1;\n}" :: "l"(dst), "r"(pend_w), "r"(pend_bal & my) : "memory");
        const uint32_t bits = pend_bal >> bsh;                    // no POPC here: its ~20-cycle latency would stall the in-order pipe every step
        wcount += (bits & 1u) + ((bits >> 1) & 1u);
    };
    // symbols are fetched two groups (16 steps, > 1500 cycles) ahead: the load never stalls the in-order pipe
    uint4 vnext = make_uint4(0, 0, 0, 0), vnext2 = make_uint4(0, 0, 0, 0);
    if (G) vnext = in16[VER == 2 ? 0 : G - 1];
    if (G > 1) vnext2 = in16[VER == 2 ? 1 : G - 2];
    for (uint32_t g = 0; g < Gmax; g++) {
        const bool gv = g < G;
        const uint32_t gi = gv ? (VER == 2 ? g : G - 1 - g) : 0u;
        uint4 v = vnext;
        vnext = vnext2;
        if (g + 2 < G) vnext2 = in16[VER == 2 ? g + 2 : G - 3 - g];
        const uint32_t nvalid = gv ? min(16u, nn - 16u * gi) : 0u;     // symbols of this group inside the stream
        const bool partial = nvalid < 16u;
        uint32_t vmask = 0xFFFFu;                                    // bit k: symbol k of the group is real
        if (__any_sync(0xffffffffu, partial)) vmask = (1u << nvalid) - 1u;   // warp-uniform branch, only near stream ends
        // my eight symbols as row byte offsets into EA (<< 8) : even positions of the group for h = 0, odd for h = 1
        const uint32_t w4[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
        for (int jj = 0; jj < 8; jj++) {
            const int j = VER == 2 ? jj : 7 - jj;
            const uint32_t word = w4[j >> 1];
            uint32_t s = (word >> (16 * (j & 1) + 8 * h)) & 0xFFu;
            s = (vmask >> (2 * j + h)) & 1u ? s : (uint32_t)NSYM;         // past the stream end: identity row
            const uint4 e = *reinterpret_cast<const uint4*>(EAb + (size_t)s * (PAIR_BLK * 16));
            const uint2 eb = *reinterpret_cast<const uint2*>(EBb + (size_t)s * (PAIR_BLK * 8));
            flush();
            const bool p = xhi >= eb.x;                               // x >= freq << (63 - pb)  (libxpng.c:370)
            pend_w = xlo;
            pend_bal = __ballot_sync(0xffffffffu, p);
            xlo = p ? xhi : xlo; xhi = p ? 0u : xhi;
            core(e, eb.y);
        }
    }
    flush();
    return wcount;
}

// ---------------------------------------------------------------------------------------------------
// v2 blocks (level 1).  id = j * ntiles + tile, c = c0 + j; 2 lanes per block.
// ---------------------------------------------------------------------------------------------------
template <int NSYM>
__global__ void __launch_bounds__(32) k_rans_v2_pair(RansV2Args A) {
    extern __shared__ __align__(16) uint4 etab[];   // EA[NSYM + 1][PAIR_BLK] then EB[NSYM + 1][PAIR_BLK]; last row = identity
    uint2* etb = reinterpret_cast<uint2*>(etab + (NSYM + 1) * PAIR_BLK);
    const uint32_t lane = threadIdx.x, h = lane & 1, blk = lane >> 1;
    if (h == 0) pair_put_ident(etab, etb, NSYM, blk);
    const uint32_t id = blockIdx.x * PAIR_BLK + blk;
    bool exists; uint32_t c, tile;
    if (A.order) {                                             // sorted work list (enc_order.cuh): longest blocks first
        const uint32_t total = *A.total;
        if (id - blk >= total) return;                         // warp-uniform
        exists = id < total;
        const uint32_t entry = exists ? A.order[id] : 0u;
        tile = entry & 0xFFFFFFu; c = exists ? entry >> 24 : A.c0;
    } else {
        exists = id < A.nc * A.ntiles;
        c = A.c0 + (exists ? id / A.ntiles : 0); tile = exists ? id % A.ntiles : 0;
    }
    const TileDesc t = A.tiles[tile];
    TileState* st = A.state + tile;
    const uint32_t n = st->len[c];
    const int pb = c == 9 ? 15 : 12;
    uint32_t* F = A.hist + (uint64_t)tile * HIST_STRIDE_M1 + (c == 9 ? HIST_ALPHA : HIST_CTX + c * 16);
    const uint8_t* in = c == 9 ? A.alpha + t.px_off : A.streams + stream_slice(t) + st->soff[c];
    uint8_t* out = A.blocks + block_slice(t, tile) + st->boff[c];
    uint32_t* o = reinterpret_cast<uint32_t*>(out);
    uint32_t cum[NSYM + 1];
    uint32_t N = 0, used = 0, nbit = 0;
    bool live = false;
    if (exists && h == 0) {
        if (c == 9 && t.pxsz != 4) st->bsize[9] = 0;
        else if (n == 0) { o[0] = 4; st->bsize[c] = 4; }                                                          // libxpng.c:313
        else {
            int top = (c == 9 ? 256 : 9); while (F[--top] == 0) {}
            N = (uint32_t)top + 1; nbit = bitlen32((uint32_t)top);
            for (uint32_t i = 0; i < N; i++) used += F[i] != 0;
            if (used == 1) { o[0] = 8u | (1u << 24); o[1] = n | ((uint32_t)in[0] << 24); st->bsize[c] = 8; }      // :318
            else {
                normalise_freqs(F, cum, N, n, pb);
                for (uint32_t i = 0; i < N; i++) pair_put_sym(etab, etb, i, blk, cum[i + 1] - cum[i], cum[i], pb);
                live = true;
            }
        }
    }
    live = __shfl_sync(0xffffffffu, (int)live, lane & 30u) != 0;
    __syncwarp();
    uint32_t xlo, xhi;
    const uint32_t words = pair_chain<2, NSYM>(etab + blk, etb + blk, in, n, live, o + 3, xlo, xhi);
    const uint32_t x1lo = __shfl_sync(0xffffffffu, xlo, lane | 1u), x1hi = __shfl_sync(0xffffffffu, xhi, lane | 1u);
    if (!live || h) return;
    uint32_t* wp = o + 3 + words;
    wp[0] = xlo; wp[1] = xhi; wp[2] = x1lo; wp[3] = x1hi; wp += 4;                                                   // :394
    const bool sparse = (N + used * (uint32_t)pb) < N * (uint32_t)pb;                                             // :396-397
    o[1] = n | ((N - 2) << 24);
    o[2] = (uint32_t)(wp - (o + 2)) | ((uint32_t)pb << 24);                                                       // :400
    BitW b{ 0, 0, wp };
    for (uint32_t k = 0; k < N; k++) {
        const uint32_t f = cum[k + 1] - cum[k];
        if (!sparse) b.put((uint32_t)pb, f);
        else if (f) b.put((uint32_t)pb + 1, f + (1u << pb));
        else b.put(1, 0);
    }
    b.end();
    uint32_t csz = (uint32_t)((uint8_t*)b.out - out);
    o[0] = csz | ((3u + (uint32_t)sparse) << 24);
    const uint64_t rawbits = (uint64_t)nbit * n;
    const uint32_t rawsz = 8 + (uint32_t)(rawbits / 32) * 4 + ((rawbits % 32) ? 4 : 0);
    if (csz >= rawsz) {                                                                                          // :417-424
        o[1] = n | (nbit << 24);
        BitW r{ 0, 0, o + 2 };
        for (uint32_t k = 0; k < n; k++) r.put(nbit, in[k]);
        r.end();
        csz = (uint32_t)((uint8_t*)r.out - out);
        o[0] = csz | (2u << 24);
    }
    st->bsize[c] = csz;
}

// ---------------------------------------------------------------------------------------------------
// v1 blocks (level 2).  Block numbering and scratch layout: see RansV1Args (enc_m2.cuh).
// ---------------------------------------------------------------------------------------------------
template <int NSYM>
__global__ void __launch_bounds__(32) k_rans_v1_pair(RansV1Args A) {
    extern __shared__ __align__(16) uint4 etab[];   // EA[NSYM + 1][PAIR_BLK] then EB[NSYM + 1][PAIR_BLK]; last row = identity
    uint2* etb = reinterpret_cast<uint2*>(etab + (NSYM + 1) * PAIR_BLK);
    const uint32_t lane = threadIdx.x, h = lane & 1, blk = lane >> 1;
    if (h == 0) pair_put_ident(etab, etb, NSYM, blk);
    const uint32_t id = blockIdx.x * PAIR_BLK + blk;
    bool exists; uint32_t c, tile;
    if (A.order) {                                             // sorted work list (enc_order.cuh): longest blocks first
        const uint32_t total = *A.total;
        if (id - blk >= total) return;                         // warp-uniform
        exists = id < total;
        const uint32_t entry = exists ? A.order[id] : 0u;
        tile = entry & 0xFFFFFFu; c = exists ? entry >> 24 : A.c0;
    } else {
        exists = id < A.nc * A.ntiles;
        c = A.c0 + (exists ? id / A.ntiles : 0); tile = exists ? id % A.ntiles : 0;
    }
    const uint8_t cls = A.tclass[tile];
    if (cls != (A.grey ? TC_GREY : TC_RGB)) exists = false;
    const TileDesc t = A.tiles[tile];
    TileState* st = A.state + tile;
    uint32_t N = 0, n = 0, rsize = 0; int pb = 14; const uint32_t* F = A.hist; const uint8_t* in = A.streams; uint8_t* region = A.blocks;
    if (exists) {
        if (A.grey) {
            N = 256; pb = 15; n = t.npx - 1;
            F = A.hist + (uint64_t)tile * HIST_STRIDE_M2 + c * 256;
            in = A.streams + t.str_off + (uint64_t)c * grey_plane_pitch(t.npx);
            rsize = align16u(2 * n + 1024);
            region = A.blocks + t.blk_off + (uint64_t)c * rsize;
            if (h == 0) st->breg[c] = c * rsize;
        } else {
            N = M2_NSYM[c]; pb = 14; n = st->len[c];
            F = A.hist + (uint64_t)tile * HIST_STRIDE_M2 + (c < 9 ? HIST_CTX + c * 16 : HIST_VAL + VAL_OFF[c - 8]);
            in = A.streams + t.str_off + st->soff[c];
            rsize = align16u(2 * n + 256);
            region = A.blocks + t.blk_off + st->breg[c];
        }
        if (N > (uint32_t)NSYM || N <= A.nmin) exists = false;   // handled by the launch with the other table size
    }
    uint32_t* rend = reinterpret_cast<uint32_t*>(region + rsize);
    uint32_t* tab = A.tabs + ((uint64_t)tile * 17 + c) * TAB_WORDS;
    const uint32_t nbit = bitlen32(N ? N - 1 : 0);
    const uint32_t breg = exists ? (A.grey ? c * rsize : st->breg[c]) : 0;
    auto finish = [&](uint32_t* start, uint32_t type, uint32_t pbits) {
        st->boff[c] = breg + (uint32_t)((uint8_t*)start - region);
        st->bsize[c] = (uint32_t)((uint8_t*)rend - (uint8_t*)start);
        st->btype[c] = type; st->pbits[c] = pbits;
    };
    uint32_t cum[NSYM + 1];
    uint32_t used = 0;
    bool live = false;
    if (exists && h == 0) {
        if (n == 0) { rend[-1] = 4; finish(rend - 1, 0, 0); }                                 // libxpng.c:167
        else {
            for (uint32_t i = 0; i < N; i++) used += F[i] != 0;
            if (used == 1) { rend[-2] = 8u | (1u << 24); rend[-1] = n | ((uint32_t)in[n - 1] << 24); finish(rend - 2, 1, 0); }   // :169-172
            else {
                normalise_freqs(F, cum, N, n, pb);
                for (uint32_t i = 0; i < N; i++) pair_put_sym(etab, etb, i, blk, cum[i + 1] - cum[i], cum[i], pb);
                live = true;
            }
        }
    }
    live = __shfl_sync(0xffffffffu, (int)live, lane & 30u) != 0;
    __syncwarp();
    uint32_t xlo, xhi;
    const uint32_t words = pair_chain<1, NSYM>(etab + blk, etb + blk, in, n, live, rend, xlo, xhi);        // :215-245, words go down from the region end
    const uint32_t x1lo = __shfl_sync(0xffffffffu, xlo, lane | 1u), x1hi = __shfl_sync(0xffffffffu, xhi, lane | 1u);
    if (!live || h) return;
    uint32_t* wp = rend - words;
    wp -= 4; wp[0] = xlo; wp[1] = xhi; wp[2] = x1lo; wp[3] = x1hi;                             // :245
    const uint32_t payload = (uint32_t)((uint8_t*)rend - (uint8_t*)wp);
    uint32_t tab_bits = (N - used) + used * ((uint32_t)pb + 1);
    const bool sparse = tab_bits < N * (uint32_t)pb;
    if (!sparse) tab_bits = N * (uint32_t)pb;
    if ((uint64_t)tab_bits + 8ull * payload >= (uint64_t)nbit * n) {                           // :250-254 raw symbols
        BitW r{ 0, 0, reinterpret_cast<uint32_t*>(region) };
        for (uint32_t k = 0; k < n; k++) r.put(nbit, in[k]);
        r.end();
        rend[-2] = 8u | (2u << 24); rend[-1] = n;
        finish(rend - 2, 2, nbit * n);
        return;
    }
    BitW b{ 0, 0, tab };                                                                      // :256-257
    for (uint32_t k = 0; k < N; k++) {
        const uint32_t f = cum[k + 1] - cum[k];
        if (!sparse) b.put((uint32_t)pb, f);
        else if (f) b.put((uint32_t)pb + 1, f + (1u << pb));
        else b.put(1, 0);
    }
    b.end();
    wp -= 2; wp[0] = (payload + 8) | ((3u + (uint32_t)sparse) << 24); wp[1] = n;               // :258-259
    finish(wp, 3 + sparse, tab_bits);
}

}  // namespace xpb
